"""`train()`: the reference's PPO entry point (ppo_imitation/train.py::train, forked from brax's PPO `train`) on the GPU.

    make_policy, params, metrics = train(environment, num_timesteps, ...)

Assembly (`Run`): reset draws for the global batch (each rank keeps its `sharding.shard_range`), the same initial networks on every
rank, RunningStatistics, the rollout policy, Rollout, PPOLearner, Trainer (metric means accumulated on the device) and, on rank 0,
the Evaluator.  Schedule (`schedule`): brax's -- an optional evaluation at step 0, then `num_evals_after_init` epochs of
`training_steps_per_epoch` training steps; after each epoch rank 0 calls `policy_params_fn`, the ranks write a checkpoint (when
`checkpoint_dir` is set), rank 0 evaluates and calls `progress_fn`.  `restore_checkpoint_path` resumes a run from a checkpoint of the
same configuration: the state is copied into the freshly built buffers and the remaining epochs of the schedule run (DESIGN §3g).

`autoreset="resample"` restarts finished training episodes from fresh draws (DESIGN §3h) instead of the first states.

Out of scope: several unrolls per training step (batch_size * num_minibatches must equal num_envs), action_repeat other than 1,
num_resets_per_eval, network depths other than 2 + 2, re-sharding a checkpoint to another world size.
"""
from __future__ import annotations

import time
from typing import Callable, Dict, Optional, Tuple

import numpy as np

from . import checkpoint as ckpt
from . import learner as lrn
from . import policy as pol
from . import sharding

POLICIES = ("3xtf32", "tf32", "bf16")
AUTORESETS = ("first", "resample")

# train()'s keyword arguments after num_timesteps (brax PPO names) and their defaults
DEFAULTS = dict(
    episode_length=150, num_envs=8192, num_eval_envs=128, unroll_length=20, batch_size=256, num_minibatches=32, num_updates_per_batch=16,
    num_evals=2, learning_rate=6e-4, entropy_cost=1e-4, discounting=0.9, reward_scaling=1.0, gae_lambda=0.95, clipping_epsilon=0.2,
    kl_weight=1e-4, normalize_advantage=True, deterministic_eval=False, encoder_layer_sizes=(256, 128), decoder_layer_sizes=(128, 256),
    latent_size=64, value_layer_sizes=(1024, 1024), policy="3xtf32", seed=0, autoreset="first")

# meta.json entries a checkpoint must share with the run that restores it (buffer sizes, sharding, schedule)
MATCH_FIELDS = ("format", "env", "obs_size", "traj_size", "action_size", "policy_shapes", "value_shapes", "world_size", "num_envs",
                "layout", "schedule")
LAYOUT_KEYS = ("episode_length", "num_eval_envs", "unroll_length", "batch_size", "num_minibatches", "num_updates_per_batch", "policy")


def schedule(num_timesteps: int, num_evals: int, batch_size: int, num_minibatches: int, unroll_length: int) -> Dict[str, int]:
    """brax PPO's schedule (one unroll per training step): the env steps of one training step, the epochs after the initial
    evaluation, and the training steps per epoch (rounded up, so at least num_timesteps env steps run)."""
    per_step = int(batch_size) * int(num_minibatches) * int(unroll_length)
    after_init = max(int(num_evals) - 1, 1)
    return dict(env_steps_per_training_step=per_step, num_evals_after_init=after_init,
                training_steps_per_epoch=-(-int(num_timesteps) // (after_init * per_step)))


def _sizes(env) -> Tuple[int, int, int]:
    return int(env.engine.obs_size), int(env.engine.traj_size), int(env.action_size)


def network_shapes(environment, cfg) -> Tuple[Dict[str, tuple], Dict[str, tuple]]:
    obs, traj, nu = _sizes(environment)
    return (pol.param_shapes(traj, obs, nu, cfg["latent_size"], cfg["encoder_layer_sizes"], cfg["decoder_layer_sizes"]),
            lrn.value_param_shapes(obs, tuple(cfg["value_layer_sizes"])))


def check_config(environment, cfg, world_size: int, eval_env=None) -> None:
    """Everything train() refuses, checked on the host before any device work; each message names the argument."""
    for name, env in (("environment", environment), ("eval_env", eval_env)):
        if env is not None and env.observation_size != env.engine.obs_size:
            raise ValueError(f"{name}: {type(env).__name__} carries its reference trajectory inside the observation, not in "
                             "info['traj']; the intention policy needs the trajectory as its own input")
    if eval_env is not None and _sizes(eval_env) != _sizes(environment):
        raise ValueError("eval_env: obs / traj / action sizes differ from environment's")
    if cfg["policy"] not in POLICIES:
        raise ValueError(f"policy must be one of {POLICIES}, not {cfg['policy']!r}")
    if cfg["autoreset"] not in AUTORESETS:
        raise ValueError(f"autoreset must be one of {AUTORESETS}, not {cfg['autoreset']!r}")
    if cfg["autoreset"] == "resample" and not hasattr(environment, "resample_spec"):
        raise ValueError(f"autoreset='resample': {type(environment).__name__} has no resample_spec() (the draws of its reset)")
    if cfg["batch_size"] * cfg["num_minibatches"] != cfg["num_envs"]:
        raise ValueError("batch_size * num_minibatches must equal num_envs: one unroll per training step (several unrolls per "
                         f"training step are not supported); got {cfg['batch_size']} * {cfg['num_minibatches']} != {cfg['num_envs']}")
    if cfg["num_envs"] % world_size:
        raise ValueError(f"num_envs ({cfg['num_envs']}) must be divisible by the world size ({world_size})")
    if cfg["batch_size"] % world_size:
        raise ValueError(f"batch_size ({cfg['batch_size']}) must be divisible by the world size ({world_size}): each rank's minibatch")
    for k in ("episode_length", "num_eval_envs", "unroll_length", "num_updates_per_batch", "num_evals"):
        if int(cfg[k]) < 1:
            raise ValueError(f"{k} must be at least 1")
    for k in ("encoder_layer_sizes", "decoder_layer_sizes", "value_layer_sizes"):
        if len(cfg[k]) != 2:
            raise ValueError(f"{k}: the networks have two hidden layers here")
    obs, traj, nu = _sizes(environment)
    (e1, e2), (d1, d2) = cfg["encoder_layer_sizes"], cfg["decoder_layer_sizes"]
    w = dict(traj=traj, obs=obs, latent=int(cfg["latent_size"]), e1=e1, e2=e2, d1=d1, d2=d2, nu=nu)  # as lrn.policy_widths reads them
    try:
        lrn.PolicyForward.check(w)
        lrn.PPOLearner.check(w, cfg["value_layer_sizes"])
    except ValueError as e:
        raise ValueError(f"encoder_layer_sizes / decoder_layer_sizes / latent_size / value_layer_sizes {w}: {e}") from None


def run_meta(environment, cfg, sched, world_size: int) -> dict:
    """meta.json of a checkpoint of this run, without the schedule position."""
    obs, traj, nu = _sizes(environment)
    shapes, vshapes = network_shapes(environment, cfg)
    layout = {k: cfg[k] for k in LAYOUT_KEYS}
    if cfg["autoreset"] == "resample":  # only then: checkpoints of the default mode keep the layout they always had
        layout["autoreset"] = "resample"
    return dict(format=ckpt.FORMAT_VERSION, env=type(environment).__name__, obs_size=obs, traj_size=traj, action_size=nu,
                policy_shapes={k: list(s) for k, s in shapes.items()}, value_shapes={k: list(s) for k, s in vshapes.items()},
                world_size=int(world_size), num_envs=int(cfg["num_envs"]), layout=layout,
                schedule=dict(sched), hyperparameters={k: list(v) if isinstance(v, tuple) else v for k, v in cfg.items()})


def _shard(state, lo: int, hi: int):
    """The rows [lo, hi) of a reset State (the fields Rollout reads), as their own tensors."""
    from .envs.base import PipelineState, State
    info = {k: state.info[k][lo:hi].clone() for k in ("cur_frame", "sub_clip_frame", "traj")}
    if state.info.get("clip_idx") is not None:
        info["clip_idx"] = state.info["clip_idx"][lo:hi].clone()
    return State(PipelineState({k: v[lo:hi].clone() for k, v in state.pipeline_state.items()}), state.obs[lo:hi].clone(), None, None,
                 {}, info)


class Run:
    """The objects of one training run on this rank, built from train()'s configuration `cfg` (DEFAULTS' keys)."""

    def __init__(self, environment, cfg, eval_env=None, rank: int = 0, world_size: int = 1, first_state=None, use_graph: bool = True,
                 learner_x3: bool = False, accumulate_metrics: bool = True, evaluate: Optional[bool] = None):
        """`first_state`: this rank's reset State (default: `environment.reset` of the global batch with numpy's default_rng(seed),
        rows `sharding.shard_range`).  `evaluate`: build the Evaluator (default: on rank 0)."""
        from . import evaluator, normalizer, rollout, trainer
        self.env, self.cfg, self.rank, self.world = environment, dict(cfg), int(rank), int(world_size)
        self.device = dev = str(environment.device)
        B = cfg["num_envs"] // self.world
        lo, hi = sharding.shard_range(cfg["num_envs"], self.rank, self.world)
        if first_state is None:
            first_state = environment.reset(np.random.default_rng(cfg["seed"]), batch_size=cfg["num_envs"])
            if (lo, hi) != (0, cfg["num_envs"]):
                first_state = _shard(first_state, lo, hi)
        shapes, vshapes = network_shapes(environment, cfg)
        rng = np.random.default_rng(cfg["seed"])  # the same initial networks on every rank (key_policy / key_value, train.py:190-192)
        pp = pol.init_params(rng, shapes)
        vp = lrn.init_value_params(rng, vshapes)
        self.stats = normalizer.RunningStatistics(environment.engine.obs_size, dev)
        self.policy = self._new_policy(pp, dev, self.stats.mean, self.stats.std)
        self.rollout = rollout.Rollout(environment, self.policy, first_state, cfg["unroll_length"], float(cfg["episode_length"]), use_graph=True,
                                       autoreset=cfg["autoreset"], seed=cfg["seed"], env_offset=lo)
        hp = {k: cfg[k] for k in ("learning_rate", "entropy_cost", "discounting", "reward_scaling", "gae_lambda", "clipping_epsilon",
                                  "normalize_advantage", "kl_weight")}
        self.learner = lrn.PPOLearner(pp, vp, cfg["unroll_length"], B // cfg["num_minibatches"], device=dev, x3=learner_x3, **hp)
        self.trainer = trainer.Trainer(environment, self.policy, self.learner, self.rollout, self.stats, cfg["num_minibatches"],
                                       cfg["num_updates_per_batch"], use_graph=use_graph, seed=cfg["seed"] + self.rank,
                                       accumulate_metrics=accumulate_metrics)
        self.evaluator = None
        if (self.rank == 0) if evaluate is None else evaluate:
            self.evaluator = evaluator.Evaluator(eval_env or environment, self.policy, cfg["num_eval_envs"], cfg["episode_length"],
                                                 seed=cfg["seed"], deterministic=cfg["deterministic_eval"])

    def _new_policy(self, params, device, mean, std):
        if self.cfg["policy"] == "bf16":
            return pol.IntentionPolicy(params, device, mean, std)
        return pol.PrecisePolicy(params, device, mean, std, precision=self.cfg["policy"])

    def make_policy(self, params, device=None):
        """A policy of the kind `policy=` selected, loaded with params = (normalizer_state, policy_params)."""
        norm, pp = params
        return self._new_policy(pp, device or self.device, norm["mean"], norm["std"])

    def params(self):
        """(normalizer_state, policy_params) on the host."""
        return self.stats.state_dict(), self.learner.policy_params()

    # ---- checkpoint ------------------------------------------------------------------------------------------------------------
    def _rank_arrays(self) -> Dict[str, np.ndarray]:
        out = {**ckpt.flatten("rollout", self.rollout.state_dict()), **ckpt.flatten("trainer", self.trainer.state_dict())}
        if self.evaluator is not None and self.rank == 0:
            out.update(ckpt.flatten("evaluator", self.evaluator.state_dict()))
        return out

    def save(self, checkpoint_dir: str, meta: dict) -> str:
        """Writes step_<meta["env_steps"]> (collective over the ranks)."""
        shared = None
        if self.rank == 0:
            norm = self.stats.state_dict()
            shared = dict(learner=self.learner.state_dict(), normalizer=norm,
                          policy=ckpt.policy_arrays(self.learner.policy_params(), norm["mean"], norm["std"]))
        return ckpt.save(checkpoint_dir, meta["env_steps"], self.rank, self._rank_arrays(), meta, shared,
                         barrier=sharding.barrier if self.world > 1 else None)

    def restore(self, path: str) -> dict:
        """Copies checkpoint `path` into this run's buffers (addresses unchanged: captured graphs stay valid; the reset kernel does
        not run).  Returns its meta."""
        c = ckpt.load(path, self.rank)
        self.learner.load_state_dict(c["learner"])
        self.stats.load_state_dict(c["normalizer"])
        self.learner.set_normalizer(self.stats.mean, self.stats.std)
        self.policy.load_params(self.learner.policy_params())
        self.rollout.load_state_dict(ckpt.unflatten(c["rank"], "rollout"))
        self.trainer.load_state_dict(ckpt.unflatten(c["rank"], "trainer"))
        if self.evaluator is not None and self.rank == 0:
            self.evaluator.load_state_dict(ckpt.unflatten(c["rank"], "evaluator"))
        return c["meta"]

    # ---- the loop ----------------------------------------------------------------------------------------------------------------
    def fit(self, num_timesteps: int, progress_fn: Callable = lambda step, metrics: None,
            policy_params_fn: Callable = lambda step, make_policy, params: None, checkpoint_dir: Optional[str] = None,
            restore_checkpoint_path: Optional[str] = None):
        """The body of train(); returns (make_policy, params, metrics)."""
        import torch
        cfg, tr = self.cfg, self.trainer
        sched = schedule(num_timesteps, cfg["num_evals"], cfg["batch_size"], cfg["num_minibatches"], cfg["unroll_length"])
        base_meta = run_meta(self.env, cfg, sched, self.world)
        per_epoch = sched["training_steps_per_epoch"] * sched["env_steps_per_training_step"]
        lead = self.rank == 0
        epoch, env_steps, train_walltime = 0, 0, 0.0
        metrics: Dict[str, float] = {}
        if restore_checkpoint_path:
            ckpt.check_meta(ckpt.read_meta(restore_checkpoint_path), base_meta, MATCH_FIELDS)
            meta = self.restore(restore_checkpoint_path)
            epoch, env_steps, train_walltime = int(meta["epoch"]), int(meta["env_steps"]), float(meta["training_walltime"])
        elif cfg["num_evals"] > 1 and lead:
            metrics = self.evaluator.run_evaluation({})
            progress_fn(0, metrics)
        self.checkpoint_log = []
        tr.epoch_metrics(reset=True)
        while epoch < sched["num_evals_after_init"]:
            torch.cuda.synchronize(self.device)
            t0 = time.perf_counter()
            for _ in range(sched["training_steps_per_epoch"]):
                tr.training_step()
            torch.cuda.synchronize(self.device)
            dt = time.perf_counter() - t0
            epoch, env_steps, train_walltime = epoch + 1, env_steps + per_epoch, train_walltime + dt
            training = {"training/sps": per_epoch / dt, "training/walltime": train_walltime}
            training.update(("training/" + k, v) for k, v in tr.epoch_metrics(reset=True).items())
            params = self.params()
            if lead:
                policy_params_fn(env_steps, self.make_policy, params)
            if checkpoint_dir:
                t1 = time.perf_counter()
                eval_walltime = self.evaluator._eval_walltime if self.evaluator is not None else 0.0
                path = self.save(checkpoint_dir, dict(base_meta, epoch=epoch, env_steps=env_steps, training_walltime=train_walltime,
                                                      eval_walltime=eval_walltime))
                self.checkpoint_log.append(dict(step=env_steps, path=path, seconds=time.perf_counter() - t1, bytes=_dir_bytes(path)))
            metrics = training
            if lead:
                metrics = self.evaluator.run_evaluation(training)
                progress_fn(env_steps, metrics)
        self.env_steps = env_steps
        return self.make_policy, self.params(), metrics


def _dir_bytes(path: str) -> int:
    import os
    return sum(os.path.getsize(os.path.join(path, n)) for n in os.listdir(path)) if os.path.isdir(path) else 0


def train(environment, num_timesteps: int, episode_length: int = 150, num_envs: int = 8192, num_eval_envs: int = 128,
          unroll_length: int = 20, batch_size: int = 256, num_minibatches: int = 32, num_updates_per_batch: int = 16, num_evals: int = 2,
          learning_rate: float = 6e-4, entropy_cost: float = 1e-4, discounting: float = 0.9, reward_scaling: float = 1.0,
          gae_lambda: float = 0.95, clipping_epsilon: float = 0.2, kl_weight: float = 1e-4, normalize_advantage: bool = True,
          deterministic_eval: bool = False, encoder_layer_sizes=(256, 128), decoder_layer_sizes=(128, 256), latent_size: int = 64,
          value_layer_sizes=(1024, 1024), policy: str = "3xtf32", seed: int = 0, autoreset: str = "first", eval_env=None,
          progress_fn: Callable = lambda step, metrics: None, policy_params_fn: Callable = lambda step, make_policy, params: None,
          checkpoint_dir: Optional[str] = None, restore_checkpoint_path: Optional[str] = None):
    """PPO training of the intention network on `environment` (RodentTracking / HumanoidTracking: an env whose info carries the
    reference trajectory).  Returns (make_policy, params, metrics): params = (normalizer_state {count, mean, summed_variance, std},
    policy_params: the flax tree); make_policy(params, device=None) builds a policy of the kind `policy=` selects ("3xtf32" /
    "tf32": policy.PrecisePolicy, "bf16": policy.IntentionPolicy), deterministic with `eps_a=None` at call time; metrics: the
    last evaluation's eval/* names with training/sps, training/walltime and training/<learner.METRIC_NAMES> (means over every
    minibatch update of the epoch).

    Under torchrun with a process group, envs are sharded over the ranks and only rank 0 evaluates and calls the callbacks.
    `checkpoint_dir`: a checkpoint after every epoch (checkpoint.py); `restore_checkpoint_path`: resume from one (same
    configuration and world size) and run the remaining epochs.  `autoreset`: "first" (the reference: a finished episode restarts
    from the env's first state, brax's AutoReset) or "resample" (from a fresh draw of clip, start frame and reset noise on the
    device, DESIGN §3h); evaluation always resets to first states."""
    cfg = {k: v for k, v in locals().items() if k in DEFAULTS}
    cfg.update((k, tuple(cfg[k])) for k in ("encoder_layer_sizes", "decoder_layer_sizes", "value_layer_sizes"))
    rank, world = _rank_world()
    check_config(environment, cfg, world, eval_env)
    if restore_checkpoint_path:
        sched = schedule(num_timesteps, num_evals, batch_size, num_minibatches, unroll_length)
        ckpt.check_meta(ckpt.read_meta(restore_checkpoint_path), run_meta(environment, cfg, sched, world), MATCH_FIELDS)
    run = Run(environment, cfg, eval_env=eval_env, rank=rank, world_size=world)
    return run.fit(num_timesteps, progress_fn, policy_params_fn, checkpoint_dir, restore_checkpoint_path)


def _rank_world() -> Tuple[int, int]:
    dist = sharding.group()
    return (dist.get_rank(), dist.get_world_size()) if dist is not None else (0, 1)
