"""`Evaluator` of the reference (ppo_imitation/acting.py:83-156): episodes of the training-wrapped env under brax's `EvalWrapper`.

    eval_env = envs.training.EvalWrapper(eval_env)                      per-episode sums of every metric + the reward while the
    eval_first_state = eval_env.reset(reset_keys)                       first episode of each env is active, its length
    generate_unroll(eval_env, first_state, policy, key, episode_length // action_repeat)
    metrics: eval/episode_<name>(_std), eval/avg_episode_length, eval/epoch_eval_time, eval/sps, eval/walltime

Here: reset, ONE unroll of `episode_length` steps through rollout.Rollout (policy kernel + `vnl_step_training`: Episode + AutoReset
wrappers fused in the step launch, the unroll replayed as one CUDA graph), then `vnl_eval_metrics` folds EvalWrapper.step over the
recorded [T, B] metrics / reward / done (one thread per env).  `deterministic_eval` = the policy's mode (eps_a = None)."""
from __future__ import annotations

import json
import time
from typing import Dict

import numpy as np

from . import train_kernels as tk
from .envs.rodent import METRIC_KEYS


class Evaluator:
    def __init__(self, eval_env, eval_policy, num_eval_envs: int, episode_length: int, action_repeat: int = 1, seed: int = 0,
                 deterministic: bool = False):
        import torch

        from .rollout import Rollout
        if action_repeat != 1:
            raise NotImplementedError("action_repeat 1 is what the reference trains and evaluates with (train.py:121)")
        self.torch, self.env, self.policy = torch, eval_env, eval_policy
        self.B, self.T = int(num_eval_envs), int(episode_length)
        self.rng = np.random.default_rng(seed)
        self.gen = torch.Generator(device=eval_env.device).manual_seed(seed)
        self.deterministic = bool(deterministic)
        self._steps_per_unroll = self.T * self.B
        self._eval_walltime = 0.0
        self._Rollout = Rollout
        dev = eval_env.device
        f = lambda *s: torch.zeros(*s, dtype=torch.float32, device=dev)
        # the env's metric names (the humanoid has no appendage term); the step kernel writes every column of METRIC_KEYS, all of
        # which are folded, and only the env's own are reported
        self.metric_keys = tuple(getattr(eval_env, "metric_keys", METRIC_KEYS))
        self.episode_metrics, self.active, self.episode_steps = f(self.B, len(METRIC_KEYS) + 1), f(self.B), f(self.B)
        self.rollout = None

    def state_dict(self) -> Dict[str, object]:
        """The two random streams (numpy for the reset draws, torch for the policy noise) and the accumulated eval walltime."""
        return {"rng": np.array(json.dumps(self.rng.bit_generator.state)), "gen": self.gen.get_state().numpy().copy(),
                "walltime": np.float64(self._eval_walltime)}

    def load_state_dict(self, sd) -> None:
        self.rng.bit_generator.state = json.loads(str(sd["rng"]))
        self.gen.set_state(self.torch.as_tensor(np.asarray(sd["gen"]), dtype=self.torch.uint8).cpu())
        self._eval_walltime = float(sd["walltime"])

    def _unroll(self):
        t = self.torch
        s0 = self.env.reset(self.rng, batch_size=self.B)  # eval_env.reset(reset_keys): fresh start frames + noise every evaluation
        if self.rollout is None:
            self.rollout = self._Rollout(self.env, self.policy, s0, self.T, float(self.T), use_graph=True)
            if self.deterministic:
                self.rollout.eps_a = None
        ro = self.rollout
        ro.reset_to(s0)
        ro.eps_z.normal_(generator=self.gen)
        if ro.eps_a is not None:
            ro.eps_a.normal_(generator=self.gen)
        tr = ro.generate_unroll()
        rc = tk.lib().vnl_eval_metrics(self.T, self.B, len(METRIC_KEYS), tr["metrics"].data_ptr(), tr["reward"].data_ptr(), ro.done.data_ptr(),
                                       self.episode_metrics.data_ptr(), self.active.data_ptr(), self.episode_steps.data_ptr(), tk.stream(self.active))
        tk.check(rc, "vnl_eval_metrics")
        return tr

    def run_evaluation(self, training_metrics: Dict[str, float], aggregate_episodes: bool = True) -> Dict[str, float]:
        """One epoch of evaluation; the reference's metric names (acting.py:133-156)."""
        t0 = time.time()
        self._unroll()
        self.torch.cuda.synchronize(self.env.device)  # eval_metrics.active_episodes.block_until_ready()
        epoch_eval_time = time.time() - t0
        em = self.episode_metrics.cpu().numpy()
        cols = [(n, METRIC_KEYS.index(n)) for n in self.metric_keys] + [("reward", len(METRIC_KEYS))]
        metrics = {}
        for fn in (np.mean, np.std):
            suffix = "_std" if fn is np.std else ""
            metrics.update({f"eval/episode_{n}{suffix}": (float(fn(em[:, i])) if aggregate_episodes else em[:, i].copy()) for n, i in cols})
        metrics["eval/avg_episode_length"] = float(np.mean(self.episode_steps.cpu().numpy()))
        metrics["eval/epoch_eval_time"] = epoch_eval_time
        metrics["eval/sps"] = self._steps_per_unroll / epoch_eval_time
        self._eval_walltime += epoch_eval_time
        return {"eval/walltime": self._eval_walltime, **training_metrics, **metrics}
