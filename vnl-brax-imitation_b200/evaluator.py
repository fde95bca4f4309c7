"""`Evaluator` of the reference (ppo_imitation/acting.py:83-156): episodes of the training-wrapped env under brax's `EvalWrapper`.

    eval_env = envs.training.EvalWrapper(eval_env)                      per-episode sums of every metric + the reward while the
    eval_first_state = eval_env.reset(reset_keys)                       first episode of each env is active, its length
    generate_unroll(eval_env, first_state, policy, key, episode_length // action_repeat)
    metrics: eval/episode_<name>(_std), eval/avg_episode_length, eval/epoch_eval_time, eval/sps, eval/walltime

Here: reset, ONE unroll of `episode_length` steps through rollout.Rollout (policy kernel + `vnl_step_training`: Episode + AutoReset
wrappers fused in the step launch, the unroll replayed as one CUDA graph), then `vnl_eval_metrics` folds EvalWrapper.step over the
recorded [T, B] metrics / reward / done (one thread per env).  `deterministic_eval` = the policy's mode (eps_a = None).

`per_clip=True` (DESIGN §3i): every evaluation resets to the same clip x start-frame sweep (`clip_sweep`) and reports, beside the
scalars, per-clip episode statistics (`vnl_eval_clip_stats`) and per-frame tracking profiles (`vnl_eval_frame_profile`)."""
from __future__ import annotations

import json
import time
from typing import Dict

import numpy as np

from . import model_blob as mb
from . import train_kernels as tk
from .envs.base import METRIC_KEYS


def clip_sweep(nclips: int, num_eval_envs: int, start_frame_hi: int):
    """The per-clip evaluation layout: (clip_id[B], start_frame[B]), int32.  W = num_eval_envs // nclips windows per clip; env b
    evaluates clip b // W (clip-major) from start frame (w * start_frame_hi) // W of its window w = b % W, so the windows spread
    evenly over [0, start_frame_hi), the range reset draws start frames from."""
    nclips, B, hi = int(nclips), int(num_eval_envs), int(start_frame_hi)
    W = B // nclips if nclips > 0 else 0
    if W < 1 or B % nclips:
        raise ValueError(f"num_eval_envs ({B}) must be a positive multiple of the clip count ({nclips}): every clip gets the same "
                         "number of start-frame windows")
    b = np.arange(B, dtype=np.int64)
    return (b // W).astype(np.int32), ((b % W) * hi // W).astype(np.int32)


def sweep_layout(env, num_eval_envs: int):
    """(nclips, clip_len, clip_id, start_frame) of `env`'s sweep: clip count and clip length from its task blob header, start
    frames over `env.resample_spec()`'s range.  Refuses an env without resample_spec (its reset draws are not known)."""
    if not hasattr(env, "resample_spec"):
        raise ValueError(f"{type(env).__name__} has no resample_spec() (the start-frame range of its reset): it cannot be swept clip by clip")
    nclips, clip_len = int(env.task_blob[mb.C["VNL_TH_NCLIPS"]]), int(env.task_blob[mb.C["VNL_TH_CLIP_LEN"]])
    clip_id, start_frame = clip_sweep(nclips, num_eval_envs, env.resample_spec()[0])
    return nclips, clip_len, clip_id, start_frame


class Evaluator:
    def __init__(self, eval_env, eval_policy, num_eval_envs: int, episode_length: int, action_repeat: int = 1, seed: int = 0,
                 deterministic: bool = False, per_clip: bool = False):
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
        self.metric_keys = tuple(eval_env.metric_keys)
        self.episode_metrics, self.active, self.episode_steps = f(self.B, len(METRIC_KEYS) + 1), f(self.B), f(self.B)
        self.rollout = None
        self.per_clip = bool(per_clip)
        if self.per_clip:
            self.nclips, self.clip_len, self.clip_id, self.start_frame = sweep_layout(eval_env, self.B)
            C, L, ncol = self.nclips, self.clip_len, len(METRIC_KEYS) + 2
            # the layout on the device once; the results in one float and one int buffer (two copies to the host)
            self.clip_id_dev = torch.as_tensor(self.clip_id, device=dev)
            self.start_frame_dev = torch.as_tensor(self.start_frame, device=dev)
            self.clip_out = torch.zeros(2 * C * ncol + C * L * (ncol - 1), dtype=torch.float32, device=dev)
            self.clip_count = torch.zeros(C + C * L, dtype=torch.int32, device=dev)
            self.clip_mean, self.clip_std, self.frame_sum, self.clip_num, self.frame_count = self._views(self.clip_out, self.clip_count)

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
        if self.per_clip:  # the sweep's clips and start frames, fresh reset noise
            kw = dict(start_frame=self.start_frame, **({"clip_id": self.clip_id} if self.nclips > 1 else {}))
            s0 = self.env.reset(self.rng, batch_size=self.B, **kw)
        else:
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
        if self.per_clip:
            L, nm, st = tk.lib(), len(METRIC_KEYS), tk.stream(self.active)
            cid = self.clip_id_dev.data_ptr() if self.nclips > 1 else None
            tk.check(L.vnl_eval_clip_stats(self.B, nm, self.episode_metrics.data_ptr(), self.episode_steps.data_ptr(), cid, self.nclips,
                                           self.clip_mean.data_ptr(), self.clip_std.data_ptr(), self.clip_num.data_ptr(), st), "vnl_eval_clip_stats")
            tk.check(L.vnl_eval_frame_profile(self.T, self.B, nm, tr["metrics"].data_ptr(), tr["reward"].data_ptr(), self.episode_steps.data_ptr(),
                                              self.start_frame_dev.data_ptr(), cid, self.nclips, self.clip_len, self.frame_sum.data_ptr(),
                                              self.frame_count.data_ptr(), st), "vnl_eval_frame_profile")
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
        if self.per_clip:
            metrics.update(self._per_clip_metrics(cols))
        self._eval_walltime += epoch_eval_time
        return {"eval/walltime": self._eval_walltime, **training_metrics, **metrics}

    def _views(self, out, counts):
        """(mean, std [nclips, nm + 2], frame_sum [nclips, clip_len, nm + 1], count [nclips], frame_count [nclips, clip_len]) of the
        flat result buffers, on the device or their host copies."""
        C, L, ncol = self.nclips, self.clip_len, len(METRIC_KEYS) + 2
        return (out[:C * ncol].reshape(C, ncol), out[C * ncol:2 * C * ncol].reshape(C, ncol), out[2 * C * ncol:].reshape(C, L, ncol - 1),
                counts[:C], counts[C:].reshape(C, L))

    def _per_clip_metrics(self, cols) -> Dict[str, np.ndarray]:
        """eval/clip/*: [nclips] statistics of the episodes of each clip; eval/frame/*: [nclips, clip_len] means per binned step
        (NaN where no step read the frame) and the step counts."""
        mean, std, fsum, num, fcount = self._views(self.clip_out.cpu().numpy(), self.clip_count.cpu().numpy())
        m = {}
        for n, i in cols:
            m[f"eval/clip/episode_{n}"], m[f"eval/clip/episode_{n}_std"] = mean[:, i].copy(), std[:, i].copy()
        m["eval/clip/avg_episode_length"] = mean[:, -1].copy()
        m["eval/clip/num_episodes"] = num.copy()
        for n, i in cols:
            m[f"eval/frame/{n}"] = (fsum[:, :, i] / np.maximum(fcount, 1)).astype(np.float32)
            m[f"eval/frame/{n}"][fcount == 0] = np.nan
        m["eval/frame/count"] = fcount.copy()
        return m
