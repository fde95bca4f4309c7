"""Host side of the observation normaliser (C ABI in include/vnl_normalizer.h): brax's
`running_statistics.RunningStatisticsState` / `init_state` / `update` as the reference uses them
(ppo_imitation/train.py:220-229 normalise, :330-334 update with `pmap_axis_name`, :405-407 init).

    stats = RunningStatistics(obs_size, device)        # count 0, mean 0, summed_variance 0, std 1  (init_state)
    policy.set_normalizer(stats.mean, stats.std)       # shares the tensors: updates are seen by the next launch
    stats.update(transition["observation"])            # once per training step, all ranks

`update` = one HBM pass over the batch on this rank's GPU (vnl_obs_stats_partial), ONE all-reduce of 2 * width + 1 floats
over the process group (NCCL over NVLink on GPUs — the rollout path's only data exchange, the `psum`s of brax's update
folded into one message), and a width-sized state epilogue (vnl_obs_stats_finish).  No CPU fallback.
"""
from __future__ import annotations

import ctypes

from . import _lib, sharding

NORMALIZER_EXPORTS = ("vnl_obs_stats_workspace_bytes", "vnl_obs_stats_partial", "vnl_obs_stats_finish",
                      "vnl_xla_obs_stats_partial", "vnl_xla_obs_stats_finish")


def _bind(lib):
    v = ctypes.c_void_p
    lib.vnl_obs_stats_workspace_bytes.argtypes = [ctypes.c_int]
    lib.vnl_obs_stats_workspace_bytes.restype = ctypes.c_size_t
    lib.vnl_obs_stats_partial.argtypes = [v, ctypes.c_longlong, ctypes.c_int, v, v, v, v]
    lib.vnl_obs_stats_finish.argtypes = [v, ctypes.c_int, v, v, v, v, ctypes.c_float, ctypes.c_float, v]
    for n in ("vnl_xla_obs_stats_partial", "vnl_xla_obs_stats_finish"):
        getattr(lib, n).argtypes = [v, ctypes.POINTER(v), ctypes.c_char_p, ctypes.c_size_t, v]
        getattr(lib, n).restype = None
    return lib


def all_reduce_sums(sums):
    """The one exchange of the update: sum the [S1 | S2 | rows] vector over the process group (identity without one)."""
    dist = sharding.group()
    if dist is not None:
        dist.all_reduce(sums, op=dist.ReduceOp.SUM)
    return sums


class RunningStatistics:
    def __init__(self, width: int, device: str = "cuda:0", std_min_value: float = 1e-6, std_max_value: float = 1e6):
        import torch

        if not torch.cuda.is_available():
            raise RuntimeError("vnl_b200 normaliser needs a CUDA device (sm_100a); there is no CPU fallback")
        self.torch = t = torch
        self.lib = _bind(_lib.load_library())
        self.device = t.device(device)
        self.width = int(width)
        nbytes = int(self.lib.vnl_obs_stats_workspace_bytes(self.width))
        if nbytes == 0:
            raise ValueError("feature width not supported (1..1024)")
        f = lambda n, v=0.0: t.full((n,), v, dtype=t.float32, device=self.device)
        self.count, self.mean, self.summed_variance, self.std = f(1), f(self.width), f(self.width), f(self.width, 1.0)
        self.workspace = t.zeros(nbytes // 4, dtype=t.float32, device=self.device)  # zero once: holds the arrival ticket
        self.sums = f(2 * self.width + 1)
        self.std_min_value, self.std_max_value = float(std_min_value), float(std_max_value)

    STATE_KEYS = ("count", "mean", "summed_variance", "std")

    def state_dict(self):
        """`RunningStatisticsState` on the host as numpy arrays."""
        return {k: getattr(self, k).detach().cpu().numpy().copy() for k in self.STATE_KEYS}

    def load_state_dict(self, sd) -> None:
        """Copies into the existing tensors: a policy that adopted `mean` / `std` (and the graphs it was captured into) sees the
        restored values."""
        import numpy as np
        for k in self.STATE_KEYS:
            x, a = getattr(self, k), np.asarray(sd[k], dtype=np.float32)
            if tuple(a.shape) != tuple(x.shape):
                raise ValueError(f"normaliser {k}: shape {a.shape} does not match {tuple(x.shape)}")
            x.copy_(self.torch.from_numpy(np.ascontiguousarray(a)))

    def update(self, batch, group_reduce: bool = True) -> None:
        """`running_statistics.update(state, batch, pmap_axis_name=...)`: batch [..., width] fp32 on this rank's GPU.
        `group_reduce=False` is brax's `pmap_axis_name=None` (statistics of this rank's batch only)."""
        t = self.torch
        if batch.dtype != t.float32 or not batch.is_contiguous() or batch.shape[-1] != self.width or batch.device != self.device:
            raise ValueError("batch must be a contiguous fp32 [..., width] tensor on the normaliser's device")
        rows = batch.numel() // self.width
        if rows == 0 and not group_reduce:
            return  # empty batch, nobody to exchange with: the state is unchanged (brax: step_increment 0)
        stream = t.cuda.current_stream(self.device).cuda_stream
        with t.cuda.device(self.device):
            rc = self.lib.vnl_obs_stats_partial(batch.data_ptr(), rows, self.width, self.mean.data_ptr(), self.workspace.data_ptr(),
                                                self.sums.data_ptr(), stream)
            if rc:
                raise RuntimeError(f"vnl_obs_stats_partial failed ({rc})")
            if group_reduce:
                all_reduce_sums(self.sums)
            rc = self.lib.vnl_obs_stats_finish(self.sums.data_ptr(), self.width, self.count.data_ptr(), self.mean.data_ptr(),
                                               self.summed_variance.data_ptr(), self.std.data_ptr(), self.std_min_value,
                                               self.std_max_value, stream)
            if rc:
                raise RuntimeError(f"vnl_obs_stats_finish failed ({rc})")
