"""brax `State` mirror (`brax/envs/base.py`): the container `Env.reset/step` return; `TrackingEnv`, the base of the tracking envs."""
from __future__ import annotations

from dataclasses import dataclass, field, replace
from typing import Any, Dict, Optional

import numpy as np

from .. import mjcf
from .. import model_blob as mb
from .._lib import STATE_F

# the columns of the step kernel's metrics output; an env reports those of its `metric_keys`
METRIC_KEYS = ("rcom", "rvel", "rtrunk", "rquat", "ract", "rapp", "termination_error")
# the `State.info` entries the step kernel carries, by their field of VnlState (include/vnl_b200.h)
ENGINE_INFO = {"cur_frame": "cur_frame", "sub_clip_frame": "sub_clip_frame", "clip_idx": "clip_id"}


class PipelineState(dict):
    """Leaves of the mjx pipeline state the reference's callers read, with attribute access
    (`state.pipeline_state.qpos`, reference train.py:293)."""

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError as e:
            raise AttributeError(k) from e

    @property
    def q(self):  # brax alias used by envs/rodent.py:314
        return self["qpos"]

    @property
    def qd(self):
        return self["qvel"]


@dataclass
class State:
    pipeline_state: PipelineState
    obs: Any
    reward: Any
    done: Any
    metrics: Dict[str, Any] = field(default_factory=dict)
    info: Dict[str, Any] = field(default_factory=dict)

    def replace(self, **kw) -> "State":
        return replace(self, **kw)


def engine_state(state: State) -> Dict[str, Any]:
    """The step kernel's state of `state`: the pipeline-state leaves and ENGINE_INFO's entries of `info` (the clip index only where
    the env carries one; without it the kernel tracks clip 0)."""
    st = {k: state.pipeline_state[k] for k in STATE_F}
    st.update((f, state.info[k]) for k, f in ENGINE_INFO.items() if k in state.info)
    return st


class TrackingEnv:
    """A reference tracking env whose `reset` / `step` run as ONE fused CUDA launch each (C ABI `vnl_reset` / `vnl_step`,
    include/vnl_b200.h).  Every leaf carries a leading batch axis B (what `VmapWrapper` would hand over) and is a torch CUDA
    tensor.  A subclass compiles its model and task tables and states its reset draws: `start_frame_hi` (None: frame 0) and
    `reset_noise` (None: no noise draw)."""

    metric_keys = METRIC_KEYS  # names of `State.metrics`: columns METRIC_KEYS.index(name) of the step kernel's metrics output

    def __init__(self, model: mjcf.Model, task_blob, ref_traj, obs_size: int, *, solver: str, iterations: int, ls_iterations: int,
                 n_frames: int, start_frame_hi: Optional[int], reset_noise: Optional[float], device: str):
        self.model = mjcf.set_solver(model, solver, iterations, ls_iterations)
        self.task_blob, self._ref_traj, self._obs_size, self._n_frames = task_blob, ref_traj, obs_size, n_frames
        self._start_frame_hi, self._reset_noise = start_frame_hi, reset_noise
        self.model_blob = mb.build_model_blob(model)
        from .._lib import Engine  # raises if the CUDA library / a GPU is missing: no CPU fallback
        self.engine = Engine(self.model_blob, self.task_blob, device=device)
        self.device = self.engine.device

    # ---- brax Env surface --------------------------------------------------------------------
    @property
    def dt(self) -> float:
        return self.model.timestep * self._n_frames

    @property
    def action_size(self) -> int:
        return self.model.nu

    @property
    def observation_size(self) -> int:
        return self._obs_size

    @property
    def backend(self) -> str:
        return "vnl_b200"

    def _wrap(self, st: Dict, out: Dict, step: bool) -> State:
        m = out["metrics"]
        metrics = {k: m[:, METRIC_KEYS.index(k)] for k in self.metric_keys}
        info = dict(cur_frame=st["cur_frame"], sub_clip_frame=st["sub_clip_frame"], traj=out["traj"],
                    termination_error=metrics["termination_error"], solver_stats=out["stats"])
        return State(PipelineState({k: st[k] for k in STATE_F}), out["obs"], out["reward"], out["done"], metrics, info)

    def reset_draws(self, rng=None, batch_size: int = 1, start_frame=None, clip_id=None):
        """The host draws of `reset`, in the reference's order: the clip (uniform, on stacked clip tables only), the start frame
        (uniform in [0, start_frame_hi), or 0), then reset_noise * N(0, 1) on all of qpos.  A given `start_frame` / `clip_id` is
        not drawn.  Returns (qpos, qvel, start_frame, clip_id) for `reset_from`."""
        if not isinstance(rng, np.random.Generator):
            rng = np.random.default_rng(rng)
        B = int(batch_size)
        rt = self._ref_traj
        stacked = np.ndim(rt.position) == 3  # [nclips, T, 3]
        if stacked and clip_id is None:
            clip_id = rng.integers(0, len(rt.position), size=B)
        if clip_id is not None:
            clip_id = np.asarray(clip_id, dtype=np.int32).reshape(B)
        if start_frame is None:
            start_frame = np.zeros(B) if self._start_frame_hi is None else rng.integers(0, self._start_frame_hi, size=B)
        start_frame = np.asarray(start_frame, dtype=np.int32).reshape(B)
        row = (clip_id, start_frame) if stacked else start_frame
        g = lambda a: np.asarray(a)[row]
        qpos = np.hstack([g(rt.position), g(rt.quaternion), g(rt.joints)]).astype(np.float32)
        qvel = np.hstack([g(rt.velocity), g(rt.angular_velocity), g(rt.joints_velocity)]).astype(np.float32)
        if self._reset_noise is not None:
            qpos = qpos + (self._reset_noise * rng.standard_normal((B, self.model.nq))).astype(np.float32)
        return qpos, qvel, start_frame, clip_id

    def reset(self, rng=None, batch_size: int = 1, start_frame=None, clip_id=None) -> State:
        """`reset(rng)` of the reference env for `batch_size` envs: `reset_draws` on the host, then `reset_from`."""
        return self.reset_from(*self.reset_draws(rng, batch_size, start_frame, clip_id))

    def reset_from(self, qpos, qvel, start_frame, clip_id=None) -> State:
        """Reset tail after the random draws: `pipeline_init` + traj / obs / termination error."""
        import torch

        dev = lambda x, dtype: torch.as_tensor(x, dtype=dtype, device=self.device).contiguous()
        st_in = dict(qpos=dev(qpos, torch.float32), qvel=dev(qvel, torch.float32), cur_frame=dev(start_frame, torch.int32))
        if clip_id is not None:
            st_in["clip_id"] = dev(clip_id, torch.int32)
        B = qpos.shape[0]
        st, out = self.engine.alloc_state(B), self.engine.alloc_outputs(B)
        self.engine.reset(st_in, st, out)
        return self._wrap(st, out, step=False)

    def step(self, state: State, action) -> State:
        import torch

        st_in = engine_state(state)
        B = st_in["qpos"].shape[0]
        action = torch.as_tensor(action, dtype=torch.float32, device=self.device).reshape(B, self.action_size).contiguous()
        st, out = self.engine.alloc_state(B), self.engine.alloc_outputs(B)
        self.engine.step(st_in, action, st, out)
        return self._wrap(st, out, step=True)
