"""`RodentTracking` -- mirror of the reference env (`envs/rodent.py:16-470`) whose `reset` / `step`
run as ONE fused CUDA launch each (C ABI `vnl_reset` / `vnl_step`, include/vnl_b200.h).

Differences from the reference that are forced by the host language, nothing else:
  * the reference env is un-batched and batched by `jax.vmap`; here every leaf carries a leading
    batch axis B (what `VmapWrapper` would hand over) and arrays are torch CUDA tensors;
  * `reset(rng)` takes a numpy `Generator` / seed instead of a jax PRNG key (bit-equal random draws
    would need jax's threefry; the distributions are the reference's: `randint(0, clip_length -
    sub_clip_length - ref_traj_length)` and `reset_noise_scale * N(0, 1)` on all of qpos).
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional, Sequence

import numpy as np

from .. import clip as clipm
from .. import mjcf
from .. import model_blob as mb
from .base import PipelineState, State

# `configs/env_config.yaml:30-106` (rodent env_args)
RODENT_ENV_ARGS = dict(
    scale_factor=0.9, solver="cg", iterations=6, ls_iterations=6, clip_length=250, sub_clip_length=10, ref_traj_length=5,
    termination_threshold=5,
    end_eff_names=["foot_L", "foot_R", "hand_L", "hand_R"],
    appendage_names=["foot_L", "foot_R", "hand_L", "hand_R", "skull"],
    walker_body_names=["torso", "pelvis", "upper_leg_L", "lower_leg_L", "foot_L", "upper_leg_R", "lower_leg_R", "foot_R",
                       "skull", "jaw", "scapula_L", "upper_arm_L", "lower_arm_L", "finger_L", "scapula_R", "upper_arm_R",
                       "lower_arm_R", "finger_R"],
    joint_names=["vertebra_1_extend", "hip_L_supinate", "hip_L_abduct", "hip_L_extend", "knee_L", "ankle_L", "toe_L",
                 "hip_R_supinate", "hip_R_abduct", "hip_R_extend", "knee_R", "ankle_R", "toe_R", "vertebra_C11_extend",
                 "vertebra_cervical_1_bend", "vertebra_axis_twist", "atlas", "mandible", "scapula_L_supinate",
                 "scapula_L_abduct", "scapula_L_extend", "shoulder_L", "shoulder_sup_L", "elbow_L", "wrist_L",
                 "scapula_R_supinate", "scapula_R_abduct", "scapula_R_extend", "shoulder_R", "shoulder_sup_R", "elbow_R",
                 "wrist_R", "finger_R"],
    center_of_mass="torso",
)

METRIC_KEYS = ("rcom", "rvel", "rtrunk", "rquat", "ract", "rapp", "termination_error")

_DATA = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "data")


def packaged_rodent():
    """(model, clip) compiled from the reference assets by tools/build_fixtures.py; lets hosts
    without the reference checkout (the GPU box) construct the env."""
    return mjcf.load_model(os.path.join(_DATA, "rodent_model.npz")), clipm.clip_from_npz(os.path.join(_DATA, "rodent_clip.npz"))


def rodent_task_tables(model: mjcf.Model, reference_clip, *, end_eff_names, appendage_names, walker_body_names, joint_names,
                       center_of_mass, clip_length=250, sub_clip_length=10, ref_traj_length=5, termination_threshold=5.0,
                       body_error_multiplier=1.0, healthy_z_range=(0.05, 0.5), n_frames=5):
    """Index arrays of `RodentTracking.__init__` (`envs/rodent.py:65-93,113-115`) + the task blob."""
    end_eff_idx = [model.body_id(n) for n in end_eff_names]
    app_idx = [model.body_id(n) for n in appendage_names]
    com_idx = model.body_id(center_of_mass)
    body_idxs = [model.body_id(n) for n in walker_body_names]
    joint_idxs = [model.jnt_id(n) for n in joint_names]
    bp = np.asarray(reference_clip.body_positions)
    filtered = bp[..., body_idxs, :] if bp.shape[-2] != len(body_idxs) else bp  # rodent.py:114 (works on stacked clips too)
    clip = reference_clip.replace(body_positions=filtered)
    nj = model.nq - 7
    obs_size = model.nq + 2 * model.nv + 3 * len(end_eff_idx)
    traj_size = ref_traj_length * (3 * len(app_idx) + 2 * 3 * len(body_idxs) + 3 + len(joint_idxs))
    blob = mb.build_task_blob(clip, body_idxs=body_idxs, end_eff_idx=end_eff_idx, app_idx=app_idx, joint_idxs=joint_idxs,
                              com_idx=com_idx, njoint_cols=nj, clip_length=clip_length, ref_traj_length=ref_traj_length,
                              sub_clip_length=sub_clip_length, healthy_z_range=healthy_z_range,
                              termination_threshold=termination_threshold, body_error_multiplier=body_error_multiplier,
                              n_frames=n_frames, torso_body=1, obs_size=obs_size, traj_size=traj_size)
    idx = dict(end_eff_idx=end_eff_idx, app_idx=app_idx, com_idx=com_idx, body_idxs=body_idxs, joint_idxs=joint_idxs)
    return blob, clip, idx, obs_size, traj_size


class _Sys:
    def __init__(self, m: mjcf.Model, n_frames: int):
        self.nq, self.nv, self.nu, self.na, self.nbody = m.nq, m.nv, m.nu, m.na, m.nbody
        self.dt = m.timestep * n_frames
        self.model = m


class RodentTracking:
    def __init__(self, reference_clip=None, end_eff_names: Sequence[str] = (), appendage_names: Sequence[str] = (),
                 walker_body_names: Sequence[str] = (), joint_names: Sequence[str] = (), center_of_mass: str = "torso",
                 mjcf_path: str = "./assets/rodent.xml", scale_factor: float = 0.9, solver: str = "cg", iterations: int = 6,
                 ls_iterations: int = 6, healthy_z_range=(0.05, 0.5), reset_noise_scale=1e-3, clip_length: int = 250,
                 sub_clip_length: int = 10, ref_traj_length: int = 5, termination_threshold: float = 5,
                 body_error_multiplier: float = 1.0, n_frames: int = 5, device: str = "cuda:0",
                 model: Optional[mjcf.Model] = None, **kwargs):
        if sub_clip_length > clip_length:
            raise ValueError("episode_length cannot be greater than clip_length!")  # rodent.py:116-117
        if model is None:
            model = mjcf.load_rodent(mjcf_path, scale_factor, solver, iterations, ls_iterations)
        else:
            model.solver = {"cg": mjcf.SOLVER_CG, "newton": mjcf.SOLVER_NEWTON}[solver.lower()]
            model.iterations, model.ls_iterations = int(iterations), int(ls_iterations)
        self.model = model
        self.sys = _Sys(model, n_frames)
        self._n_frames = n_frames
        self._healthy_z_range = healthy_z_range
        self._reset_noise_scale = reset_noise_scale
        self._termination_threshold = termination_threshold
        self._body_error_multiplier = body_error_multiplier
        self._clip_length = clip_length
        self._sub_clip_length = sub_clip_length
        self._ref_traj_length = ref_traj_length
        self.task_blob, self._ref_traj, idx, self._obs_size, self._traj_size = rodent_task_tables(
            model, reference_clip, end_eff_names=end_eff_names, appendage_names=appendage_names,
            walker_body_names=walker_body_names, joint_names=joint_names, center_of_mass=center_of_mass,
            clip_length=clip_length, sub_clip_length=sub_clip_length, ref_traj_length=ref_traj_length,
            termination_threshold=termination_threshold, body_error_multiplier=body_error_multiplier,
            healthy_z_range=healthy_z_range, n_frames=n_frames)
        self._end_eff_idx, self._app_idx, self._com_idx = idx["end_eff_idx"], idx["app_idx"], idx["com_idx"]
        self._body_idxs, self._joint_idxs = idx["body_idxs"], idx["joint_idxs"]
        self.model_blob = mb.build_model_blob(model)
        from .._lib import Engine  # raises if the CUDA library / a GPU is missing: no CPU fallback
        self.engine = Engine(self.model_blob, self.task_blob, device=device)
        self.device = self.engine.device

    # ---- brax Env surface --------------------------------------------------------------------
    @property
    def dt(self) -> float:
        return self.sys.dt

    @property
    def action_size(self) -> int:
        return self.sys.nu

    @property
    def observation_size(self) -> int:
        return self._obs_size

    @property
    def metric_keys(self):
        """Names of `State.metrics` (columns METRIC_KEYS.index(name) of the step kernel's metrics output)."""
        return METRIC_KEYS

    @property
    def backend(self) -> str:
        return "vnl_b200"

    def _wrap(self, st: Dict, out: Dict) -> State:
        ps = PipelineState({k: st[k] for k in ("qpos", "qvel", "act", "qacc_warmstart", "xpos", "xquat", "subtree_com",
                                              "qfrc_actuator")})
        m = out["metrics"]
        metrics = {k: m[:, i] for i, k in enumerate(METRIC_KEYS)}
        info = dict(cur_frame=st["cur_frame"], sub_clip_frame=st["sub_clip_frame"], traj=out["traj"],
                    termination_error=m[:, 6], solver_stats=out["stats"], clip_idx=st["clip_id"])
        return State(ps, out["obs"], out["reward"], out["done"], metrics, info)

    def reset(self, rng, batch_size: int = 1, start_frame=None) -> State:
        """`RodentTracking.reset` (`envs/rodent.py:119-176`) for `batch_size` envs."""
        import torch

        if not isinstance(rng, np.random.Generator):
            rng = np.random.default_rng(rng)
        B = int(batch_size)
        hi = self._clip_length - self._sub_clip_length - self._ref_traj_length
        if start_frame is None:
            start_frame = rng.integers(0, hi, size=B)
        start_frame = np.asarray(start_frame, dtype=np.int32).reshape(B)
        noise = (self._reset_noise_scale * rng.standard_normal((B, self.sys.nq))).astype(np.float32)
        rt = self._ref_traj
        qpos = np.hstack([rt.position[start_frame], rt.quaternion[start_frame], rt.joints[start_frame]]).astype(np.float32)
        qvel = np.hstack([rt.velocity[start_frame], rt.angular_velocity[start_frame], rt.joints_velocity[start_frame]]).astype(np.float32)
        return self.reset_from(qpos + noise, qvel, start_frame)

    def resample_spec(self):
        """(start_frame_hi, noise_scale) of `reset`'s draws, for the resampling AutoReset on the GPU (rollout.Rollout(...,
        autoreset="resample")): start frame uniform in [0, start_frame_hi), qpos += noise_scale * N(0, 1), clip uniform over
        the task's clips."""
        return self._clip_length - self._sub_clip_length - self._ref_traj_length, float(self._reset_noise_scale)

    def reset_from(self, qpos, qvel, start_frame, clip_id=None) -> State:
        """Reset tail after the random draws: `pipeline_init` + traj / obs / termination error."""
        import torch

        dev = self.device
        B = qpos.shape[0]
        st_in = dict(qpos=torch.as_tensor(qpos, dtype=torch.float32, device=dev).contiguous(),
                     qvel=torch.as_tensor(qvel, dtype=torch.float32, device=dev).contiguous(),
                     cur_frame=torch.as_tensor(start_frame, dtype=torch.int32, device=dev).contiguous())
        if clip_id is not None:
            st_in["clip_id"] = torch.as_tensor(clip_id, dtype=torch.int32, device=dev).contiguous()
        st, out = self.engine.alloc_state(B), self.engine.alloc_outputs(B)
        self.engine.reset(st_in, st, out)
        return self._wrap(st, out)

    def step(self, state: State, action) -> State:
        """`RodentTracking.step` (`envs/rodent.py:178-239`): one fused launch."""
        import torch

        ps = state.pipeline_state
        B = ps["qpos"].shape[0]
        st_in = dict(ps)
        st_in["cur_frame"] = state.info["cur_frame"]
        st_in["sub_clip_frame"] = state.info["sub_clip_frame"]
        st_in["clip_id"] = state.info.get("clip_idx")
        action = torch.as_tensor(action, dtype=torch.float32, device=self.device).reshape(B, self.sys.nu).contiguous()
        st, out = self.engine.alloc_state(B), self.engine.alloc_outputs(B)
        self.engine.step(st_in, action, st, out)
        return self._wrap(st, out)


def stack_clips(clips):
    """[ReferenceClip] (equal lengths) -> one ReferenceClip whose fields carry a leading clip axis [nclips, T, ...]."""
    from dataclasses import fields
    out = {}
    for f in fields(clipm.ReferenceClip):
        vals = [getattr(c, f.name) for c in clips]
        if all(v is not None for v in vals):
            out[f.name] = np.stack([np.asarray(v) for v in vals])
    return clipm.ReferenceClip(**out)


class RodentMultiClipTracking(RodentTracking):
    """The env the reference only stubs (`envs/rodent.py:473-475`): `RodentTracking` over a SET of clips.  The clip tables
    are stacked `[nclips, T, ...]` in one task blob (VNL_TH_NCLIPS); every env carries `info["clip_idx"]` (VnlState.clip_id),
    drawn uniformly at reset; everything else (`step`, rewards, termination, quirks) is `RodentTracking` on that env's
    clip, in the same fused launch.  `reference_clips`: a list of ReferenceClip of equal length, or one already stacked."""

    def __init__(self, reference_clips=None, **kw):
        if isinstance(reference_clips, (list, tuple)):
            reference_clips = stack_clips(reference_clips)
        super().__init__(reference_clip=reference_clips, **kw)
        self.nclips = int(np.asarray(self._ref_traj.position).shape[0])

    def reset(self, rng, batch_size: int = 1, start_frame=None, clip_id=None) -> State:
        if not isinstance(rng, np.random.Generator):
            rng = np.random.default_rng(rng)
        B = int(batch_size)
        if clip_id is None:
            clip_id = rng.integers(0, self.nclips, size=B)
        clip_id = np.asarray(clip_id, dtype=np.int32).reshape(B)
        hi = self._clip_length - self._sub_clip_length - self._ref_traj_length
        if start_frame is None:
            start_frame = rng.integers(0, hi, size=B)
        start_frame = np.asarray(start_frame, dtype=np.int32).reshape(B)
        noise = (self._reset_noise_scale * rng.standard_normal((B, self.sys.nq))).astype(np.float32)
        rt = self._ref_traj
        g = lambda a: np.asarray(a)[clip_id, start_frame]
        qpos = np.hstack([g(rt.position), g(rt.quaternion), g(rt.joints)]).astype(np.float32)
        qvel = np.hstack([g(rt.velocity), g(rt.angular_velocity), g(rt.joints_velocity)]).astype(np.float32)
        return self.reset_from(qpos + noise, qvel, start_frame, clip_id)


def process_clips_gpu(model: mjcf.Model, mocap_qpos, max_qvel: float = 20.0, dt: float = 0.02, device: str = "cuda:0"):
    """`process_clip` (`preprocessing/mjx_preprocess.py:43-107`) for a stack of clips `[nclips, T, nq]` (or one `[T, nq]`)
    on the GPU: `vnl_process_clip` = the env kernel's kinematics pass per frame + the finite-difference velocity kernel.
    Returns a ReferenceClip with a leading clip axis (squeezed for a single 2-D input)."""
    import ctypes

    import torch

    from .._lib import Engine
    q = np.asarray(mocap_qpos, dtype=np.float32)
    single = q.ndim == 2
    if single:
        q = q[None]
    n, T, nq = q.shape
    eng = Engine(mb.build_model_blob(model), None, device=device)
    dev = eng.device
    qd = torch.as_tensor(q, device=dev).contiguous()
    f = lambda *s: torch.empty(*s, dtype=torch.float32, device=dev)
    qo, bp, bq, qv = f(n, T, nq), f(n, T, model.nbody, 3), f(n, T, model.nbody, 4), f(n, T, nq - 1)
    with torch.cuda.device(dev):
        rc = eng.lib.vnl_process_clip(ctypes.byref(eng.ctx), eng.model_dev.data_ptr(), n, T, qd.data_ptr(), float(dt), float(max_qvel),
                                      qo.data_ptr(), bp.data_ptr(), bq.data_ptr(), qv.data_ptr(), eng._stream())
    if rc:
        raise RuntimeError(f"vnl_process_clip failed ({rc})")
    torch.cuda.synchronize(dev)
    qo, bp, bq, qv = (x.cpu().numpy() for x in (qo, bp, bq, qv))
    sq = (lambda a: a[0]) if single else (lambda a: a)
    c = np.ascontiguousarray
    return clipm.ReferenceClip(position=c(sq(qo[..., :3])), quaternion=c(sq(qo[..., 3:7])), joints=c(sq(qo[..., 7:])),
                               body_positions=c(sq(bp)), velocity=c(sq(qv[..., :3])), joints_velocity=c(sq(qv[..., 6:])),
                               angular_velocity=c(sq(qv[..., 3:6])), body_quaternions=c(sq(bq)))
