"""`AntTracking` -- mirror of the reference env (`envs/ant.py:25-438`) over the fused CUDA step.

BASELINE configs[0]: ant.xml loaded the brax way (jointless bodies fused: 10 bodies, nq 15, nv 14, nu 8, four foot
spheres against the floor), Newton solver with one iteration and four line-search iterations
(`configs/env_config.yaml:17-23`), eulerdamp disabled, timestep 0.01 x 5 substeps.  Same kernel as the rodent; the
task-blob switches select the ant semantics:

* every reward term and the healthy test read the PRE-step state (`ant.py:229 data_c = state.pipeline_state`);
* termination error = mean |.| over joints and over ALL body coordinates, threshold 0.9, `done = rtrunk < 0`
  (`ant.py:196,222-226`);
* reward = 0.05 rcom + 0.01 rvel + 0.20 rtrunk + 0.01 rquat + 0.001 ract with ract = 0.01 * -0.015 * sum(action^2) / nu
  (`ant.py:186-192,251`); the metrics hold the UNWEIGHTED terms (`ant.py:203-210`);
* the reference window of a step starts at OLD cur_frame + 1 (`ant.py:182` passes `state.info` before the increment) and
  the egocentric rotation is `data.xmat[0]`, the world body's, i.e. the identity (`ant.py:333`);
* obs = [bodies local, bodies global, root local, joints | qpos, qvel] in ONE vector (`ant.py:300-309`): the kernel's
  `traj` output is exactly the first block, so the host side only concatenates (and applies the reference's
  `nan_to_num` to that block too); `info` carries no traj.

The reference's `clips/ant_traj_still.p` is absent; as in its notebook the clip is the `init_qpos` pose (ant.xml:11)
tiled, zero velocities.
"""
from __future__ import annotations

import os
from typing import Optional

import numpy as np

from .. import clip as clipm
from .. import mjcf
from .. import model_blob as mb
from .base import State, TrackingEnv

_DATA = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "data")

ANT_ENV_ARGS = dict(solver="newton", iterations=1, ls_iterations=4)  # configs/env_config.yaml:17-23
ANT_METRIC_KEYS = ("rcom", "rvel", "rtrunk", "rquat", "ract", "termination_error")  # ant.py:148-155


def packaged_ant():
    """(model, clip): ant.xml compiled by tools/build_fixtures.py (brax-style fused) and the still clip."""
    model = mjcf.load_model(os.path.join(_DATA, "ant_model.npz"))
    return model, clipm.tiled_clip(model, model.arrays["init_qpos"], 256)


def ant_task_tables(model: mjcf.Model, reference_clip, *, clip_length=250, episode_length=150, ref_traj_length=5,
                    termination_threshold=0.9, body_error_multiplier=1.0, healthy_z_range=(0.2, 1.0), n_frames=5):
    nb, nj = model.nbody, model.nq - 7
    body_idxs = list(range(nb))      # ant.py:224 compares the clip against data.xpos: every body, world included
    joint_idxs = list(range(nj))     # ant.py:386: all joints
    state_size = model.nq + model.nv
    traj_size = ref_traj_length * (2 * 3 * nb + 3 + nj)
    blob = mb.build_task_blob(reference_clip, body_idxs=body_idxs, end_eff_idx=[], app_idx=[], joint_idxs=joint_idxs, com_idx=0,
                              njoint_cols=nj, clip_length=clip_length, ref_traj_length=ref_traj_length,
                              sub_clip_length=episode_length, healthy_z_range=healthy_z_range,
                              termination_threshold=termination_threshold, body_error_multiplier=body_error_multiplier,
                              n_frames=n_frames, torso_body=1, obs_size=state_size, traj_size=traj_size, kind=2,
                              reward_old_state=True, term_mean=True, use_subclip=False, obs_qfrc=False, com_from_field=True,
                              done_rtrunk=0.0, rot_body=0, traj_old_frame=True, ract_action=True, metrics_raw=True,
                              weights=(0.05, 0.01, 0.20, 0.01, 0.001, 0.0))
    return blob, state_size, traj_size


class AntTracking(TrackingEnv):
    """`reset`: `AntTracking.reset` (`ant.py:76-123`), start frame 0 and no reset noise, no draws; `step`: `AntTracking.step`
    (`ant.py:167-216`), one fused launch + the obs concatenation."""

    metric_keys = ANT_METRIC_KEYS

    def __init__(self, params=None, healthy_z_range=(0.2, 1.0), reset_noise_scale=1e-2, clip_length: int = 250,
                 episode_length: int = 150, ref_traj_length: int = 5, termination_threshold: float = 0.9,
                 body_error_multiplier: float = 1.0, n_frames: int = 5, device: str = "cuda:0",
                 model: Optional[mjcf.Model] = None, reference_clip=None, mjcf_path: str = "./assets/ant.xml", **kwargs):
        params = dict(ANT_ENV_ARGS, **(params or {}))
        if episode_length > clip_length:
            raise ValueError("episode_length cannot be greater than clip_length!")  # ant.py:73-74
        if model is None:
            model = mjcf.load_ant(mjcf_path)
        if reference_clip is None:
            if "clip_path" in params and os.path.exists(params["clip_path"]):
                reference_clip = clipm.load_pickle(params["clip_path"])  # ant.py:70-71
            else:
                reference_clip = clipm.tiled_clip(model, model.arrays["init_qpos"], 256)
        task_blob, state_size, traj_size = ant_task_tables(
            model, reference_clip, clip_length=clip_length, episode_length=episode_length, ref_traj_length=ref_traj_length,
            termination_threshold=termination_threshold, body_error_multiplier=body_error_multiplier,
            healthy_z_range=healthy_z_range, n_frames=n_frames)
        super().__init__(model, task_blob, reference_clip, traj_size + state_size, solver=params["solver"],
                         iterations=params["iterations"], ls_iterations=params["ls_iterations"], n_frames=n_frames,
                         start_frame_hi=None, reset_noise=None, device=device)

    def _wrap(self, st, out, step: bool) -> State:
        import torch
        state = super()._wrap(st, out, step)
        traj = state.info.pop("traj")
        traj = torch.nan_to_num(traj) if step else traj  # ant.py:199 nan_to_num(obs); reset applies none
        return state.replace(obs=torch.cat([traj, state.obs], dim=1))  # ant.py:300-309

    def reset_to_frame(self, start_frame, batch_size: int = 1) -> State:  # ant.py:125-165
        return self.reset(batch_size=batch_size, start_frame=np.full(int(batch_size), int(start_frame), dtype=np.int32))
