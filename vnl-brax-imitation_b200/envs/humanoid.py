"""`HumanoidTracking` -- mirror of the reference env (`envs/humanoid.py:25-466`) over the fused CUDA step.

Same kernel as the rodent; the task blob switches select the humanoid semantics (SURVEY Appendix B):
every reward term and the healthy test read the PRE-step state (`humanoid.py:275,304`), the termination error is a
mean |.| over joints and over ALL body coordinates with threshold 0.9 and `done = rtrunk < 0.5` before scaling
(`humanoid.py:199,256-260`), no appendage term, no sub-clip episode, obs = [qpos, qvel] (55), traj = bodies local /
global + root local + all joints (630), COM reference from the clip's `center_of_mass` field (`humanoid.py:279`).
"""
from __future__ import annotations

import os
from typing import Optional

from .. import clip as clipm
from .. import mjcf
from .. import model_blob as mb
from .base import METRIC_KEYS, TrackingEnv

_DATA = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "data")

HUMANOID_ENV_ARGS = dict(solver="cg", iterations=6, ls_iterations=6)  # configs/env_config.yaml:1-8
# the episode metrics of the reference env (humanoid.py:121-128): the rodent's without the appendage term; the step kernel still
# writes all of METRIC_KEYS (column "rapp" unused)
HUMANOID_METRIC_KEYS = tuple(k for k in METRIC_KEYS if k != "rapp")


def packaged_humanoid(moving: bool = False):
    """(model, clip): humanoid.xml compiled by tools/build_fixtures.py and a stand-in for the reference's `clips/humanoid_traj_stand.p`
    (git-ignored and absent).  Default: `qpos0` tiled x256, zero velocities.  `moving=True`: 256 frames of states of a physics rollout
    (a PD-held humanoid dipping 20 cm with swinging arms, played forwards and backwards so that it stays inside the healthy range),
    processed like the rodent's clips -- tools/build_humanoid_moving_clip.py."""
    model = mjcf.load_model(os.path.join(_DATA, "humanoid_model.npz"))
    if moving:
        return model, clipm.clip_from_npz(os.path.join(_DATA, "humanoid_moving_clip.npz"))
    return model, clipm.tiled_clip(model, model.arrays["qpos0"], 256)


def humanoid_task_tables(model: mjcf.Model, reference_clip, *, clip_length=250, episode_length=150, ref_traj_length=5,
                         termination_threshold=0.9, body_error_multiplier=1.0, healthy_z_range=(1.0, 2.0), n_frames=5):
    nb, nj = model.nbody, model.nq - 7
    body_idxs = list(range(nb))       # humanoid.py:257 compares the clip against data.xpos: every body, world included
    joint_idxs = list(range(nj))      # humanoid.py:419: all joints, no index list
    obs_size = model.nq + model.nv    # humanoid.py:359-366
    traj_size = ref_traj_length * (2 * 3 * nb + 3 + nj)
    blob = mb.build_task_blob(reference_clip, body_idxs=body_idxs, end_eff_idx=[], app_idx=[], joint_idxs=joint_idxs, com_idx=0,
                              njoint_cols=nj, clip_length=clip_length, ref_traj_length=ref_traj_length,
                              sub_clip_length=episode_length, healthy_z_range=healthy_z_range,
                              termination_threshold=termination_threshold, body_error_multiplier=body_error_multiplier,
                              n_frames=n_frames, torso_body=1, obs_size=obs_size, traj_size=traj_size, kind=1,
                              reward_old_state=True, term_mean=True, use_subclip=False, obs_qfrc=False, com_from_field=True,
                              done_rtrunk=0.5)
    return blob, obs_size, traj_size


class HumanoidTracking(TrackingEnv):
    """`reset`: `HumanoidTracking.reset` (`humanoid.py:78-136`), a start frame and no reset noise (the reference applies none)."""

    metric_keys = HUMANOID_METRIC_KEYS

    def __init__(self, params=None, healthy_z_range=(1.0, 2.0), reset_noise_scale=1e-2, clip_length: int = 250,
                 episode_length: int = 150, ref_traj_length: int = 5, termination_threshold: float = 0.9,
                 body_error_multiplier: float = 1.0, n_frames: int = 5, device: str = "cuda:0",
                 model: Optional[mjcf.Model] = None, reference_clip=None, mjcf_path: str = "./assets/humanoid.xml", **kwargs):
        params = dict(HUMANOID_ENV_ARGS, **(params or {}))
        if episode_length > clip_length:
            raise ValueError("episode_length cannot be greater than clip_length!")  # humanoid.py:75-76
        if model is None:
            model = mjcf.load_humanoid(mjcf_path)
        if reference_clip is None:
            if "clip_path" in params and os.path.exists(params["clip_path"]):
                reference_clip = clipm.load_pickle(params["clip_path"])  # humanoid.py:72-73
            else:
                reference_clip = clipm.tiled_clip(model, model.arrays["qpos0"], 256)
        task_blob, obs_size, _ = humanoid_task_tables(
            model, reference_clip, clip_length=clip_length, episode_length=episode_length, ref_traj_length=ref_traj_length,
            termination_threshold=termination_threshold, body_error_multiplier=body_error_multiplier,
            healthy_z_range=healthy_z_range, n_frames=n_frames)
        super().__init__(model, task_blob, reference_clip, obs_size, solver=params["solver"], iterations=params["iterations"],
                         ls_iterations=params["ls_iterations"], n_frames=n_frames,
                         start_frame_hi=clip_length - episode_length - ref_traj_length, reset_noise=None, device=device)

    def resample_spec(self):
        """(start_frame_hi, noise_scale) of `reset`'s draws for the resampling AutoReset: no noise, as the reference."""
        return self._start_frame_hi, 0.0
