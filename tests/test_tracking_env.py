"""The host half of every tracking env's reset (`TrackingEnv.reset_draws`), seeded, against an inline restatement of the
reference's reset draws: which numbers are drawn, in which order, and the qpos / qvel gathered from the clip tables.  The
evaluator's and train()'s seeded streams depend on that order.  The draws need no GPU: the Engine is stubbed out."""
import types

import numpy as np
import pytest

from conftest import pkg

B = 16


@pytest.fixture
def no_engine(monkeypatch):
    monkeypatch.setattr(pkg("_lib"), "Engine", lambda model_blob, task_blob, device: types.SimpleNamespace(device=device))


def _gather(rt, row):
    g = lambda a: np.asarray(a)[row]
    qpos = np.hstack([g(rt.position), g(rt.quaternion), g(rt.joints)]).astype(np.float32)
    qvel = np.hstack([g(rt.velocity), g(rt.angular_velocity), g(rt.joints_velocity)]).astype(np.float32)
    return qpos, qvel


def _check(env, seed, want):
    """`want(rng)` -> (qpos, qvel, start_frame, clip_id); both streams must also end in the same state."""
    rng_got, rng_want = np.random.default_rng(seed), np.random.default_rng(seed)
    got, ref = env.reset_draws(rng_got, batch_size=B), want(rng_want)
    for g, w in zip(got, ref):
        assert (g is None) == (w is None)
        if w is not None:
            assert g.dtype == w.dtype and np.array_equal(g, w)
    assert rng_got.integers(1 << 62) == rng_want.integers(1 << 62)


def test_rodent_reset_draws_start_frame_then_noise(no_engine):
    envs, rod = pkg("envs"), pkg("envs.rodent")
    model, clip = rod.packaged_rodent()
    env = envs.RodentTracking(reference_clip=clip, model=model, device="cuda:0", **rod.RODENT_ENV_ARGS)

    def want(rng):  # envs/rodent.py:119-176
        start = rng.integers(0, 250 - 10 - 5, size=B).astype(np.int32)
        qpos, qvel = _gather(env._ref_traj, start)
        return qpos + (1e-3 * rng.standard_normal(qpos.shape)).astype(np.float32), qvel, start, None
    _check(env, 3, want)


def test_multiclip_reset_draws_clip_then_start_frame_then_noise(no_engine):
    envs, rod = pkg("envs"), pkg("envs.rodent")
    model, clip = rod.packaged_rodent()
    clips = [clip.replace(position=clip.position + np.float32(0.01 * i), joints=clip.joints * np.float32(1 - 0.05 * i)) for i in range(4)]
    env = envs.RodentMultiClipTracking(reference_clips=clips, model=model, device="cuda:0", **rod.RODENT_ENV_ARGS)

    def want(rng):
        clip_id = rng.integers(0, 4, size=B).astype(np.int32)
        start = rng.integers(0, 250 - 10 - 5, size=B).astype(np.int32)
        qpos, qvel = _gather(env._ref_traj, (clip_id, start))
        return qpos + (1e-3 * rng.standard_normal(qpos.shape)).astype(np.float32), qvel, start, clip_id
    _check(env, 4, want)


def test_humanoid_reset_draws_start_frame_only(no_engine):
    envs, hum = pkg("envs"), pkg("envs.humanoid")
    model, clip = hum.packaged_humanoid(moving=True)
    env = envs.HumanoidTracking(model=model, reference_clip=clip, device="cuda:0")

    def want(rng):  # humanoid.py:78-136: no reset noise
        start = rng.integers(0, 250 - 150 - 5, size=B).astype(np.int32)
        return (*_gather(env._ref_traj, start), start, None)
    _check(env, 5, want)


def test_ant_reset_draws_nothing(no_engine):
    envs, ant = pkg("envs"), pkg("envs.ant")
    model, clip = ant.packaged_ant()
    env = envs.AntTracking(model=model, reference_clip=clip, device="cuda:0")

    def want(rng):  # ant.py:76-123: frame 0, no noise
        start = np.zeros(B, dtype=np.int32)
        return (*_gather(env._ref_traj, start), start, None)
    _check(env, 6, want)
