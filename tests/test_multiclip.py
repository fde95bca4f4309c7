"""SURVEY 8 row f4: multi-clip task tables + clip preprocessing on the GPU.

The reference stubs `RodentMultiClipTracking` (envs/rodent.py:473-475) and processes one clip at a time on the host
(preprocessing/mjx_preprocess.py:43-107).  Checkers: the single-clip oracle run per clip (a multi-clip env step must equal
the single-clip env step of that env's clip, bit for bit on the GPU and within tolerance against the CPU oracle), the
host restatement `clip.process_clip_qpos` and the reference's own pickle (golden fixture) for the preprocessing."""
import numpy as np
import pytest

from conftest import pkg, start_states


def _variants(clip, n):
    """n clips of the packaged clip's length: the clip itself, then time-reversed / shifted / scaled-joint variants."""
    out = [clip]
    T = clip.position.shape[0]
    for i in range(1, n):
        idx = (np.arange(T)[::-1] if i % 3 == 1 else np.roll(np.arange(T), 17 * i)) if i % 3 else np.arange(T)
        sc = 1.0 - 0.05 * i
        out.append(clip.replace(position=clip.position[idx] + np.float32(0.001 * i), quaternion=clip.quaternion[idx],
                                joints=(clip.joints[idx] * np.float32(sc)), body_positions=clip.body_positions[idx] + np.float32(0.001 * i),
                                velocity=clip.velocity[idx] * np.float32(sc), angular_velocity=clip.angular_velocity[idx],
                                joints_velocity=clip.joints_velocity[idx] * np.float32(sc),
                                body_quaternions=None if clip.body_quaternions is None else clip.body_quaternions[idx]))
    return out


def test_multiclip_blob_layout(rodent):
    """Host logic: stacked clips are stored clip-major, NCLIPS / CLIP_LEN in the header, index tables unchanged."""
    rod, mb = pkg("envs.rodent"), pkg("model_blob")
    clips = _variants(rodent["clip"], 3)
    args = {k: rod.RODENT_ENV_ARGS[k] for k in ("end_eff_names", "appendage_names", "walker_body_names", "joint_names", "center_of_mass")}
    blob, fclip, idx, obs_size, traj_size = rod.rodent_task_tables(rodent["model"], rod.stack_clips(clips), **args)
    C = mb.C
    assert blob[C["VNL_TH_NCLIPS"]] == 3 and blob[C["VNL_TH_CLIP_LEN"]] == 250 and (obs_size, traj_size) == (232, 795)
    single = rod.rodent_task_tables(rodent["model"], clips[1], **args)[0]
    assert single[C["VNL_TH_NCLIPS"]] == 1

    def field(b, name, dt=np.float32):
        off, n = int(b[C["VNL_TABLE_OFF"] + 2 * C[name]]), int(b[C["VNL_TABLE_OFF"] + 2 * C[name] + 1])
        return b[off:off + n].view(dt)
    for name in ("VNL_T_POSITION", "VNL_T_JOINTS", "VNL_T_BODY_POSITIONS", "VNL_T_JOINTS_VELOCITY"):
        m, s = field(blob, name), field(single, name)
        assert m.size == 3 * s.size and np.array_equal(m[s.size:2 * s.size], s), name
    assert np.array_equal(field(blob, "VNL_T_BODY_IDXS", np.int32), field(single, "VNL_T_BODY_IDXS", np.int32))


@pytest.mark.gpu
def test_multiclip_step_equals_single_clip_step_of_each_envs_clip(rodent, oracle_mod):
    import torch
    envs, rod, mb = pkg("envs"), pkg("envs.rodent"), pkg("model_blob")
    clips = _variants(rodent["clip"], 4)
    multi = envs.RodentMultiClipTracking(reference_clips=clips, model=rodent["model"], device="cuda:0", **rod.RODENT_ENV_ARGS)
    assert multi.nclips == 4
    B = 96
    rng = np.random.default_rng(5)
    # the draws of RodentMultiClipTracking.reset, done here so that the single-clip envs see the very same raw inputs
    clip_id = rng.integers(0, 4, size=B).astype(np.int32)
    start = rng.integers(0, 235, size=B).astype(np.int32)
    rt = multi._ref_traj
    g = lambda a: np.asarray(a)[clip_id, start]
    qpos = np.hstack([g(rt.position), g(rt.quaternion), g(rt.joints)]).astype(np.float32)
    qpos += (1e-3 * rng.standard_normal(qpos.shape)).astype(np.float32)
    qvel = np.hstack([g(rt.velocity), g(rt.angular_velocity), g(rt.joints_velocity)]).astype(np.float32)
    s = multi.reset_from(qpos, qvel, start, clip_id)
    assert np.array_equal(s.info["clip_idx"].cpu().numpy(), clip_id) and set(clip_id.tolist()) == {0, 1, 2, 3}
    s2 = multi.reset(np.random.default_rng(6), batch_size=B)  # the public reset draws clips itself
    assert s2.info["clip_idx"].min() >= 0 and s2.info["clip_idx"].max() <= 3 and torch.isfinite(s2.obs).all()
    singles = [envs.RodentTracking(reference_clip=c, model=rodent["model"], device="cuda:0", **rod.RODENT_ENV_ARGS) for c in clips]
    acts = torch.tensor(rng.uniform(-1, 1, size=(3, B, 30)).astype(np.float32), device="cuda")
    # reset parity: the multi-clip reset equals each clip's own reset from the same qpos / qvel / frame
    for c in range(4):
        mi = np.nonzero(clip_id == c)[0]
        m = torch.tensor(mi, device="cuda")
        one = singles[c].reset_from(qpos[mi], qvel[mi], start[mi])
        assert torch.equal(one.obs, s.obs[m])
        assert torch.equal(one.info["traj"], s.info["traj"][m])
        assert torch.equal(one.metrics["termination_error"], s.metrics["termination_error"][m])
    st = s
    for t in range(3):
        nxt = multi.step(st, acts[t])
        torch.cuda.synchronize()
        assert torch.equal(nxt.info["clip_idx"], st.info["clip_idx"])  # a step never changes the clip
        for c in range(4):
            m = torch.tensor(np.nonzero(clip_id == c)[0], device="cuda")
            sub = envs.State(pkg("envs.base").PipelineState({k: v[m].clone() for k, v in st.pipeline_state.items()}), st.obs[m], st.reward[m],
                             st.done[m], {}, {"cur_frame": st.info["cur_frame"][m].clone(), "sub_clip_frame": st.info["sub_clip_frame"][m].clone()})
            one = singles[c].step(sub, acts[t][m])
            for k in ("qpos", "qvel", "xpos"):
                assert torch.equal(one.pipeline_state[k], nxt.pipeline_state[k][m]), (t, c, k)
            assert torch.equal(one.reward, nxt.reward[m]) and torch.equal(one.done, nxt.done[m]), (t, c)
            assert torch.equal(one.obs, nxt.obs[m]) and torch.equal(one.info["traj"], nxt.info["traj"][m]), (t, c)
            for k in one.metrics:
                assert torch.equal(one.metrics[k], nxt.metrics[k][m]), (t, c, k)
        st = nxt
    # and against the CPU oracle's single-clip task logic for one of the non-trivial clips (clip 2)
    c = 2
    m = np.nonzero(clip_id == c)[0]
    args = {k: rod.RODENT_ENV_ARGS[k] for k in ("end_eff_names", "appendage_names", "walker_body_names", "joint_names", "center_of_mass")}
    tb = rod.rodent_task_tables(rodent["model"], clips[c], **args)[0]
    st_np = {k: s.pipeline_state[k].cpu().numpy()[m].astype(np.float64) for k in s.pipeline_state}
    st_np["cur_frame"] = s.info["cur_frame"].cpu().numpy()[m]
    st_np["sub_clip_frame"] = s.info["sub_clip_frame"].cpu().numpy()[m]
    so, oo = oracle_mod.step(rodent["model_blob"], tb, st_np, acts[0].cpu().numpy()[m].astype(np.float64), precision=32, dims=rodent["dims"],
                             obs_size=232, traj_size=795)
    first = multi.step(s, acts[0])
    assert np.array_equal(first.done.cpu().numpy()[m], oo["done"])
    assert np.abs(first.reward.cpu().numpy()[m] - oo["reward"]).max() < 2e-4
    assert np.abs(first.info["traj"].cpu().numpy()[m] - oo["traj"]).max() < 2e-3


@pytest.mark.gpu
def test_host_stepper_on_multiclip_env_equals_env_step(rodent):
    """hostio.HostStepper steps every env against its own clip, as env.step does: the same obs / traj / reward / done, bit for bit."""
    import torch
    envs, rod = pkg("envs"), pkg("envs.rodent")
    multi = envs.RodentMultiClipTracking(reference_clips=_variants(rodent["clip"], 4), model=rodent["model"], device="cuda:0",
                                         **rod.RODENT_ENV_ARGS)
    B, K = 96, 4
    s = multi.reset(np.random.default_rng(8), batch_size=B)
    assert set(s.info["clip_idx"].tolist()) == {0, 1, 2, 3}
    stepper = pkg("hostio").HostStepper(multi, s, autoreset=False)
    acts = torch.tensor(np.random.default_rng(9).uniform(-1, 1, size=(K, B, multi.action_size)).astype(np.float32)).pin_memory()
    for t in range(K):
        host = stepper.step(acts[t])
        s = multi.step(s, acts[t].cuda())
        torch.cuda.synchronize()
        for k, want in (("obs", s.obs), ("traj", s.info["traj"]), ("reward", s.reward), ("done", s.done)):
            assert torch.equal(host[k], want.cpu()), (t, k)


@pytest.mark.gpu
def test_process_clip_on_gpu_matches_host_restatement_and_reference_pickle(rodent, golden):
    """`vnl_process_clip` (kinematics pass of the env kernel per frame + finite-difference velocity kernel) against
    (a) `clip.process_clip_qpos` (float64 FK, the host restatement of mjx_preprocess.py:43-107) and (b) the fields of the
    reference's own pickle `clips/transform_snips_groom.p` (tests/golden/rodent_clip_golden.npz), for a stack of clips."""
    rod, clipm, mjcf = pkg("envs.rodent"), pkg("clip"), pkg("mjcf")
    clip = rodent["clip"]
    q0 = np.hstack([golden["position"], golden["quaternion"], golden["joints"]]).astype(np.float32)
    rng = np.random.default_rng(3)
    q1 = q0[::-1].copy()
    q2 = q0.copy(); q2[:, 3:7] *= np.float32(1.7)            # un-normalised root quaternion: kinematics normalises it
    q2[:, 7:] += (0.01 * rng.standard_normal(q2[:, 7:].shape)).astype(np.float32)
    stack = np.stack([q0, q1, q2])
    model = rodent["model"]
    got = rod.process_clips_gpu(model, stack)
    assert got.position.shape == (3, 250, 3) and got.body_positions.shape == (3, 250, model.nbody, 3)
    for c in range(3):
        want = clipm.process_clip_qpos(model, stack[c])
        for f, tol in (("position", 1e-7), ("quaternion", 2e-7), ("joints", 0.0), ("body_positions", 2e-6), ("body_quaternions", 2e-6),
                       ("velocity", 2e-4), ("angular_velocity", 2e-3), ("joints_velocity", 1e-3)):
            a, b = getattr(got, f)[c], getattr(want, f)
            err = float(np.abs(a - b).max())
            assert err <= tol * max(1.0, float(np.abs(b).max())), (c, f, err)
    # the reference pickle's own derived fields (FK of the 18 tracked bodies is what its body_positions holds)
    bidx = rodent["idx"]["body_idxs"]
    gb = np.asarray(golden["body_positions"])
    if gb.shape[1] == len(bidx):
        assert np.abs(got.body_positions[0][:, bidx] - gb).max() < 2e-6
    assert np.abs(got.velocity[0] - golden["velocity"]).max() < 1e-4
    assert np.abs(got.joints_velocity[0] - golden["joints_velocity"]).max() < 2e-3
    # single 2-D input: squeezed result, equal to clip 0 of the stack
    one = rod.process_clips_gpu(model, q0)
    assert one.position.shape == (250, 3) and np.array_equal(one.body_positions, got.body_positions[0])
    assert np.array_equal(one.joints_velocity, got.joints_velocity[0])
