"""The resampling AutoReset (DESIGN §3h): `vnl_step_training_resample`, `Rollout(..., autoreset="resample")` and
`train(..., autoreset="resample")`.

The checker is a numpy restatement of the draw (Philox4x32-10, the block layout of include/vnl_b200.h `VnlResample`) and
the two entry points the new one is made of: `vnl_step_training` for the step (bit for bit wherever no episode ends) and
`vnl_reset` of the restated draw for the envs whose episode ends.

CPU: the restatement against Philox's published known-answer vectors, the C ABI's argument refusals, train()'s refusals and
checkpoint layout.  GPU: the rodent in all four kernel builds (as tests/test_inertia_solves.py forces them), the humanoid and
a 4-clip RodentMultiClipTracking, at a ragged B larger than the resident envs, with no env, some envs and every env done;
the rollout loop (graph == eager == a step-by-step loop); a small train() with checkpoint / restore.
"""
import ctypes
import os
import shutil

import numpy as np
import pytest

from conftest import pkg

libm, mb = pkg("_lib"), pkg("model_blob")

M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
MASK = 0xFFFFFFFF


# ---- numpy restatement of the draw ----------------------------------------------------------------------------------------------
def philox(ctr, key):
    """Philox4x32-10 on uint32 arrays: ctr [..., 4], key [..., 2] -> [..., 4]."""
    x = [np.asarray(ctr[..., i], dtype=np.uint64) for i in range(4)]
    k0, k1 = np.asarray(key[..., 0], dtype=np.uint64), np.asarray(key[..., 1], dtype=np.uint64)
    for _ in range(10):
        p0, p1 = np.uint64(M0) * x[0], np.uint64(M1) * x[2]
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & np.uint64(MASK), p1 >> np.uint64(32), p1 & np.uint64(MASK)
        x = [hi1 ^ x[1] ^ k0, lo1, hi0 ^ x[3] ^ k1, lo0]
        k0, k1 = (k0 + np.uint64(W0)) & np.uint64(MASK), (k1 + np.uint64(W1)) & np.uint64(MASK)
    return np.stack(x, axis=-1).astype(np.uint32)


def draw(seed, g, n, nclips, hi, nq, noise_scale):
    """(clip, start, normals [len(g), nq] in float64 or None) of the envs with global index g and reset counter n."""
    g, n = np.asarray(g, np.uint64), np.asarray(n, np.uint64)
    key = np.broadcast_to(np.array([seed & MASK, (seed >> 32) & MASK], np.uint64), g.shape + (2,))
    blk = lambda j: philox(np.stack([g, n, np.full_like(g, j), np.zeros_like(g)], axis=-1), key).astype(np.uint64)
    x = blk(0)
    clip = ((x[:, 0] * np.uint64(nclips)) >> np.uint64(32)).astype(np.int32)
    start = ((x[:, 1] * np.uint64(hi)) >> np.uint64(32)).astype(np.int32)
    if noise_scale == 0:
        return clip, start, None
    cols = []
    for j in range(1, (nq + 3) // 4 + 1):
        u = (((blk(j) >> np.uint64(8)) + np.uint64(1)).astype(np.float64)) * 2.0 ** -24
        for a, b in ((0, 1), (2, 3)):
            r, th = np.sqrt(-2.0 * np.log(u[:, a])), 2.0 * np.pi * u[:, b]
            cols += [r * np.cos(th), r * np.sin(th)]
    return clip, start, np.stack(cols, axis=1)[:, :nq]


def test_philox_known_answers():
    """Random123's known-answer vectors for philox4x32-10."""
    cases = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
             ((MASK,) * 4, (MASK, MASK), (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
             ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]
    for ctr, key, want in cases:
        got = philox(np.array([ctr], np.uint64), np.array([key], np.uint64))[0]
        assert [int(v) for v in got] == list(want), [hex(int(v)) for v in got]


def test_draw_distribution():
    """The restated draws are the distributions the env classes' reset() use: clip and start uniform, noise N(0, 1)."""
    g = np.arange(20000)
    clip, start, z = draw(12345, g, np.zeros_like(g), 4, 235, 74, 1e-3)
    assert clip.min() == 0 and clip.max() == 3 and start.min() == 0 and start.max() == 234
    assert abs(np.bincount(clip).std() / 5000) < 0.05 and abs(z.mean()) < 0.01 and abs(z.std() - 1) < 0.01
    clip1 = draw(12345, g, np.ones_like(g), 4, 235, 74, 0)[0]
    assert (clip1 != clip).mean() > 0.7  # the reset counter gives a new draw


# ---- CPU: refusals ------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(libm.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return libm.load_library()


def test_capi_refuses_bad_arguments(lib, rodent):
    """Argument errors come back as negative codes before any CUDA call (this runs without a GPU)."""
    ctx = libm.VnlContext()
    m, t = rodent["model_blob"], rodent["task_blob"]
    assert lib.vnl_context_init(ctypes.byref(ctx), m.ctypes.data, m.nbytes, t.ctypes.data, t.nbytes) == 0
    T, ref_len = int(t[mb.C["VNL_TH_CLIP_LEN"]]), int(t[mb.C["VNL_TH_REF_LEN"]])
    fake = 0x10000  # device addresses are never touched by a refused call
    st, out = libm.VnlState(*([fake] * 11)), libm.VnlState(*([fake] * 11))
    o = libm.VnlOutputs(*([fake] * 6))
    ep = libm.VnlEpisode(fake, fake, fake, fake, 150.0)

    def call(B=64, ctx_=ctx, st_=st, o_=o, ep_=ep, action=fake, **rs_kw):
        kw = dict(seed=1, env_offset=0, start_frame_hi=235, noise_scale=1e-3, reset_count=fake, scratch=fake)
        kw.update(rs_kw)
        rs = libm.VnlResample(**kw)
        return lib.vnl_step_training_resample(None if ctx_ is None else ctypes.byref(ctx_), fake, fake, B,
                                              None if st_ is None else ctypes.byref(st_), action, ctypes.byref(out),
                                              None if o_ is None else ctypes.byref(o_), None if ep_ is None else ctypes.byref(ep_),
                                              ctypes.byref(rs), None)
    bad = [call(B=0), call(B=-3), call(st_=None), call(o_=None), call(ep_=None), call(action=None), call(reset_count=None),
           call(scratch=None), call(start_frame_hi=0), call(start_frame_hi=-5), call(noise_scale=-1.0),
           call(noise_scale=float("nan")), call(noise_scale=float("inf")), call(start_frame_hi=T - ref_len + 1), call(ctx_=None), call(ep_=libm.VnlEpisode(fake, None, fake, fake, 150.0))]
    assert all(rc < 0 for rc in bad), bad
    rs_null = lib.vnl_step_training_resample(ctypes.byref(ctx), fake, fake, 64, ctypes.byref(st), fake, ctypes.byref(out), ctypes.byref(o),
                                             ctypes.byref(ep), None, None)
    assert rs_null < 0


def _stub_env(resample=True):
    """The sizes train() reads before any device work, with or without resample_spec."""
    import types
    attrs = {"resample_spec": lambda self: (235, 1e-3)} if resample else {}
    env = type("RodentTracking" if resample else "AntTracking", (), attrs)()
    env.engine = types.SimpleNamespace(obs_size=107, traj_size=795)
    env.observation_size, env.action_size, env.device = 107, 30, "cuda:0"
    return env


def test_train_refuses_unknown_or_unsupported_autoreset(monkeypatch):
    import torch
    trn = pkg("train")
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    assert trn.DEFAULTS["autoreset"] == "first"
    with pytest.raises(ValueError, match="autoreset"):
        trn.train(_stub_env(), 1000, autoreset="always")
    with pytest.raises(ValueError, match="autoreset.*resample_spec"):
        trn.train(_stub_env(resample=False), 1000, autoreset="resample")


def test_checkpoint_layout_names_autoreset_only_when_resampling(tmp_path):
    trn, ck = pkg("train"), pkg("checkpoint")

    def meta(**kw):
        cfg = dict(trn.DEFAULTS, **kw)
        return trn.run_meta(_stub_env(), cfg, trn.schedule(10 ** 6, cfg["num_evals"], cfg["batch_size"], cfg["num_minibatches"],
                                                             cfg["unroll_length"]), 1)
    first, res = meta(), meta(autoreset="resample")
    assert "autoreset" not in first["layout"] and set(first["layout"]) == set(trn.LAYOUT_KEYS)
    assert res["layout"]["autoreset"] == "resample"
    ck.check_meta(first, meta(), trn.MATCH_FIELDS)
    for saved, current in ((first, res), (res, first)):
        with pytest.raises(ValueError, match=r"layout\[autoreset\]"):
            ck.check_meta(saved, current, trn.MATCH_FIELDS)


# ---- GPU fixtures ---------------------------------------------------------------------------------------------------------------
EP = 150.0
BUILDS = ("ew1s0", "ew1s1", "ew2s0", "ew2s1")


def _variants(clip, n):
    """n clips of the packaged clip's length: the clip, then time-reversed / shifted copies with small offsets."""
    T = clip.position.shape[0]
    out = [clip]
    for i in range(1, n):
        idx = np.arange(T)[::-1] if i % 2 else np.roll(np.arange(T), 31 * i)
        out.append(clip.replace(position=clip.position[idx] + np.float32(0.002 * i), quaternion=clip.quaternion[idx],
                                joints=clip.joints[idx], body_positions=clip.body_positions[idx] + np.float32(0.002 * i),
                                velocity=clip.velocity[idx], angular_velocity=clip.angular_velocity[idx],
                                joints_velocity=clip.joints_velocity[idx],
                                body_quaternions=None if clip.body_quaternions is None else clip.body_quaternions[idx]))
    return out


@pytest.fixture(scope="module")
def lib_copies(tmp_path_factory):
    """home ("0" resident, "1" streamed) -> a private copy of libvnl_b200.so with VNL_STREAM latched (test_inertia_solves.py)."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    rod = pkg("envs.rodent")
    model, _ = rod.packaged_rodent()
    out = {}
    for stream in ("0", "1"):
        path = str(tmp_path_factory.mktemp("vnl_rs" + stream) / "libvnl_b200.so")
        shutil.copy(libm.LIB_PATH, path)
        with pytest.MonkeyPatch.context() as mp:
            mp.setenv("VNL_STREAM", stream)
            lib = libm.load_library(path)
            for ew in (1, 2):
                lib.vnl_dump_size(mb.build_model_blob(model, env_warps=ew).ctypes.data)
        out[stream] = path
    return out


def _field(blob, name):
    C = mb.C
    off, n = int(blob[C["VNL_TABLE_OFF"] + 2 * C[name]]), int(blob[C["VNL_TABLE_OFF"] + 2 * C[name] + 1])
    return blob[off:off + n].view(np.float32)


class Case:
    """An engine plus what the restatement needs: the task blob's clip tables, the draw parameters and a reset start state."""

    def __init__(self, eng, task_blob, hi, noise, subclip):
        self.eng, self.hi, self.noise, self.subclip = eng, int(hi), float(noise), subclip
        C = mb.C
        self.nclips, self.T = max(1, int(task_blob[C["VNL_TH_NCLIPS"]])), int(task_blob[C["VNL_TH_CLIP_LEN"]])
        d = eng.dims
        self.nq, self.nv = d["nq"], d["nv"]
        f = lambda n, w: _field(task_blob, n).reshape(-1, w)
        self.qpos_rows = np.hstack([f("VNL_T_POSITION", 3), f("VNL_T_QUATERNION", 4), f("VNL_T_JOINTS", self.nq - 7)])
        self.qvel_rows = np.hstack([f("VNL_T_VELOCITY", 3), f("VNL_T_ANGULAR_VELOCITY", 3), f("VNL_T_JOINTS_VELOCITY", self.nv - 6)])

    def restated(self, seed, g, n, noise=None):
        """(qpos float32, qvel, start, clip, normals) of the restated draws."""
        noise = self.noise if noise is None else noise
        clip, start, z = draw(seed, g, n, self.nclips, self.hi, self.nq, noise)
        row = clip * self.T + start
        q = self.qpos_rows[row]
        if z is not None:
            q = (q.astype(np.float64) + noise * z).astype(np.float32)
        return q, self.qvel_rows[row], start, clip, z

    def reset(self, qpos, qvel, start, clip):
        t = _torch()
        st_in = dict(qpos=_t(qpos), qvel=_t(qvel), cur_frame=_t(start), clip_id=_t(clip))
        st, out = self.eng.alloc_state(len(start)), self.eng.alloc_outputs(len(start))
        self.eng.reset(st_in, st, out)
        t.cuda.synchronize()
        return st, out


def _torch():
    import torch
    return torch


def _t(a):
    return _torch().tensor(np.ascontiguousarray(a), device="cuda")


def _h(x):
    return x.detach().cpu().numpy()


_CASES = {}


def _case(name, rodent, lib_copies):
    if name in _CASES:
        return _CASES[name]
    rod, hum = pkg("envs.rodent"), pkg("envs.humanoid")
    args = {k: rod.RODENT_ENV_ARGS[k] for k in ("end_eff_names", "appendage_names", "walker_body_names", "joint_names",
                                                "center_of_mass", "clip_length", "sub_clip_length", "ref_traj_length",
                                                "termination_threshold")}
    if name.startswith("rodent_ew"):  # one kernel build forced: blob width + library copy with the inertia home latched
        build = name.split("_")[1]
        ew, stream = int(build[2]), build[4]
        blob = mb.build_model_blob(rodent["model"], env_warps=ew)
        eng = libm.Engine(blob, rodent["task_blob"], device="cuda:0", lib_path=lib_copies[stream])
        assert eng.dims["env_warps"] == ew and (eng.ctx.workspace_bytes > 0) == (stream == "1"), name
        c = Case(eng, rodent["task_blob"], 235, 1e-3, True)
    elif name == "rodent_nonoise":
        env = pkg("envs").RodentTracking(reference_clip=rodent["clip"], model=rodent["model"], device="cuda:0",
                                         **dict(rod.RODENT_ENV_ARGS, reset_noise_scale=0.0))
        c = Case(env.engine, env.task_blob, *env.resample_spec(), True)
    elif name == "multiclip":
        env = pkg("envs").RodentMultiClipTracking(reference_clips=_variants(rodent["clip"], 4), model=rodent["model"], device="cuda:0",
                                                  **rod.RODENT_ENV_ARGS)
        assert env.nclips == 4
        c = Case(env.engine, env.task_blob, *env.resample_spec(), True)
        c.env = env
    else:
        model, clip = hum.packaged_humanoid(moving=True)
        env = pkg("envs").HumanoidTracking(model=model, reference_clip=clip, device="cuda:0")
        hi, noise = env.resample_spec()
        assert noise == 0.0 and hi == 250 - 150 - 5
        c = Case(env.engine, env.task_blob, hi, noise, False)
    _CASES[name] = c
    return c


def _inputs(c, B, which, seed):
    """A reset state of B envs, random actions, and episode inputs that end the episodes of `which` ("none" / "some" / "all")."""
    rng = np.random.default_rng(seed)
    g0 = rng.integers(0, 1000)
    q, v, start, clip, _ = c.restated(seed, np.arange(B) + g0, np.zeros(B, np.int64))
    st, _ = c.reset(q, v, start, clip)
    act = _t(rng.uniform(-1, 1, size=(B, c.eng.dims["nu"])).astype(np.float32))
    steps = np.zeros(B, np.float32)
    if which == "some":
        steps[::3] = EP - 1
        if c.subclip:
            st["sub_clip_frame"][1::5] = 9  # sub_clip_length - 1
    elif which == "all":
        steps[:] = EP - 1
    count = _t(rng.integers(0, 7, size=B).astype(np.int32))
    return st, act, _t(steps), count


def _run_resample(c, st, act, steps, count, seed, offset=0, lo=0, hi=None, noise=None):
    """vnl_step_training_resample on rows [lo, hi) (global env offset `offset`): (out state, outputs, steps, truncation, count)."""
    t = _torch()
    hi = st["qpos"].shape[0] if hi is None else hi
    B = hi - lo
    sl = {k: v[lo:hi].contiguous() for k, v in st.items()}
    out, o = c.eng.alloc_state(B), c.eng.alloc_outputs(B)
    so, tr, cnt = steps[lo:hi].clone(), t.zeros(B, device="cuda"), count[lo:hi].clone()
    scratch = t.full((B + 1,), -7, dtype=t.int32, device="cuda")
    c.eng.step_training_resample(sl, act[lo:hi].contiguous(), out, o, steps[lo:hi].contiguous(), t.zeros(B, device="cuda"), so, tr, EP, cnt,
                                 scratch, seed, offset, c.hi, c.noise if noise is None else noise)
    t.cuda.synchronize()
    return out, o, so, tr, cnt


STATE_KEYS = ("qpos", "qvel", "act", "qacc_warmstart", "xpos", "xquat", "subtree_com", "qfrc_actuator", "cur_frame", "sub_clip_frame",
              "clip_id")


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["none", "some", "all"])
@pytest.mark.parametrize("name", ["rodent_" + b for b in BUILDS] + ["rodent_nonoise", "humanoid", "multiclip"])
def test_resample_step_is_the_training_step_then_the_restated_reset(name, which, rodent, lib_copies):
    t = _torch()
    c = _case(name, rodent, lib_copies)
    B = c.eng.resident_envs + 37  # more than one round of the persistent grid, the last one ragged
    seed = 0x1234_5678_9ABC + len(name)
    st, act, steps, count0 = _inputs(c, B, which, 7 + len(which))
    # the reference: the training step with the first-state restore (the restored rows are not compared)
    first = {k: st[k].clone() for k in STATE_KEYS[:8]}
    ref, ro = c.eng.alloc_state(B), c.eng.alloc_outputs(B)
    rsteps, rtr = steps.clone(), t.zeros(B, device="cuda")
    c.eng.step_training(st, act, ref, ro, first, t.zeros(B, c.eng.obs_size, device="cuda"), steps, t.zeros(B, device="cuda"), rsteps, rtr, EP)
    out, o, so, tr, cnt = _run_resample(c, st, act, steps, count0, seed)
    done = _h(ro["done"]) > 0
    n_done = int(done.sum())
    if which == "all":
        assert done.all()
    elif which == "none":
        assert n_done == 0
    else:
        assert 0 < n_done < B and done[::3].all()
    keep = ~done
    # every env: the step's reward / done / metrics / truncation / steps / stats
    for a, b in ((o["reward"], ro["reward"]), (o["done"], ro["done"]), (o["metrics"], ro["metrics"]), (tr, rtr), (so, rsteps),
                 (o["stats"], ro["stats"])):
        assert np.array_equal(_h(a), _h(b))
    # envs that go on: bit-equal to the training step on every leaf
    for k in STATE_KEYS:
        assert np.array_equal(_h(out[k])[keep], _h(ref[k])[keep]), k
    for k in ("obs", "traj"):
        assert np.array_equal(_h(o[k])[keep], _h(ro[k])[keep]), k
    # the counters: +1 on exactly the done envs
    assert np.array_equal(_h(cnt), _h(count0) + done)
    if n_done:
        idx = np.nonzero(done)[0]
        q, v, start, clip, _ = c.restated(seed, idx, _h(count0)[idx])
        assert np.array_equal(_h(out["cur_frame"])[idx], start) and (_h(out["sub_clip_frame"])[idx] == 0).all()
        assert np.array_equal(_h(out["clip_id"])[idx], clip if c.nclips > 1 else np.zeros_like(clip))
        rst, rout = c.reset(q, v, start, clip)
        for k, a in [(k, out[k]) for k in STATE_KEYS[:8]] + [("obs", o["obs"]), ("traj", o["traj"])]:
            want = _h(rst[k]) if k in rst else _h(rout[k])
            got = _h(a)[idx]
            if c.noise == 0.0:
                assert np.array_equal(got, want), k
            else:
                assert np.abs(got - want).max() <= 1e-5 * max(1.0, float(np.abs(want).max())), k
    if which == "all":
        # the noise itself, at a scale where float32 rounding of qpos is far below 1e-5 * scale
        out1 = _run_resample(c, st, act, steps, count0, seed, noise=1.0)[0]
        q1, _, _, _, z = c.restated(seed, np.arange(B), _h(count0), noise=1.0)
        nq_cols = [i for i in range(c.nq) if not 3 <= i < 7]
        assert np.abs(_h(out1["qpos"])[:, nq_cols] - q1[:, nq_cols]).max() <= 1e-5
        # layout independence: two halves with their global offsets == the whole batch; a second run == the first
        h = B // 2
        halves = [_run_resample(c, st, act, steps, count0, seed, offset=lo, lo=lo, hi=hi) for lo, hi in ((0, h), (h, B))]
        again = _run_resample(c, st, act, steps, count0, seed)
        for k in STATE_KEYS:
            whole = _h(out[k])
            assert np.array_equal(np.concatenate([_h(x[0][k]) for x in halves]), whole), k
            assert np.array_equal(_h(again[0][k]), whole), k
        for k in ("obs", "traj"):
            assert np.array_equal(np.concatenate([_h(x[1][k]) for x in halves]), _h(o[k])), k
            assert np.array_equal(_h(again[1][k]), _h(o[k])), k


@pytest.mark.gpu
def test_start_frame_bound_keeps_the_reference_window_in_the_clip(rodent, lib_copies):
    """start_frame_hi = clip length - ref_traj_length + 1 would draw a start whose reference window runs past the clip: refused."""
    t = _torch()
    c = _case("multiclip", rodent, lib_copies)
    ref_len = int(c.eng.task_host[mb.C["VNL_TH_REF_LEN"]])
    B = 8
    st = c.eng.alloc_state(B)
    z = t.zeros(B, device="cuda")
    cnt, scratch = t.zeros(B, dtype=t.int32, device="cuda"), t.zeros(B + 1, dtype=t.int32, device="cuda")
    act = t.zeros(B, c.eng.dims["nu"], device="cuda")
    with pytest.raises(RuntimeError, match="-1"):
        c.eng.step_training_resample(st, act, c.eng.alloc_state(B), c.eng.alloc_outputs(B), z, z, z.clone(), z.clone(), EP, cnt, scratch,
                                     0, 0, c.T - ref_len + 1, 0.0)


# ---- rollout ------------------------------------------------------------------------------------------------------------------
RT, RB, RU = 20, 256, 3


def _policy(eng, seed):
    import torch
    pol = pkg("policy")
    params = pol.init_params(np.random.default_rng(seed), pol.param_shapes(eng.traj_size, eng.obs_size, eng.dims["nu"]), perturb=0.1)
    g = torch.Generator(device="cuda").manual_seed(seed)
    mean = torch.randn(eng.obs_size, device="cuda", generator=g) * 0.1
    std = torch.rand(eng.obs_size, device="cuda", generator=g) + 0.5
    draws = [(torch.randn(RT, RB, 64, device="cuda", generator=g), torch.randn(RT, RB, eng.dims["nu"], device="cuda", generator=g))
             for _ in range(RU)]
    return pol.IntentionPolicy(params, "cuda:0", mean, std), draws


@pytest.mark.gpu
def test_rollout_resamples_finished_episodes(rodent, lib_copies):
    t = _torch()
    c = _case("multiclip", rodent, lib_copies)
    env = c.env
    eng, seed, offset = env.engine, 99, 1000
    s0 = env.reset(np.random.default_rng(3), batch_size=RB)
    policy, draws = _policy(eng, 11)
    Rollout = pkg("rollout").Rollout
    eager = Rollout(env, policy, s0, RT, EP, use_graph=False, autoreset="resample", seed=seed, env_offset=offset)
    graph = Rollout(env, policy, s0, RT, EP, use_graph=True, autoreset="resample", seed=seed, env_offset=offset)
    assert eager.first is None and "reset_count" in eager.state_dict() and not any(k.startswith("first") for k in eager.state_dict())
    # the step-by-step loop over the C entry point, checking the episode bookkeeping at every step
    st = dict({k: v.clone() for k, v in s0.pipeline_state.items()}, cur_frame=s0.info["cur_frame"].clone(),
              sub_clip_frame=s0.info["sub_clip_frame"].clone(), clip_id=s0.info["clip_idx"].clone())
    obs, traj = s0.obs.clone(), s0.info["traj"].clone()
    steps, done, count = t.zeros(RB, device="cuda"), t.zeros(RB, device="cuda"), t.zeros(RB, dtype=t.int32, device="cuda")
    scratch = t.zeros(RB + 1, dtype=t.int32, device="cuda")
    pairs = set(zip(_h(st["clip_id"]).tolist(), _h(st["cur_frame"]).tolist()))
    resets = 0
    for u in range(RU):
        a, b = eager.generate_unroll(*draws[u]), graph.generate_unroll(*draws[u])
        t.cuda.synchronize()
        for k in ("observation", "next_observation", "action", "reward", "discount", "metrics"):
            assert t.equal(a[k], b[k]), (u, k)
        for grp in ("policy_extras", "state_extras"):
            for k in a[grp]:
                assert t.equal(a[grp][k], b[grp][k]), (u, grp, k)
        for k, v in eager.env_state.items():
            assert t.equal(graph.env_state[k], v), (u, k)
        assert t.equal(eager.reset_count, graph.reset_count)
        for s in range(RT):
            act, _ = policy(traj, obs, draws[u][0][s], draws[u][1][s])
            nxt, out, trunc = eng.alloc_state(RB), eng.alloc_outputs(RB), t.zeros(RB, device="cuda")
            before = _h(count)
            eng.step_training_resample(st, act, nxt, out, steps, done, steps, trunc, EP, count, scratch, seed, offset, *env.resample_spec())
            t.cuda.synchronize()
            assert t.equal(a["observation"][s], obs) and t.equal(a["reward"][s], out["reward"]), (u, s)
            assert t.equal(a["next_observation"][s], out["obs"]) and t.equal(a["state_extras"]["traj"][s], out["traj"]), (u, s)
            d = _h(out["done"]) > 0
            scf, cf, cl = _h(nxt["sub_clip_frame"]), _h(nxt["cur_frame"]), _h(nxt["clip_id"])
            assert scf.max() <= 10, (u, s)
            idx = np.nonzero(d)[0]
            _, _, start, clip, _ = c.restated(seed, idx + offset, before[idx])
            assert (scf[idx] == 0).all() and np.array_equal(cf[idx], start) and np.array_equal(cl[idx], clip), (u, s)
            pairs |= set(zip(clip.tolist(), start.tolist()))
            resets += len(idx)
            st, obs, traj, done = nxt, out["obs"], out["traj"], out["done"].clone()
        for k, v in st.items():
            assert t.equal(eager.env_state[k], v), (u, k)
        assert t.equal(eager.reset_count, count)
    assert resets > RB and len(pairs) > RB, (resets, len(pairs))
    # the default mode, by contrast: the sub-clip counter is never reset, so from the tenth step on every env is done
    first = Rollout(env, policy, s0, RT, EP, use_graph=True)
    for u in range(RU):
        tr = first.generate_unroll(*draws[u])
        t.cuda.synchronize()
        dn = 1 - tr["discount"]
        assert bool((dn[9:] == 1).all()) if u == 0 else bool((dn == 1).all()), u


# ---- train() -------------------------------------------------------------------------------------------------------------------
SMALL = dict(num_envs=256, batch_size=64, num_minibatches=4, unroll_length=4, num_updates_per_batch=2, num_eval_envs=16)
S = 2 * 64 * 4 * 4  # env steps of one epoch of 2 training steps


@pytest.mark.gpu
def test_train_with_resampling_follows_the_schedule_and_resumes(rodent, lib_copies, tmp_path):
    import torch
    trn, ck = pkg("train"), pkg("checkpoint")
    env = _case("multiclip", rodent, lib_copies).env
    seen = []
    _, _, metrics = trn.train(env, 2 * S, progress_fn=lambda s, m: seen.append(s), autoreset="resample", num_evals=3, **SMALL)
    assert seen == [0, S, 2 * S] and all(np.isfinite(v) for v in metrics.values())
    cfg = dict(trn.DEFAULTS, **SMALL, num_evals=2, autoreset="resample")
    a = trn.Run(env, cfg)
    a.fit(S, checkpoint_dir=str(tmp_path))
    assert a.rollout.autoreset == "resample" and a.evaluator.rollout.autoreset == "first"
    path = ck.latest(str(tmp_path))
    assert ck.read_meta(path)["layout"]["autoreset"] == "resample"
    assert int(a.rollout.reset_count.sum()) > 0
    with pytest.raises(ValueError, match=r"layout\[autoreset\]"):
        trn.train(env, S, restore_checkpoint_path=path, num_evals=2, **SMALL)
    b = trn.Run(env, cfg)
    b.trainer.training_step()  # graphs captured before the restore
    torch.cuda.synchronize()
    b.restore(path)
    torch.cuda.synchronize()
    sa, sb = a.rollout.state_dict(), b.rollout.state_dict()
    assert set(sa) == set(sb) and "reset_count" in sb
    for k in sa:
        assert sa[k].tobytes() == sb[k].tobytes(), k
    # b's next unroll (graph replay) == an eager loop of the entry point from the restored carry: env outputs bit for bit
    for r in (a, b):
        r.rollout.eps_z.normal_(generator=r.trainer.gen)
        r.rollout.eps_a.normal_(generator=r.trainer.gen)
    start = b.rollout.state_dict()
    tb = b.rollout.generate_unroll()
    torch.cuda.synchronize()
    d = lambda k: torch.as_tensor(start[k], device="cuda")
    st = {k[6:]: d(k) for k in start if k.startswith("state/")}
    steps, done, count, obs = d("steps"), d("done_prev"), d("reset_count"), d("obs")
    scratch = torch.zeros(257, dtype=torch.int32, device="cuda")
    for s in range(b.rollout.T):
        assert torch.equal(tb["observation"][s], obs), s
        nxt, out, trunc = env.engine.alloc_state(256), env.engine.alloc_outputs(256), torch.zeros(256, device="cuda")
        env.engine.step_training_resample(st, tb["action"][s].contiguous(), nxt, out, steps, done, steps, trunc, EP, count, scratch,
                                          cfg["seed"], 0, *env.resample_spec())
        torch.cuda.synchronize()
        assert torch.equal(tb["reward"][s], out["reward"]) and torch.equal(tb["discount"][s], 1 - out["done"]), s
        assert torch.equal(tb["next_observation"][s], out["obs"]) and torch.equal(tb["state_extras"]["traj"][s], out["traj"]), s
        assert torch.equal(tb["state_extras"]["truncation"][s], trunc), s
        st, obs, done = nxt, out["obs"], out["done"].clone()
    assert torch.equal(b.rollout.reset_count, count)
