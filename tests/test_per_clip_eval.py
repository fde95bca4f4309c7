"""Per-clip evaluation: the clip x start-frame sweep (evaluator.clip_sweep), the two reductions vnl_eval_clip_stats and
vnl_eval_frame_profile (include/vnl_train.h) against float64, `Evaluator(per_clip=True)` against numpy restatements over the same
rollout, and `train(per_clip_eval=True)`.  Tolerances follow tests/test_train_kernels.py (u = 2^-24): the kernels accumulate in
double, so what remains is the final rounding to fp32 plus the double sums' own error."""
import os
import types

import numpy as np
import pytest

from conftest import pkg
from test_multiclip import _variants

tk = pkg("train_kernels")
libm = pkg("_lib")

U = 2.0 ** -24
TINY = 2.0 ** -126
SENTINEL = 12345.0
NM = len(pkg("envs.rodent").METRIC_KEYS)


# ---- CPU: layout, refusals, configuration ------------------------------------------------------------------------------------------
def test_clip_sweep_layout_and_refusals():
    ev = pkg("evaluator")
    cid, sf = ev.clip_sweep(4, 32, 235)
    assert cid.dtype == np.int32 and sf.dtype == np.int32 and cid.shape == sf.shape == (32,)
    assert np.array_equal(cid, np.repeat(np.arange(4), 8))                            # clip-major
    assert np.array_equal(sf, np.tile([(w * 235) // 8 for w in range(8)], 4))       # windows spread over [0, 235)
    assert sf.min() == 0 and sf.max() < 235
    cid, sf = ev.clip_sweep(1, 5, 100)
    assert np.array_equal(cid, np.zeros(5)) and np.array_equal(sf, [0, 20, 40, 60, 80])
    cid, sf = ev.clip_sweep(3, 3, 235)                                                # one window: every clip from frame 0
    assert np.array_equal(cid, [0, 1, 2]) and np.array_equal(sf, [0, 0, 0])
    for nclips, B in ((4, 30), (4, 2), (0, 8)):
        with pytest.raises(ValueError, match=r"num_eval_envs \(%d\).*clip count \(%d\)" % (B, nclips)):
            ev.clip_sweep(nclips, B, 235)
    with pytest.raises(ValueError, match="resample_spec"):
        ev.sweep_layout(types.SimpleNamespace(task_blob=_task_header(1, 250)), 8)


def _task_header(nclips, clip_len):
    C = pkg("model_blob").C
    blob = np.zeros(C["VNL_DATA_OFF"], dtype=np.uint32)
    blob[C["VNL_TH_NCLIPS"]], blob[C["VNL_TH_CLIP_LEN"]] = nclips, clip_len
    return blob


def _stub_env(nclips=None, name="RodentMultiClipTracking"):
    """The sizes train() reads before any device work; with `nclips`, a task blob header and the rodent's resample_spec."""
    attrs = {} if nclips is None else {"resample_spec": lambda self: (235, 1e-3)}
    env = type(name, (), attrs)()
    env.engine = types.SimpleNamespace(obs_size=107, traj_size=795)
    env.observation_size, env.action_size, env.device = 107, 30, "cuda:0"
    if nclips is not None:
        env.task_blob = _task_header(nclips, 250)
    return env


def test_per_clip_eval_is_refused_before_any_device_work(monkeypatch):
    import torch
    trn = pkg("train")
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    with pytest.raises(ValueError, match="per_clip_eval.*AntTracking has no resample_spec"):
        trn.train(_stub_env(name="AntTracking"), 1000, per_clip_eval=True)
    with pytest.raises(ValueError, match=r"per_clip_eval.*num_eval_envs \(128\).*clip count \(3\)"):
        trn.train(_stub_env(3), 1000, per_clip_eval=True)
    with pytest.raises(ValueError, match=r"per_clip_eval.*clip count \(3\)"):  # the eval env is the one swept
        trn.train(_stub_env(4), 1000, per_clip_eval=True, eval_env=_stub_env(3))
    trn.check_config(_stub_env(4), dict(trn.DEFAULTS, per_clip_eval=True), 1)
    trn.check_config(_stub_env(name="AntTracking"), dict(trn.DEFAULTS), 1)  # the default never asks for a sweep


def test_per_clip_eval_is_not_part_of_the_checkpoint_layout():
    trn, ck = pkg("train"), pkg("checkpoint")
    assert "per_clip_eval" in trn.DEFAULTS and "per_clip_eval" not in trn.LAYOUT_KEYS and "per_clip_eval" not in trn.MATCH_FIELDS
    env = _stub_env(4)

    def meta(flag):
        cfg = dict(trn.DEFAULTS, per_clip_eval=flag)
        return trn.run_meta(env, cfg, trn.schedule(10 ** 6, cfg["num_evals"], cfg["batch_size"], cfg["num_minibatches"], cfg["unroll_length"]), 1)
    ck.check_meta(meta(False), meta(True), trn.MATCH_FIELDS)
    ck.check_meta(meta(True), meta(False), trn.MATCH_FIELDS)


@pytest.fixture(scope="module")
def host_lib():
    if not os.path.exists(libm.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return tk.lib()


def test_per_clip_exports_refuse_bad_arguments_before_any_cuda_call(host_lib):
    """Every refusal returns -1 before the library touches CUDA; the fake addresses are never dereferenced."""
    L = host_lib
    P = 0x7000000000
    cs = lambda B=1536, nm=7, em=P, st=P, cid=P, nclips=64, mean=P, std=P, count=P: L.vnl_eval_clip_stats(B, nm, em, st, cid, nclips, mean, std,
                                                                                                            count, None)
    fp = lambda T=150, B=1536, nm=7, m=P, r=P, st=P, sf=P, cid=P, nclips=64, L_=250, fs=P, fc=P: L.vnl_eval_frame_profile(
        T, B, nm, m, r, st, sf, cid, nclips, L_, fs, fc, None)
    refusals = {
        "clip_stats B 0": cs(B=0), "clip_stats nm -1": cs(nm=-1), "clip_stats nm 16": cs(nm=16), "clip_stats nclips 0": cs(nclips=0),
        "clip_stats NULL episode_metrics": cs(em=None), "clip_stats NULL episode_steps": cs(st=None), "clip_stats NULL mean": cs(mean=None),
        "clip_stats NULL std": cs(std=None), "clip_stats NULL count": cs(count=None),
        "frame_profile T 0": fp(T=0), "frame_profile B 0": fp(B=0), "frame_profile nm -1": fp(nm=-1), "frame_profile nm 16": fp(nm=16),
        "frame_profile nclips 0": fp(nclips=0), "frame_profile clip_len 0": fp(L_=0),
        "frame_profile NULL metrics": fp(m=None), "frame_profile NULL metrics nm 0": fp(nm=0, m=None), "frame_profile NULL reward": fp(r=None),
        "frame_profile NULL episode_steps": fp(st=None), "frame_profile NULL start_frame": fp(sf=None),
        "frame_profile NULL frame_sum": fp(fs=None), "frame_profile NULL frame_count": fp(fc=None),
    }
    assert {k: v for k, v in refusals.items() if v != -1} == {}


# ---- GPU: the kernels against float64 -----------------------------------------------------------------------------------------------
def _check(name, got, want, bound):
    """|got - want| <= bound elementwise (float64), as tests/test_train_kernels.py checks."""
    import torch
    got, want = got.double(), want.double()
    bound = torch.as_tensor(bound, dtype=torch.float64, device=want.device).expand_as(want)
    assert torch.isfinite(got).all(), name
    r = (got - want).abs() / bound
    ratio, i = float(r.max()), int(r.argmax())
    print("%-44s worst error / tolerance %.3g" % (name, ratio))
    assert ratio <= 1.0, (name, ratio, float(got.flatten()[i]), float(want.flatten()[i]), float(bound.flatten()[i]))


@pytest.mark.gpu
@pytest.mark.parametrize("nm,null_ids", [(0, False), (15, False), (7, True)], ids=["nm0", "nm15", "nm7-null-clip-id"])
def test_clip_kernels_match_float64(nm, null_ids):
    """B = 8193 (a ragged last chunk), 37 clips of which three are empty, ids -1 and 37 (counted nowhere), start frames near both ends
    of a 40-frame clip (the clamp bins several steps into the first and the last frame).  The episode sums come from
    vnl_eval_metrics over the same unroll, so the profile must add up to them."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    K = tk.lib()
    st_ = torch.cuda.current_stream().cuda_stream
    T, B, C, L = 20, 8193, 37, 40
    rng = np.random.default_rng(nm)
    g = torch.Generator(device="cuda").manual_seed(nm)
    metrics = torch.randn(T, B, max(nm, 1), device="cuda", generator=g)[:, :, :nm].contiguous()
    reward = torch.randn(T, B, device="cuda", generator=g)
    done = (torch.rand(T, B, device="cuda", generator=g) > 0.93).float()
    done[:, :64] = 0.0  # a few envs run the whole unroll
    mp = metrics.data_ptr() if nm else reward.data_ptr()  # nm = 0: never read, but not NULL
    em, active, steps = torch.zeros(B, nm + 1, device="cuda"), torch.zeros(B, device="cuda"), torch.zeros(B, device="cuda")
    tk.check(K.vnl_eval_metrics(T, B, nm, mp, reward.data_ptr(), done.data_ptr(), em.data_ptr(), active.data_ptr(), steps.data_ptr(), st_),
             "eval_metrics")
    clip = rng.choice(np.setdiff1d(np.arange(C), [5, 17, 36]), size=B).astype(np.int32)
    bad = rng.choice(B, 80, replace=False)
    clip[bad[:40]], clip[bad[40:]] = -1, C
    start = rng.integers(0, L, size=B).astype(np.int32)
    start[rng.choice(B, 300, replace=False)] = rng.integers(L - 4, L + 3, size=300)  # near / past the end: clamped to L - 1
    start[rng.choice(B, 50, replace=False)] = -3                                       # before the start: clamped to 0
    clip_d, start_d = torch.as_tensor(clip, device="cuda"), torch.as_tensor(start, device="cuda")
    cid = None if null_ids else clip_d.data_ptr()

    def run():
        ncol = nm + 2
        mean, sd = torch.full((C * ncol + 1,), SENTINEL, device="cuda"), torch.full((C * ncol + 1,), SENTINEL, device="cuda")
        count = torch.full((C + 1,), -7, dtype=torch.int32, device="cuda")
        fsum = torch.full((C * L * (nm + 1) + 1,), SENTINEL, device="cuda")
        fcount = torch.full((C * L + 1,), -7, dtype=torch.int32, device="cuda")
        tk.check(K.vnl_eval_clip_stats(B, nm, em.data_ptr(), steps.data_ptr(), cid, C, mean.data_ptr(), sd.data_ptr(), count.data_ptr(), st_),
                 "clip_stats")
        tk.check(K.vnl_eval_frame_profile(T, B, nm, mp, reward.data_ptr(), steps.data_ptr(), start_d.data_ptr(), cid, C, L, fsum.data_ptr(),
                                          fcount.data_ptr(), st_), "frame_profile")
        torch.cuda.synchronize()
        for buf, s in ((mean, SENTINEL), (sd, SENTINEL), (count, -7), (fsum, SENTINEL), (fcount, -7)):
            assert buf[-1] == s, "written past the end"
        return [x[:-1].cpu() for x in (mean, sd, count, fsum, fcount)]

    mean, sd, count, fsum, fcount = first = run()
    again = run()
    for a, b in zip(first, again):  # bit-identical, NaN included
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))

    # float64 reference
    c_ref = np.zeros(B, np.int32) if null_ids else clip
    em64, st64 = em.double().cpu().numpy(), steps.double().cpu().numpy()
    vals = np.concatenate([em64, st64[:, None]], 1)                        # [B, nm + 2]
    mean, sd = mean.view(C, nm + 2).double(), sd.view(C, nm + 2).double()
    count = count.numpy()
    empty = [c for c in range(C) if not (c_ref == c).any()]
    assert (5 in empty and 17 in empty and 36 in empty) and (len(empty) == C - 1 if null_ids else len(empty) == 3)
    assert count.sum() == (B if null_ids else B - 80)  # ids -1 and C are counted nowhere
    for c in range(C):
        v = vals[c_ref == c]
        assert count[c] == len(v)
        if not len(v):
            assert torch.isnan(mean[c]).all() and torch.isnan(sd[c]).all()
            continue
        mu, s = torch.as_tensor(v.mean(0)), torch.as_tensor(v.std(0))
        _check("clip_stats nm %d clip %d mean" % (nm, c), mean[c], mu, 2 * U * torch.as_tensor(np.abs(v).mean(0)) + TINY)
        _check("clip_stats nm %d clip %d std" % (nm, c), sd[c], s, 2 * U * s + 2.0 ** -40 * torch.as_tensor(np.abs(v).mean(0)) + TINY)
    # the profile: every (env, step < min(steps, T)) binned at clamp(start + t, 0, L - 1)
    n = np.minimum(st64.astype(np.int64), T)
    bb, tt = np.nonzero(np.arange(T)[None, :] < n[:, None])
    keep = (c_ref[bb] >= 0) & (c_ref[bb] < C)
    bb, tt = bb[keep], tt[keep]
    cc, ff = c_ref[bb], np.clip(start[bb] + tt, 0, L - 1)
    step_vals = np.concatenate([metrics.double().cpu().numpy(), reward.double().cpu().numpy()[:, :, None]], 2)[tt, bb]  # [steps, nm + 1]
    want, mag, wcount = np.zeros((C, L, nm + 1)), np.zeros((C, L, nm + 1)), np.zeros((C, L), np.int64)
    np.add.at(want, (cc, ff), step_vals)
    np.add.at(mag, (cc, ff), np.abs(step_vals))
    np.add.at(wcount, (cc, ff), 1)
    fsum, fcount = fsum.view(C, L, nm + 1), fcount.view(C, L).numpy()
    assert np.array_equal(fcount, wcount)
    assert (fcount[:, L - 1] > fcount[:, L - 2]).any() and (fcount[:, 0] > 0).any()  # the clamps did bin several steps
    _check("frame_profile nm %d" % nm, fsum, torch.as_tensor(want), 2 * U * torch.as_tensor(mag) + TINY)
    # per clip: the frame counts are the clip's episode steps, the frame sums its episode sums
    for c in range(C):
        m = c_ref == c
        assert fcount[c].sum() == n[m].sum()
        if m.any():
            ep = torch.as_tensor(em64[m].sum(0))
            _check("frame_profile nm %d clip %d sums" % (nm, c), fsum[c].double().sum(0), ep,
                   (L + T + 2) * U * torch.as_tensor(mag[c].sum(0)) + TINY)


# ---- GPU: the evaluator ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def multi(rodent):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    rod = pkg("envs.rodent")
    return pkg("envs").RodentMultiClipTracking(reference_clips=_variants(rodent["clip"], 4), model=rodent["model"], device="cuda:0",
                                              **rod.RODENT_ENV_ARGS)


def _policy(env):
    pol = pkg("policy")
    eng = env.engine
    params = pol.init_params(np.random.default_rng(7), pol.param_shapes(eng.traj_size, eng.obs_size, env.action_size))
    return pol.PrecisePolicy(params, "cuda:0")


def _first_episode_steps(done):
    """[B] steps of each env's first episode in an unroll that starts at reset (its first done, inclusive; T if none)."""
    T = done.shape[0]
    d = done > 0
    return np.where(d.any(0), d.argmax(0) + 1, T)


@pytest.mark.gpu
def test_evaluator_per_clip_matches_numpy_over_the_same_rollout(multi, monkeypatch):
    import torch
    ev = pkg("evaluator")
    B, T = 32, 30
    resets = []
    real = multi.reset
    monkeypatch.setattr(multi, "reset", lambda *a, **k: resets.append(real(*a, **k)) or resets[-1])
    e = ev.Evaluator(multi, _policy(multi), num_eval_envs=B, episode_length=T, seed=7, per_clip=True)
    assert (e.nclips, e.clip_len) == (4, 250)
    cid, sf = ev.clip_sweep(4, B, multi.resample_spec()[0])
    names = list(multi.metric_keys) + ["reward"]
    cols = [pkg("envs.rodent").METRIC_KEYS.index(n) for n in multi.metric_keys] + [NM]
    for epoch in range(2):  # the second evaluation replays the captured graph from a fresh reset: the same layout
        out = e.run_evaluation({"training/sps": 1.0})
        s0 = resets[-1]
        assert np.array_equal(s0.info["clip_idx"].cpu().numpy(), cid) and np.array_equal(s0.info["cur_frame"].cpu().numpy(), sf)
        ro = e.rollout
        em, steps = e.episode_metrics.cpu().numpy().astype(np.float64), e.episode_steps.cpu().numpy().astype(np.float64)
        # scalars: still over every env
        for i, n in zip(cols, names):
            assert abs(out[f"eval/episode_{n}"] - em[:, i].mean()) < 1e-5 and abs(out[f"eval/episode_{n}_std"] - em[:, i].std()) < 1e-5
        assert out["eval/avg_episode_length"] == steps.mean()
        # per clip: a numpy grouping of the same episode sums
        assert out["eval/clip/num_episodes"].shape == (4,) and np.array_equal(out["eval/clip/num_episodes"], [8] * 4)
        assert np.issubdtype(out["eval/clip/num_episodes"].dtype, np.integer)
        for i, n in zip(cols, names):
            g = em[:, i].reshape(4, 8)
            for key, want in ((f"eval/clip/episode_{n}", g.mean(1)), (f"eval/clip/episode_{n}_std", g.std(1))):
                assert out[key].shape == (4,) and np.abs(out[key] - want).max() <= 1e-6 * max(1.0, np.abs(g).max()), (key, out[key], want)
        assert np.abs(out["eval/clip/avg_episode_length"] - steps.reshape(4, 8).mean(1)).max() < 1e-6
        # per frame: a numpy restatement over the rollout's buffers
        met, rew, done = ro.metrics.cpu().numpy().astype(np.float64), ro.reward.cpu().numpy().astype(np.float64), ro.done.cpu().numpy()
        n_steps = _first_episode_steps(done)
        assert np.array_equal(n_steps, steps)
        vals = np.concatenate([met, rew[:, :, None]], 2)
        fsum, fcount = np.zeros((4, 250, NM + 1)), np.zeros((4, 250), np.int64)
        for b in range(B):
            for t in range(n_steps[b]):
                f = min(max(sf[b] + t, 0), 249)
                fsum[cid[b], f] += vals[t, b]
                fcount[cid[b], f] += 1
        assert out["eval/frame/count"].shape == (4, 250) and np.array_equal(out["eval/frame/count"], fcount)
        assert np.array_equal(fcount.sum(1), steps.reshape(4, 8).sum(1))
        with np.errstate(invalid="ignore"):
            for i, n in zip(cols, names):
                want = fsum[:, :, i] / fcount
                got = out[f"eval/frame/{n}"]
                assert got.shape == (4, 250) and np.array_equal(np.isnan(got), fcount == 0), n
                assert np.nanmax(np.abs(got - want)) <= 1e-5 * max(1.0, np.nanmax(np.abs(want))), n
    assert len(resets) == 2


@pytest.mark.gpu
def test_single_clip_envs_sweep_one_clip(gpu_env):
    """The rodent's and the moving humanoid's packaged clip: one clip, whose statistics are the scalar aggregates."""
    ev, hum = pkg("evaluator"), pkg("envs.humanoid")
    model, clip = hum.packaged_humanoid(moving=True)
    humanoid = pkg("envs").HumanoidTracking(model=model, reference_clip=clip, device="cuda:0")
    for env, clip_len in ((gpu_env, 250), (humanoid, 256)):
        B = 16
        e = ev.Evaluator(env, _policy(env), num_eval_envs=B, episode_length=30, seed=3, per_clip=True)
        out = e.run_evaluation({})
        assert (e.nclips, e.clip_len) == (1, clip_len)
        assert np.array_equal(out["eval/clip/num_episodes"], [B]) and out["eval/frame/count"].shape == (1, clip_len)
        for n in list(env.metric_keys) + ["reward"]:
            for s in ("", "_std"):
                a, b = float(out[f"eval/clip/episode_{n}{s}"][0]), out[f"eval/episode_{n}{s}"]
                assert abs(a - b) <= 1e-6 * max(1.0, abs(b)), (type(env).__name__, n, s, a, b)
        assert abs(float(out["eval/clip/avg_episode_length"][0]) - out["eval/avg_episode_length"]) < 1e-5
        assert out["eval/frame/count"].sum() == e.episode_steps.sum().item()
        assert ("eval/frame/rapp" in out) == ("eval/clip/episode_rapp" in out) == (env is gpu_env)  # the humanoid has no appendage term


# ---- GPU: train() ----------------------------------------------------------------------------------------------------------------
SMALL = dict(num_envs=256, batch_size=64, num_minibatches=4, unroll_length=4, num_updates_per_batch=2, num_eval_envs=16)
S = 2 * 64 * 4 * 4  # env steps of one epoch of 2 training steps


def _per_clip_shapes(metrics, env, nclips, clip_len):
    names = list(env.metric_keys) + ["reward"]
    want = {f"eval/clip/episode_{n}{s}": (nclips,) for n in names for s in ("", "_std")}
    want.update({"eval/clip/avg_episode_length": (nclips,), "eval/clip/num_episodes": (nclips,), "eval/frame/count": (nclips, clip_len)})
    want.update({f"eval/frame/{n}": (nclips, clip_len) for n in names})
    got = {k: np.shape(v) for k, v in metrics.items() if k.startswith(("eval/clip/", "eval/frame/"))}
    assert got == want


@pytest.mark.gpu
def test_train_reports_per_clip_results_and_resumes_across_the_setting(multi, tmp_path):
    trn = pkg("train")
    seen = []
    trn.train(multi, S, progress_fn=lambda s, m: seen.append((s, m)), num_evals=2, per_clip_eval=True, **SMALL)
    assert [s for s, _ in seen] == [0, S]
    for _, m in seen:
        _per_clip_shapes(m, multi, 4, 250)
        assert np.array_equal(m["eval/clip/num_episodes"], [4] * 4)
        assert all(np.isfinite(v) for k, v in m.items() if not k.startswith(("eval/clip/", "eval/frame/")))
    # a checkpoint of a run without per-clip evaluation resumes with it
    kw = dict(SMALL, num_evals=3)
    trn.train(multi, 2 * S, checkpoint_dir=str(tmp_path), **kw)
    resumed = []
    trn.train(multi, 2 * S, progress_fn=lambda s, m: resumed.append((s, m)), per_clip_eval=True,
              restore_checkpoint_path=os.path.join(tmp_path, "step_%d" % S), **kw)
    assert [s for s, _ in resumed] == [2 * S]
    _per_clip_shapes(resumed[0][1], multi, 4, 250)
