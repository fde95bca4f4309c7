"""The env step's joint-space inertia code (csrc/vnl_kernels.cu: the M build, `factor`, `solve_m`, `solve_ld`) against a
float64 restatement of the same linear algebra, per env, in all four kernel builds and on every packaged tree.

vnl_kernels.cu is compiled four times: ew<W>s<S> with W = 1 or 2 warps per env (lane programs, how a level's rows are dealt
to the warps, shuffle groups) and S = the home of M and of its inverse factor K (1: the global workspace, addressed by
`slot_work`; 0: shared memory, `Ms` / `Ks`).  The library picks one home per model (`decide_stream`) and the blob one width
(`choose_env_warps`), so a packaged model runs one build.  Here every build runs: the width comes from
`build_model_blob(env_warps=W)`, the home from `VNL_STREAM`, which the library reads once per loaded instance and width
(each width has its own decide_stream), so each home gets its own copy of libvnl_b200.so.  `_engine` asserts that the requested build is the one that ran (layout, workspace,
env_warps).  Every packaged model fits in every build, which `_engine` asserts too (fewest envs per CTA: the rodent_pair
with resident inertia, 3; the Newton rodent in ew2s1, 2); the launch refuses a build that does not fit
(cudaErrorInvalidConfiguration), so a model that outgrew a build would fail here, not skip.

Checks, per env (every env of a batch of B_SMALL = 35 >= 2 * envs_per_cta + 3 envs: several CTAs, the last one ragged;
plus streamed cases with B > resident_envs, where the persistent grid reuses workspace slots):
  1. M build: the dumped qM against the fp64 oracle's at the same qpos, each entry scaled by its own size
     |dM_ij| / sqrt(M_ii M_jj) (not by max |M|, which hides the toes and fingers); exactly symmetric, exactly 0 off the
     tree pattern.  Bound: MBUILD_K times the fp32 oracle's error on the same states (both build M in fp32 from the same
     kinematics; the cancellation in the composite inertias of the small distal bodies is physics, not the kernel).
  2. smooth solve (factor with inversion + solve_m): qacc_smooth against numpy.linalg.solve of the dumped qM and
     qfrc_smooth in float64.  Componentwise backward error max_i |M x - b|_i / (|M||x| + |b|)_i <= BWD_K * u * (depth + 2),
     u = 2^-24, depth = the tree's dof depth (`maxdepth`); forward error max_i sqrt(M_ii) |x - x64|_i / sqrt(x64' M x64)
     no worse than FWD_RATIO times the fp32 oracle's (LDL' substitution, backward stable) on its own qM.
  3. integrator solve: from qvel = 0, one forward dump and one substep (pipeline_step, nsteps = 1) from the same state;
     x = qvel' / dt is the acceleration euler applied, to one rounding.  With eulerdamp it solves
     (qM + dt diag(dof_damping)) x = qfrc_smooth + qfrc_constraint (factor(damp=true): M restored from the workspace copy
     or from Ms, the damped diagonal, both solve_ld sweeps) to the same backward-error bound as check 2; without it
     x == qacc to one rounding.  The dump launch and the step launch compute the same forward pass bit for bit.
  4. cross-build: the two homes of one width differ only in where M and K are stored.  spmv_section and spmv_stream_g
     walk the same lane program in the same order (one accumulator, one flush per slot; the streamed walk of mul_m only
     runs the descendant section behind the ancestor one, with the accumulator flushed at every row end in between), and
     spill_section / restore_section copy values without arithmetic.  So qM, qacc_smooth, qacc and the post-substep state
     are asserted bit-identical between s0 and s1.  Across widths the active sets are identical and checks 1-3 hold for
     each build on its own.
The constraint force map (qfrc_constraint = J' f over the active rows) is not checked here: the kernel never materialises
efc_J or efc_force (contact rows are applied through the ancestor chain), so its dump has no rows to restate it from.

Models: rodent (CG, eulerdamp, depth 35: rows longer than a warp, the `n > 32` branch of factor), rodent with the Newton
solver, humanoid, ant (Newton), rodent_pair (two trees, nv 146), and copies of the humanoid and the ant with eulerdamp on
(solve_ld on shallow trees, where a warp packs several rows per level).  States: half the batch in contact, half in flight.

Measured on an NVIDIA B200 (power limit 1000 W), worst over the four builds and every env, bounds in brackets; every build
of every model ran the build it was asked for.  Check 3 is backward error / u / (depth + 2) with eulerdamp, |x - qacc| / u
|qacc| without:
  model            depth  M build / fp32 oracle [4]  check 2 backward [4]  check 2 fwd / fp32 oracle [4]  check 3
  rodent             35          1.92                      0.061                     1.56                0.073 [4]
  rodent (Newton)    35          1.92                      0.061                     1.56                0.073 [4]
  humanoid           14          0.67                      0.138                     0.98                0.978 [1]
  ant                 7          0.84                      0.211                     0.29                0.934 [1]
  rodent_pair        35          0.92                      0.082                     0.64                0.072 [4]
  humanoid, damped   14          0.67                      0.138                     0.98                0.115 [4]
  ant, damped         7          0.84                      0.211                     0.29                0.238 [4]
  B > resident_envs: rodent ew1s1 (B 2103, 2072 resident) 0.100 / 1.11 / 0.089, rodent_pair ew2s1 (B 903, 888 resident)
  0.104 / 0.98 / 0.086 (check 2 backward / fwd ratio / check 3).
The fp32 oracle's own check 2 backward error on the same states is 0.19 - 0.69: the explicit inverse factor with rsqrtf is
no worse than its LDL' substitution on these trees.  Deliberate defects, one at a time: dropping the last level of the K
inversion fails check 2 in every model and build (backward error ~1e5 in these units); leaving dt * dof_damping out of the
damped diagonal fails check 3 in every eulerdamp model and build; swapping the two columns of factor's n > 32 branch fails
check 2 on the rodent, the Newton rodent and the rodent_pair (the trees deep enough to have such rows), in every build;
spilling K to the next env's workspace slot fails check 2 and the bit-identity check in every streamed build.  Shifting
every use of `slot_work` by one env (modulo the grid) keeps each slot private to one env and changes no result: that is
not a defect the numbers can or should show.
"""
import copy
import ctypes
import functools
import os
import shutil

import numpy as np
import pytest

from conftest import ROOT, pkg, start_states

mb, mj, libm = pkg("model_blob"), pkg("mjcf"), pkg("_lib")

U = 2.0 ** -24
BWD_K = 4.0        # check 2 / 3: componentwise backward error <= BWD_K * u * (depth + 2)
FWD_RATIO = 4.0    # check 2: kernel forward error <= FWD_RATIO * the fp32 oracle's (worst env against worst env)
MBUILD_K = 4.0     # check 1: kernel M entry error <= MBUILD_K * the fp32 oracle's (worst env against worst env)

# every build of every model runs the same states: 2 * 16 + 3 envs, >= 2 * envs_per_cta + 3 for every build (16 is the
# most envs a CTA holds), so several CTAs run and the last one is ragged
B_SMALL = 35
MODELS = ("rodent", "rodent_newton", "humanoid", "ant", "rodent_pair", "humanoid_damped", "ant_damped")
BUILDS = ("ew1s0", "ew1s1", "ew2s0", "ew2s1")


# ---------------------------------------------------------------------------------------------------------------------
# float64 residuals (the checker; tested against the oracle's fp64 and fp32 builds in the CPU test below)
# ---------------------------------------------------------------------------------------------------------------------
def tree_pattern(blob):
    """[nv, nv] bool: the dof pairs (i, ancestor of i) and their mirror images, from the blob's sparse-inertia tables."""
    d = mb.read_dims(blob)
    madr = mb.read_field(blob, "VNL_F_DOF_MADR", np.int32)
    mcol = mb.read_field(blob, "VNL_F_M_COL", np.int32)
    pat = np.zeros((d["nv"], d["nv"]), dtype=bool)
    for i in range(d["nv"]):
        pat[i, mcol[madr[i]:madr[i + 1]]] = True
    return pat | pat.T


def mbuild_error(M, M64):
    """Per env: max_ij |M - M64|_ij / sqrt(M64_ii M64_jj)."""
    s = np.sqrt(np.diagonal(M64, axis1=-2, axis2=-1))
    return (np.abs(M - M64) / (s[:, :, None] * s[:, None, :])).max(axis=(1, 2))


def backward_error(M, x, b):
    """Per env: componentwise backward error max_i |M x - b|_i / (|M| |x| + |b|)_i, in float64."""
    r = np.einsum("bij,bj->bi", M, x) - b
    den = np.einsum("bij,bj->bi", np.abs(M), np.abs(x)) + np.abs(b)
    return (np.abs(r) / np.where(den > 0, den, 1.0)).max(axis=1)


def forward_error(M, x, b):
    """Per env: max_i sqrt(M_ii) |x - x64|_i / sqrt(x64' M x64), x64 = the float64 solve of M x = b."""
    x64 = np.linalg.solve(M, b[..., None])[..., 0]
    s = np.sqrt(np.diagonal(M, axis1=-2, axis2=-1))
    energy = np.sqrt(np.einsum("bi,bij,bj->b", x64, M, x64))
    return (s * np.abs(x - x64)).max(axis=1) / energy


def damped(M, damping, dt):
    return M + np.diag(dt * damping)[None]


# ---------------------------------------------------------------------------------------------------------------------
# models, states
# ---------------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _model(name):
    base = name.split("_")[0] if name != "rodent_pair" else name
    m = mj.load_model(os.path.join(ROOT, "vnl-brax-imitation_b200", "data", base + "_model.npz"))
    m = copy.deepcopy(m)
    if name == "rodent_newton":  # as test_gpu_parity.test_rodent_newton_solver_matches_oracle sets it
        m.solver, m.iterations, m.ls_iterations = mj.SOLVER_NEWTON, 2, 4
    if name.endswith("_damped"):
        m.eulerdamp = True
    return m


def _states(name, rodent, B, seed):
    """(qpos, qvel, act, qacc_warmstart, ctrl) in float32; even envs in contact, odd envs in flight."""
    m = _model(name)
    rng = np.random.default_rng(seed)
    fly = np.arange(B) % 2 == 1
    if name.startswith("rodent") and name != "rodent_pair":  # clip starts (tail a few cm inside the floor)
        qpos, qvel, _ = start_states(rodent, B, seed=seed)
        qpos[fly, 2] = 0.45
        qvel = qvel + (0.5 * rng.standard_normal(qvel.shape)).astype(np.float32)
    elif name == "rodent_pair":  # perturbed qpos0, as test_gpu_parity.test_rodent_pair_physics_matches_oracle
        qpos = np.tile(m.arrays["qpos0"], (B, 1)).astype(np.float32)
        qpos[:, 7:74] += (0.05 * rng.standard_normal((B, 67))).astype(np.float32)
        qpos[:, 81:] += (0.05 * rng.standard_normal((B, 67))).astype(np.float32)
        qpos[:, 2] -= 0.02; qpos[:, 76] -= 0.015
        qpos[fly, 2] += 0.5; qpos[fly, 76] += 0.5
        qvel = (0.1 * rng.standard_normal((B, m.nv))).astype(np.float32)
    else:  # the humanoid's / ant's reset pose with random joint offsets and velocities
        q0 = m.arrays["init_qpos"] if name.startswith("ant") else m.arrays["qpos0"]
        qpos = np.tile(q0, (B, 1)).astype(np.float32)
        qpos[:, 7:] += (0.1 * rng.standard_normal((B, m.nq - 7))).astype(np.float32)
        qpos[:, 2] -= 0.03
        qpos[fly, 2] += 1.0
        qvel = (0.3 * rng.standard_normal((B, m.nv))).astype(np.float32)
    act = rng.uniform(0, 1, size=(B, m.na)).astype(np.float32)
    warm = rng.standard_normal((B, m.nv)).astype(np.float32)
    ctrl = rng.uniform(-1, 1, size=(B, m.nu)).astype(np.float32)
    return qpos, qvel, act, warm, ctrl


def _oracle_dump(oracle_mod, blob, st, ctrl, precision):
    ost = {k: np.asarray(v, np.float64) for k, v in st.items()}
    return oracle_mod.forward_dump(blob, ost, np.asarray(ctrl, np.float64), precision=precision, dims=mb.read_dims(blob))


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the checker against the oracle's fp64 and fp32 builds
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["rodent", "humanoid_damped", "ant", "rodent_pair"])
def test_residuals_on_oracle_dumps(name, rodent, oracle_mod):
    """fp64 oracle: every residual of the checker <= 1e-12.  fp32 oracle (LDL' substitution on its own fp32 qM): the
    backward error of the smooth solve sits inside the error model BWD_K * u * (depth + 2) the GPU tests hold the kernel
    to, and is an fp32-sized number (not 0: the checker sees fp32 rounding)."""
    m = _model(name)
    blob = mb.build_model_blob(m, env_warps=1)
    dims = mb.read_dims(blob)
    qpos, qvel, act, warm, ctrl = _states(name, rodent, 6, seed=3)
    st = dict(qpos=qpos, qvel=qvel, act=act, qacc_warmstart=warm)
    o64 = _oracle_dump(oracle_mod, blob, st, ctrl, 64)
    o32 = _oracle_dump(oracle_mod, blob, st, ctrl, 32)
    pat = tree_pattern(blob)
    for o in (o64, o32):
        assert (o["qM"][:, ~pat] == 0).all() and (o["qM"] == np.swapaxes(o["qM"], 1, 2)).all()
    bound = BWD_K * U * (dims["maxdepth"] + 2)
    assert backward_error(o64["qM"], o64["qacc_smooth"], o64["qfrc_smooth"]).max() <= 1e-12
    assert forward_error(o64["qM"], o64["qacc_smooth"], o64["qfrc_smooth"]).max() <= 1e-12
    b32 = backward_error(o32["qM"], o32["qacc_smooth"], o32["qfrc_smooth"])
    assert (b32 <= bound).all() and b32.max() > 1e-3 * U, (b32.max() / U, dims["maxdepth"])
    assert forward_error(o32["qM"], o32["qacc_smooth"], o32["qfrc_smooth"]).max() < 1e-3
    assert mbuild_error(o32["qM"], o64["qM"]).max() < 1e-4
    # the damped system of the integrator, restated on the fp64 oracle's own arrays: M x = b is solved exactly, so the
    # residual of (M + dt D) x against b + dt D x is rounding only (this exercises `damped` and the checker's scaling)
    D = m.arrays["dof_damping"]
    x = o64["qacc_smooth"]
    assert backward_error(damped(o64["qM"], D, m.timestep), x, o64["qfrc_smooth"] + m.timestep * D * x).max() <= 1e-12


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib_copies(tmp_path_factory):
    """home ("0" resident, "1" streamed) -> a private copy of libvnl_b200.so whose VNL_STREAM is latched to that home.
    Each width has its own instantiation of decide_stream, and each reads VNL_STREAM on its first call: both are made here,
    with the variable set (a blob of either width asks the library for its dump size)."""
    out = {}
    for stream in ("0", "1"):
        path = str(tmp_path_factory.mktemp("vnl_s" + stream) / "libvnl_b200.so")
        shutil.copy(libm.LIB_PATH, path)
        with pytest.MonkeyPatch.context() as mp:
            mp.setenv("VNL_STREAM", stream)
            lib = libm.load_library(path)
            for ew in (1, 2):
                lib.vnl_dump_size(mb.build_model_blob(_model("ant"), env_warps=ew).ctypes.data)
        out[stream] = path
    return out


def _layout_sizes(lib, blob):
    names, offs, sizes = (ctypes.c_char_p * 64)(), (ctypes.c_int32 * 64)(), (ctypes.c_int32 * 64)()
    n = lib.vnl_debug_layout(blob.ctypes.data, names, offs, sizes, 64)
    return {names[i].decode(): sizes[i] for i in range(n)}


_ENGINES = {}


def _engine(name, build, lib_copies):
    """An Engine that runs kernel build `build` on model `name`; asserts which build that is."""
    key = (name, build)
    if key not in _ENGINES:
        ew, stream = int(build[2]), build[4]
        blob = mb.build_model_blob(_model(name), env_warps=ew)
        eng = libm.Engine(blob, None, device="cuda:0", lib_path=lib_copies[stream])
        lay = _layout_sizes(eng.lib, eng.model_host)
        assert eng.dims["env_warps"] == ew and eng.envs_per_cta >= 1, (name, build)
        if stream == "0":
            assert lay["Ms"] > 0 and lay["Ks"] > 0 and eng.ctx.workspace_bytes == 0, (name, build)
        else:
            assert lay["Ms"] == 0 and lay["Ks"] == 0 and eng.ctx.workspace_bytes > 0, (name, build)
        _ENGINES[key] = eng
    return _ENGINES[key]


def _t(a):
    import torch
    return torch.tensor(np.ascontiguousarray(a), device="cuda")


_RUNS = {}


def _run(name, build, lib_copies, rodent, oracle_mod, B=B_SMALL, seed=11):
    """One forward dump and one substep of build `build` from the states of `_states`, and one forward dump and one
    substep from the same states with qvel = 0.  Returns the split dumps and the post-substep states (float64)."""
    key = (name, build, B, seed)
    if key in _RUNS:
        return _RUNS[key]
    import torch
    eng = _engine(name, build, lib_copies)
    assert B >= 2 * eng.envs_per_cta + 3
    qpos, qvel, act, warm, ctrl = _states(name, rodent, B, seed)
    dims = eng.dims
    split = lambda t: {k: v.astype(np.float64) for k, v in oracle_mod.split_dump(dims, t.cpu().numpy()).items()}
    out = dict(B=B, qpos=qpos, qvel=qvel, act=act, warm=warm, ctrl=ctrl)
    for tag, v in (("", qvel), ("0", np.zeros_like(qvel))):
        st = dict(qpos=_t(qpos), qvel=_t(v), act=_t(act), qacc_warmstart=_t(warm))
        c = _t(ctrl)
        out["dump" + tag] = split(eng.forward_dump(st, c))
        nxt = eng.alloc_state(B)
        eng.pipeline_step(st, c, nxt, 1)
        torch.cuda.synchronize()
        out["next" + tag] = {k: nxt[k].cpu().numpy().astype(np.float64) for k in ("qpos", "qvel", "act", "qacc_warmstart")}
    _RUNS[key] = out
    return out


def _check_build(name, build, lib_copies, rodent, oracle_mod, B=B_SMALL):
    m = _model(name)
    eng = _engine(name, build, lib_copies)
    r = _run(name, build, lib_copies, rodent, oracle_mod, B)
    blob, dims, B = eng.model_host, eng.dims, r["B"]
    depth = dims["maxdepth"]
    g, g0 = r["dump"], r["dump0"]
    assert (g["counters"][:, 2] > 0).any() and (g["counters"][:, 2] == 0).any()  # contact and flight in the batch
    st = dict(qpos=r["qpos"], qvel=r["qvel"], act=r["act"], qacc_warmstart=r["warm"])
    o64 = _oracle_dump(oracle_mod, blob, st, r["ctrl"], 64)
    o32 = _oracle_dump(oracle_mod, blob, st, r["ctrl"], 32)
    res = {}
    # 1. M build
    pat = tree_pattern(blob)
    M = g["qM"]
    assert np.isfinite(M).all() and (M[:, ~pat] == 0).all() and (M == np.swapaxes(M, 1, 2)).all()
    em, eo = mbuild_error(M, o64["qM"]), mbuild_error(o32["qM"], o64["qM"])
    res["mbuild"] = (em.max(), eo.max())
    assert em.max() <= MBUILD_K * max(eo.max(), U), (name, build, em.max(), eo.max(), int(em.argmax()))
    # 2. smooth solve
    bound = BWD_K * U * (depth + 2)
    bk = backward_error(M, g["qacc_smooth"], g["qfrc_smooth"])
    fk = forward_error(M, g["qacc_smooth"], g["qfrc_smooth"])
    fo = forward_error(o32["qM"], o32["qacc_smooth"], o32["qfrc_smooth"])
    res["smooth"] = (bk.max() / (U * (depth + 2)), fk.max() / fo.max())
    assert (bk <= bound).all(), (name, build, bk.max() / (U * (depth + 2)), int(bk.argmax()))
    assert fk.max() <= FWD_RATIO * fo.max(), (name, build, fk.max(), fo.max(), int(fk.argmax()))
    # 3. integrator solve, from qvel = 0: x = qvel' / dt is euler's acceleration to one rounding
    dt = float(np.float32(m.timestep))
    x = r["next0"]["qvel"] / dt
    if dims["eulerdamp"]:
        D = m.arrays["dof_damping"].astype(np.float32).astype(np.float64)
        bi = backward_error(damped(g0["qM"], D, dt), x, g0["qfrc_smooth"] + g0["qfrc_constraint"])
        res["integrator"] = bi.max() / (U * (depth + 2))
        assert (bi <= bound).all(), (name, build, bi.max() / (U * (depth + 2)), int(bi.argmax()))
    else:
        qacc = g0["qacc"]
        err = np.abs(x - qacc) / np.maximum(np.abs(qacc), 1e-30)
        res["integrator"] = err.max() / U
        assert (err <= U * (1 + 1e-6)).all(), (name, build, err.max() / U)
    return res


@pytest.mark.gpu
@pytest.mark.parametrize("build", BUILDS)
@pytest.mark.parametrize("name", MODELS)
def test_inertia_solves_match_float64(name, build, lib_copies, rodent, oracle_mod):
    res = _check_build(name, build, lib_copies, rodent, oracle_mod)
    print("inertia %-16s %s depth %2d  M build %.2e (oracle32 %.2e)  smooth bwd/u/(d+2) %.3f fwd ratio %.3f  integrator %.3f"
          % (name, build, _engine(name, build, lib_copies).dims["maxdepth"], res["mbuild"][0], res["mbuild"][1],
             res["smooth"][0], res["smooth"][1], res["integrator"]))


@pytest.mark.gpu
@pytest.mark.parametrize("name,build", [("rodent", "ew1s1"), ("rodent_pair", "ew2s1")])
def test_streamed_slots_reused_past_the_first_wave(name, build, lib_copies, rodent, oracle_mod):
    """B > resident_envs on the streamed home: every workspace slot serves a second env, and every env is checked."""
    eng = _engine(name, build, lib_copies)
    B = eng.resident_envs + 2 * eng.envs_per_cta + 3
    res = _check_build(name, build, lib_copies, rodent, oracle_mod, B=B)
    print("inertia %s %s B %d (resident %d): %s" % (name, build, B, eng.resident_envs, res))


@pytest.mark.gpu
@pytest.mark.parametrize("ew", ["ew1", "ew2"])
@pytest.mark.parametrize("name", MODELS)
def test_inertia_home_changes_no_bit(name, ew, lib_copies, rodent, oracle_mod):
    """s0 against s1 of one width: same program order for every mat-vec and copy-only spills / restores, so the stage
    arrays and the post-substep state are bit-identical."""
    a, b = _run(name, ew + "s0", lib_copies, rodent, oracle_mod), _run(name, ew + "s1", lib_copies, rodent, oracle_mod)
    for tag in ("", "0"):
        for k in ("qM", "qacc_smooth", "qacc", "qfrc_constraint", "counters"):
            assert np.array_equal(a["dump" + tag][k], b["dump" + tag][k]), (tag, k)
        for k, v in a["next" + tag].items():
            assert np.array_equal(v, b["next" + tag][k]), (tag, k)


@pytest.mark.gpu
@pytest.mark.parametrize("name", MODELS)
def test_widths_share_active_sets(name, lib_copies, rodent, oracle_mod):
    """ew1 against ew2 (same home): identical constraint activity; the floats differ by the grouping of partial sums."""
    a, b = _run(name, "ew1s1", lib_copies, rodent, oracle_mod), _run(name, "ew2s1", lib_copies, rodent, oracle_mod)
    assert np.array_equal(a["dump"]["counters"][:, 2:4], b["dump"]["counters"][:, 2:4])
