"""The C-ABI library loads and exports every symbol include/vnl_b200.h declares; host-side entry
points (blob validation, sizing) behave.  No compute calls: this file runs without a GPU."""
import ctypes
import os
import re

import numpy as np
import pytest

from conftest import ROOT, pkg

libm = pkg("_lib")


def _declared_functions():
    txt = open(os.path.join(ROOT, "include", "vnl_b200.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(vnl_[a-z_0-9]+)\s*\(", txt)))


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(libm.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return libm.load_library()


def test_header_and_binding_agree():
    assert set(_declared_functions()) == set(libm.EXPORTS)


def test_exports(lib):
    for name in _declared_functions():
        assert getattr(lib, name) is not None, name
    assert b"sm_100a" in lib.vnl_version()


def test_library_embeds_sm100a_code():
    import subprocess
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-lelf", libm.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out, out


def test_blob_validation(lib, rodent):
    m, t = rodent["model_blob"], rodent["task_blob"]
    assert lib.vnl_check_model(m.ctypes.data, m.nbytes) == 0
    assert lib.vnl_check_task(t.ctypes.data, t.nbytes) == 0
    assert lib.vnl_check_model(t.ctypes.data, t.nbytes) != 0  # wrong magic
    assert lib.vnl_check_model(m.ctypes.data, m.nbytes - 4) != 0  # truncated
    bad = m.copy(); bad[1] += 1
    assert lib.vnl_check_model(bad.ctypes.data, bad.nbytes) != 0  # wrong version
    bad = m.copy(); bad[pkg("model_blob").C["VNL_TABLE_OFF"]] = 2 ** 31
    assert lib.vnl_check_model(bad.ctypes.data, bad.nbytes) != 0  # field out of range
    assert lib.vnl_check_model(None, 0) != 0


def test_sizes(lib, rodent, oracle_mod):
    m = rodent["model_blob"]
    smem = lib.vnl_step_smem_bytes(m.ctypes.data)
    assert 0 < smem <= 227 * 1024
    assert lib.vnl_dump_size(m.ctypes.data) == oracle_mod.lib().vnl_oracle_dump_size(m.ctypes.data_as(ctypes.c_void_p))


def _ctx(lib, m, t=None):
    ctx = libm.VnlContext()
    rc = lib.vnl_context_init(ctypes.byref(ctx), m.ctypes.data, m.nbytes, None if t is None else t.ctypes.data, 0 if t is None else t.nbytes)
    return rc, ctx


def test_bad_context_is_an_argument_error(lib, rodent):
    st = libm.VnlState(); out = libm.VnlOutputs()
    dummy = np.zeros(8, dtype=np.float32)
    empty = libm.VnlContext()  # never initialised: no model header
    rc = lib.vnl_step(ctypes.byref(empty), dummy.ctypes.data, dummy.ctypes.data, 4, ctypes.byref(st), dummy.ctypes.data, ctypes.byref(st),
                      ctypes.byref(out), None)
    assert rc == -11  # never launches
    assert lib.vnl_step(None, None, None, 0, None, None, None, None, None) < 0
    bad = rodent["model_blob"].copy(); bad[0] ^= 1
    assert _ctx(lib, bad)[0] == -2
    rc, ctx = _ctx(lib, rodent["model_blob"], rodent["task_blob"])
    assert rc == 0 and ctx.workspace is None and ctx.model_hdr[0] == rodent["model_blob"][0] and ctx.task_hdr[0] == rodent["task_blob"][0]
    badt = rodent["task_blob"].copy(); badt[1] += 1
    assert _ctx(lib, rodent["model_blob"], badt)[0] == -103


def test_workspace_is_required_and_sized(lib, rodent):
    """Stateless boundary: the workspace is an ARGUMENT (VnlContext).  The step entry points refuse to launch (-20 / -21,
    before any device access) without one that is big enough for the geometry of THIS call; sizing follows the resident-env
    count and both lane-program lengths.  Nothing is registered: the same host context serves any device address."""
    mb = pkg("model_blob")
    m, t = rodent["model_blob"], rodent["task_blob"]
    need = lib.vnl_workspace_bytes(m.ctypes.data)
    d = mb.model_dims(rodent["model"])
    per_env = (2 * (d["TA"] + d["TD"]) * 32 + 31) // 32 * 32 * 4  # M and K, one copy per lane program each
    assert need == lib.vnl_resident_envs(m.ctypes.data) * per_env and per_env == 20480
    assert lib.vnl_resident_envs(m.ctypes.data) % lib.vnl_envs_per_cta(m.ctypes.data) == 0 and lib.vnl_envs_per_cta(m.ctypes.data) == 14
    fake_model, fake_task, fake_work = 0x7000000000, 0x7100000000, 0x7200000000  # never dereferenced on these paths
    rc, ctx = _ctx(lib, m, t)
    assert rc == 0
    st = libm.VnlState(); out = libm.VnlOutputs()
    dummy = np.zeros(8, dtype=np.float32)
    call = lambda B=4096, model=fake_model: lib.vnl_step(ctypes.byref(ctx), model, fake_task, B, ctypes.byref(st), dummy.ctypes.data,
                                                         ctypes.byref(st), ctypes.byref(out), None)
    assert call() == -20
    ctx.workspace, ctx.workspace_bytes = fake_work, need - 4
    assert call() == -21 and call(model=fake_model + 4096) == -21   # no dependence on the blob's device address
    ctx.workspace_bytes = 4 * per_env
    assert call(B=4096) == -21  # checked against the geometry of the actual batch: 4 env slots are not enough for 4096 envs
    ctx.workspace = None
    assert call() == -20
    # the XLA trampolines carry the same bytes in `opaque`: a short or wrong-version opaque never launches
    op = libm.VnlXlaOpaque()
    ctx.workspace_bytes = need
    assert lib.vnl_xla_make_opaque(ctypes.byref(ctx), 4096, ctypes.byref(op)) == 0 and op.B == 4096 and op.version == 2
    bufs = (ctypes.c_void_p * libm.VNL_XLA_STEP_NBUF)()
    raw = bytes(op)
    assert lib.vnl_xla_step_rc(None, bufs, raw[:100], 100) == -30
    op.version = 1
    assert lib.vnl_xla_step_rc(None, bufs, bytes(op), len(bytes(op))) == -31
    assert lib.vnl_xla_reset_rc(None, bufs, raw, len(raw)) == -10  # NULL model buffer: argument error, still no launch


def test_no_mutable_globals_in_the_abi():
    """SURVEY 8(b): no registry / lock / global state behind the C ABI (round-1 kept pointer-keyed maps)."""
    src = open(os.path.join(ROOT, "vnl-brax-imitation_b200", "csrc", "vnl_capi.cu")).read()
    for needle in ("std::mutex", "unordered_map", "g_headers", "g_work", "vnl_register_blob", "vnl_set_workspace"):
        assert needle not in src, needle
    hdr = open(os.path.join(ROOT, "include", "vnl_b200.h")).read()
    assert "vnl_register_blob" not in hdr and "vnl_set_workspace" not in hdr


def test_env_warps_follow_the_shared_memory_residency(monkeypatch):
    """model_blob.choose_env_warps: one warp per env unless shared memory leaves <= 8 envs on an SM (then the second warp is free):
    rodent / humanoid / ant keep one, rodent_pair (nv 146, 6 envs per SM) gets two; VNL_ENV_WARPS overrides."""
    mb, mj = pkg("model_blob"), pkg("mjcf")
    monkeypatch.delenv("VNL_ENV_WARPS", raising=False)
    want = {"rodent": 1, "humanoid": 1, "ant": 1, "rodent_pair": 2}
    for name, ew in want.items():
        model = mj.load_model(os.path.join(ROOT, "vnl-brax-imitation_b200", "data", name + "_model.npz"))
        assert mb.choose_env_warps(model) == ew, name
        assert mb.read_dims(mb.build_model_blob(model))["env_warps"] == ew, name
    monkeypatch.setenv("VNL_ENV_WARPS", "1")
    assert mb.choose_env_warps(model) == 1  # (model = rodent_pair)


def test_two_warp_blob_has_wider_lane_programs(rodent):
    mb = pkg("model_blob")
    b1, b2 = mb.build_model_blob(rodent["model"], 1), mb.build_model_blob(rodent["model"], 2)
    d1, d2 = mb.read_dims(b1), mb.read_dims(b2)
    assert (d1["env_warps"], d2["env_warps"]) == (1, 2)
    t1, t2 = mb.derived_tables(rodent["model"], 1), mb.derived_tables(rodent["model"], 2)
    assert t2["TA"] < t1["TA"] and t2["TD"] < t1["TD"] and t1["TA"] % 8 == 0 and t2["TD"] % 8 == 0
    # every off-diagonal inertia entry appears exactly once in each ancestor program, whatever the lane count
    C = mb.C
    for tb, nl in ((t1, 32), (t2, 64)):
        kt = tb["ktab"]
        off = kt[C["VNL_KT_PROG_A"]] // 4
        prog = kt[off:off + tb["TA"] * nl]
        ent = (prog & 0x3FFC) >> 2
        nM = len(tb["m_col"])
        real = ent[ent != nM]
        assert len(real) == nM - rodent["model"].nv and len(set(real.tolist())) == len(real)


def test_engine_refuses_to_run_without_gpu(rodent, monkeypatch):
    import torch
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)  # also on a GPU machine
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        libm.Engine(rodent["model_blob"], rodent["task_blob"])


def test_product_package_never_imports_the_oracle():
    pk = os.path.join(ROOT, "vnl-brax-imitation_b200")
    for dp, _, fs in os.walk(pk):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dp, f)).read()
                for needle in ("import oracle", "from oracle", "libvnl_oracle", "vnl_oracle_"):
                    assert needle not in src, (f, needle)
