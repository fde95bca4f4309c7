"""Intention-network policy forward (SURVEY section 8 row f1, include/vnl_policy.h).

CPU (`-m "not gpu"`): the library exports every symbol the header declares, the size checks, the packed operand image
of `vnl_policy_pack` (bf16 round-to-nearest-even at the documented byte offsets), and the torch restatement against a
hand-written numpy forward of intention_policy_network.py.
GPU (`-m gpu`): `vnl_policy_forward` (tcgen05) against the torch restatement with bf16-rounded dense operands and fp32
accumulation (tolerances below), per-layer accumulators, ragged batch sizes, identity normaliser, and bounds against
the plain fp32 forward.
"""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT, pkg

pol = pkg("policy")
libm = pkg("_lib")

RODENT = dict(traj_size=795, obs_size=232, action_size=30)  # SURVEY App. A; latent 64, [256,128] / [128,256]


def _declared():
    txt = open(os.path.join(ROOT, "include", "vnl_policy.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(vnl_(?:xla_)?policy_[a-z_0-9]+)\s*\(", txt)))


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(libm.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return pol._bind(libm.load_library())


def test_header_and_binding_agree(lib):
    assert set(_declared()) == set(pol.POLICY_EXPORTS)
    for n in _declared():
        assert getattr(lib, n) is not None


def test_size_checks(lib):
    ok = pol.VnlPolicyDims(795, 232, 64, 256, 128, 128, 256, 30)
    assert lib.vnl_policy_check(ctypes.byref(ok)) == 0
    assert lib.vnl_policy_blob_bytes(ctypes.byref(ok)) > 0
    hum = pol.VnlPolicyDims(630, 55, 64, 256, 128, 128, 256, 21)  # humanoid sizes (SURVEY App. A)
    assert lib.vnl_policy_check(ctypes.byref(hum)) == 0
    for bad in (pol.VnlPolicyDims(795, 232, 60, 256, 128, 128, 256, 30),   # latent not a multiple of 16
                pol.VnlPolicyDims(795, 232, 64, 1024, 1024, 128, 256, 30),  # the factory defaults (1024,1024): too wide
                pol.VnlPolicyDims(795, 232, 64, 256, 100, 128, 256, 30),
                pol.VnlPolicyDims(795, 232, 64, 256, 128, 128, 256, 0)):
        assert lib.vnl_policy_check(ctypes.byref(bad)) < 0
        assert lib.vnl_policy_blob_bytes(ctypes.byref(bad)) == 0


def _bf16_bits(x):
    return (torch.from_numpy(np.ascontiguousarray(x)).to(torch.bfloat16).view(torch.int16).numpy().astype(np.uint16))


def test_pack_image(lib):
    """Element (k, n) of layer i sits at offW[i] + (k // 8) * (16 N_i + 16) + n * 16 + (k % 8) * 2, rounded RNE to bf16; the
    two encoder heads share one operand (mean rows first); padding is zero; the fp32 vectors follow."""
    rng = np.random.default_rng(3)
    shapes = pol.param_shapes(**RODENT)
    params = pol.init_params(rng, shapes, perturb=0.2)
    d = pol.VnlPolicyDims(795, 232, 64, 256, 128, 128, 256, 30)
    n = lib.vnl_policy_blob_bytes(ctypes.byref(d))
    blob = np.zeros(n, dtype=np.uint8)
    arrs = [np.ascontiguousarray(params[k], dtype=np.float32) for k in pol.PARAM_ORDER]
    ptrs = (ctypes.c_void_p * len(arrs))(*[a.ctypes.data for a in arrs])
    assert lib.vnl_policy_pack(ctypes.byref(d), ptrs, blob.ctypes.data, n) == 0
    assert lib.vnl_policy_pack(ctypes.byref(d), ptrs, blob.ctypes.data, n - 1) < 0
    K = [832, 256, 128, 304, 128, 256]
    N = [256, 128, 128, 128, 256, 64]
    mats = [params["encoder/hidden_0/kernel"], params["encoder/hidden_1/kernel"],
            np.concatenate([params["encoder/fc2_mean/kernel"], params["encoder/fc2_logvar/kernel"]], 1),
            params["decoder/hidden_0/kernel"], params["decoder/hidden_1/kernel"], params["decoder/hidden_2/kernel"]]
    off = 64
    for i in range(6):
        lbo = 16 * N[i] + 16
        img = blob[off:off + (K[i] // 8) * lbo].reshape(K[i] // 8, lbo)
        assert not img[:, 16 * N[i]:].any()
        w = img[:, :16 * N[i]].copy().view(np.uint16).reshape(K[i] // 8, N[i], 8)  # [kg, n, k % 8]
        w = w.transpose(0, 2, 1).reshape(K[i], N[i])
        kt, nt = mats[i].shape
        assert (w[:kt, :nt] == _bf16_bits(mats[i])).all(), i
        assert not w[kt:].any() and not w[:, nt:].any()
        off += (K[i] // 8) * lbo
    vec = blob[off:].view(np.float32)
    assert vec.size == 3 * 256 + 3 * 128 + 128 + 3 * 128 + 3 * 256 + 64
    np.testing.assert_array_equal(vec[:256], params["encoder/hidden_0/bias"])
    np.testing.assert_array_equal(vec[256:512], params["encoder/LayerNorm_0/scale"])
    np.testing.assert_array_equal(vec[3 * 256 + 3 * 128:3 * 256 + 3 * 128 + 64], params["encoder/fc2_mean/bias"])
    np.testing.assert_array_equal(vec[-64:-4], params["decoder/hidden_2/bias"])


def _numpy_forward(p, traj, obs, eps_z, eps_a):
    """Independent float64 numpy forward of intention_policy_network.py:20-105 + NormalTanhDistribution."""
    def ln(x, s, b):
        m = x.mean(-1, keepdims=True)
        v = np.maximum((x * x).mean(-1, keepdims=True) - m * m, 0)
        return (x - m) / np.sqrt(v + 1e-6) * s + b
    g = lambda k: p[k].astype(np.float64)
    h = traj
    for i in range(2):
        h = ln(np.maximum(h @ g(f"encoder/hidden_{i}/kernel") + g(f"encoder/hidden_{i}/bias"), 0),
               g(f"encoder/LayerNorm_{i}/scale"), g(f"encoder/LayerNorm_{i}/bias"))
    mean = h @ g("encoder/fc2_mean/kernel") + g("encoder/fc2_mean/bias")
    logvar = h @ g("encoder/fc2_logvar/kernel") + g("encoder/fc2_logvar/bias")
    h = np.concatenate([mean + eps_z * np.exp(0.5 * logvar), obs], -1)
    for i in range(2):
        h = ln(np.maximum(h @ g(f"decoder/hidden_{i}/kernel") + g(f"decoder/hidden_{i}/bias"), 0),
               g(f"decoder/LayerNorm_{i}/scale"), g(f"decoder/LayerNorm_{i}/bias"))
    logits = h @ g("decoder/hidden_2/kernel") + g("decoder/hidden_2/bias")
    nu = logits.shape[-1] // 2
    scale = np.logaddexp(0, logits[:, nu:]) + 1e-3
    raw = logits[:, :nu] + scale * eps_a
    lp = (-0.5 * eps_a ** 2 - np.log(scale) - 0.5 * np.log(2 * np.pi) - 2 * (np.log(2) - raw - np.logaddexp(0, -2 * raw))).sum(-1)
    return np.tanh(raw), logits, lp


def test_torch_restatement_matches_numpy():
    rng = np.random.default_rng(5)
    params = pol.init_params(rng, pol.param_shapes(**RODENT), perturb=0.1)
    B = 7
    traj, obs, ez, ea = (rng.standard_normal((B, w)) for w in (795, 232, 64, 30))
    t = lambda x: torch.from_numpy(x.astype(np.float32))
    r = pol.reference_forward(params, t(traj), t(obs), t(ez), t(ea))
    act, logits, lp = _numpy_forward(params, *(x.astype(np.float32).astype(np.float64) for x in (traj, obs, ez, ea)))
    np.testing.assert_allclose(r["logits"].numpy(), logits, atol=2e-5)
    np.testing.assert_allclose(r["action"].numpy(), act, atol=2e-5)
    np.testing.assert_allclose(r["log_prob"].numpy(), lp, atol=5e-4)


def test_policy_refuses_to_run_without_gpu(monkeypatch):
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)  # also on a GPU machine
    params = pol.init_params(np.random.default_rng(0), pol.param_shapes(**RODENT))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pol.IntentionPolicy(params)


# ---------------------------------------------------------------------------------------------------------------------
def _case(B, seed, normalise=True, sizes=RODENT):
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(seed)
    params = pol.init_params(rng, pol.param_shapes(**sizes), perturb=0.1)
    g = torch.Generator().manual_seed(seed)
    mk = lambda *s: torch.randn(*s, generator=g).to(dev)
    x = dict(traj=mk(B, sizes["traj_size"]), obs=mk(B, sizes["obs_size"]) * 2 + 0.5, eps_z=mk(B, 64), eps_a=mk(B, sizes["action_size"]),
             rand=(torch.rand(B, sizes["action_size"], generator=g) * 2 - 1).to(dev))
    mean = std = None
    if normalise:
        mean, std = mk(sizes["obs_size"]) * 0.3, torch.rand(sizes["obs_size"], generator=g).to(dev) + 0.5
    return params, x, mean, std


# The kernel rounds the operands of each dense layer to bf16 and accumulates in fp32 (tensor cores); against a torch
# forward that rounds the same operands the differences are accumulation order and the occasional bf16 rounding flip of
# an activation (one flip = 2^-9 relative on one of <= 304 inputs).  Against plain fp32 the gap is the bf16 operand
# rounding itself.
TOL_BF16REF = dict(logits=2e-2, action=2e-2, raw_action=3e-2, log_prob=0.25, rand_log_prob=0.6, z_mean=1e-2, z_logvar=1e-2)
TOL_FP32 = dict(logits=0.12, action=0.12)


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 127, 128, 300, 1024])
def test_policy_forward_matches_restatement(B):
    params, x, mean, std = _case(B, seed=B)
    p = pol.IntentionPolicy(params, "cuda:0", mean, std)
    act, out = p(x["traj"], x["obs"], x["eps_z"], x["eps_a"], x["rand"], heads=True)
    torch.cuda.synchronize()
    ref = pol.reference_forward(params, x["traj"], x["obs"], x["eps_z"], x["eps_a"], x["rand"], mean, std, operand_dtype=torch.bfloat16)
    ref32 = pol.reference_forward(params, x["traj"], x["obs"], x["eps_z"], x["eps_a"], x["rand"], mean, std)
    for k, tol in TOL_BF16REF.items():
        assert torch.isfinite(out[k]).all(), k
        err = float((out[k] - ref[k]).abs().max())
        if k == "rand_log_prob":  # -z^2 / 2 with z = (u - loc) / scale up to ~50: the bound is relative
            tol += 2e-3 * float(ref[k].abs().max())
        assert err < tol, (k, err)
    for k, tol in TOL_FP32.items():
        err = float((out[k] - ref32[k]).abs().max())
        assert err < tol, (k, err)
    assert act.data_ptr() == out["action"].data_ptr() and p.launches == 1
    assert float(act.abs().max()) <= 1.0


@pytest.mark.gpu
def test_policy_layer_accumulators():
    """Raw tcgen05 accumulators of every layer (first tile) against the restatement's pre-activations minus bias: the first
    layer sees identical operands, so only the accumulation order differs."""
    params, x, mean, std = _case(200, seed=11)
    p = pol.IntentionPolicy(params, "cuda:0", mean, std)
    ref = pol.reference_forward(params, x["traj"], x["obs"], x["eps_z"], x["eps_a"], None, mean, std, operand_dtype=torch.bfloat16)
    bias = [params["encoder/hidden_0/bias"], params["encoder/hidden_1/bias"],
            np.concatenate([params["encoder/fc2_mean/bias"], params["encoder/fc2_logvar/bias"]]),
            params["decoder/hidden_0/bias"], params["decoder/hidden_1/bias"], params["decoder/hidden_2/bias"]]
    for layer in range(6):
        d = p.debug_layer(x["traj"], x["obs"], x["eps_z"], layer)
        torch.cuda.synchronize()
        r = ref["pre"][layer][:128] - torch.as_tensor(bias[layer], device=d.device)
        w = r.shape[1]
        err = float((d[:128, :w] - r).abs().max())
        assert err < (2e-4 if layer == 0 else 2e-2), (layer, err)
        assert not d[128:].any() and not d[:, w:].any()


@pytest.mark.gpu
def test_policy_identity_normaliser_and_humanoid_sizes():
    sizes = dict(traj_size=630, obs_size=55, action_size=21)  # humanoid: obs not a multiple of 8, K padding on both inputs
    params, x, _, _ = _case(130, seed=2, normalise=False, sizes=sizes)
    p = pol.IntentionPolicy(params, "cuda:0")
    _, out = p(x["traj"], x["obs"], x["eps_z"], x["eps_a"])
    torch.cuda.synchronize()
    ref = pol.reference_forward(params, x["traj"], x["obs"], x["eps_z"], x["eps_a"], None, operand_dtype=torch.bfloat16)
    for k in ("logits", "action", "log_prob"):
        assert float((out[k] - ref[k]).abs().max()) < TOL_BF16REF[k], k


@pytest.mark.gpu
def test_policy_rows_are_independent_and_deterministic():
    """A row's outputs do not depend on its neighbours or its tile position (per-env contraction, no cross-row reduction)."""
    params, x, mean, std = _case(384, seed=4)
    p = pol.IntentionPolicy(params, "cuda:0", mean, std)
    _, a = p(x["traj"], x["obs"], x["eps_z"], x["eps_a"])
    a = {k: v.clone() for k, v in a.items()}
    perm = torch.randperm(384, device="cuda:0")
    _, b = p(*(x[k][perm].contiguous() for k in ("traj", "obs", "eps_z", "eps_a")))
    torch.cuda.synchronize()
    for k in ("logits", "action", "log_prob"):
        assert torch.equal(a[k][perm], b[k]), k


@pytest.mark.gpu
def test_xla_custom_call_trampoline_equals_direct_call():
    """`vnl_xla_policy_forward(stream, buffers, opaque, len)` (legacy XLA custom-call ABI) == vnl_policy_forward."""
    import struct
    params, x, mean, std = _case(257, seed=9)
    p = pol.IntentionPolicy(params, "cuda:0", mean, std)
    _, a = p(x["traj"], x["obs"], x["eps_z"], x["eps_a"], x["rand"])
    a = {k: v.clone() for k, v in a.items()}
    b = p.alloc_outputs(257)
    bufs = [p.blob_dev, x["traj"], x["obs"], mean, std, x["eps_z"], x["eps_a"], x["rand"],
            b["action"], b["raw_action"], b["logits"], b["log_prob"], b["rand_log_prob"]]
    arr = (ctypes.c_void_p * len(bufs))(*[t.data_ptr() for t in bufs])
    d = p.dims
    opaque = struct.pack("<9i", d.traj, d.obs, d.latent, d.e1, d.e2, d.d1, d.d2, d.nu, 257)
    p.lib.vnl_xla_policy_forward(torch.cuda.current_stream().cuda_stream, arr, opaque, len(opaque), None)
    torch.cuda.synchronize()
    for k in ("action", "raw_action", "logits", "log_prob", "rand_log_prob"):
        assert torch.equal(a[k], b[k]), k


@pytest.mark.gpu
def test_empty_batch_and_argument_errors(lib):
    params, x, mean, std = _case(4, seed=1)
    p = pol.IntentionPolicy(params, "cuda:0", mean, std)
    z = lambda w: torch.zeros(0, w, device="cuda")
    act, out = p(z(795), z(232), z(64), z(30))  # B = 0: nothing is launched, nothing fails
    torch.cuda.synchronize()
    assert act.shape == (0, 30)
    with pytest.raises(ValueError):
        p(x["traj"][:, :100].contiguous(), x["obs"], x["eps_z"], x["eps_a"])
    with pytest.raises(ValueError):
        p(x["traj"].double(), x["obs"], x["eps_z"], x["eps_a"])
    d = p.dims
    assert lib.vnl_policy_forward(None, ctypes.byref(d), 4, *([None] * 15)) < 0  # null blob: argument error, no launch
    ptr = lambda t: t.data_ptr()
    assert lib.vnl_policy_forward(ptr(p.blob_dev) + 4, ctypes.byref(d), 4, ptr(x["traj"]), ptr(x["obs"]), None, None, ptr(x["eps_z"]),
                                  *([None] * 10)) == -10  # misaligned blob: refused, not mis-streamed


@pytest.mark.gpu
def test_deterministic_mode_is_tanh_of_loc():
    """make_policy(params, deterministic=True) (ppo_networks.py:63-64): action = distribution.mode(logits) = tanh(loc)."""
    params, x, mean, std = _case(200, seed=13)
    p = pol.IntentionPolicy(params, "cuda:0", mean, std)
    act, out = p(x["traj"], x["obs"], x["eps_z"], None)
    torch.cuda.synchronize()
    loc = out["logits"][:, :30]
    assert float((act - torch.tanh(loc)).abs().max()) < 2e-6 and torch.equal(out["raw_action"], loc)


# ---- the fp32-accurate rollout policy (VERDICT r1 item 5 / ADVICE r1 medium) -------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("precision,tol_logits,tol_lp", [("3xtf32", 3e-5, 1e-3), ("tf32", 1e-2, 1.5e-1)])
@pytest.mark.parametrize("B", [1, 130, 4096])
def test_precise_policy_matches_fp32_network(B, precision, tol_logits, tol_lp):
    """policy.PrecisePolicy (tcgen05 TF32 GEMMs + row kernels) against the float64 evaluation of the reference network with NO operand
    rounding.  3xTF32: logits 3e-5, log_prob 1e-3 absolute (the bound the PPO importance ratio needs: rho within 0.1 % of 1 at update 0,
    against a clip range of 0.2); the bf16 one-launch kernel above is at 2.4e-2 / 0.18.  `rand_log_prob` uses the reference's ONE
    uniform draw of shape (action_size,) broadcast over the batch (ppo_networks.py:68-73)."""
    params, x, mean, std = _case(B, seed=20 + B % 7)
    traj, obs, eps_z, eps_a, rand = x["traj"], x["obs"], x["eps_z"], x["eps_a"], x["rand"]
    p = pol.PrecisePolicy(params, "cuda:0", mean, std, precision=precision)
    rand1 = rand[0].contiguous()  # shape (nu,)
    act, out = p(traj, obs, eps_z, eps_a, rand1, heads=True)
    torch.cuda.synchronize()
    ref = pol.reference_forward(params, traj.double(), obs.double(), eps_z.double(), eps_a.double(), rand1.double()[None].expand(B, -1), mean.double(), std.double())
    assert float((out["logits"].double() - ref["logits"]).abs().max()) < tol_logits * max(1.0, float(ref["logits"].abs().max()))
    assert float((out["log_prob"].double() - ref["log_prob"]).abs().max()) < tol_lp
    # rand_log_prob = -z^2 / 2 with z = (u - loc) / scale up to ~50 (values of -100 .. -1000): the bound is relative
    assert float((out["rand_log_prob"].double() - ref["rand_log_prob"]).abs().max()) < tol_lp + (5e-5 if precision == "3xtf32" else 2e-2) * float(ref["rand_log_prob"].abs().max())
    assert float((act.double() - ref["action"]).abs().max()) < 10 * tol_logits and float(act.abs().max()) <= 1.0
    assert float((out["z_mean"].double() - ref["z_mean"]).abs().max()) < tol_logits * 10
    # deterministic mode (evaluation): action = tanh(loc)
    act_d, out_d = p(traj, obs, eps_z, None)
    torch.cuda.synchronize()
    nu = act.shape[1]
    assert torch.allclose(act_d, torch.tanh(out_d["logits"][:, :nu]), atol=1e-6)


@pytest.mark.gpu
def test_precise_policy_reloads_in_place_and_is_graph_capturable():
    params, x, mean, std = _case(256, seed=31)
    traj, obs, eps_z, eps_a = x["traj"], x["obs"], x["eps_z"], x["eps_a"]
    p = pol.PrecisePolicy(params, "cuda:0", mean, std)
    out = p.alloc_outputs(256)
    p(traj, obs, eps_z, eps_a, out=out)  # warm-up allocates the per-batch buffers
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        p(traj, obs, eps_z, eps_a, out=out)
    g.replay()
    torch.cuda.synchronize()
    first = out["log_prob"].clone()
    eager = p(traj, obs, eps_z, eps_a)[1]["log_prob"]
    assert torch.allclose(first, eager, atol=1e-4)  # split-K red.adds land in any order: equal to rounding (log-probs of magnitude 10-100)
    new = pol.init_params(np.random.default_rng(99), pol.param_shapes(795, 232, 30), perturb=0.1)
    ptr = p.blob_dev.data_ptr()
    p.load_params(new)
    assert p.blob_dev.data_ptr() == ptr
    g.replay()  # the captured launches read the refreshed weights and splits
    torch.cuda.synchronize()
    want = pol.reference_forward(new, traj.double(), obs.double(), eps_z.double(), eps_a.double(), None, mean.double(), std.double())["log_prob"]
    assert float((out["log_prob"].double() - want).abs().max()) < 1e-3 and not torch.allclose(out["log_prob"], first)
