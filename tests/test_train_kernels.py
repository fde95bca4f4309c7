"""The non-GEMM kernels of the PPO update (include/vnl_train.h), each called through the C ABI on CUDA tensors and compared with a
few lines of float64 torch, at the sizes training runs (5120 rows per minibatch update) and on both sides of every kernel's regime
boundary:
  * 1184 rows: vnl_relu_ln_bwd and vnl_ppo_loss_bwd cap their grid at 148 blocks of 8 warps; above it a warp sums several rows
    (dscale / dbias / dbias_pre, the loss metrics) in registers;
  * 303,104 elements: grid_for's cap of 1184 blocks of 256 threads; above it the elementwise kernels go round their grid-stride
    loop (vnl_heads_bwd then also adds several KL terms per thread);
  * 9472 rows: the same cap for the one-warp-per-row kernels (relu_ln_fwd, rowdot, ppo_rows, policy_sample);
  * the advantage mean / std of vnl_ppo_loss_bwd is one block of 1024 threads: above 1024 rows each thread sums several values.

Tolerances, u = 2^-24 (half an fp32 ulp):
  * elementwise results: a few u of the magnitudes that enter them, more where expf / log1pf / logf / tanhf (each <= 2 ulp) appear;
    a result below the normal range (2^-126) carries no relative precision, so that is the floor;
  * reductions: k u sum|terms| with k the number of terms a thread or an atomic chain adds one after the other, bounded by the
    number of terms summed: n for a row sum, rows for a column sum or an atomic sum over rows (plus a few for the roundings
    of the terms).  An output that accumulates counts its initial value among the terms: every atomic add rounds the running
    total.  That leaves room for any order of summation; a dropped row, an overwritten partial or a wrong column
    break it by orders of magnitude at the row counts where they can happen.
Inputs carry NaN in their padding columns (it must not reach a result); outputs that have padding carry a sentinel there (it must
stay).  vnl_gather_rows is the exception: its contract zero-fills the padding.

The refusal test at the end needs the built library but no device: every refusal returns before any CUDA call."""
import ctypes
import math
import os

import numpy as np
import pytest

from conftest import pkg

tk = pkg("train_kernels")
libm = pkg("_lib")

U = 2.0 ** -24
TINY = 2.0 ** -126
SENTINEL = 12345.0
SQUARE_ROWS = (1, 1184, 1185, 5120)


@pytest.fixture(scope="module")
def K():
    return tk.lib()


def _dev():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda")


def _gen(seed):
    import torch
    return torch.Generator(device="cuda").manual_seed(seed)


def _st():
    import torch
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return None if t is None else t.data_ptr()


def _rows(rows, n, ld, g, scale=1.0):
    """[rows, n] fp32 view of a [rows, ld] buffer with NaN in the padding columns."""
    import torch
    buf = torch.full((rows, ld), float("nan"), device="cuda")
    buf[:, :n] = scale * torch.randn(rows, n, device="cuda", generator=g)
    return buf, buf[:, :n]


def _out(rows, n, ld):
    """[rows, ld] output buffer filled with the sentinel (the kernel writes [:, :n])."""
    import torch
    return torch.full((rows, ld), SENTINEL, device="cuda")


def _check(name, got, want, bound):
    """|got - want| <= bound elementwise (float64); returns the worst error / bound, printed for the record."""
    import torch
    got, want = got.double(), want.double()
    bound = torch.as_tensor(bound, dtype=torch.float64, device=want.device).expand_as(want)
    assert torch.isfinite(got).all(), name
    r = (got - want).abs() / bound
    ratio, i = float(r.max()), int(r.argmax())
    print("%-44s worst error / tolerance %.3g" % (name, ratio))
    assert ratio <= 1.0, (name, ratio, float(got.flatten()[i]), float(want.flatten()[i]), float(bound.flatten()[i]))
    return ratio


def _sentinel_kept(buf, n):
    assert bool((buf[:, n:] == SENTINEL).all()), "output padding written"


# ---- split, gather, normalise -----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 255, 303105, 5120 * 1024])
def test_split_tf32_is_exact(K, n):
    """hi = x with its low 13 mantissa bits cleared, lo = x - hi exactly: bitwise, over every exponent, subnormals and signed zeros."""
    import torch
    _dev()
    g = _gen(n)
    bits = torch.randint(-2 ** 31, 2 ** 31 - 1, (n + 1,), dtype=torch.int64, device="cuda", generator=g).to(torch.int32)
    bits = torch.where((bits & 0x7F800000) == 0x7F800000, bits & ~0x40000000, bits)  # no inf / NaN; every other exponent
    edges = torch.tensor([0x00000000, 0x80000000, 0x00000001, 0x807FFFFF, 0x00800000, 0x7F7FFFFF, 0x3F800000, 0x00001FFF],
                         dtype=torch.int64, device="cuda").to(torch.int32)
    bits[:min(n, len(edges))] = edges[:min(n, len(edges))]
    x = bits.view(torch.float32)
    hi, lo = torch.full_like(x, SENTINEL), torch.full_like(x, SENTINEL)
    tk.check(K.vnl_split_tf32(x.data_ptr(), n, hi.data_ptr(), lo.data_ptr(), _st()), "split")
    torch.cuda.synchronize()
    assert torch.equal(hi[:n].view(torch.int32), bits[:n] & ~0x1FFF)
    assert torch.equal((hi[:n].double() + lo[:n].double()), x[:n].double())  # lo exact: hi + lo == x
    assert torch.equal(hi[:n] + lo[:n], x[:n])  # and in fp32
    assert hi[n] == SENTINEL and lo[n] == SENTINEL


@pytest.mark.gpu
@pytest.mark.parametrize("width,ld", [(795, 796), (232, 236)])
def test_gather_rows_is_bitwise_with_zeroed_padding(K, width, ld):
    import torch
    _dev()
    T, B, Bm = 20, 8192, 256
    g = _gen(width)
    src = torch.randn(T * B, width, device="cuda", generator=g)
    idx = torch.randint(0, B, (Bm,), dtype=torch.int32, device="cuda", generator=g)
    idx[1], idx[2], idx[-1] = idx[0], B - 1, 0  # repeated indices, the first and the last env
    dst = torch.full((T * Bm, ld), float("nan"), device="cuda")
    tk.check(K.vnl_gather_rows(src.data_ptr(), T, B, width, idx.data_ptr(), Bm, dst.data_ptr(), ld, _st()), "gather_rows")
    torch.cuda.synchronize()
    want = src.view(T, B, width)[:, idx.long()].reshape(T * Bm, width)
    assert torch.equal(dst[:, :width], want)
    assert bool((dst[:, width:] == 0).all())


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 3, 4])
def test_gather_scalars_is_bitwise(K, n):
    import torch
    _dev()
    T, B, Bm = 20, 8192, 256
    g = _gen(10 + n)
    src = [torch.randn(T * B, device="cuda", generator=g) for _ in range(n)]
    dst = [torch.full((T * Bm + 1,), SENTINEL, device="cuda") for _ in range(n)]
    idx = torch.randint(0, B, (Bm,), dtype=torch.int32, device="cuda", generator=g)
    idx[1], idx[-1] = idx[0], B - 1
    ps = lambda ts: (ctypes.c_void_p * n)(*[t.data_ptr() for t in ts])
    tk.check(K.vnl_gather_scalars(n, ps(src), ps(dst), T, B, idx.data_ptr(), Bm, _st()), "gather_scalars")
    torch.cuda.synchronize()
    for s, d in zip(src, dst):
        assert torch.equal(d[:T * Bm], s.view(T, B)[:, idx.long()].reshape(-1)) and d[-1] == SENTINEL


@pytest.mark.gpu
@pytest.mark.parametrize("rows,width", [(5120, 232), (256, 55)])
def test_obs_normalize_into_an_offset_of_the_decoder_input(K, rows, width):
    """out = (obs - mean) / std written at column 64 of a padded [rows, 64 + ld4(width) + 4] buffer (the decoder input [z | obs])."""
    import torch
    _dev()
    g = _gen(rows + width)
    _, obs = _rows(rows, width, tk.ld4(width) + 4, g, 3.0)
    mean = 0.5 * torch.randn(width, device="cuda", generator=g)
    sd = 0.1 + torch.rand(width, device="cuda", generator=g)
    ld_out = 64 + tk.ld4(width) + 4
    out = _out(rows, ld_out, ld_out)
    tk.check(K.vnl_obs_normalize(obs.data_ptr(), obs.stride(0), rows, width, mean.data_ptr(), sd.data_ptr(), out[:, 64:].data_ptr(), ld_out,
                                 _st()), "obs_normalize")
    torch.cuda.synchronize()
    want = (obs.double() - mean.double()) / sd.double()
    # one rounding of the difference (u |obs - mean|), one of the IEEE division: (1 + u)^2 - 1 > 2 u, so 3 u
    _check("obs_normalize %dx%d" % (rows, width), out[:, 64:64 + width], want, 3 * U * want.abs() + TINY)
    assert bool((out[:, :64] == SENTINEL).all()) and bool((out[:, 64 + width:] == SENTINEL).all())


# ---- relu + LayerNorm ---------------------------------------------------------------------------------------------------------
def _ln_stats64(pre):
    """flax LayerNorm statistics of relu(pre) with the fast variance, float64."""
    import torch
    x = torch.relu(pre.double())
    mu = x.mean(-1)
    var = torch.clamp((x * x).mean(-1) - mu * mu, min=0.0)
    return x, mu, var, 1.0 / torch.sqrt(var + 1e-6)


def _pre(rows, n, g):
    """Pre-activations with row 0 all <= 0 (one exact zero: relu'(0) = 0) and a few exact zeros elsewhere."""
    buf, pre = _rows(rows, n, tk.ld4(n) + 4, g)
    pre[0] = -pre[0].abs()
    pre[0, 0] = 0.0
    if rows > 2:
        pre[rows // 2, : (n + 1) // 2] = 0.0
    return buf, pre


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 31, 33, 126, 256, 1000, 1024])
def test_relu_ln_fwd_matches_float64(K, n):
    import torch
    _dev()
    for rows in (1, 480, 9473):
        g = _gen(rows * 7 + n)
        _, pre = _pre(rows, n, g)
        scale, bias = 1.0 + 0.3 * torch.randn(n, device="cuda", generator=g), 0.3 * torch.randn(n, device="cuda", generator=g)
        ld_out = tk.ld4(n) + 4
        out, stats = _out(rows, n, ld_out), torch.full((rows + 1, 2), SENTINEL, device="cuda")
        tk.check(K.vnl_relu_ln_fwd(pre.data_ptr(), pre.stride(0), rows, n, scale.data_ptr(), bias.data_ptr(), out.data_ptr(), ld_out,
                                   stats.data_ptr(), _st()), "relu_ln_fwd")
        torch.cuda.synchronize()
        x, mu, var, rstd = _ln_stats64(pre)
        want = (x - mu[:, None]) * rstd[:, None] * scale.double() + bias.double()
        # mean: an n-term sum and a division; fast variance: an n-term sum of squares minus mu^2 (both <= mean(x^2)); rstd moves by
        # 0.5 rstd^3 of the variance's error; the output by scale (|err mu| rstd + |x - mu| |err rstd|) plus its own 4 roundings
        k = n + 4
        e_mu = k * U * x.abs().mean(-1)
        e_var = 3 * k * U * (x * x).mean(-1)
        e_rstd = 0.5 * rstd ** 3 * e_var + 2 * U * rstd
        e_out = (scale.double().abs() * (e_mu[:, None] * rstd[:, None] + (x - mu[:, None]).abs() * e_rstd[:, None])
                 + 4 * U * ((x - mu[:, None]).abs() * rstd[:, None] * scale.double().abs() + bias.double().abs()))
        tag = "relu_ln_fwd rows %d n %d" % (rows, n)
        _check(tag + " mean", stats[:rows, 0], mu, e_mu + TINY)
        _check(tag + " rstd", stats[:rows, 1], rstd, e_rstd)
        _check(tag + " out", out[:, :n], want, e_out + TINY)
        _sentinel_kept(out, n)
        assert bool((stats[rows] == SENTINEL).all())
        # the row of non-positive pre-activations: mean 0, variance 0, rstd = 1 / sqrt(1e-6), out = bias exactly
        assert stats[0, 0] == 0 and abs(float(stats[0, 1]) - 1000.0) < 1e-3 and torch.equal(out[0, :n], bias)


def _ln_bwd64(pre, stats, scale, dy):
    """float64 autograd of h = LayerNorm(relu(pre)) w.r.t. pre, scale and bias, with the mean and rstd the kernel is given
    (the fp32 statistics of the forward): dpre, dscale, dbias."""
    import torch
    p = pre.double().clone().requires_grad_(True)
    sc = scale.double().clone().requires_grad_(True)
    b = torch.zeros_like(sc, requires_grad=True)
    x = torch.relu(p)
    mu = x.mean(-1, keepdim=True)
    var = torch.clamp((x * x).mean(-1, keepdim=True) - mu * mu, min=0.0)
    rstd = torch.rsqrt(var + 1e-6)
    # the kernel is handed fp32 statistics: move the float64 ones onto those values, keeping their derivatives
    mu = mu + (stats[:, :1].double() - mu).detach()
    rstd = rstd + (stats[:, 1:].double() - rstd).detach()
    h = (x - mu) * rstd * sc + b
    h.backward(dy.double())
    return p.grad, sc.grad, b.grad


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 33, 126, 250, 256])
def test_relu_ln_bwd_matches_float64_autograd(K, n):
    """dpre and the accumulated dscale / dbias / dbias_pre, with and without dbias_pre, onto outputs that start non-zero."""
    import torch
    _dev()
    for rows in SQUARE_ROWS:
        for with_pre in (True, False):
            g = _gen(rows * 11 + n + with_pre)
            _, pre = _pre(rows, n, g)
            _, dy = _rows(rows, n, tk.ld4(n) + 8, g)
            scale = 1.0 + 0.3 * torch.randn(n, device="cuda", generator=g)
            _, mu, _, rstd = _ln_stats64(pre)
            stats = torch.stack([mu, rstd], 1).float().contiguous()
            ld_d = tk.ld4(n) + 4
            dpre = _out(rows, n, ld_d)
            init = [torch.randn(n, device="cuda", generator=g) for _ in range(3)]
            dscale, dbias, dbias_pre = [t.clone() for t in init]
            tk.check(K.vnl_relu_ln_bwd(dy.data_ptr(), dy.stride(0), pre.data_ptr(), pre.stride(0), stats.data_ptr(), scale.data_ptr(), rows, n,
                                       dpre.data_ptr(), ld_d, dscale.data_ptr(), dbias.data_ptr(), dbias_pre.data_ptr() if with_pre else None,
                                       _st()), "relu_ln_bwd")
            torch.cuda.synchronize()
            w_pre, w_scale, w_bias = _ln_bwd64(pre, stats, scale, dy)
            # error model of dpre = rstd (gg - mean(gg) - xh mean(gg xh)), gg = dy scale, xh = (relu(pre) - mu) rstd: two n-term row
            # means and a few roundings, on the magnitudes of the terms; xh is known to u (|x| + |mu|) rstd
            x = torch.relu(pre.double())
            m, r = stats[:, :1].double(), stats[:, 1:].double()
            gg = (dy.double() * scale.double()).abs()
            X = (x + m.abs()) * r
            e_dpre = (n + 8) * U * r * (gg + gg.mean(-1, keepdim=True) + X * (gg * X).mean(-1, keepdim=True)) * (pre > 0)
            tag = "relu_ln_bwd rows %d n %d%s" % (rows, n, "" if with_pre else " (no dbias_pre)")
            _check(tag + " dpre", dpre[:, :n], w_pre, e_dpre + TINY)
            _sentinel_kept(dpre, n)
            # column sums over the rows, onto the initial values
            k = rows + 4
            xh_abs = (x - m).abs() * r
            _check(tag + " dscale", dscale, init[0].double() + w_scale,
                   k * U * ((dy.double().abs() * (xh_abs + X)).sum(0) + init[0].double().abs()) + TINY)
            _check(tag + " dbias", dbias, init[1].double() + w_bias, k * U * (dy.double().abs().sum(0) + init[1].double().abs()) + TINY)
            if with_pre:
                _check(tag + " dbias_pre", dbias_pre, init[2].double() + w_pre.sum(0),
                       k * U * (w_pre.abs().sum(0) + init[2].double().abs()) + e_dpre.sum(0) + TINY)
            else:
                assert torch.equal(dbias_pre, init[2])


# ---- swish ----------------------------------------------------------------------------------------------------------------------
# below x = -88.72 expf(-x) overflows and the fp32 sigmoid is 0; there the exact |swish| and |swish'| are below 89 * 2^-128 < 2^-121
SWISH_FLOOR = 2.0 ** -121


def _swish_inputs(n, g):
    import torch
    x = 4.0 * torch.randn(n, device="cuda", generator=g)
    edges = torch.tensor([100.0, -100.0, 88.7, -88.7, 88.73, -88.73, 89.0, -89.0, 0.0, -1.2785, 1e-30, -1e-30], device="cuda")
    x[:len(edges)] = edges
    return x


def _swish_d64(x):
    """(swish, swish') in float64 and the envelope of swish''s fp32 error: 1 - s loses u of s, multiplied by |x| s."""
    import torch
    x = x.double()
    s = torch.sigmoid(x)
    return x * s, s + x * s * (1 - s), s + x.abs() * s * (1 - s), x.abs() * s


@pytest.mark.gpu
def test_swish_fwd_bwd_match_float64(K):
    """Above 303,104 elements (the grid-stride regime), with x = +-100 and around +-88.7 where expf(-x) overflows and sigmoid -> 0."""
    import torch
    _dev()
    n = 2 * 303104 + 7
    g = _gen(5)
    x = _swish_inputs(n, g)
    dy = torch.randn(n, device="cuda", generator=g)
    out, dpre = torch.full((n + 1,), SENTINEL, device="cuda"), torch.full((n + 1,), SENTINEL, device="cuda")
    tk.check(K.vnl_swish_fwd(x.data_ptr(), n, out.data_ptr(), _st()), "swish_fwd")
    tk.check(K.vnl_swish_bwd(dy.data_ptr(), x.data_ptr(), n, dpre.data_ptr(), _st()), "swish_bwd")
    torch.cuda.synchronize()
    sw, d, env, env1 = _swish_d64(x)
    # sigmoid through expf (2 ulp), an add and a division: 8 u of every term; 1 - s in fp32 loses u of s (2 u |x| s below)
    _check("swish_fwd", out[:n], sw, 8 * U * sw.abs() + SWISH_FLOOR)
    _check("swish_bwd", dpre[:n], dy.double() * d, dy.double().abs() * (8 * U * env + 2 * U * env1 + SWISH_FLOOR) + TINY)
    assert out[n] == SENTINEL and dpre[n] == SENTINEL


@pytest.mark.gpu
def test_outer_swish_bwd_matches_float64(K):
    """dpre[r, c] = dv[r] w[c] swish'(pre[r, c]) over 320 x 1024 = 327,680 elements (the value MLP's last hidden layer)."""
    import torch
    _dev()
    rows, n = 320, 1024
    g = _gen(6)
    pre = _swish_inputs(rows * n, g).view(rows, n)
    dv, w = torch.randn(rows, device="cuda", generator=g), torch.randn(n, device="cuda", generator=g)
    dpre = torch.full((rows * n + 1,), SENTINEL, device="cuda")
    tk.check(K.vnl_outer_swish_bwd(dv.data_ptr(), rows, w.data_ptr(), n, pre.data_ptr(), dpre.data_ptr(), _st()), "outer_swish_bwd")
    torch.cuda.synchronize()
    _, d, env, env1 = _swish_d64(pre)
    dw = (dv.double()[:, None] * w.double()).abs()
    _check("outer_swish_bwd", dpre[:-1].view(rows, n), dv.double()[:, None] * w.double() * d, dw * (10 * U * env + 2 * U * env1 + SWISH_FLOOR) + TINY)
    assert dpre[-1] == SENTINEL


# ---- value head: rowdot, colsum -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("rows", [5376, 20000])
@pytest.mark.parametrize("n,ld", [(1024, 1028), (1, 1)])
def test_rowdot_and_colsum_match_float64(K, rows, n, ld):
    """5376 = R + Bm rows (the value of every transition and of the bootstrap observations), 20000 rows (above colsum's 512-chunk
    cap); n = 1 with ld = 1 is the value bias gradient.  b NULL and set; w NULL and set; colsum accumulates onto its output."""
    import torch
    _dev()
    g = _gen(rows + n)
    if ld == n:
        x = torch.randn(rows, n, device="cuda", generator=g)
    else:
        _, x = _rows(rows, n, ld, g)
    w, wr, b = torch.randn(n, device="cuda", generator=g), torch.randn(rows, device="cuda", generator=g), torch.randn(1, device="cuda", generator=g)
    x64 = x.double()
    for bias in (None, b):
        out = torch.full((rows + 1,), SENTINEL, device="cuda")
        tk.check(K.vnl_rowdot(x.data_ptr(), ld, rows, n, w.data_ptr(), _p(bias), out.data_ptr(), _st()), "rowdot")
        torch.cuda.synchronize()
        b64 = 0.0 if bias is None else float(bias)
        _check("rowdot rows %d n %d b %s" % (rows, n, bias is not None), out[:rows], x64 @ w.double() + b64,
               (n + 2) * U * (x64.abs() @ w.double().abs() + abs(b64)) + TINY)
        assert out[rows] == SENTINEL
    for weights in (None, wr):
        init = torch.randn(n + 1, device="cuda", generator=g)
        init[n] = SENTINEL
        out = init.clone()
        tk.check(K.vnl_colsum(x.data_ptr(), ld, rows, n, _p(weights), out.data_ptr(), _st()), "colsum")
        torch.cuda.synchronize()
        wt = torch.ones(rows, dtype=torch.float64, device="cuda") if weights is None else weights.double()
        _check("colsum rows %d n %d w %s" % (rows, n, weights is not None), out[:n], init[:n].double() + wt @ x64,
               (rows + 4) * U * (wt.abs() @ x64.abs() + init[:n].double().abs()) + TINY)
        assert out[n] == SENTINEL


# ---- reparameterisation and its backward with the KL term ---------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("rows,L", [(5120, 64), (20000, 64), (1, 2)])
def test_reparam_and_heads_bwd_match_float64(K, rows, L):
    """5120 x 64 = 327,680 elements is above grid_for's cap (each thread then adds two KL terms); logvar in [-20, 10]."""
    import torch
    _dev()
    g = _gen(rows + L)
    heads = torch.cat([torch.randn(rows, L, device="cuda", generator=g), -20.0 + 30.0 * torch.rand(rows, L, device="cuda", generator=g)], 1)
    heads[0, L:] = torch.linspace(-20.0, 10.0, L, device="cuda")
    eps = torch.randn(rows, L, device="cuda", generator=g)
    ld = L + 232 + 8
    dec_in = _out(rows, ld, ld)
    tk.check(K.vnl_reparam_fwd(heads.data_ptr(), eps.data_ptr(), rows, L, dec_in.data_ptr(), ld, _st()), "reparam_fwd")
    torch.cuda.synchronize()
    m, lv, e64 = heads[:, :L].double(), heads[:, L:].double(), eps.double()
    sd = torch.exp(0.5 * lv)
    _check("reparam_fwd rows %d L %d" % (rows, L), dec_in[:, :L], m + e64 * sd, 4 * U * (m.abs() + 2 * (e64 * sd).abs()) + TINY)
    assert bool((dec_in[:, L:] == SENTINEL).all())

    ddec_buf, ddec = _rows(rows, L, ld, g)  # columns [L, ld) are the observation part of the decoder input's gradient: NaN here
    kl_coef = 1e-4 / (rows * L)
    for with_kl in (True, False):
        dheads = torch.full((rows * 2 * L + 1,), SENTINEL, device="cuda")
        kl = torch.tensor([0.25, SENTINEL], device="cuda")
        tk.check(K.vnl_heads_bwd(ddec.data_ptr(), ld, heads.data_ptr(), eps.data_ptr(), rows, L, kl_coef, dheads.data_ptr(),
                                 kl.data_ptr() if with_kl else None, _st()), "heads_bwd")
        torch.cuda.synchronize()
        dz, el = ddec.double(), torch.exp(lv)
        kc = float(np.float32(kl_coef))
        want_m = dz + kc * m
        want_lv = dz * 0.5 * e64 * sd - 0.5 * kc * (1 - el)
        tag = "heads_bwd rows %d L %d" % (rows, L)
        got = dheads[:-1].view(rows, 2 * L)
        _check(tag + " dmean", got[:, :L], want_m, 3 * U * (dz.abs() + kc * m.abs()) + TINY)
        _check(tag + " dlogvar", got[:, L:], want_lv, 8 * U * ((dz * e64 * sd).abs() + kc * (1 + el)) + TINY)
        assert dheads[-1] == SENTINEL
        terms = -0.5 * kc * (1 + lv - m * m - el)
        if with_kl:
            # rows * L terms, each thread adds <= 5 in order, then a block tree and one atomic per block: fewer than `rows` in a chain
            e_terms = 8 * U * 0.5 * kc * (1 + lv.abs() + m * m + el)
            _check(tag + " kl_loss", kl[:1], 0.25 + terms.sum().reshape(1),
                   (rows + 8) * U * (terms.abs().sum() + 0.25) + e_terms.sum())
        else:
            assert float(kl[0]) == 0.25
        assert kl[1] == SENTINEL


# ---- brax NormalTanhDistribution: ppo_rows, policy_sample -----------------------------------------------------------------------
def _softplus(x):
    import torch
    return torch.nn.functional.softplus(x)


def _ldj(x):
    """brax TanhBijector.forward_log_det_jacobian and its magnitude envelope |x| + |softplus(-2x)| + log 2."""
    return 2.0 * (math.log(2.0) - x - _softplus(-2.0 * x)), x.abs() + _softplus(-2.0 * x) + 1.0


def _logits(rows, nu, g):
    """[rows, 2 nu] logits in a [rows, ld4(2 nu)] buffer (NaN padding): loc ~ N(0, 1), scale logits ~ N(0, 2) with +-30 entries
    (softplus(-30) + 0.001: the 0.001 floor)."""
    buf, lg = _rows(rows, 2 * nu, tk.ld4(2 * nu), g)
    lg[:, nu:] *= 2.0
    lg[::7, nu] = 30.0
    lg[::5, 2 * nu - 1] = -30.0
    return lg


def _lp64(lg, a):
    """float64 log-prob of raw action a under logits lg, and the per-lane magnitudes of its terms."""
    import torch
    nu = a.shape[1]
    loc, scale = lg[:, :nu].double(), _softplus(lg[:, nu:].double()) + 0.001
    z = (a.double() - loc) / scale
    ldj, env = _ldj(a.double())
    lanes = -0.5 * z * z - torch.log(scale) - 0.5 * math.log(2 * math.pi) - ldj
    mag = 0.5 * z * z + torch.log(scale).abs() + 1.0 + env
    return lanes.sum(-1), mag, loc, scale


def _row_sum_tol(mag, c=16):
    """Tolerance of a warp sum over the action lanes: each lane's term carries c u of its magnitudes (expf / log1pf / logf chains),
    the nu-term sum adds nu u of the sum of their magnitudes."""
    nu = mag.shape[1]
    return (c + nu) * U * mag.sum(-1) + TINY


@pytest.mark.gpu
@pytest.mark.parametrize("nu", [1, 21, 30, 32])
def test_ppo_rows_matches_float64(K, nu):
    import torch
    _dev()
    rows = 9473
    g = _gen(nu)
    lg = _logits(rows, nu, g)
    raw = (15.0 * (2 * torch.rand(rows, nu, device="cuda", generator=g) - 1)).contiguous()  # |raw| up to 15: the tail of log_det_jac
    eps_ent = torch.randn(rows, nu, device="cuda", generator=g)
    disc = (torch.rand(rows, device="cuda", generator=g) > 0.1).float()
    trunc = (torch.rand(rows, device="cuda", generator=g) > 0.9).float()
    rew = torch.randn(rows, device="cuda", generator=g)
    outs = [torch.full((rows + 1,), SENTINEL, device="cuda") for _ in range(4)]
    tk.check(K.vnl_ppo_rows(lg.data_ptr(), lg.stride(0), raw.data_ptr(), eps_ent.data_ptr(), rows, nu, disc.data_ptr(), trunc.data_ptr(),
                            rew.data_ptr(), 0.37, *[o.data_ptr() for o in outs], _st()), "ppo_rows")
    torch.cuda.synchronize()
    lp, mag, loc, scale = _lp64(lg, raw)
    _check("ppo_rows nu %d target_lp" % nu, outs[0][:rows], lp, _row_sum_tol(mag))
    s = loc + scale * eps_ent.double()
    ldj, env = _ldj(s)
    ent = (0.5 + 0.5 * math.log(2 * math.pi) + torch.log(scale) + ldj).sum(-1)
    # the sample loc + scale eps is itself rounded (u of |loc| + |scale eps|); log_det_jac's slope is at most 2
    mag_e = torch.log(scale).abs() + 2.0 + env + 2 * (loc.abs() + (scale * eps_ent.double()).abs())
    _check("ppo_rows nu %d entropy" % nu, outs[1][:rows], ent, _row_sum_tol(mag_e))
    assert torch.equal(outs[2][:rows], (1 - disc) * (1 - trunc))
    assert torch.equal(outs[3][:rows], rew * np.float32(0.37))
    assert all(o[rows] == SENTINEL for o in outs)


@pytest.mark.gpu
@pytest.mark.parametrize("nu", [1, 21, 30, 32])
def test_policy_sample_matches_float64(K, nu):
    """The sample (eps_a set) and the mode (eps_a NULL); rand_action NULL (rand_log_prob untouched) and set."""
    import torch
    _dev()
    rows = 9473
    g = _gen(100 + nu)
    lg = _logits(rows, nu, g)
    eps = torch.randn(rows, nu, device="cuda", generator=g)
    ra = 2 * torch.rand(nu, device="cuda", generator=g) - 1
    for eps_a, rand in ((eps, ra), (None, None), (eps, None), (None, ra)):
        act, raw = [torch.full((rows * nu + 1,), SENTINEL, device="cuda") for _ in range(2)]
        lp, rlp = [torch.full((rows + 1,), SENTINEL, device="cuda") for _ in range(2)]
        tk.check(K.vnl_policy_sample(lg.data_ptr(), lg.stride(0), _p(eps_a), _p(rand), rows, nu, act.data_ptr(), raw.data_ptr(), lp.data_ptr(),
                                     rlp.data_ptr(), _st()), "policy_sample")
        torch.cuda.synchronize()
        tag = "policy_sample nu %d %s%s" % (nu, "sample" if eps_a is not None else "mode", " rand" if rand is not None else "")
        raw2 = raw[:-1].view(rows, nu)
        loc, scale = lg[:, :nu].double(), _softplus(lg[:, nu:].double()) + 0.001
        if eps_a is None:
            assert torch.equal(raw2, lg[:, :nu])
        else:
            _check(tag + " raw", raw2, loc + scale * eps.double(), 8 * U * (loc.abs() + (scale * eps.double()).abs()) + TINY)
        # log_prob and tanh at the raw action the kernel drew (z = (raw - loc) / scale is eps up to that rounding)
        _check(tag + " action", act[:-1].view(rows, nu), torch.tanh(raw2.double()), 4 * U * torch.tanh(raw2.double()).abs() + TINY)
        want, mag, _, _ = _lp64(lg, raw2)
        _check(tag + " log_prob", lp[:rows], want, _row_sum_tol(mag))
        if rand is not None:
            want, mag, _, _ = _lp64(lg, rand.expand(rows, nu))
            _check(tag + " rand_log_prob", rlp[:rows], want, _row_sum_tol(mag))
        else:
            assert bool((rlp == SENTINEL).all())
        assert act[-1] == SENTINEL and raw[-1] == SENTINEL and lp[rows] == SENTINEL and rlp[rows] == SENTINEL


# ---- the PPO loss and its gradients -----------------------------------------------------------------------------------------------
def _loss_inputs(rows, nu, clip, g):
    """Logits, actions drawn from them, and log rho = target_lp - behaviour_lp on both sides of the clip range and inside it, each at
    least 1e-3 away from log(1 +- eps) so that fp32 rounding cannot move a row across a clip boundary."""
    import torch
    lg = _logits(rows, nu, g)
    loc, scale = lg[:, :nu].double(), _softplus(lg[:, nu:].double()) + 0.001
    raw = (loc + scale * torch.randn(rows, nu, device="cuda", generator=g).double()).float().contiguous()
    eps_ent = torch.randn(rows, nu, device="cuda", generator=g)
    tlp = _lp64(lg, raw)[0].float()
    log_rho = 0.4 * torch.randn(rows, device="cuda", generator=g).double()
    for edge in (math.log(1 - clip), math.log(1 + clip)):
        near = (log_rho - edge).abs() < 1e-3
        log_rho = torch.where(near, edge + torch.sign(log_rho - edge + 1e-12) * 2e-3, log_rho)
    blp = (tlp.double() - log_rho).float()
    adv = torch.randn(rows, device="cuda", generator=g)
    vs, baseline = torch.randn(rows, device="cuda", generator=g), torch.randn(rows, device="cuda", generator=g)
    return lg, raw, eps_ent, tlp, blp, adv, vs, baseline


@pytest.mark.gpu
@pytest.mark.parametrize("nu", [21, 30])
@pytest.mark.parametrize("normalize", [1, 0])
def test_ppo_loss_bwd_matches_float64_autograd(K, nu, normalize):
    """dlogits, dvalue, the advantage mean / std in scratch2 and the accumulated loss metrics against float64 autograd of the
    clipped surrogate, the value loss and the entropy loss (the KL term is vnl_heads_bwd's); rows = 1 has std 0."""
    import torch
    _dev()
    clip, ent_cost = 0.3, 1e-4
    for rows in (1, 480, 1184, 1185, 5120, 20000):
        g = _gen(rows + 31 * nu + normalize)
        lg, raw, eps_ent, tlp, blp, adv, vs, baseline = _loss_inputs(rows, nu, clip, g)
        _, _, loc, scale = _lp64(lg, raw)
        s = loc + scale * eps_ent.double()
        ent = (0.5 + 0.5 * math.log(2 * math.pi) + torch.log(scale) + _ldj(s)[0]).sum(-1).float()  # what vnl_ppo_rows hands over
        ld_d = tk.ld4(2 * nu) + 4
        dl = _out(rows, 2 * nu, ld_d)
        dvalue = torch.full((rows + 1,), SENTINEL, device="cuda")
        metrics0 = torch.tensor([0.5, -0.25, 0.125, 1.0, 7.0, 2.0, 0.75, SENTINEL], device="cuda")
        metrics, scratch = metrics0.clone(), torch.full((3,), SENTINEL, device="cuda")
        tk.check(K.vnl_ppo_loss_bwd(lg.data_ptr(), lg.stride(0), raw.data_ptr(), eps_ent.data_ptr(), rows, nu, tlp.data_ptr(), blp.data_ptr(),
                                    ent.data_ptr(), adv.data_ptr(), vs.data_ptr(), baseline.data_ptr(), clip, ent_cost, normalize, dl.data_ptr(),
                                    ld_d, dvalue.data_ptr(), metrics.data_ptr(), scratch.data_ptr(), _st()), "ppo_loss_bwd")
        torch.cuda.synchronize()
        tag = "ppo_loss_bwd rows %d nu %d norm %d" % (rows, nu, normalize)

        # float64 autograd; the loss is evaluated at the fp32 target_lp / entropy the kernel is handed, with their derivatives
        L64 = lg.double().clone().requires_grad_(True)
        b64 = baseline.double().clone().requires_grad_(True)
        loc_, scale_ = L64[:, :nu], _softplus(L64[:, nu:]) + 0.001
        t_lp = _lp64(L64, raw)[0]
        t_lp = t_lp + (tlp.double() - t_lp).detach()
        en = (0.5 + 0.5 * math.log(2 * math.pi) + torch.log(scale_) + _ldj(loc_ + scale_ * eps_ent.double())[0]).sum(-1)
        en = en + (ent.double() - en).detach()
        A = adv.double()
        amu, asd = A.mean(), A.std(unbiased=False)
        An = (A - amu) / (asd + 1e-8) if normalize else A
        rho = torch.exp(t_lp - blp.double())
        s1, s2 = rho * An, torch.clamp(rho, 1 - clip, 1 + clip) * An
        pol = -torch.minimum(s1, s2).mean()
        v_loss = ((vs.double() - b64) ** 2).mean() * 0.25
        ent_loss = -ent_cost * en.mean()
        (pol + v_loss + ent_loss).backward()

        # scratch2: mean and population std, summed in double and rounded once
        want_stats = torch.stack([amu, asd])
        _check(tag + " adv mean/std", scratch[:2], want_stats, 2 * U * want_stats.abs() + TINY)
        assert scratch[2] == SENTINEL
        # dlogits: error envelope of g_lp = -A rho / R (normalised A to 3 u of (|A| + |mean|) / std, rho = expf of a difference of two
        # log-probs to u (|t| + |b|) + 2 ulp) times d / scale^2 (scale to 4 u), plus the entropy terms (tanh of a rounded sample)
        invR = 1.0 / rows
        r64 = rho.detach()
        d, inv = raw.double() - loc, 1.0 / scale
        Amag = (An.abs() + ((A.abs() + amu.abs()) / (asd + 1e-8) if normalize else 0.0)) * r64 * invR * (1 + tlp.double().abs() + blp.double().abs())
        e_s = ent_cost * invR * 2.0 * (1.0 + loc.abs() + (scale * eps_ent.double()).abs())
        Mloc = Amag[:, None] * d.abs() * inv * inv + e_s
        Mscale = (Amag[:, None] * (d * d * inv ** 3 + inv) + ent_cost * invR * inv + e_s * eps_ent.double().abs()) * torch.sigmoid(lg[:, nu:].double())
        _check(tag + " dlogits", dl[:, :2 * nu], L64.grad, 16 * U * torch.cat([Mloc, Mscale], 1) + TINY)
        _sentinel_kept(dl, 2 * nu)
        _check(tag + " dvalue", dvalue[:rows], b64.grad, 4 * U * b64.grad.abs() + TINY)
        assert dvalue[rows] == SENTINEL
        # metrics: atomic sums over the rows onto the initial values
        m0 = metrics0.double()
        k = rows + 16
        t_pol = -torch.minimum(s1, s2).detach() * invR
        e_pol = k * U * t_pol.abs().sum() + 16 * U * Amag.sum()
        t_v = 0.25 * (vs.double() - baseline.double()) ** 2 * invR
        e_v = k * U * t_v.abs().sum() + 4 * U * t_v.sum()
        t_e = -ent_cost * ent.double() * invR
        e_e = k * U * t_e.abs().sum()
        t_r = r64 * invR
        e_r = k * U * t_r.sum() + 16 * U * (t_r * (1 + tlp.double().abs() + blp.double().abs())).sum()
        outside = (r64 < 1 - clip) | (r64 > 1 + clip)
        t_c = outside.double() * invR
        want = torch.stack([m0[0] + t_pol.sum() + t_v.sum() + t_e.sum(), m0[1] + t_pol.sum(), m0[2] + t_v.sum(), m0[3] + t_e.sum(),
                            m0[5] + t_r.sum(), m0[6] + t_c.sum()])
        bound = torch.stack([e_pol + e_v + e_e, e_pol, e_v, e_e, e_r, k * U * t_c.sum()]) + k * U * m0[[0, 1, 2, 3, 5, 6]].abs() + TINY
        for i, (slot, what) in enumerate(zip((0, 1, 2, 3, 5, 6), ("total", "policy_loss", "v_loss", "entropy_loss", "mean rho", "clipped"))):
            _check(tag + " metrics " + what, metrics[slot:slot + 1], want[i:i + 1], bound[i:i + 1])
        assert metrics[4] == metrics0[4] and metrics[7] == SENTINEL
        if rows >= 480:
            assert 0.05 < float(t_c.sum()) < 0.95  # both branches of the clipped surrogate


# ---- evaluation metrics ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("nm", [0, 15])
def test_eval_metrics_matches_the_eval_wrapper(K, nm):
    """brax EvalWrapper over an unroll from reset, B = 8193 (ragged last block): envs done at t = 0, never, and mid-unroll."""
    import torch
    _dev()
    T, B = 20, 8193
    g = _gen(nm)
    metrics = torch.randn(T, B, max(nm, 1), device="cuda", generator=g)[:, :, :nm].contiguous()
    reward = torch.randn(T, B, device="cuda", generator=g)
    done = (torch.rand(T, B, device="cuda", generator=g) > 0.93).float()
    done[:, 1] = 0.0          # never done
    done[0, 0] = 1.0          # done at the first step
    done[:, 2] = 0.0
    done[7, 2] = 1.0          # mid-unroll
    done[T - 1, 3] = 1.0      # at the last step
    em = torch.full((B * (nm + 1) + 1,), SENTINEL, device="cuda")
    active, steps = torch.full((B + 1,), SENTINEL, device="cuda"), torch.full((B + 1,), SENTINEL, device="cuda")
    mp = metrics.data_ptr() if nm else reward.data_ptr()  # nm = 0: never read, but the pointer must not be NULL
    tk.check(K.vnl_eval_metrics(T, B, nm, mp, reward.data_ptr(), done.data_ptr(), em.data_ptr(), active.data_ptr(), steps.data_ptr(), _st()),
             "eval_metrics")
    torch.cuda.synchronize()
    vals = torch.cat([metrics.double(), reward.double()[:, :, None]], 2)  # [T, B, nm + 1]
    act = torch.ones(B, dtype=torch.float64, device="cuda")
    acc = torch.zeros(B, nm + 1, dtype=torch.float64, device="cuda")
    mag = torch.zeros_like(acc)
    st = torch.zeros(B, dtype=torch.float64, device="cuda")
    for t in range(T):
        st = torch.where(act != 0, torch.full_like(st, t + 1), st)
        acc += vals[t] * act[:, None]
        mag += vals[t].abs() * act[:, None]
        act = act * (1 - done[t].double())
    _check("eval_metrics nm %d" % nm, em[:-1].view(B, nm + 1), acc, (T + 1) * U * mag + TINY)
    assert torch.equal(active[:B].double(), act) and torch.equal(steps[:B].double(), st)
    assert (float(steps[0]), float(active[0]), float(steps[1]), float(active[1]), float(steps[2])) == (1.0, 0.0, T, 1.0, 8.0)
    assert em[-1] == SENTINEL and active[B] == SENTINEL and steps[B] == SENTINEL


# ---- Adam ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", [1630397, 1])
def test_adam_matches_float64(K, n):
    """optax.adam on the 1.63 M-parameter buffer and on one value: bias corrections from the host and from vnl_adam_tick's device
    counter, at step 1 and at step 10^5, with grad_scale 0.5.  The float64 reference uses the fp32 values of b1, b2, eps, lr."""
    import torch
    _dev()
    f32 = lambda v: float(np.float32(v))
    lr, b1, b2, eps = 3e-4, 0.9, 0.999, 1e-8
    lr_, b1_, b2_, eps_ = f32(lr), f32(b1), f32(b2), f32(eps)
    g = _gen(n % 1000)
    for step in (1, 100000):
        for device_bc in (False, True):
            p = torch.randn(n + 1, device="cuda", generator=g)
            gr = torch.randn(n + 1, device="cuda", generator=g) * (10.0 ** torch.randint(-4, 2, (n + 1,), device="cuda", generator=g))
            m = torch.zeros(n + 1, device="cuda") if step == 1 else 0.1 * torch.randn(n + 1, device="cuda", generator=g)
            v = torch.zeros(n + 1, device="cuda") if step == 1 else 0.01 * torch.rand(n + 1, device="cuda", generator=g)
            p[n] = m[n] = v[n] = SENTINEL
            p0, m0, v0 = p.double(), m.double(), v.double()
            bc = None
            if device_bc:
                ctr = torch.tensor([step - 1], dtype=torch.int32, device="cuda")
                bc = torch.full((2,), SENTINEL, device="cuda")
                tk.check(K.vnl_adam_tick(ctr.data_ptr(), b1, b2, bc.data_ptr(), _st()), "adam_tick")
            tk.check(K.vnl_adam(p.data_ptr(), gr.data_ptr(), m.data_ptr(), v.data_ptr(), n, lr, b1, b2, eps, 0 if device_bc else step, 0.5,
                                _p(bc), _st()), "adam")
            torch.cuda.synchronize()
            tag = "adam n %d step %d %s" % (n, step, "device bc" if device_bc else "host bc")
            # bias corrections 1 - b^t from fp32 powf: b^t to 2 ulp, then one subtraction
            bc1, bc2 = 1 - b1_ ** step, 1 - b2_ ** step
            e_bc1, e_bc2 = U * (1 + 4 * b1_ ** step / bc1), U * (1 + 4 * b2_ ** step / bc2)
            if device_bc:
                assert int(ctr.item()) == step
                _check(tag + " bias corrections", bc, torch.tensor([bc1, bc2], dtype=torch.float64, device="cuda"),
                       torch.tensor([e_bc1 * bc1, e_bc2 * bc2], dtype=torch.float64, device="cuda") + TINY)
            gs = 0.5 * gr.double()[:n]
            m_ = b1_ * m0[:n] + (1 - b1_) * gs
            v_ = b2_ * v0[:n] + (1 - b2_) * gs * gs
            upd = lr_ * (m_ / bc1) / (torch.sqrt(v_ / bc2) + eps_)
            p_ = p0[:n] - upd
            # m, v: 4 roundings of their two terms; the update: m's error through the ratio, 8 u of its own roundings, and the
            # relative errors of the bias corrections (1 / bc1 and sqrt(bc2))
            Mm = (b1_ * m0[:n]).abs() + ((1 - b1_) * gs).abs()
            env = lr_ * (Mm / bc1) / (torch.sqrt(v_ / bc2) + eps_)
            _check(tag + " m", m[:n], m_, 4 * U * Mm + TINY)
            _check(tag + " v", v[:n], v_, 4 * U * v_ + TINY)
            _check(tag + " params", p[:n], p_, 2 * U * p_.abs() + (16 * U + e_bc1 + 0.5 * e_bc2) * env + TINY)
            assert p[n] == SENTINEL and m[n] == SENTINEL and v[n] == SENTINEL


# ---- argument checks (no device needed) -------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def host_lib():
    if not os.path.exists(libm.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return tk.lib()


def test_exports_refuse_bad_arguments_before_any_cuda_call(host_lib):
    """Every refusal returns -1 before the library touches CUDA (so this runs on a host without a device); n == 0 is a no-op that
    returns 0 for split, swish and Adam.  The fake addresses are never dereferenced on these paths."""
    L = host_lib
    P = 0x7000000000  # a non-NULL device address
    PP = (ctypes.c_void_p * 4)(P, P, P, P)
    NUL = (ctypes.c_void_p * 4)(P, None, P, P)
    refusals = {
        "split NULL": L.vnl_split_tf32(None, 8, P, P, None),
        "split NULL lo": L.vnl_split_tf32(P, 8, P, None, None),
        "gather_rows NULL idx": L.vnl_gather_rows(P, 20, 8192, 795, None, 256, P, 796, None),
        "gather_rows ld < width": L.vnl_gather_rows(P, 20, 8192, 795, P, 256, P, 794, None),
        "gather_rows rows 0": L.vnl_gather_rows(P, 0, 8192, 795, P, 256, P, 796, None),
        "gather_rows Bm 0": L.vnl_gather_rows(P, 20, 8192, 795, P, 0, P, 796, None),
        "obs_normalize NULL": L.vnl_obs_normalize(P, 232, 5120, 232, P, None, P, 296, None),
        "obs_normalize ld_obs < width": L.vnl_obs_normalize(P, 231, 5120, 232, P, P, P, 296, None),
        "obs_normalize ld_out < width": L.vnl_obs_normalize(P, 232, 5120, 232, P, P, P, 231, None),
        "obs_normalize rows 0": L.vnl_obs_normalize(P, 232, 0, 232, P, P, P, 296, None),
        "relu_ln_fwd n 1025": L.vnl_relu_ln_fwd(P, 1028, 5120, 1025, P, P, P, 1028, P, None),
        "relu_ln_fwd ld_pre < n": L.vnl_relu_ln_fwd(P, 255, 5120, 256, P, P, P, 256, P, None),
        "relu_ln_fwd ld_out < n": L.vnl_relu_ln_fwd(P, 256, 5120, 256, P, P, P, 255, P, None),
        "relu_ln_fwd NULL stats": L.vnl_relu_ln_fwd(P, 256, 5120, 256, P, P, P, 256, None, None),
        "relu_ln_fwd rows 0": L.vnl_relu_ln_fwd(P, 256, 0, 256, P, P, P, 256, P, None),
        "relu_ln_bwd n 257": L.vnl_relu_ln_bwd(P, 260, P, 260, P, P, 5120, 257, P, 260, P, P, P, None),
        "relu_ln_bwd ld_dy < n": L.vnl_relu_ln_bwd(P, 255, P, 256, P, P, 5120, 256, P, 256, P, P, P, None),
        "relu_ln_bwd ld_pre < n": L.vnl_relu_ln_bwd(P, 256, P, 255, P, P, 5120, 256, P, 256, P, P, P, None),
        "relu_ln_bwd ld_dpre < n": L.vnl_relu_ln_bwd(P, 256, P, 256, P, P, 5120, 256, P, 255, P, P, P, None),
        "relu_ln_bwd NULL dscale": L.vnl_relu_ln_bwd(P, 256, P, 256, P, P, 5120, 256, P, 256, None, P, P, None),
        "relu_ln_bwd rows 0": L.vnl_relu_ln_bwd(P, 256, P, 256, P, P, 0, 256, P, 256, P, P, P, None),
        "swish_fwd NULL": L.vnl_swish_fwd(None, 8, P, None),
        "swish_bwd NULL": L.vnl_swish_bwd(P, P, 8, None, None),
        "reparam_fwd ld < L": L.vnl_reparam_fwd(P, P, 5120, 64, P, 63, None),
        "reparam_fwd NULL eps": L.vnl_reparam_fwd(P, None, 5120, 64, P, 296, None),
        "reparam_fwd rows 0": L.vnl_reparam_fwd(P, P, 0, 64, P, 296, None),
        "heads_bwd ld < L": L.vnl_heads_bwd(P, 63, P, P, 5120, 64, 1e-4, P, P, None),
        "heads_bwd NULL dheads": L.vnl_heads_bwd(P, 296, P, P, 5120, 64, 1e-4, None, P, None),
        "heads_bwd rows 0": L.vnl_heads_bwd(P, 296, P, P, 0, 64, 1e-4, P, P, None),
        "colsum ld < n": L.vnl_colsum(P, 1023, 5120, 1024, None, P, None),
        "colsum NULL out": L.vnl_colsum(P, 1024, 5120, 1024, None, None, None),
        "colsum rows 0": L.vnl_colsum(P, 1024, 0, 1024, None, P, None),
        "rowdot ld < n": L.vnl_rowdot(P, 1023, 5120, 1024, P, None, P, None),
        "rowdot NULL w": L.vnl_rowdot(P, 1024, 5120, 1024, None, None, P, None),
        "rowdot rows 0": L.vnl_rowdot(P, 1024, 0, 1024, P, None, P, None),
        "outer_swish_bwd NULL pre": L.vnl_outer_swish_bwd(P, 5120, P, 1024, None, P, None),
        "outer_swish_bwd rows 0": L.vnl_outer_swish_bwd(P, 0, P, 1024, P, P, None),
        "gather_scalars n 0": L.vnl_gather_scalars(0, PP, PP, 20, 8192, P, 256, None),
        "gather_scalars n 5": L.vnl_gather_scalars(5, PP, PP, 20, 8192, P, 256, None),
        "gather_scalars NULL src[1]": L.vnl_gather_scalars(4, NUL, PP, 20, 8192, P, 256, None),
        "gather_scalars NULL dst[1]": L.vnl_gather_scalars(2, PP, NUL, 20, 8192, P, 256, None),
        "gather_scalars rows 0": L.vnl_gather_scalars(4, PP, PP, 0, 8192, P, 256, None),
        "policy_sample nu 33": L.vnl_policy_sample(P, 68, P, P, 8192, 33, P, P, P, P, None),
        "policy_sample ld < 2 nu": L.vnl_policy_sample(P, 59, P, P, 8192, 30, P, P, P, P, None),
        "policy_sample NULL log_prob": L.vnl_policy_sample(P, 60, P, P, 8192, 30, P, P, None, P, None),
        "policy_sample rows 0": L.vnl_policy_sample(P, 60, P, P, 0, 30, P, P, P, P, None),
        "eval_metrics nm 16": L.vnl_eval_metrics(20, 8192, 16, P, P, P, P, P, P, None),
        "eval_metrics nm -1": L.vnl_eval_metrics(20, 8192, -1, P, P, P, P, P, P, None),
        "eval_metrics NULL done": L.vnl_eval_metrics(20, 8192, 15, P, P, None, P, P, P, None),
        "eval_metrics T 0": L.vnl_eval_metrics(0, 8192, 15, P, P, P, P, P, P, None),
        "ppo_rows nu 33": L.vnl_ppo_rows(P, 68, P, P, 5120, 33, P, P, P, 1.0, P, P, P, P, None),
        "ppo_rows ld < 2 nu": L.vnl_ppo_rows(P, 59, P, P, 5120, 30, P, P, P, 1.0, P, P, P, P, None),
        "ppo_rows NULL eps_ent": L.vnl_ppo_rows(P, 60, P, None, 5120, 30, P, P, P, 1.0, P, P, P, P, None),
        "ppo_rows rows 0": L.vnl_ppo_rows(P, 60, P, P, 0, 30, P, P, P, 1.0, P, P, P, P, None),
        "ppo_loss_bwd nu 33": L.vnl_ppo_loss_bwd(P, 68, P, P, 5120, 33, P, P, P, P, P, P, 0.3, 1e-4, 1, P, 68, P, P, P, None),
        "ppo_loss_bwd ld_d < 2 nu": L.vnl_ppo_loss_bwd(P, 60, P, P, 5120, 30, P, P, P, P, P, P, 0.3, 1e-4, 1, P, 59, P, P, P, None),
        "ppo_loss_bwd NULL scratch2": L.vnl_ppo_loss_bwd(P, 60, P, P, 5120, 30, P, P, P, P, P, P, 0.3, 1e-4, 1, P, 60, P, P, None, None),
        "ppo_loss_bwd rows 0": L.vnl_ppo_loss_bwd(P, 60, P, P, 0, 30, P, P, P, P, P, P, 0.3, 1e-4, 1, P, 60, P, P, P, None),
        "adam_tick NULL": L.vnl_adam_tick(None, 0.9, 0.999, P, None),
        "adam step 0 without device bias corrections": L.vnl_adam(P, P, P, P, 8, 3e-4, 0.9, 0.999, 1e-8, 0, 1.0, None, None),
        "adam NULL v": L.vnl_adam(P, P, P, None, 8, 3e-4, 0.9, 0.999, 1e-8, 1, 1.0, None, None),
        "metrics_accumulate n 1025": L.vnl_metrics_accumulate(P, 1025, P, None),
        "metrics_accumulate n 0": L.vnl_metrics_accumulate(P, 0, P, None),
    }
    assert {k: v for k, v in refusals.items() if v != -1} == {}
    noops = {
        "split": L.vnl_split_tf32(P, 0, P, P, None),
        "swish_fwd": L.vnl_swish_fwd(P, 0, P, None),
        "swish_bwd": L.vnl_swish_bwd(P, P, 0, P, None),
        "adam host bias corrections": L.vnl_adam(P, P, P, P, 0, 3e-4, 0.9, 0.999, 1e-8, 1, 1.0, None, None),
        "adam device bias corrections": L.vnl_adam(P, P, P, P, 0, 3e-4, 0.9, 0.999, 1e-8, 0, 1.0, P, None),
    }
    assert {k: v for k, v in noops.items() if v != 0} == {}
