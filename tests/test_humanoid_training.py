"""Training `HumanoidTracking` end to end: the PPO update, the fp32-class rollout policy, the rollout, the training step and the
evaluator at the humanoid's sizes (obs 55, nu 21: 42 logits, decoder input 64 + 55 = 119, traj 630).  None of these widths is a
multiple of 4 floats, which a TMA tensor map needs for its row stride: such operands live in zeroed buffers with rows of
`train_kernels.ld4(n)` floats (learner.flat_layout for the flat parameter buffer).  Checkers and tolerances are the rodent tests'
(tests/test_gemm.py, test_learner.py, test_policy.py, test_rollout.py, test_trainer.py, test_evaluator.py)."""
import numpy as np
import pytest

from conftest import pkg

HUMANOID = dict(traj_size=630, obs_size=55, action_size=21)


def _rodent_parent_layout(lrn, pol):
    """Offsets and size of the flat buffer as the layout was before padded row strides: (numel + 3) // 4 * 4 floats per tensor."""
    P, V = pol.param_shapes(795, 232, 30), lrn.value_param_shapes(232, (1024, 1024))
    shapes = {}
    for k in lrn._POLICY_TENSORS:
        shapes["policy/" + k] = {"encoder/heads/kernel": (128, 128), "encoder/heads/bias": (128,)}.get(k, P.get(k))
    for k in lrn.VALUE_ORDER:
        shapes["value/" + k] = V[k]
    offsets, off = {}, 0
    for k, s in shapes.items():
        offsets[k] = off
        off += (int(np.prod(s)) + 3) // 4 * 4
    return shapes, offsets, off


def test_flat_layout_keeps_the_rodent_layout():
    lrn, pol = pkg("learner"), pkg("policy")
    want_shapes, want_offsets, want_n = _rodent_parent_layout(lrn, pol)
    shapes = lrn.learner_shapes(pol.param_shapes(795, 232, 30), lrn.value_param_shapes(232, (1024, 1024)))
    assert shapes == want_shapes and list(shapes) == list(want_shapes)
    offsets, strides, n = lrn.flat_layout(shapes)
    assert offsets == want_offsets and list(offsets) == list(want_offsets) and n == want_n == 1630400
    assert all(strides[k] == s[-1] for k, s in shapes.items())  # every row stride is the width: nothing is padded


def test_flat_layout_pads_only_the_humanoid_logit_kernel():
    lrn, pol, tk = pkg("learner"), pkg("policy"), pkg("train_kernels")
    shapes = lrn.learner_shapes(pol.param_shapes(630, 55, 21), lrn.value_param_shapes(55))
    offsets, strides, n = lrn.flat_layout(shapes)
    padded = {k: strides[k] for k, s in shapes.items() if strides[k] != s[-1]}
    assert padded == {"policy/decoder/hidden_2/kernel": 44} and shapes["policy/decoder/hidden_2/kernel"] == (256, 42)
    assert shapes["value/hidden_2/kernel"] == (1024, 1) and strides["value/hidden_2/kernel"] == 1  # read by row kernels: dense
    off = 0
    for k, s in shapes.items():  # in order, 16-byte aligned, rows x stride floats each
        assert offsets[k] == off and off % 4 == 0
        off += tk.ld4(s[0] * strides[k] if len(s) == 2 else s[0])
    assert n == off
    assert [tk.ld4(w) for w in (55, 119, 42, 630, 232, 60)] == [56, 120, 44, 632, 232, 60]


@pytest.mark.parametrize("dims", [(795, 232, 30), (630, 55, 21)], ids=["rodent", "humanoid"])
def test_precise_policy_layout_is_the_learners_policy_bucket(dims, monkeypatch):
    """PrecisePolicy's flat parameter buffer has the keys, offsets and row strides of the learner's policy bucket, and its size
    n_policy (the policy is built on the CPU in one-pass TF32: laying out and packing needs no kernel)."""
    import torch
    lrn, pol = pkg("learner"), pkg("policy")
    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    shapes = pol.param_shapes(*dims)
    p = pol.PrecisePolicy(pol.init_params(np.random.default_rng(0), shapes), device="cpu", precision="tf32")
    offsets, strides, _ = lrn.flat_layout(lrn.learner_shapes(shapes, lrn.value_param_shapes(dims[1])))
    bucket = [k for k in offsets if k.startswith("policy/")]
    assert ["policy/" + k for k in p.p] == bucket and p.blob_dev.numel() == offsets["value/hidden_0/kernel"]
    for k, x in p.p.items():
        assert x.data_ptr() - p.blob_dev.data_ptr() == 4 * offsets["policy/" + k], k
        assert x.dim() == 1 or x.stride(0) == strides["policy/" + k], k


def test_learner_size_checks_keep_the_real_limits(monkeypatch):
    """Odd widths are accepted; what the kernels cannot do is refused before any device work."""
    import torch
    lrn, pol = pkg("learner"), pkg("policy")
    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)  # reach the size check without a device
    rng = np.random.default_rng(0)
    V = lrn.init_value_params(rng, lrn.value_param_shapes(55))
    for kw in (dict(latent=63), dict(decoder_layer_sizes=(128, 300))):  # odd latent (dense [mean | logvar] rows); width > 256
        P = pol.init_params(rng, pol.param_shapes(630, 55, 21, **kw))
        with pytest.raises(ValueError):
            lrn.PPOLearner(P, V, 2, 8, device="cpu")
    P = pol.init_params(rng, pol.param_shapes(630, 55, 21))
    with pytest.raises(ValueError):
        lrn.PPOLearner(P, lrn.init_value_params(rng, lrn.value_param_shapes(55, (1022, 1024))), 2, 8, device="cpu")


# ---- GEMM at the humanoid's operand shapes ------------------------------------------------------------------------------
# (name, M, N, K, a_mn, b_mn, splitk)
GEMM_CASES = [
    ("value fwd K=55", 600, 1024, 55, 0, 1, 1),
    ("decoder fwd K=119", 600, 128, 119, 0, 1, 1),
    ("logits fwd N=42", 600, 42, 256, 0, 1, 1),
    ("logits dgrad K=42", 600, 256, 42, 0, 0, 1),
    ("value wgrad M=55", 55, 1024, 640, 1, 1, 4),
    ("decoder wgrad M=119", 119, 128, 640, 1, 1, 4),
    ("logits wgrad N=42", 256, 42, 640, 1, 1, 4),
]


def _padded_operand(rows, cols, g):
    """[rows, cols] view of a [rows, ld4(cols)] buffer whose padding holds NaN: the GEMM must never read it."""
    import torch
    tk = pkg("train_kernels")
    buf = torch.full((rows, tk.ld4(cols)), float("nan"), device="cuda")
    x = buf[:, :cols]
    x.copy_(torch.randn(rows, cols, device="cuda", generator=g))
    return x


@pytest.mark.gpu
@pytest.mark.parametrize("case", GEMM_CASES, ids=[c[0] for c in GEMM_CASES])
def test_gemm_with_padded_row_strides(case):
    """Against float64 matmuls: TF32 5e-3, 3xTF32 1e-4 of the largest entry (tests/test_gemm.py).  The operands' padding columns
    hold NaN (never read), C's padding holds a sentinel (never written, split-K included)."""
    import torch
    tk = pkg("train_kernels")
    _, M, N, K, a_mn, b_mn, sk = case
    g = torch.Generator(device="cuda").manual_seed(M + 3 * N + 7 * K)
    A = _padded_operand(K, M, g) if a_mn else _padded_operand(M, K, g)
    B = _padded_operand(K, N, g) if b_mn else _padded_operand(N, K, g)
    assert A.stride(0) % 4 == 0 and B.stride(0) % 4 == 0 and (A.stride(0) != A.shape[1] or B.stride(0) != B.shape[1])
    bias = torch.randn(N, device="cuda", generator=g)
    Ad, Bd = (A.T if a_mn else A).double(), (B.T if b_mn else B).double()
    want = Ad @ Bd.T + bias.double()
    scale = float(want.abs().max())
    Cbuf = torch.full((M, tk.ld4(N)), 7.0, device="cuda")
    C = Cbuf[:, :N]
    C.fill_(-5.0)  # poisoned: every element must be written (or zeroed + added)
    tk.gemm(A, a_mn, B, b_mn, C, M, N, K, bias=bias, splitk=sk)
    torch.cuda.synchronize()
    e1 = float((C.double() - want).abs().max()) / scale
    assert e1 < 5e-3, e1
    assert bool((Cbuf[:, N:] == 7.0).all())
    # 3xTF32 (the operands are split over their padded storage, hi / lo keep the row stride) into a dense C (ldc = N, as the
    # fp32-class policy's logits)
    C3 = torch.full((M, N), -3.0, device="cuda")
    tk.gemm(A, a_mn, B, b_mn, C3, M, N, K, bias=bias, x3=True, splitk=max(sk, (K + 255) // 256))
    torch.cuda.synchronize()
    e3 = float((C3.double() - want).abs().max()) / scale
    assert e3 < 1e-4, e3
    hi, lo = tk.split(A)
    assert hi.stride() == A.stride() and lo.stride() == A.stride() and torch.equal(hi + lo, A)


# ---- the PPO update -----------------------------------------------------------------------------------------------------
T, BM = 5, 96  # 480 rows: ragged last tile


def _params(seed, enc=(256, 128), dec=(128, 256), last_scale=1.0):
    pol, lrn = pkg("policy"), pkg("learner")
    rng = np.random.default_rng(seed)
    P = pol.init_params(rng, pol.param_shapes(630, 55, 21, encoder_layer_sizes=enc, decoder_layer_sizes=dec), perturb=0.05)
    P["decoder/hidden_2/kernel"] = P["decoder/hidden_2/kernel"] * np.float32(last_scale)
    V = lrn.init_value_params(rng, lrn.value_param_shapes(55), perturb=0.05)
    return P, V


def _batch(seed, P, V, T=T, BM=BM, clip=0.3):
    """A humanoid minibatch as tests/test_learner.py builds the rodent's: actions sampled from the policy's own distribution,
    behaviour log-probs = the target's plus noise (rho on both sides of the clip range, no row within 2e-3 of a clip boundary in
    log rho), some truncations / terminations."""
    import torch
    from test_learner import keep_off_clip_edges
    lrn = pkg("learner")
    g = torch.Generator(device="cuda").manual_seed(seed)
    R, nu = T * BM, 21
    rn = lambda *s: torch.randn(*s, device="cuda", generator=g)
    traj = torch.zeros(R, 632, device="cuda")
    traj[:, :630] = 0.3 * rn(R, 630)
    batch = dict(traj=traj, observation=rn(R, 55), next_observation_last=rn(BM, 55), reward=0.05 * torch.rand(R, device="cuda", generator=g),
                 discount=(torch.rand(R, device="cuda", generator=g) > 0.1).float(),
                 truncation=(torch.rand(R, device="cuda", generator=g) > 0.93).float(), raw_action=0.7 * rn(R, nu), eps_z=rn(R, 64),
                 eps_ent=rn(R, nu), log_prob=torch.zeros(R, device="cuda"))
    mean, std = 0.1 * rn(55), 0.5 + torch.rand(55, device="cuda", generator=g)
    _, _, _, _, aux = lrn.reference_loss(P, V, batch, T, BM, mean, std)
    loc, scale = aux["logits"][:, :nu], torch.nn.functional.softplus(aux["logits"][:, nu:]) + 0.001
    batch["raw_action"] = (loc + scale * rn(R, nu).double()).float().contiguous()
    _, _, _, _, aux = lrn.reference_loss(P, V, batch, T, BM, mean, std)
    log_rho = keep_off_clip_edges(-0.25 * rn(R).double(), clip)
    batch["log_prob"] = (aux["target_lp"].reshape(-1) - log_rho).float().contiguous()
    return batch, mean, std


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / (np.abs(b).max() + 1e-30))


def _padding(L, flat):
    """The padding columns of every row-padded tensor of a flat buffer."""
    out = []
    for k, s in L.shapes.items():
        if len(s) == 2 and L.strides[k] != s[1]:
            o = L.offsets[k]
            out.append(flat[o:o + s[0] * L.strides[k]].view(s[0], L.strides[k])[:, s[1]:])
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("T_,BM_", [(T, BM), (20, 256)], ids=["480rows", "5120rows"])
@pytest.mark.parametrize("x3", [True, False], ids=["3xtf32", "tf32"])
@pytest.mark.parametrize("sizes", [((256, 128), (128, 256)), ((250, 126), (126, 250))], ids=["humanoid", "odd-hidden-widths"])
def test_humanoid_loss_and_gradients_match_autograd(sizes, x3, T_, BM_):
    """Against learner.reference_loss in float64 on the kernel's relu branches (test_learner.reference_on_kernel_branches), with
    test_learner's tolerances: 3xTF32 loss terms 1e-5, every gradient tensor 5e-4 of its largest entry; TF32 (what train() runs) loss
    2e-3, gradients 1e-1 in Frobenius norm, logits of std 0.2 and the clip range opened wide (the reasons are given there).  The second
    case also pads the hidden activations and kernels (widths 250 / 126); 5120 rows is the minibatch training runs."""
    import torch
    from test_learner import reference_on_kernel_branches
    lrn = pkg("learner")
    P, V = _params(1, *sizes, last_scale=1.0 if x3 else 0.2)
    clip = 0.3 if x3 else 1e3
    tol_loss, tol_grad, tol_fwd = (1e-5, 5e-4, 2e-5) if x3 else (2e-3, 1e-1, 5e-3)
    batch, mean, std = _batch(2, P, V, T=T_, BM=BM_, clip=clip)
    L = lrn.PPOLearner(P, V, T_, BM_, x3=x3, clipping_epsilon=clip)
    L.set_normalizer(mean, std)
    m = L.metrics_dict(L.loss_and_grads(batch))
    torch.cuda.synchronize()
    want, gP, gV, aux, flips = reference_on_kernel_branches(L, P, V, batch, T_, BM_, mean, std, x3, clip)
    assert L.ws["logits"].stride(0) == 44 and L.ws["dec_in"].stride(0) == 120 and L.ws["vin"].stride(0) == 56
    for k in ("total_loss", "policy_loss", "v_loss", "entropy_loss", "kl_loss_intention", "mean_rho"):
        assert abs(m[k] - want[k]) < tol_loss * max(1.0, abs(want[k])), (k, m[k], want[k])
    assert (0.05 < m["clip_fraction"] < 0.95) if x3 else m["clip_fraction"] == 0
    assert _rel(L.ws["logits"].cpu().numpy(), aux["logits"].cpu().numpy()) < tol_fwd
    assert _rel(L.ws["val"][:T_ * BM_].cpu().numpy(), aux["baseline"].reshape(-1).cpu().numpy()) < tol_fwd
    assert _rel(L.ws["dlogits"].cpu().numpy(), aux["dlogits"].cpu().numpy()) < tol_grad
    got_p, got_v = L.policy_grads(), L.value_grads()
    fro = lambda a, b: float(np.linalg.norm(np.asarray(a, np.float64) - np.asarray(b, np.float64)) / (np.linalg.norm(np.asarray(b, np.float64)) + 1e-30))
    err = _rel if x3 else fro
    worst = {"policy/" + k: err(got_p[k], g.cpu().numpy()) for k, g in gP.items()}
    worst.update({"value/" + k: err(got_v[k], g.cpu().numpy()) for k, g in gV.items()})
    bad = {k: v for k, v in worst.items() if v > tol_grad}
    assert not bad, bad
    assert len(worst) == 28
    print("sizes %s x3=%s rows %d: %d relu flips, worst gradient error %.2e (%s)" % (sizes, x3, T_ * BM_, flips, max(worst.values()),
                                                                                     max(worst, key=worst.get)))


@pytest.mark.gpu
def test_humanoid_updates_keep_the_padding_zero():
    """8 updates on changing batches: the padding columns of parameters, gradients and both Adam moments stay exactly 0, the
    exported trees keep the flax shapes and the parameters moved."""
    import torch
    lrn, pol = pkg("learner"), pkg("policy")
    P, V = _params(3)
    L = lrn.PPOLearner(P, V, T, BM, x3=True, learning_rate=6e-4)
    assert L.strides["policy/decoder/hidden_2/kernel"] == 44 and L.p["policy/decoder/hidden_2/kernel"].stride(0) == 44
    for step in range(8):
        batch, mean, std = _batch(20 + step, L.policy_params(), L.value_params())
        L.set_normalizer(mean, std)
        L.update(batch)
    torch.cuda.synchronize()
    assert L.updates == 8 and int(L.step_dev.item()) == 8
    for name, flat in (("params", L.params), ("grads", L.grads), ("m", L.m), ("v", L.v)):
        pads = _padding(L, flat)
        assert len(pads) == 1 and all(bool((p == 0).all()) for p in pads), name
    assert float(L.grads.abs().max()) > 0 and float(L.v.abs().max()) > 0
    want = pol.param_shapes(630, 55, 21)
    for tree in (L.policy_params(), L.policy_grads()):
        assert {k: v.shape for k, v in tree.items()} == want
        assert all(v.flags["C_CONTIGUOUS"] for v in tree.values())
    for tree in (L.value_params(), L.value_grads()):
        assert {k: v.shape for k, v in tree.items()} == lrn.value_param_shapes(55)
    assert not np.array_equal(L.policy_params()["decoder/hidden_2/kernel"], P["decoder/hidden_2/kernel"])
    assert torch.isfinite(L.params).all()


@pytest.mark.gpu
def test_precise_policy_parameters_equal_the_learners_policy_bucket():
    """After two updates, `policy.load_params(learner.policy_params())` on a policy built from other parameters leaves its flat
    parameter buffer equal to the learner's [0, n_policy) bit for bit, padding included, and its 3xTF32 splits equal to the split
    of that bucket."""
    import torch
    lrn, pol, tk = pkg("learner"), pkg("policy"), pkg("train_kernels")
    P, V = _params(4)
    L = lrn.PPOLearner(P, V, T, BM, x3=True)
    for step in range(2):
        batch, mean, std = _batch(30 + step, L.policy_params(), L.value_params())
        L.set_normalizer(mean, std)
        L.update(batch)
    p = pol.PrecisePolicy(_params(5)[0], "cuda:0")
    p.load_params(L.policy_params())
    torch.cuda.synchronize()
    bits = lambda x: x.view(torch.int32)
    bucket = L.params[:L.n_policy]
    assert p.blob_dev.shape == bucket.shape and torch.equal(bits(p.blob_dev), bits(bucket))
    for got, want in zip(p.blob_split, tk.split(bucket)):
        assert torch.equal(bits(got), bits(want))


# ---- the fp32-class rollout policy --------------------------------------------------------------------------------------
def _policy_case(B, seed):
    import torch
    pol = pkg("policy")
    params = pol.init_params(np.random.default_rng(seed), pol.param_shapes(**HUMANOID), perturb=0.1)
    g = torch.Generator().manual_seed(seed)
    mk = lambda *s: torch.randn(*s, generator=g).cuda()
    x = dict(traj=mk(B, 630), obs=mk(B, 55) * 2 + 0.5, eps_z=mk(B, 64), eps_a=mk(B, 21), rand=(torch.rand(21, generator=g) * 2 - 1).cuda())
    mean, std = mk(55) * 0.3, torch.rand(55, generator=g).cuda() + 0.5
    return params, x, mean, std


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 130, 4096])
def test_humanoid_precise_policy_in_the_learners_layout_matches_fp32_network(B):
    """3xTF32 against the float64 network: logits 3e-5, log-prob 1e-3 (tests/test_policy.py).  The logit kernel keeps its padded
    row stride in the flat parameter buffer and both split buffers, and so does the cached forward's decoder input."""
    import torch
    pol = pkg("policy")
    params, x, mean, std = _policy_case(B, 40 + B % 7)
    p = pol.PrecisePolicy(params, "cuda:0", mean, std)
    k = "decoder/hidden_2/kernel"
    assert p.p[k].stride(0) == 44 and p.splits[0][k].stride(0) == 44 and p.splits[1][k].stride(0) == 44
    act, out = p(x["traj"], x["obs"], x["eps_z"], x["eps_a"], x["rand"])
    torch.cuda.synchronize()
    assert p.bufs[B]["fwd"].ws["dec_in"].stride(0) == 120 and out["logits"].is_contiguous()
    d = lambda k: x[k].double()
    ref = pol.reference_forward(params, d("traj"), d("obs"), d("eps_z"), d("eps_a"), d("rand")[None].expand(B, -1), mean.double(), std.double())
    assert float((out["logits"].double() - ref["logits"]).abs().max()) < 3e-5 * max(1.0, float(ref["logits"].abs().max()))
    assert float((out["log_prob"].double() - ref["log_prob"]).abs().max()) < 1e-3
    assert float((act.double() - ref["action"]).abs().max()) < 3e-4 and float(act.abs().max()) <= 1.0


@pytest.mark.gpu
def test_humanoid_precise_policy_reloads_in_place_and_is_graph_capturable():
    import torch
    pol = pkg("policy")
    params, x, mean, std = _policy_case(256, 31)
    args = (x["traj"], x["obs"], x["eps_z"], x["eps_a"])
    p = pol.PrecisePolicy(params, "cuda:0", mean, std)
    out = p.alloc_outputs(256)
    p(*args, out=out)  # warm-up allocates the per-batch buffers
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        p(*args, out=out)
    g.replay()
    torch.cuda.synchronize()
    first = out["log_prob"].clone()
    assert torch.allclose(first, p(*args)[1]["log_prob"], atol=1e-4)  # split-K red.adds land in any order
    new = pol.init_params(np.random.default_rng(99), pol.param_shapes(**HUMANOID), perturb=0.1)
    ptr = p.blob_dev.data_ptr()
    p.load_params(new)
    assert p.blob_dev.data_ptr() == ptr
    g.replay()  # the captured launches read the refreshed weights and their splits
    torch.cuda.synchronize()
    want = pol.reference_forward(new, *(a.double() for a in args), None, mean.double(), std.double())["log_prob"]
    assert float((out["log_prob"].double() - want).abs().max()) < 1e-3 and not torch.allclose(out["log_prob"], first)


# ---- rollout, training step and evaluation on HumanoidTracking (the moving stand-in clip) -------------------------------
@pytest.fixture(scope="module")
def hum_env():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    model, clip = pkg("envs.humanoid").packaged_humanoid(moving=True)
    return pkg("envs").HumanoidTracking(model=model, reference_clip=clip, device="cuda:0")


RT, RB, EP = 6, 200, 4.0  # episode_length 4 < unroll: truncation + restore happen inside an unroll


def _make_policy(kind, params, mean, std):
    """kind: "bf16" (IntentionPolicy), "precise-tf32" / "precise-3xtf32" (PrecisePolicy in that precision)."""
    pol = pkg("policy")
    if kind == "bf16":
        return pol.IntentionPolicy(params, "cuda:0", mean, std)
    return pol.PrecisePolicy(params, "cuda:0", mean, std, precision=kind.split("-")[1])


def _rollout_setup(env, seed, kind):
    import torch
    pol = pkg("policy")
    s0 = env.reset(np.random.default_rng(seed), batch_size=RB)
    params = pol.init_params(np.random.default_rng(seed), pol.param_shapes(**HUMANOID), perturb=0.1)
    g = torch.Generator(device="cuda").manual_seed(seed)
    mean = torch.randn(55, device="cuda", generator=g) * 0.1
    std = torch.rand(55, device="cuda", generator=g) + 0.5
    draws = [(torch.randn(RT, RB, 64, device="cuda", generator=g), torch.randn(RT, RB, 21, device="cuda", generator=g)) for _ in range(3)]
    return s0, _make_policy(kind, params, mean, std), draws


# The bitwise comparisons need a deterministic policy: the bf16 kernel, and PrecisePolicy in its one-pass TF32 mode (no split-K).
# In 3xTF32 mode its split-K partial sums land in any order; that mode runs the rollout of the training-step tests below.
POLICY_KINDS = ["bf16", "precise-tf32"]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", POLICY_KINDS)
def test_humanoid_unroll_equals_stepwise_loop(hum_env, kind):
    import torch
    s0, policy, draws = _rollout_setup(hum_env, 71, kind)
    eng = hum_env.engine
    ro = pkg("rollout").Rollout(hum_env, policy, s0, RT, EP, use_graph=False)
    first, first_obs = dict(s0.pipeline_state), s0.obs
    st = dict({k: v.clone() for k, v in first.items()}, cur_frame=s0.info["cur_frame"].clone(), sub_clip_frame=s0.info["sub_clip_frame"].clone())
    obs, traj = s0.obs.clone(), s0.info["traj"].clone()
    steps, done = torch.zeros(RB, device="cuda"), torch.zeros(RB, device="cuda")
    seen_trunc = False
    for u in range(2):
        tr = ro.generate_unroll(*draws[u])
        torch.cuda.synchronize()
        for t in range(RT):
            act, ex = policy(traj, obs, draws[u][0][t], draws[u][1][t])
            nxt, out, trunc = eng.alloc_state(RB), eng.alloc_outputs(RB), torch.zeros(RB, device="cuda")
            eng.step_training(st, act, nxt, out, first, first_obs, steps, done, steps, trunc, EP)
            torch.cuda.synchronize()
            assert torch.equal(tr["observation"][t], obs) and torch.equal(tr["action"][t], act), (u, t)
            for k in ("log_prob", "raw_action", "logits"):
                assert torch.equal(tr["policy_extras"][k][t], ex[k]), (u, t, k)
            assert torch.equal(tr["reward"][t], out["reward"]) and torch.equal(tr["discount"][t], 1 - out["done"])
            assert torch.equal(tr["next_observation"][t], out["obs"]) and torch.equal(tr["state_extras"]["traj"][t], out["traj"])
            assert torch.equal(tr["state_extras"]["truncation"][t], trunc)
            seen_trunc = seen_trunc or bool((trunc > 0).any())
            st, obs, traj, done = nxt, out["obs"], out["traj"], out["done"].clone()
        for k, v in ro.env_state.items():
            assert torch.equal(v, st[k]), k
    assert seen_trunc and float(steps.max()) <= EP and ro.launches == 4 * RT


@pytest.mark.gpu
def test_humanoid_unroll_with_3xtf32_policy_equals_teacher_forced_loop(hum_env):
    """The training loop's rollout policy (PrecisePolicy, 3xTF32) inside the captured unroll.  Its split-K partial sums land in any
    order, so its outputs are compared within the bars of test_precise_policy_matches_fp32_network (logits 3e-5 of the largest entry,
    log-prob 1e-3) on the unroll's own inputs; the loop then steps the env with the unroll's recorded actions, so everything the
    deterministic env kernel produces is compared bit for bit."""
    import torch
    s0, policy, draws = _rollout_setup(hum_env, 74, "precise-3xtf32")
    eng = hum_env.engine
    ro = pkg("rollout").Rollout(hum_env, policy, s0, RT, EP, use_graph=True)
    first, first_obs = dict(s0.pipeline_state), s0.obs
    st = dict({k: v.clone() for k, v in first.items()}, cur_frame=s0.info["cur_frame"].clone(), sub_clip_frame=s0.info["sub_clip_frame"].clone())
    obs, traj = s0.obs.clone(), s0.info["traj"].clone()
    steps, done = torch.zeros(RB, device="cuda"), torch.zeros(RB, device="cuda")
    seen_trunc, worst = False, 0.0
    for u in range(2):
        tr = ro.generate_unroll(*draws[u])
        torch.cuda.synchronize()
        for t in range(RT):
            assert torch.equal(tr["observation"][t], obs), (u, t)
            act, ex = policy(traj, obs, draws[u][0][t], draws[u][1][t])
            torch.cuda.synchronize()
            lg = tr["policy_extras"]["logits"][t]
            assert float((ex["logits"] - lg).abs().max()) < 3e-5 * max(1.0, float(lg.abs().max())), (u, t)
            err = float((ex["log_prob"] - tr["policy_extras"]["log_prob"][t]).abs().max())
            worst = max(worst, err)
            assert err < 1e-3, (u, t, err)
            assert float((act - tr["action"][t]).abs().max()) < 3e-4, (u, t)
            nxt, out, trunc = eng.alloc_state(RB), eng.alloc_outputs(RB), torch.zeros(RB, device="cuda")
            eng.step_training(st, tr["action"][t].contiguous(), nxt, out, first, first_obs, steps, done, steps, trunc, EP)
            torch.cuda.synchronize()
            assert torch.equal(tr["reward"][t], out["reward"]) and torch.equal(tr["discount"][t], 1 - out["done"]), (u, t)
            assert torch.equal(tr["next_observation"][t], out["obs"]) and torch.equal(tr["state_extras"]["traj"][t], out["traj"]), (u, t)
            assert torch.equal(tr["state_extras"]["truncation"][t], trunc), (u, t)
            seen_trunc = seen_trunc or bool((trunc > 0).any())
            st, obs, traj, done = nxt, out["obs"], out["traj"], out["done"].clone()
        for k, v in ro.env_state.items():
            assert torch.equal(v, st[k]), k
    assert seen_trunc and float(steps.max()) <= EP
    print("3xTF32 rollout policy vs eager: worst log-prob difference %.2e" % worst)


HUM_STATE_KEYS = ("qpos", "qvel", "act", "qacc_warmstart", "xpos", "xquat", "subtree_com", "qfrc_actuator")


@pytest.mark.gpu
def test_humanoid_fused_training_wrappers_equal_brax_semantics(hum_env):
    """vnl_step_training on the humanoid == AutoResetWrapper(EpisodeWrapper(env)).step of brax (envs/wrappers/training.py) with
    action_repeat 1, restated in torch around vnl_step step by step, as test_fused_training_wrappers_equal_brax_semantics does for the
    rodent.  The humanoid has no sub-clip episode: its own done comes from the termination error and the healthy range, so a few envs
    start below healthy_z_range (done on step 1, counter restarts) and the episode length 7 truncates the others."""
    import torch
    B, K, EP_ = 64, 16, 7.0
    eng = hum_env.engine
    s0 = hum_env.reset(np.random.default_rng(41), batch_size=B)
    first, first_obs = dict(s0.pipeline_state), s0.obs
    mk = lambda: dict({k: v.clone() for k, v in first.items()}, cur_frame=s0.info["cur_frame"].clone(),
                      sub_clip_frame=s0.info["sub_clip_frame"].clone())
    ref, fus = mk(), mk()
    ref["qpos"][5::9, 2] = 0.6; fus["qpos"][5::9, 2] = 0.6  # torso below healthy_z_range (1.0, 2.0)
    z = lambda: torch.zeros(B, device="cuda")
    r_steps, r_done = z(), z()
    f_steps, f_done, f_trunc = z(), z(), z()
    rng = np.random.default_rng(42)
    seen_trunc = seen_restart = seen_env_done = False
    for it in range(K):
        a = torch.tensor(rng.uniform(-1, 1, size=(B, 21)).astype(np.float32), device="cuda")
        # --- reference: AutoResetWrapper.step { steps = where(done, 0, steps); EpisodeWrapper.step { env.step } ; restore }
        r_steps = torch.where(r_done > 0, torch.zeros_like(r_steps), r_steps)
        nxt, out = eng.alloc_state(B), eng.alloc_outputs(B)
        eng.step(ref, a, nxt, out)
        r_steps = r_steps + 1
        over = r_steps >= EP_
        trunc = torch.where(over, 1 - out["done"], torch.zeros_like(r_steps))
        done = torch.where(over, torch.ones_like(r_steps), out["done"])
        for k in HUM_STATE_KEYS:
            nxt[k] = torch.where(done.reshape((B,) + (1,) * (nxt[k].dim() - 1)) > 0, first[k], nxt[k])
        obs = torch.where(done[:, None] > 0, first_obs, out["obs"])
        ref, r_done = nxt, done
        # --- fused
        fn, fo = eng.alloc_state(B), eng.alloc_outputs(B)
        eng.step_training(fus, a, fn, fo, first, first_obs, f_steps, f_done, f_steps, f_trunc, EP_)  # steps updated in place
        torch.cuda.synchronize()
        assert torch.equal(f_steps, r_steps) and torch.equal(f_trunc, trunc) and torch.equal(fo["done"], done), it
        assert torch.equal(fo["obs"], obs) and torch.equal(fo["reward"], out["reward"]) and torch.equal(fo["traj"], out["traj"])
        assert torch.equal(fo["metrics"], out["metrics"]), it
        for k in HUM_STATE_KEYS + ("cur_frame", "sub_clip_frame"):
            assert torch.equal(fn[k], ref[k]), (it, k)
        fus, f_done = fn, fo["done"].clone()
        seen_trunc = seen_trunc or bool((trunc > 0).any())
        seen_env_done = seen_env_done or bool(((out["done"] > 0) & ~over).any())
        seen_restart = seen_restart or bool(((r_steps == 1) & (torch.tensor(it > 0, device="cuda"))).any())
    assert float(r_steps.max()) <= EP_ and seen_trunc and seen_restart and seen_env_done  # every wrapper path was exercised


@pytest.mark.gpu
@pytest.mark.parametrize("kind", POLICY_KINDS)
def test_humanoid_graph_replay_equals_eager(hum_env, kind):
    import torch
    s0, policy, draws = _rollout_setup(hum_env, 72, kind)
    eager = pkg("rollout").Rollout(hum_env, policy, s0, RT, EP, use_graph=False)
    graph = pkg("rollout").Rollout(hum_env, policy, s0, RT, EP, use_graph=True)
    for u in range(3):
        a = eager.generate_unroll(*draws[u])
        b = graph.generate_unroll(*draws[u])
        torch.cuda.synchronize()
        for k in ("observation", "next_observation", "action", "reward", "discount", "metrics"):
            assert torch.equal(a[k], b[k]), (u, k)
        for grp in ("policy_extras", "state_extras"):
            for k in a[grp]:
                assert torch.equal(a[grp][k], b[grp][k]), (u, grp, k)
        for k, v in eager.env_state.items():
            assert torch.equal(graph.env_state[k], v), (u, k)
    assert graph.graph is not None


@pytest.mark.gpu
def test_humanoid_odd_unroll_length_carries_state(hum_env):
    """An odd unroll hands the ping-pong state back to the buffer the launches read first.  The humanoid's first state has no clip
    index (single clip), so that buffer has no clip_id while the other one does."""
    import torch
    s0, policy, draws = _rollout_setup(hum_env, 73, "bf16")
    a = pkg("rollout").Rollout(hum_env, policy, s0, 3, EP, use_graph=False)
    b = pkg("rollout").Rollout(hum_env, policy, s0, 6, EP, use_graph=False)
    assert "clip_id" not in a.state[0] and "clip_id" in a.state[1]
    z, e = draws[0]
    a.generate_unroll(z[:3], e[:3])
    ta = {k: v.clone() for k, v in a.generate_unroll(z[3:], e[3:]).items() if k in ("reward", "action", "observation")}
    tb = b.generate_unroll(z, e)
    torch.cuda.synchronize()
    for k in ta:
        assert torch.equal(ta[k], tb[k][3:]), k
    for k, v in a.env_state.items():
        assert torch.equal(v, b.env_state[k]), k


def _trainer(env, B, T_, nmb, nup, graph, seed=0, x3=False, precise=True):
    pol, lrn = pkg("policy"), pkg("learner")
    s0 = env.reset(np.random.default_rng(seed), batch_size=B)
    rng = np.random.default_rng(seed)
    pp = pol.init_params(rng, pol.param_shapes(**HUMANOID), perturb=0.02)
    vp = lrn.init_value_params(rng, lrn.value_param_shapes(55))
    stats = pkg("normalizer").RunningStatistics(55)
    policy = (pol.PrecisePolicy if precise else pol.IntentionPolicy)(pp, "cuda:0", stats.mean, stats.std)
    ro = pkg("rollout").Rollout(env, policy, s0, T_, 150.0, use_graph=True)
    learner = lrn.PPOLearner(pp, vp, T_, B // nmb, x3=x3, clipping_epsilon=0.2)
    return pkg("trainer").Trainer(env, policy, learner, ro, stats, nmb, nup, use_graph=graph, seed=seed), pp


@pytest.mark.gpu
def test_humanoid_learner_reevaluates_the_rollouts_log_probs(hum_env):
    """Same parameters, normaliser and latent noise as the rollout: the learner's target log-prob (3xTF32) equals the behaviour
    log-prob PrecisePolicy wrote to 1e-3, so rho ~ 1 and nothing is clipped."""
    import torch
    B, T_ = 256, 4
    tr, _ = _trainer(hum_env, B, T_, 2, 1, graph=False, seed=3, x3=True)
    ro, L = tr.rollout, tr.learner
    g = torch.Generator(device="cuda").manual_seed(3)
    ro.eps_z.normal_(generator=g); ro.eps_a.normal_(generator=g)
    data = ro.generate_unroll()
    tr.discount_buf.copy_(data["discount"])
    data = dict(data, state_extras_traj_in=ro.traj[:T_])
    tr.idx.copy_(torch.arange(0, B, 2, device="cuda", dtype=torch.int32))
    tr._gather(data)
    tk = pkg("train_kernels")
    tk.check(tk.lib().vnl_gather_rows(ro.eps_z.data_ptr(), T_, B, L.L, tr.idx.data_ptr(), tr.Bm, tr.mb["eps_z"].data_ptr(), L.L, tk.stream(tr.idx)), "gather")
    tr.mb["eps_ent"].normal_(generator=g)
    L.set_normalizer(tr.stats.mean, tr.stats.std)
    m = L.metrics_dict(L.loss_and_grads(tr.mb))
    torch.cuda.synchronize()
    rows = (torch.arange(T_, device="cuda")[:, None] * B + tr.idx[None, :].long()).reshape(-1)
    assert torch.equal(tr.mb["observation"], data["observation"].reshape(T_ * B, -1)[rows])
    assert torch.equal(tr.mb["traj"][:, :630], ro.traj[:T_].reshape(T_ * B, -1)[rows]) and float(tr.mb["traj"][:, 630:].abs().max()) == 0
    behaviour = data["policy_extras"]["log_prob"].reshape(-1)[rows]
    diff = (L.ws["target_lp"] - behaviour).abs()
    assert float(diff.max()) < 1e-3, float(diff.max())
    assert float((L.ws["logits"] - data["policy_extras"]["logits"].reshape(T_ * B, -1)[rows]).abs().max()) < 5e-5
    assert abs(m["mean_rho"] - 1.0) < 1e-4 and m["clip_fraction"] == 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [False, True])
def test_humanoid_training_step_runs_and_updates_everything(hum_env, graph):
    import torch
    B, T_, nmb, nup = 512, 5, 4, 2
    tr, pp = _trainer(hum_env, B, T_, nmb, nup, graph=graph, seed=4)
    blob_ptr = tr.policy.blob_dev.data_ptr()
    p0 = tr.learner.params.clone()
    for _ in range(2):
        m = tr.training_step()
        torch.cuda.synchronize()
        assert all(np.isfinite(v) for v in m.values()), m
    assert tr.learner.updates == 2 * nup * nmb and int(tr.learner.step_dev.item()) == 2 * nup * nmb
    assert tr.env_steps == 2 * B * T_ and float(tr.stats.count) == 2 * B * T_
    assert float((tr.learner.params - p0).abs().max()) > 1e-4 and torch.isfinite(tr.learner.params).all()
    assert tr.policy.blob_dev.data_ptr() == blob_ptr
    new = tr.learner.policy_params()
    assert not np.array_equal(new["decoder/hidden_2/kernel"], pp["decoder/hidden_2/kernel"])
    assert all(bool((p == 0).all()) for p in _padding(tr.learner, tr.learner.params))
    if graph:
        assert tr.graph is not None


@pytest.mark.gpu
def test_humanoid_graph_replay_equals_eager_update(hum_env):
    """The bars of test_graph_replay_equals_eager_update: split-K partial sums land in any order, so gradients agree to rounding and
    Adam turns that into O(lr) differences on entries whose gradient is at rounding level.  The rollout policy is the deterministic
    bf16 kernel (as there), so that both trainers see the same unroll."""
    import torch
    B, T_ = 256, 4
    a, _ = _trainer(hum_env, B, T_, 2, 1, graph=False, seed=5, precise=False)
    b, _ = _trainer(hum_env, B, T_, 2, 1, graph=True, seed=5, precise=False)
    for tr in (a, b):
        tr.training_step()
    torch.cuda.synchronize()
    assert torch.equal(a.rollout.obs, b.rollout.obs) and torch.equal(a.rollout.log_prob, b.rollout.log_prob)
    d = (a.learner.params - b.learner.params).abs()
    assert float(torch.quantile(d[::7].float(), 0.99)) < 2e-4 and float(d.max()) < 2 * 2 * 6e-4 + 1e-6


@pytest.mark.gpu
def test_humanoid_evaluator_reports_the_humanoids_metrics(hum_env):
    """Evaluator names the episode metrics after the env: the humanoid's (no appendage term `rapp`), each the EvalWrapper fold of its
    own column of the step kernel's metrics."""
    import torch
    pol, ev, rod = pkg("policy"), pkg("evaluator"), pkg("envs.rodent")
    B, T_ = 64, 30
    names = pkg("envs.humanoid").HUMANOID_METRIC_KEYS
    assert hum_env.metric_keys == names and "rapp" not in names and len(names) == 6
    policy = pol.PrecisePolicy(pol.init_params(np.random.default_rng(7), pol.param_shapes(**HUMANOID)), "cuda:0")
    e = ev.Evaluator(hum_env, policy, num_eval_envs=B, episode_length=T_, seed=7)
    out = e.run_evaluation({})
    ro = e.rollout
    met, rew, done = (x.cpu().numpy().astype(np.float64) for x in (ro.metrics, ro.reward, ro.done))
    ep, active = np.zeros((B, met.shape[2] + 1)), np.ones(B)
    for t in range(T_):  # brax EvalWrapper.step
        ep += np.concatenate([met[t], rew[t][:, None]], 1) * active[:, None]
        active = active * (1 - done[t])
    assert np.abs(e.episode_metrics.cpu().numpy() - ep).max() < 1e-5
    episode = sorted(k for k in out if k.startswith("eval/episode_") and not k.endswith("_std"))
    assert episode == sorted("eval/episode_" + n for n in names + ("reward",)) and "eval/episode_rapp" not in out
    for n in names + ("reward",):
        i = rod.METRIC_KEYS.index(n) if n != "reward" else len(rod.METRIC_KEYS)
        assert abs(out[f"eval/episode_{n}"] - ep[:, i].mean()) < 1e-5 and abs(out[f"eval/episode_{n}_std"] - ep[:, i].std()) < 1e-5
    assert torch.isfinite(ro.action).all()
