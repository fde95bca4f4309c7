"""SURVEY 8 row f2: the PPO update.  One `minibatch_step` of the reference (ppo_imitation/train.py:251-268) on the GPU --
loss forward / backward through the intention policy network and the value MLP on the tcgen05 TF32 GEMM, Adam -- against the
torch-autograd restatement of `compute_ppo_intention_loss` (learner.reference_loss, float64).  Tolerances (written here):
  * 3xTF32 mode (the parity mode): every loss term 1e-5 absolute, every gradient tensor 1e-4 of its largest entry;
  * TF32 mode (one tensor-core pass, the reference's own GPU arithmetic): loss 2e-3, gradients 3e-2.
The gradient exchange (one SUM all-reduce + 1 / world folded into Adam = lax.pmean) is driven on CPU by a 2-rank gloo group."""
import math
import os

import numpy as np
import pytest

from conftest import pkg

T, BM = 5, 96  # 480 rows: not a multiple of 128 (ragged last tile)
TRAIN_T, TRAIN_BM = 20, 256  # 5120 rows: unroll 20 x 8192 envs / 32 minibatches, what train() and bench.py run per update


def _params(seed, perturb=0.05, last_scale=1.0):
    pol, lrn = pkg("policy"), pkg("learner")
    rng = np.random.default_rng(seed)
    P = pol.init_params(rng, pol.param_shapes(795, 232, 30), perturb=perturb)
    P["decoder/hidden_2/kernel"] = (P["decoder/hidden_2/kernel"] * np.float32(last_scale))
    V = lrn.init_value_params(rng, lrn.value_param_shapes(232), perturb=perturb)
    return P, V


def keep_off_clip_edges(log_rho, clip, margin=2e-3):
    """log rho moved at least `margin` away from log(1 +- clip): a row within rounding of a clip boundary could take the other branch
    of the clipped surrogate in the kernel and in the float64 checker, and a row that changes branch changes its whole gradient."""
    import torch
    for edge in [math.log(1 + clip)] + ([math.log(1 - clip)] if clip < 1 else []):
        d = log_rho - edge
        log_rho = torch.where(d.abs() < margin, edge + torch.where(d < 0, -margin, margin), log_rho)
    return log_rho


def _batch(seed, P, V, device="cuda", T=T, BM=BM, clip=0.3):
    """A transition minibatch with plausible statistics: behaviour log-probs from a slightly different policy (rho spread over
    both sides of the clip range, no row within 2e-3 of a clip boundary in log rho), some truncations / terminations."""
    import torch
    lrn = pkg("learner")
    g = torch.Generator(device=device).manual_seed(seed)
    R = T * BM
    rn = lambda *s: torch.randn(*s, device=device, generator=g)
    traj = torch.zeros(R, 796, device=device)
    traj[:, :795] = 0.3 * rn(R, 795)
    obs = rn(R, 232)
    batch = dict(traj=traj, observation=obs, next_observation_last=rn(BM, 232), reward=0.05 * torch.rand(R, device=device, generator=g),
                 discount=(torch.rand(R, device=device, generator=g) > 0.1).float(),
                 truncation=(torch.rand(R, device=device, generator=g) > 0.93).float(), raw_action=0.7 * rn(R, 30), eps_z=rn(R, 64), eps_ent=rn(R, 30),
                 log_prob=torch.zeros(R, device=device))
    mean, std = 0.1 * rn(232), 0.5 + torch.rand(232, device=device, generator=g)
    # actions as a rollout produces them: sampled from the policy's own distribution (raw = loc + scale * eps), so log-probs
    # are O(nu) like real PPO data (iid actions under scales of ~0.03 give log-probs of -3000 and rho at the mercy of rounding)
    _, _, _, _, aux = lrn.reference_loss(P, V, batch, T, BM, mean, std)
    nu = 30
    loc, scale = aux["logits"][:, :nu], torch.nn.functional.softplus(aux["logits"][:, nu:]) + 0.001
    batch["raw_action"] = (loc + scale * rn(R, nu).double()).float().contiguous()
    # behaviour log-prob: the target's own log-prob plus noise, so that rho = exp(-noise) straddles [1 - eps, 1 + eps]
    _, _, _, _, aux = lrn.reference_loss(P, V, batch, T, BM, mean, std)
    log_rho = keep_off_clip_edges(-0.25 * rn(R).double(), clip)
    batch["log_prob"] = (aux["target_lp"].reshape(-1) - log_rho).float().contiguous()
    return batch, mean, std


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / (np.abs(b).max() + 1e-30))


PRE = ("h0pre", "h1pre", "d0pre", "d1pre")


def reference_on_kernel_branches(L, P, V, batch, T_, BM_, mean, std, x3, clip):
    """learner.reference_loss in float64 on the kernel's own relu branches (its pre-activation signs as `relu_masks`): relu'(0) is a
    discontinuity, and at thousands of rows some pre-activations lie within the GEMM's rounding of zero, where one flipped element
    moves a bias-gradient entry by ~1 / sqrt(rows) of its size.  Asserts what makes that legitimate: every pre-activation agrees with
    float64 to the GEMM's rounding (2e-5 of the tensor's largest entry in 3xTF32, 5e-3 in TF32; a flipped element is within that of
    zero), and every row takes the same branch of the clipped surrogate in the kernel and in float64.  Returns reference_loss's
    results and the number of flipped elements."""
    import torch
    lrn = pkg("learner")
    masks = [L.ws[n] > 0 for n in PRE]
    _, want, gP, gV, aux = lrn.reference_loss(P, V, batch, T_, BM_, mean, std, clipping_epsilon=clip, relu_masks=masks)
    tol_pre = 2e-5 if x3 else 5e-3
    flips = 0
    for n, mask, ref in zip(PRE, masks, aux["pre"]):
        err = float((L.ws[n].double() - ref).abs().max())
        assert err <= tol_pre * float(ref.abs().max()), (n, err, float(ref.abs().max()))
        flips += int((mask != (ref > 0)).sum())
    rho_k = torch.exp(L.ws["target_lp"].double() - batch["log_prob"].double())
    inside = lambda r: (r >= 1 - clip) & (r <= 1 + clip)
    assert torch.equal(inside(rho_k), inside(aux["rho"].reshape(-1))), "a row changed its clip decision"
    return want, gP, gV, aux, flips


@pytest.mark.gpu
@pytest.mark.parametrize("T_,BM_", [(T, BM), (TRAIN_T, TRAIN_BM)], ids=["480rows", "5120rows"])
@pytest.mark.parametrize("x3,tol_loss,tol_grad", [(True, 1e-5, 5e-4), (False, 2e-3, 1e-1)], ids=["3xtf32", "tf32"])
def test_loss_and_gradients_match_autograd(x3, tol_loss, tol_grad, T_, BM_):
    """3xTF32: loss terms 1e-5, every gradient tensor 5e-4 of its largest entry (measured 2.8e-4 at 480 rows) (what is left is the ~5e-6
    relative error of the logits amplified by 1 / scale^2 of the tanh-normal log-prob on rows with scale ~0.03).  The float64 checker
    follows the kernel's relu branches (reference_on_kernel_branches: flips are allowed only within the GEMM's rounding of zero).
    TF32: one tensor-core pass, the arithmetic XLA uses for the reference on a GPU and the one train() runs: loss 2e-3, gradients 1e-1
    (measured 6e-2 on the encoder at 480 rows) -- with the clip range opened wide: at TF32 resolution (log-prob errors ~2e-2) a few
    rows land on the other side of rho = 1 +- eps than in float64, and a row that changes its clip decision changes its whole gradient
    (10-25 % of the largest entry of every policy tensor on this batch).  That is a property of the clipped objective at this
    precision, the reference's own GPU runs included; the clipped branch itself is covered by the 3xTF32 case.
    5120 rows (T, Bm = 20, 256) is the minibatch training runs: _wgrad's split-K and big-tile choices, and every row kernel above its
    single-pass regime (tests/test_train_kernels.py)."""
    import torch
    lrn = pkg("learner")
    # TF32 case: logits of std 0.2 (action scales 0.5 .. 0.9): with unit-variance logits the rows with scale ~0.03 carry the largest
    # gradient entries and amplify the TF32 log-prob error by 1 / scale^2 (sup-norm errors of 10-17 % on this batch)
    P, V = _params(1, last_scale=1.0 if x3 else 0.2)
    clip = 0.3 if x3 else 1e3
    batch, mean, std = _batch(2, P, V, T=T_, BM=BM_, clip=clip)
    L = lrn.PPOLearner(P, V, T_, BM_, x3=x3, clipping_epsilon=clip)
    L.set_normalizer(mean, std)
    m = L.metrics_dict(L.loss_and_grads(batch))
    torch.cuda.synchronize()
    want, gP, gV, aux, flips = reference_on_kernel_branches(L, P, V, batch, T_, BM_, mean, std, x3, clip)
    for k in ("total_loss", "policy_loss", "v_loss", "entropy_loss", "kl_loss_intention", "mean_rho"):
        assert abs(m[k] - want[k]) < tol_loss * max(1.0, abs(want[k])), (k, m[k], want[k])
    assert (0.05 < m["clip_fraction"] < 0.95) if x3 else m["clip_fraction"] == 0  # 3xTF32: both branches of the clipped surrogate
    assert _rel(L.ws["logits"].cpu().numpy(), aux["logits"].cpu().numpy()) < (2e-5 if x3 else 5e-3)
    assert _rel(L.ws["val"][:T_ * BM_].cpu().numpy(), aux["baseline"].reshape(-1).cpu().numpy()) < (2e-5 if x3 else 5e-3)
    assert _rel(L.ws["vs"].cpu().numpy(), aux["vs"].reshape(-1).cpu().numpy()) < (2e-5 if x3 else 5e-3)
    assert _rel(L.ws["dlogits"].cpu().numpy(), aux["dlogits"].cpu().numpy()) < tol_grad
    got_p, got_v = L.policy_grads(), L.value_grads()
    # 3xTF32: sup norm relative to the largest entry; TF32: Frobenius norm (single relu flips / low-scale rows move single entries
    # of a weight gradient by > 10 % of the largest one at TF32 resolution, the tensor as a whole by a few per cent)
    fro = lambda a, b: float(np.linalg.norm(np.asarray(a, np.float64) - np.asarray(b, np.float64)) / (np.linalg.norm(np.asarray(b, np.float64)) + 1e-30))
    err = _rel if x3 else fro
    worst = {}
    for k, gw in gP.items():
        worst["policy/" + k] = err(got_p[k], gw.cpu().numpy())
    for k, gw in gV.items():
        worst["value/" + k] = err(got_v[k], gw.cpu().numpy())
    bad = {k: v for k, v in worst.items() if v > tol_grad}
    assert not bad, bad
    assert len(worst) == 28
    print("x3=%s rows %d: %d relu flips, worst gradient error %.2e (%s), loss error %.2e" % (
        x3, T_ * BM_, flips, max(worst.values()), max(worst, key=worst.get), abs(m["total_loss"] - want["total_loss"])))


@pytest.mark.gpu
def test_adam_updates_match_optax_semantics():
    """Three updates on changing batches: parameters, first and second moments follow optax.adam (bias-corrected, eps outside the
    square root) to fp32 rounding of the same gradients; the device-side step counter drives the bias corrections."""
    import torch
    lrn = pkg("learner")
    P, V = _params(3)
    L = lrn.PPOLearner(P, V, T, BM, x3=True, learning_rate=6e-4)
    p = L.params.clone().double()
    m = torch.zeros_like(p)
    v = torch.zeros_like(p)
    for step in range(1, 4):
        batch, mean, std = _batch(10 + step, L.policy_params(), L.value_params())
        L.set_normalizer(mean, std)
        L.loss_and_grads(batch)
        g = L.grads.clone().double()
        L.apply_gradients()
        torch.cuda.synchronize()
        p, m, v = lrn.reference_adam(p, g, m, v, step, 6e-4)
        assert float((L.params.double() - p).abs().max()) < 2e-7
        assert float((L.m.double() - m).abs().max()) < 1e-7 * max(1.0, float(m.abs().max()))
        p = L.params.clone().double()  # fp32 state is the truth for the next step
        m, v = L.m.clone().double(), L.v.clone().double()
    assert int(L.step_dev.item()) == 3 and L.updates == 3
    # exported trees round-trip (the rollout policy re-packs from them)
    P2 = L.policy_params()
    assert set(P2) == set(P) and P2["encoder/fc2_logvar/kernel"].shape == (128, 64)
    assert not np.array_equal(P2["decoder/hidden_2/kernel"], P["decoder/hidden_2/kernel"])


@pytest.mark.gpu
def test_update_feeds_the_rollout_policy():
    """After an update the rollout policy re-packs from the learner's tree into the SAME device blob (captured graphs keep working)."""
    import torch
    lrn, pol = pkg("learner"), pkg("policy")
    P, V = _params(4)
    L = lrn.PPOLearner(P, V, T, BM)
    policy = pol.IntentionPolicy(P, "cuda:0")
    ptr = policy.blob_dev.data_ptr()
    batch, mean, std = _batch(5, P, V)
    L.set_normalizer(mean, std)
    L.update(batch)
    policy.load_params(L.policy_params())
    assert policy.blob_dev.data_ptr() == ptr
    g = torch.Generator(device="cuda").manual_seed(0)
    traj, obs = batch["traj"][:64, :795].contiguous(), batch["observation"][:64].contiguous()
    act, out = policy(traj, obs, torch.randn(64, 64, device="cuda", generator=g), torch.randn(64, 30, device="cuda", generator=g))
    torch.cuda.synchronize()
    assert torch.isfinite(act).all() and torch.isfinite(out["log_prob"]).all()


def _gloo_worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    lrn = pkg("learner")
    g = torch.Generator().manual_seed(100 + rank)
    grads = torch.randn(1000, generator=g)
    mine = grads.clone()
    scale = lrn.all_reduce_gradients(grads)
    q.put((rank, mine.numpy(), (grads * scale).numpy()))
    dist.destroy_process_group()


def test_gradient_all_reduce_is_the_mean_over_ranks_gloo():
    """world_size 2, gloo, CPU: the whole-buffer SUM all-reduce with its scale (folded into Adam) == lax.pmean."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 500
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=120) for _ in procs], key=lambda x: x[0])
    for p in procs:
        p.join(timeout=60)
    mean = 0.5 * (res[0][1] + res[1][1])
    for _, _, got in res:
        assert np.allclose(got, mean, rtol=0, atol=1e-7)


def test_value_param_shapes_and_exports():
    lrn, tk = pkg("learner"), pkg("train_kernels")
    sh = lrn.value_param_shapes(232)
    assert sh["hidden_0/kernel"] == (232, 1024) and sh["hidden_1/kernel"] == (1024, 1024) and sh["hidden_2/kernel"] == (1024, 1)
    n = sum(int(np.prod(s)) for s in sh.values())
    pol = pkg("policy")
    npol = sum(int(np.prod(s)) for s in pol.param_shapes(795, 232, 30).values())
    assert n + npol == 1630397  # the 1.63 M parameters whose gradients the reference `pmean`s (SURVEY 8d config 4: 6.5 MB)
    import re
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "vnl_train.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    assert sorted(set(re.findall(r"\b(vnl_[a-z_0-9]+)\s*\(", hdr))) == sorted(tk.TRAIN_EXPORTS)
    L = tk.lib()
    for name in tk.TRAIN_EXPORTS:
        assert getattr(L, name) is not None
