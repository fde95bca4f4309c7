"""The PPO update on the GPU (SURVEY section 8 row f2): one `minibatch_step` of the reference (ppo_imitation/train.py:251-268) =
`jax.value_and_grad(compute_ppo_intention_loss)` (ppo_imitation/intention_losses.py:91-202) over the intention policy network
(intention_policy_network.py:20-105) and the brax value MLP (ppo_networks.py:114-118: hidden (1024, 1024), swish), the gradient
`pmean` over devices (`all_reduce_gradients`: one SUM all-reduce of the whole flat gradient buffer, 1 / world applied by Adam) and
`optax.adam` (train.py:231-232).

Everything numeric runs in libvnl_b200.so (include/vnl_train.h): the dense contractions on the tensor cores
(`vnl_gemm_tf32`: tcgen05 kind::tf32, TMA tensor maps, K-major / MN-major operands so that forward, dgrad and wgrad need no
transposed copies), the rest as fp32 row kernels.  torch is device memory, streams and `torch.distributed`; there is no torch
or CPU fallback on this path.  `reference_loss` below is the torch-autograd restatement of the reference loss the tests compare
against (never the product).

Precision: `x3=False` runs one TF32 pass per product -- what XLA executes for the reference's f32 dots on an NVIDIA GPU
(jax default matmul precision); `x3=True` runs the 3xTF32 split (hi.hi + hi.lo + lo.hi, split-K chains of <= 8 K blocks because
the tensor core's accumulator truncates) and reproduces fp32 autograd to ~1e-5: the parity mode.
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import numpy as np

from . import ppo as gae_mod
from . import sharding
from . import train_kernels as tk

VALUE_ORDER = ("hidden_0/kernel", "hidden_0/bias", "hidden_1/kernel", "hidden_1/bias", "hidden_2/kernel", "hidden_2/bias")
METRIC_NAMES = ("total_loss", "policy_loss", "v_loss", "entropy_loss", "kl_loss_intention", "mean_rho", "clip_fraction")


def value_param_shapes(obs_size: int, hidden=(1024, 1024)) -> Dict[str, tuple]:
    """flax tree of brax `networks.make_value_network` (MLP layer_sizes = hidden + [1]; ppo_networks.py:114-118)."""
    sizes = [obs_size] + list(hidden) + [1]
    out = {}
    for i in range(len(sizes) - 1):
        out[f"hidden_{i}/kernel"], out[f"hidden_{i}/bias"] = (sizes[i], sizes[i + 1]), (sizes[i + 1],)
    return out


def init_value_params(rng: np.random.Generator, shapes, perturb: float = 0.0):
    """brax MLP init: lecun_uniform kernels, zero biases (`perturb` jitters the biases for tests)."""
    out = {}
    for k, s in shapes.items():
        if k.endswith("/kernel"):
            lim = math.sqrt(3.0 / s[0])
            out[k] = rng.uniform(-lim, lim, size=s).astype(np.float32)
        else:
            out[k] = (perturb * rng.standard_normal(s)).astype(np.float32)
    return out


# the two encoder heads are ONE tensor in the learner ([e2, 2 L]: mean | logvar columns), as in the rollout kernel
_POLICY_TENSORS = ("encoder/hidden_0/kernel", "encoder/hidden_0/bias", "encoder/LayerNorm_0/scale", "encoder/LayerNorm_0/bias",
                   "encoder/hidden_1/kernel", "encoder/hidden_1/bias", "encoder/LayerNorm_1/scale", "encoder/LayerNorm_1/bias",
                   "encoder/heads/kernel", "encoder/heads/bias",
                   "decoder/hidden_0/kernel", "decoder/hidden_0/bias", "decoder/LayerNorm_0/scale", "decoder/LayerNorm_0/bias",
                   "decoder/hidden_1/kernel", "decoder/hidden_1/bias", "decoder/LayerNorm_1/scale", "decoder/LayerNorm_1/bias",
                   "decoder/hidden_2/kernel", "decoder/hidden_2/bias")


def policy_widths(policy_params) -> Dict[str, int]:
    """Layer widths of the intention network, read from its flax tree."""
    traj, e1 = policy_params["encoder/hidden_0/kernel"].shape
    e2, latent = policy_params["encoder/fc2_mean/kernel"].shape
    k4, d1 = policy_params["decoder/hidden_0/kernel"].shape
    d2, nlog = policy_params["decoder/hidden_2/kernel"].shape
    return dict(traj=traj, obs=k4 - latent, latent=latent, e1=e1, e2=e2, d1=d1, d2=d2, nu=nlog // 2)


def policy_tensor_shapes(policy_shapes: Dict[str, tuple]) -> Dict[str, tuple]:
    """Shapes of _POLICY_TENSORS from the flax tree's: the two encoder heads as one [e2, 2 L] tensor."""
    e2, L = policy_shapes["encoder/fc2_mean/kernel"]
    heads = {"encoder/heads/kernel": (e2, 2 * L), "encoder/heads/bias": (2 * L,)}
    return {k: heads[k] if k in heads else tuple(policy_shapes[k]) for k in _POLICY_TENSORS}


def learner_shapes(policy_shapes: Dict[str, tuple], value_shapes: Dict[str, tuple]) -> Dict[str, tuple]:
    """Shapes of the learner's tensors in flat-buffer order: "policy/" + _POLICY_TENSORS (policy_tensor_shapes), then
    "value/" + VALUE_ORDER."""
    shapes = {"policy/" + k: s for k, s in policy_tensor_shapes(policy_shapes).items()}
    shapes.update(("value/" + k, tuple(value_shapes[k])) for k in VALUE_ORDER)
    return shapes


def flat_layout(shapes: Dict[str, tuple]):
    """(offsets, row strides, total floats) of the flat parameter buffer.  Every tensor starts 16-byte aligned; a matrix whose
    column count is not a multiple of 4 is a GEMM operand with rows of tk.ld4(cols) floats (the padding columns are never written
    and stay 0 in parameters, gradients and Adam moments).  A single-column matrix (the value head [n, 1]) is read by row kernels,
    not by TMA, and stays dense.  A 1-D tensor counts as one row."""
    offsets, strides, off = {}, {}, 0
    for k, s in shapes.items():
        ld = tk.ld4(s[1]) if len(s) == 2 and s[1] > 1 else s[-1]
        offsets[k], strides[k] = off, ld
        off += tk.ld4(s[0] * ld if len(s) == 2 else s[0])
    return offsets, strides, off


def flat_views(flat, shapes: Dict[str, tuple]) -> Dict[str, "torch.Tensor"]:
    """The tensors of a flat buffer laid out by flat_layout(shapes), as views in their shapes with the layout's row strides."""
    offsets, strides, _ = flat_layout(shapes)
    out = {}
    for k, s in shapes.items():
        o = offsets[k]
        out[k] = flat[o:o + s[0] * strides[k]].view(s[0], strides[k])[:, :s[1]] if len(s) == 2 else flat[o:o + s[0]]
    return out


def pack_policy(views: Dict[str, "torch.Tensor"], policy_params: Dict[str, np.ndarray]) -> None:
    """Copies a flax tree into the policy views (keyed by _POLICY_TENSORS), fc2_mean | fc2_logvar merged into the encoder heads."""
    import torch
    for k, x in views.items():
        a = np.concatenate([policy_params[k.replace("heads", h)] for h in ("fc2_mean", "fc2_logvar")], -1) if "/heads/" in k else policy_params[k]
        x.copy_(torch.as_tensor(np.ascontiguousarray(a, dtype=np.float32), device=x.device))


def export_policy(views: Dict[str, "torch.Tensor"]) -> Dict[str, np.ndarray]:
    """The flax tree of the policy views (keyed by _POLICY_TENSORS) on the host, the encoder heads split into fc2_mean | fc2_logvar."""
    out = {}
    for k, x in views.items():
        a = x.detach().cpu().numpy()
        if "/heads/" in k:
            L = a.shape[-1] // 2
            out[k.replace("heads", "fc2_mean")], out[k.replace("heads", "fc2_logvar")] = a[..., :L].copy(), a[..., L:].copy()
        else:
            out[k] = a.copy()
    return out


def splitk(K: int, x3: bool) -> int:
    """Split-K of a product over K: 3xTF32 accumulates in chains of <= 8 K blocks of 32 (the tensor core's accumulator truncates)."""
    return max(1, ((K + 31) // 32 + 7) // 8) if x3 else 1


class PolicyForward:
    """The intention network's forward pass over `rows` rows, for the learner's minibatch and policy.PrecisePolicy's rollout call.
    Owns the workspaces `ws` (GEMM operands with tk.ld4 row strides) and, in 3xTF32, the hi / lo copies of each GEMM's left operand."""
    LAUNCHES = 12  # normalise, 6 GEMMs (3xTF32 splits counted with their GEMM), 4 relu + LayerNorm, reparameterisation

    @staticmethod
    def check(w: Dict[str, int]) -> None:
        # the forward kernels' limits: vnl_relu_ln_fwd rows of <= 1024 floats, vnl_policy_sample <= 32 actions; the encoder heads
        # [mean | logvar] are read as dense rows of 2 latent floats by the reparameterisation kernels (latent even)
        if max(w["e1"], w["e2"], 2 * w["latent"], w["d1"], w["d2"]) > 1024 or w["nu"] > 32 or w["latent"] % 2:
            raise ValueError("layer sizes not supported by the policy forward kernels")

    def __init__(self, widths: Dict[str, int], rows: int, device, x3: bool):
        import torch
        self.check(widths)
        self.w = w = widths
        self.rows, self.x3 = int(rows), bool(x3)
        f = lambda n: torch.zeros(self.rows, n, dtype=torch.float32, device=device)
        fp = lambda n: tk.padded(self.rows, n, device)
        self.ws = dict(h0pre=fp(w["e1"]), h0=fp(w["e1"]), s0=f(2), h1pre=fp(w["e2"]), h1=fp(w["e2"]), s1=f(2), heads=f(2 * w["latent"]),
                       dec_in=fp(w["latent"] + w["obs"]), d0pre=fp(w["d1"]), d0=fp(w["d1"]), s2=f(2), d1pre=fp(w["d2"]), d1=fp(w["d2"]), s3=f(2))
        self.hilo = {}
        if self.x3:
            lhs = {k: self.ws[k] for k in ("h0", "h1", "dec_in", "d0", "d1")}
            lhs["traj"] = torch.empty(self.rows, tk.ld4(w["traj"]), dtype=torch.float32, device=device)  # the callers' traj rows
            self.hilo = {k: (tk.like(x), tk.like(x)) for k, x in lhs.items()}

    def __call__(self, P, traj, obs, mean, std, eps_z, logits, splits=None) -> None:
        """Enqueues normalise, e0, e1, heads, reparam, d0, d1, d2 (relu + LayerNorm after the hidden layers) on the current stream.
        P: parameter views keyed by _POLICY_TENSORS; traj: rows of stride tk.ld4(traj); logits [rows, 2 nu]: the output, any row
        stride; splits: (hi, lo) views of P in 3xTF32 (without them each GEMM splits its weight)."""
        L_, ws, w, R, chk, st = tk.lib(), self.ws, self.w, self.rows, tk.check, tk.stream(logits)
        ptr = lambda x: x.data_ptr()
        ld = lambda x: x.stride(0)  # every row stride comes from the tensor (padded operands: tk.ld4 of the width)
        lhs = dict(ws, traj=traj)

        def dense(src, name, out):
            x, W = lhs[src], P[name + "/kernel"]
            K, N = W.shape
            parts = None
            if self.x3:
                xs = tk.split_into(x, *self.hilo[src])
                parts = (xs, (splits[0][name + "/kernel"], splits[1][name + "/kernel"]) if splits else tk.split(W))
            tk.gemm(x, 0, W, 1, out, R, N, K, bias=P[name + "/bias"], x3=self.x3, splitk=splitk(K, self.x3), parts=parts)

        def hidden(src, net, i, pre, out, stats):  # net/hidden_i, then relu + net/LayerNorm_i
            pre, out, ln = ws[pre], ws[out], f"{net}/LayerNorm_{i}"
            dense(src, f"{net}/hidden_{i}", pre)
            chk(L_.vnl_relu_ln_fwd(ptr(pre), ld(pre), R, pre.shape[1], ptr(P[ln + "/scale"]), ptr(P[ln + "/bias"]), ptr(out), ld(out),
                                   ptr(ws[stats]), st), "relu_ln_fwd")
        dec_in = ws["dec_in"]
        chk(L_.vnl_obs_normalize(ptr(obs), ld(obs), R, w["obs"], ptr(mean), ptr(std), ptr(dec_in) + 4 * w["latent"], ld(dec_in), st), "normalize")
        hidden("traj", "encoder", 0, "h0pre", "h0", "s0")
        hidden("h0", "encoder", 1, "h1pre", "h1", "s1")
        dense("h1", "encoder/heads", ws["heads"])
        chk(L_.vnl_reparam_fwd(ptr(ws["heads"]), ptr(eps_z), R, w["latent"], ptr(dec_in), ld(dec_in), st), "reparam")
        hidden("dec_in", "decoder", 0, "d0pre", "d0", "s2")
        hidden("d0", "decoder", 1, "d1pre", "d1", "s3")
        dense("d1", "decoder/hidden_2", logits)


class PPOLearner:
    """Flat parameter / gradient / Adam buffers + the workspaces of one minibatch shape (T x Bm rows).

    `loss_and_grads(batch)` -> metrics; `apply_gradients(scale)` = Adam; `update(batch)` = loss_and_grads, all_reduce_gradients
    (if a process group exists), apply_gradients.  `policy_params()` / `value_params()` export the flax trees (the rollout policy
    re-packs from them)."""

    @staticmethod
    def check(widths: Dict[str, int], value_hidden) -> None:
        # the backward kernels' limits (PolicyForward checks the forward's): any policy width up to 256 (tk.ld4 row strides), value
        # hidden widths multiples of 4 (the swish passes are elementwise over dense rows)
        if max(widths["e1"], widths["e2"], widths["d1"], widths["d2"]) > 256 or any(v % 4 for v in value_hidden):
            raise ValueError("layer sizes not supported by the update kernels")

    def __init__(self, policy_params: Dict[str, np.ndarray], value_params: Dict[str, np.ndarray], T: int, Bm: int, device: str = "cuda:0",
                 learning_rate: float = 6e-4, entropy_cost: float = 1e-4, discounting: float = 0.9, reward_scaling: float = 1.0,
                 gae_lambda: float = 0.95, clipping_epsilon: float = 0.3, normalize_advantage: bool = True, kl_weight: float = 1e-4,
                 x3: bool = False, adam_b1: float = 0.9, adam_b2: float = 0.999, adam_eps: float = 1e-8):
        import torch

        if not torch.cuda.is_available():
            raise RuntimeError("vnl_b200 learner needs a CUDA device (sm_100a); there is no CPU fallback")
        self.torch = t = torch
        self.device = dev = t.device(device)
        self.T, self.Bm, self.R = int(T), int(Bm), int(T) * int(Bm)
        self.hp = dict(learning_rate=learning_rate, entropy_cost=entropy_cost, discounting=discounting, reward_scaling=reward_scaling,
                       gae_lambda=gae_lambda, clipping_epsilon=clipping_epsilon, normalize_advantage=normalize_advantage, kl_weight=kl_weight,
                       b1=adam_b1, b2=adam_b2, eps=adam_eps)
        self.x3 = bool(x3)
        self.widths = w = policy_widths(policy_params)
        self.traj, self.obs, self.L, self.nu = w["traj"], w["obs"], w["latent"], w["nu"]
        e1, e2, d1, d2 = w["e1"], w["e2"], w["d1"], w["d2"]
        self.vh = [value_params["hidden_0/kernel"].shape[1], value_params["hidden_1/kernel"].shape[1]]
        self.check(w, self.vh)
        self.fwd = PolicyForward(w, self.R, dev, self.x3)
        # ---- flat buffers -------------------------------------------------------------------------------------------------
        shapes = learner_shapes({k: v.shape for k, v in policy_params.items()}, {k: v.shape for k, v in value_params.items()})
        self.shapes = shapes
        self.offsets, self.strides, off = flat_layout(shapes)
        self.nparams = off
        self.n_policy = self.offsets["value/hidden_0/kernel"]  # the policy tensors = [0, n_policy)
        z = lambda n, dt=t.float32: t.zeros(n, dtype=dt, device=dev)
        self.params, self.grads, self.m, self.v = z(off), z(off), z(off), z(off)
        self.step_dev, self.bc_dev = z(1, t.int32), z(2)
        self.p, self.g = flat_views(self.params, shapes), flat_views(self.grads, shapes)
        self.pp, self.gp = ({k: views["policy/" + k] for k in _POLICY_TENSORS} for views in (self.p, self.g))  # keyed as the policy's
        self.load_params(policy_params, value_params)
        # ---- workspaces of one minibatch ---------------------------------------------------------------------------------
        R, Bm, L, nu = self.R, self.Bm, self.L, self.nu
        f = lambda *s: t.zeros(*s, dtype=t.float32, device=dev)
        fp = lambda rows, n: tk.padded(rows, n, dev)  # TMA operands of any width (row stride tk.ld4(n))
        self.ld_traj = tk.ld4(self.traj)
        self.ws = dict(
            self.fwd.ws, logits=fp(R, 2 * nu),
            vin=fp(R + Bm, self.obs), v0pre=f(R + Bm, self.vh[0]), v0=f(R + Bm, self.vh[0]), v1pre=f(R + Bm, self.vh[1]), v1=f(R + Bm, self.vh[1]),
            val=f(R + Bm), target_lp=f(R), ent=f(R), termination=f(R), rewards_s=f(R), vs=f(R), adv=f(R),
            dlogits=fp(R, 2 * nu), dval=f(R), dd1=fp(R, d2), dd1pre=fp(R, d2), dd0=fp(R, d1), dd0pre=fp(R, d1), ddec_in=fp(R, L + self.obs),
            dheads=f(R, 2 * L), dh1=fp(R, e2), dh1pre=fp(R, e2), dh0=fp(R, e1), dh0pre=fp(R, e1),
            dv1pre=f(R, self.vh[1]), dv0=f(R, self.vh[0]), dv0pre=f(R, self.vh[0]),
            metrics=f(8), scratch2=f(2))
        self.obs_mean, self.obs_std = f(self.obs), t.ones(self.obs, dtype=t.float32, device=dev)
        self.updates = 0
        self.launches = 0
        self.branch = t.cuda.Stream(device=dev)  # the value network's forward / backward, beside the policy's
        self.leaf_p, self.leaf_v = t.cuda.Stream(device=dev), t.cuda.Stream(device=dev)  # weight / bias gradients: leaves of the backward chains
        self._gae = gae_mod._bind(tk.lib())

    # ---- parameters -----------------------------------------------------------------------------------------------------
    @staticmethod
    def _value(views) -> Dict[str, np.ndarray]:
        return {k: views["value/" + k].detach().cpu().numpy().copy() for k in VALUE_ORDER}

    def load_params(self, policy_params, value_params) -> None:
        pack_policy(self.pp, policy_params)
        for k in VALUE_ORDER:
            self.p["value/" + k].copy_(self.torch.as_tensor(np.ascontiguousarray(value_params[k], dtype=np.float32), device=self.device))

    def set_normalizer(self, mean, std) -> None:
        self.obs_mean.copy_(self.torch.as_tensor(mean, dtype=self.torch.float32))
        self.obs_std.copy_(self.torch.as_tensor(std, dtype=self.torch.float32))

    def policy_params(self):
        return export_policy(self.pp)

    def value_params(self):
        return self._value(self.p)

    def policy_grads(self):
        return export_policy(self.gp)

    def value_grads(self):
        return self._value(self.g)

    # ---- checkpoint ------------------------------------------------------------------------------------------------------------
    STATE_KEYS = ("params", "m", "v", "step_dev", "bc_dev")

    def state_dict(self) -> Dict[str, np.ndarray]:
        """The optimiser state on the host: the flat params and Adam moments (padding included) and the device step counter /
        bias corrections."""
        return {k: getattr(self, k).detach().cpu().numpy().copy() for k in self.STATE_KEYS}

    def load_state_dict(self, sd) -> None:
        """Copies into the existing buffers (captured SGD graphs keep their addresses)."""
        for k in self.STATE_KEYS:
            x, a = getattr(self, k), np.asarray(sd[k])
            if tuple(a.shape) != tuple(x.shape) or a.dtype != np.dtype(str(x.dtype).replace("torch.", "")):
                raise ValueError(f"learner state {k}: {a.dtype}{tuple(a.shape)} does not match this learner's {x.dtype}{tuple(x.shape)}")
            x.copy_(self.torch.from_numpy(np.ascontiguousarray(a)))

    # ---- the three products of a dense layer -------------------------------------------------------------------------------
    def _fwd(self, x, rows, W, b, out, act):  # out[rows, out] = x[rows, in] . W[in, out] + b;  act = swish(out) from the same epilogue
        K, N = W.shape
        sk = splitk(K, self.x3)
        fused = sk <= 1 and N % 32 == 0
        tk.gemm(x, 0, W, 1, out, rows, N, K, bias=b, x3=self.x3, splitk=sk, epilogue=1 if fused else 0, aux=act if fused else None)
        self.launches += 1
        if not fused:
            tk.check(tk.lib().vnl_swish_fwd(out.data_ptr(), rows * N, act.data_ptr(), tk.stream(out)), "swish")
            self.launches += 1

    def _dgrad(self, dy, rows, W, out, pre=None, tmp=None):  # out[rows, in] = dy[rows, out] . W[in, out]^T  (* swish'(pre) in the epilogue)
        N, K = W.shape
        sk = splitk(K, self.x3)
        if pre is None:
            tk.gemm(dy, 0, W, 0, out, rows, N, K, x3=self.x3, splitk=sk)
        elif sk <= 1 and N % 32 == 0:
            tk.gemm(dy, 0, W, 0, out, rows, N, K, x3=self.x3, splitk=sk, epilogue=2, aux=pre)
        else:
            tk.gemm(dy, 0, W, 0, tmp, rows, N, K, x3=self.x3, splitk=sk)
            tk.check(tk.lib().vnl_swish_bwd(tmp.data_ptr(), pre.data_ptr(), rows * N, out.data_ptr(), tk.stream(out)), "swish_bwd")
            self.launches += 1
        self.launches += 1

    def _wgrad(self, x, dy, rows, gW):  # gW[in, out] = x[rows, in]^T . dy[rows, out]
        M, N = gW.shape
        tiles = ((M + 127) // 128) * ((N + (127 if N > 64 else 63)) // (128 if N > 64 else 64))
        kb = (rows + 31) // 32
        sk = max(splitk(rows, self.x3), min(max(1, 148 // tiles), max(1, kb // 4)))
        if N % 256 == 0 and M >= 256:  # 256 x 256 tiles (vnl_gemm.cu picks them when tiles x splits still fill the machine)
            tb = ((M + 255) // 256) * (N // 256)
            skb = min(max(1, 148 // tb), max(1, kb // 4))
            if tb * skb >= 96:
                sk = max(splitk(rows, self.x3), skb)
        tk.gemm(x, 1, dy, 1, gW, M, N, rows, x3=self.x3, splitk=sk, zero=False)  # self.grads was zeroed at the top of the evaluation
        self.launches += 1

    # ---- one loss + gradient evaluation ------------------------------------------------------------------------------------
    def loss_and_grads(self, batch: Dict[str, "torch.Tensor"]):
        """batch (time-major, contiguous fp32 CUDA tensors, R = T * Bm rows):
        traj [R, ld_traj] (row stride padded to a multiple of 4: vnl_gather_rows does it), observation [R, obs],
        next_observation_last [Bm, obs], reward / discount / truncation / log_prob [R], raw_action [R, nu],
        eps_z [R, L] (the encoder's reparameterisation noise, `policy_rng`), eps_ent [R, nu] (the entropy sample, `rng`).
        Returns the metrics tensor (device; names in METRIC_NAMES); gradients are left in self.grads."""
        t, L_, ws, p, g, R, Bm, nu = self.torch, tk.lib(), self.ws, self.p, self.g, self.R, self.Bm, self.nu
        st = tk.stream(self.params)
        hp = self.hp
        P = lambda k: p["policy/" + k]
        G = lambda k: g["policy/" + k]
        chk = tk.check
        ptr = lambda x: x.data_ptr()
        self.grads.zero_()
        ws["metrics"].zero_()
        traj, obs = batch["traj"], batch["observation"]
        assert traj.shape == (R, self.ld_traj) and obs.shape == (R, self.obs) and traj.is_contiguous() and obs.is_contiguous()
        # ---- forward: policy --------------------------------------------------------------------------------------------
        # The two networks are independent up to the loss rows and again after them: the value network runs on `self.branch`
        # (fork / join by stream events, which a CUDA-graph capture records as two parallel chains), so the policy's small,
        # latency-bound GEMMs (40-80 CTAs each) fill the SMs the value GEMMs leave idle between their waves.
        main = t.cuda.current_stream(self.device)
        V = lambda k: p["value/" + k]
        GV = lambda k: g["value/" + k]
        RB = R + Bm
        ld = lambda x: x.stride(0)  # every row stride comes from the tensor (padded operands: tk.ld4 of the width)
        nxt, vin, dec_in = batch["next_observation_last"], ws["vin"], ws["dec_in"]
        self.branch.wait_stream(main)
        with t.cuda.stream(self.branch):
            sb = tk.stream(self.params)
            chk(L_.vnl_obs_normalize(ptr(obs), ld(obs), R, self.obs, ptr(self.obs_mean), ptr(self.obs_std), ptr(vin), ld(vin), sb), "normalize")
            chk(L_.vnl_obs_normalize(ptr(nxt), ld(nxt), Bm, self.obs, ptr(self.obs_mean), ptr(self.obs_std), ptr(vin) + 4 * R * ld(vin), ld(vin), sb),
                "normalize")
            # value forward (baseline rows + the Bm bootstrap rows in one pass)
            self._fwd(vin, RB, V("hidden_0/kernel"), V("hidden_0/bias"), ws["v0pre"], act=ws["v0"])  # swish in the GEMM epilogue
            self._fwd(ws["v0"], RB, V("hidden_1/kernel"), V("hidden_1/bias"), ws["v1pre"], act=ws["v1"])
            chk(L_.vnl_rowdot(ptr(ws["v1"]), ld(ws["v1"]), RB, self.vh[1], ptr(V("hidden_2/kernel")), ptr(V("hidden_2/bias")), ptr(ws["val"]), sb), "rowdot")
        self.fwd(self.pp, traj, obs, self.obs_mean, self.obs_std, batch["eps_z"], ws["logits"])
        self.launches += PolicyForward.LAUNCHES
        # ---- loss -------------------------------------------------------------------------------------------------------------
        chk(L_.vnl_ppo_rows(ptr(ws["logits"]), ld(ws["logits"]), ptr(batch["raw_action"]), ptr(batch["eps_ent"]), R, nu, ptr(batch["discount"]),
                            ptr(batch["truncation"]), ptr(batch["reward"]), float(hp["reward_scaling"]), ptr(ws["target_lp"]), ptr(ws["ent"]),
                            ptr(ws["termination"]), ptr(ws["rewards_s"]), st), "ppo_rows")
        main.wait_stream(self.branch)  # join: GAE needs the values
        chk(self._gae.vnl_gae(self.T, Bm, ptr(batch["truncation"]), ptr(ws["termination"]), ptr(ws["rewards_s"]), ptr(ws["val"]), ptr(ws["val"]) + 4 * R,
                         float(hp["gae_lambda"]), float(hp["discounting"]), ptr(ws["vs"]), ptr(ws["adv"]), st), "gae")
        chk(L_.vnl_ppo_loss_bwd(ptr(ws["logits"]), ld(ws["logits"]), ptr(batch["raw_action"]), ptr(batch["eps_ent"]), R, nu, ptr(ws["target_lp"]),
                                ptr(batch["log_prob"]), ptr(ws["ent"]), ptr(ws["adv"]), ptr(ws["vs"]), ptr(ws["val"]), float(hp["clipping_epsilon"]),
                                float(hp["entropy_cost"]), int(bool(hp["normalize_advantage"])), ptr(ws["dlogits"]), ld(ws["dlogits"]), ptr(ws["dval"]),
                                ptr(ws["metrics"]), ptr(ws["scratch2"]), st), "ppo_loss_bwd")
        self.launches += 7  # row kernels of the value forward and the loss, and the zeroing (GEMMs and the policy forward count themselves)
        colsum = lambda x, n, out, w=None: chk(L_.vnl_colsum(ptr(x), ld(x) if x.dim() == 2 else n, R, n, None if w is None else ptr(w), ptr(out),
                                                             tk.stream(self.params)), "colsum")
        # ---- backward ------------------------------------------------------------------------------------------------------------
        # Each network's backward is a serial CHAIN (dgrad -> activation backward -> dgrad ...) with LEAVES hanging off it (the weight
        # and bias gradients of every layer, which nothing downstream reads).  Chains run on `main` (policy) and `self.branch`
        # (value); leaves go to `leaf_p` / `leaf_v` as soon as their operand exists, so a chain never queues behind a leaf.
        def leaf(stream, after, fn):
            stream.wait_stream(after)
            with t.cuda.stream(stream):
                fn()

        # value (only the R baseline rows carry gradient; the bootstrap rows feed the stop-gradient GAE)
        self.branch.wait_stream(main)

        def value_head_leaves():
            sl = tk.stream(self.params)
            chk(L_.vnl_colsum(ptr(ws["v1"]), ld(ws["v1"]), R, self.vh[1], ptr(ws["dval"]), ptr(GV("hidden_2/kernel")), sl), "colsum")
            chk(L_.vnl_colsum(ptr(ws["dval"]), 1, R, 1, None, ptr(GV("hidden_2/bias")), sl), "colsum")
        leaf(self.leaf_v, main, value_head_leaves)
        with t.cuda.stream(self.branch):
            sb = tk.stream(self.params)
            chk(L_.vnl_outer_swish_bwd(ptr(ws["dval"]), R, ptr(V("hidden_2/kernel")), self.vh[1], ptr(ws["v1pre"]), ptr(ws["dv1pre"]), sb), "outer_swish_bwd")
        leaf(self.leaf_v, self.branch, lambda: (self._wgrad(ws["v0"], ws["dv1pre"], R, GV("hidden_1/kernel")),
                                                colsum(ws["dv1pre"], self.vh[1], GV("hidden_1/bias"))))
        with t.cuda.stream(self.branch):
            self._dgrad(ws["dv1pre"], R, V("hidden_1/kernel"), ws["dv0pre"], pre=ws["v0pre"], tmp=ws["dv0"])  # swish' in the GEMM epilogue
            self._wgrad(vin, ws["dv0pre"], R, GV("hidden_0/kernel"))
            colsum(ws["dv0pre"], self.vh[0], GV("hidden_0/bias"))

        # policy
        def relu_ln_bwd(dy, pre, stats, name, dpre, dense):  # also leaves the bias gradient of the dense layer in front (column sums of dpre)
            n = pre.shape[1]
            chk(L_.vnl_relu_ln_bwd(ptr(dy), ld(dy), ptr(pre), ld(pre), ptr(stats), ptr(P(name + "/scale")), R, n, ptr(dpre), ld(dpre), ptr(G(name + "/scale")),
                                   ptr(G(name + "/bias")), ptr(G(dense + "/bias")), st), "relu_ln_bwd")
        lp = lambda fn: leaf(self.leaf_p, main, fn)
        lp(lambda: (self._wgrad(ws["d1"], ws["dlogits"], R, G("decoder/hidden_2/kernel")), colsum(ws["dlogits"], 2 * nu, G("decoder/hidden_2/bias"))))
        self._dgrad(ws["dlogits"], R, P("decoder/hidden_2/kernel"), ws["dd1"])
        relu_ln_bwd(ws["dd1"], ws["d1pre"], ws["s3"], "decoder/LayerNorm_1", ws["dd1pre"], "decoder/hidden_1")
        lp(lambda: self._wgrad(ws["d0"], ws["dd1pre"], R, G("decoder/hidden_1/kernel")))
        self._dgrad(ws["dd1pre"], R, P("decoder/hidden_1/kernel"), ws["dd0"])
        relu_ln_bwd(ws["dd0"], ws["d0pre"], ws["s2"], "decoder/LayerNorm_0", ws["dd0pre"], "decoder/hidden_0")
        lp(lambda: self._wgrad(dec_in, ws["dd0pre"], R, G("decoder/hidden_0/kernel")))
        self._dgrad(ws["dd0pre"], R, P("decoder/hidden_0/kernel"), ws["ddec_in"])
        kl_coef = float(hp["kl_weight"]) / float(R * self.L)
        chk(L_.vnl_heads_bwd(ptr(ws["ddec_in"]), ld(ws["ddec_in"]), ptr(ws["heads"]), ptr(batch["eps_z"]), R, self.L, kl_coef, ptr(ws["dheads"]),
                             ptr(ws["metrics"]) + 16, st), "heads_bwd")
        lp(lambda: (self._wgrad(ws["h1"], ws["dheads"], R, G("encoder/heads/kernel")), colsum(ws["dheads"], 2 * self.L, G("encoder/heads/bias"))))
        self._dgrad(ws["dheads"], R, P("encoder/heads/kernel"), ws["dh1"])
        relu_ln_bwd(ws["dh1"], ws["h1pre"], ws["s1"], "encoder/LayerNorm_1", ws["dh1pre"], "encoder/hidden_1")
        lp(lambda: self._wgrad(ws["h0"], ws["dh1pre"], R, G("encoder/hidden_1/kernel")))
        self._dgrad(ws["dh1pre"], R, P("encoder/hidden_1/kernel"), ws["dh0"])
        relu_ln_bwd(ws["dh0"], ws["h0pre"], ws["s0"], "encoder/LayerNorm_0", ws["dh0pre"], "encoder/hidden_0")
        self._wgrad(traj, ws["dh0pre"], R, G("encoder/hidden_0/kernel"))
        main.wait_stream(self.leaf_p)  # join: all gradients are in self.grads
        main.wait_stream(self.branch)
        main.wait_stream(self.leaf_v)
        self.launches += 12  # row kernels of the backward pass
        return ws["metrics"]

    # ---- optimiser -------------------------------------------------------------------------------------------------------------
    def apply_gradients(self, scale: float = 1.0):
        """optax.adam on the flat buffers, the gradients multiplied by `scale` (1 / world after all_reduce_gradients: the mean over
        ranks folded into Adam)."""
        L_ = tk.lib()
        st = tk.stream(self.params)
        hp = self.hp
        tk.check(L_.vnl_adam_tick(self.step_dev.data_ptr(), float(hp["b1"]), float(hp["b2"]), self.bc_dev.data_ptr(), st), "adam_tick")
        tk.check(L_.vnl_adam(self.params.data_ptr(), self.grads.data_ptr(), self.m.data_ptr(), self.v.data_ptr(), self.nparams, float(hp["learning_rate"]),
                             float(hp["b1"]), float(hp["b2"]), float(hp["eps"]), 0, float(scale), self.bc_dev.data_ptr(), st), "adam")
        self.updates += 1
        self.launches += 2

    def update(self, batch):
        m = self.loss_and_grads(batch)
        self.apply_gradients(all_reduce_gradients(self.grads))
        return m

    def metrics_dict(self, m=None) -> Dict[str, float]:
        a = (self.ws["metrics"] if m is None else m).detach().cpu().numpy()
        out = {k: float(a[i]) for i, k in enumerate(METRIC_NAMES)}
        out["total_loss"] = float(a[0] + a[4])  # the KL term is accumulated by its own kernel
        return out


# -------------------------------------------------------------------------------------------------------------------------------
# gradient exchange (device-agnostic: the 2-rank gloo test on CPU drives it on a CPU tensor)
# -------------------------------------------------------------------------------------------------------------------------------
def all_reduce_gradients(grads) -> float:
    """`lax.pmean` of the gradients (gradients.gradient_update_fn with pmap_axis_name, ppo_imitation/train.py:251): one in-place
    SUM all-reduce of the whole flat buffer over the process group.  Returns the factor that turns the SUMs into the mean, which
    Adam applies (vnl_adam grad_scale): 1 / world, or 1.0 without a group (nothing is exchanged)."""
    dist = sharding.group()
    if dist is None:
        return 1.0
    dist.all_reduce(grads, op=dist.ReduceOp.SUM)
    return 1.0 / dist.get_world_size()


# -------------------------------------------------------------------------------------------------------------------------------
# checker: torch-autograd restatement of the reference loss (tests / tools only)
# -------------------------------------------------------------------------------------------------------------------------------
def reference_loss(policy_params, value_params, batch, T: int, Bm: int, obs_mean, obs_std, *, entropy_cost=1e-4, discounting=0.9,
                   reward_scaling=1.0, gae_lambda=0.95, clipping_epsilon=0.3, normalize_advantage=True, kl_weight=1e-4, dtype=None,
                   relu_masks=None):
    """`compute_ppo_intention_loss` (ppo_imitation/intention_losses.py:91-202) restated in torch with autograd, line by line:
    policy_apply (intention_policy_network.py:82-105 with the reparameterisation noise `eps_z`), value_apply (brax MLP, swish),
    NormalTanhDistribution.log_prob / entropy (sample from `eps_ent`), compute_gae (:26-89, stop-gradient), advantage
    normalisation, clipped surrogate, v_loss * 0.5 * 0.5, entropy_cost, kl_weight * kl_divergence.
    relu_masks: optional [h0pre, h1pre, d0pre, d1pre] sign masks (pre-activation > 0) of another evaluation, the kernels' own: relu(x)
    becomes x * mask, so that an element whose pre-activation lies within rounding of zero takes the same branch in both.
    Returns (total, metrics dict, policy grads dict, value grads dict) with parameters as leaf tensors."""
    import torch

    dtype = dtype or torch.float64
    dev = batch["observation"].device
    Pp = {k: torch.as_tensor(v, dtype=dtype, device=dev).clone().requires_grad_(True) for k, v in policy_params.items()}
    Vp = {k: torch.as_tensor(v, dtype=dtype, device=dev).clone().requires_grad_(True) for k, v in value_params.items()}
    R = T * Bm
    c = lambda x: x.to(dtype)
    mean, std = c(torch.as_tensor(obs_mean, device=dev)), c(torch.as_tensor(obs_std, device=dev))
    traj = c(batch["traj"])[:, :Pp["encoder/hidden_0/kernel"].shape[0]]
    obs_n = (c(batch["observation"]) - mean) / std
    nobs_n = (c(batch["next_observation_last"]) - mean) / std

    def ln(x, name):
        m = x.mean(-1, keepdim=True)
        var = torch.clamp((x * x).mean(-1, keepdim=True) - m * m, min=0.0)
        return (x - m) * torch.rsqrt(var + 1e-6) * Pp[name + "/scale"] + Pp[name + "/bias"]
    dense = lambda x, name: x @ Pp[name + "/kernel"] + Pp[name + "/bias"]
    relu = lambda x: torch.relu(x) if relu_masks is None else x * c(relu_masks[len(pres) - 1])
    h = traj
    pres = []
    for i in range(2):
        pres.append(dense(h, f"encoder/hidden_{i}"))
        h = ln(relu(pres[-1]), f"encoder/LayerNorm_{i}")
    zm, zlv = dense(h, "encoder/fc2_mean"), dense(h, "encoder/fc2_logvar")
    z = zm + c(batch["eps_z"]) * torch.exp(0.5 * zlv)
    h = torch.cat([z, obs_n], -1)
    for i in range(2):
        pres.append(dense(h, f"decoder/hidden_{i}"))
        h = ln(relu(pres[-1]), f"decoder/LayerNorm_{i}")
    logits = dense(h, "decoder/hidden_2")
    logits.retain_grad()

    def value(x):
        nl = len(Vp) // 2
        for i in range(nl):
            x = x @ Vp[f"hidden_{i}/kernel"] + Vp[f"hidden_{i}/bias"]
            if i < nl - 1:
                x = x * torch.sigmoid(x)
        return x.squeeze(-1)
    baseline = value(obs_n).reshape(T, Bm)
    baseline.retain_grad()
    bootstrap = value(nobs_n)
    tm = lambda k: c(batch[k]).reshape(T, Bm)
    rewards = tm("reward") * reward_scaling
    truncation = tm("truncation")
    termination = (1 - tm("discount")) * (1 - truncation)
    nu = logits.shape[-1] // 2
    loc, scale = logits[..., :nu], torch.nn.functional.softplus(logits[..., nu:]) + 0.001
    ldj = lambda x: 2.0 * (math.log(2.0) - x - torch.nn.functional.softplus(-2.0 * x))
    raw = c(batch["raw_action"])
    target_lp = (-0.5 * ((raw - loc) / scale) ** 2 - torch.log(scale) - 0.5 * math.log(2 * math.pi) - ldj(raw)).sum(-1).reshape(T, Bm)
    behaviour_lp = tm("log_prob")
    # compute_gae (stop-gradient)
    with torch.no_grad():
        vals = baseline.detach()
        tmask = 1 - truncation
        v_tp1 = torch.cat([vals[1:], bootstrap.detach()[None]], 0)
        deltas = (rewards + discounting * (1 - termination) * v_tp1 - vals) * tmask
        acc = torch.zeros_like(bootstrap)
        out = []
        for t_ in range(T - 1, -1, -1):
            acc = deltas[t_] + discounting * (1 - termination[t_]) * tmask[t_] * gae_lambda * acc
            out.append(acc)
        vs = torch.stack(out[::-1]) + vals
        vs_tp1 = torch.cat([vs[1:], bootstrap.detach()[None]], 0)
        adv = (rewards + discounting * (1 - termination) * vs_tp1 - vals) * tmask
        if normalize_advantage:
            adv = (adv - adv.mean()) / (adv.std(unbiased=False) + 1e-8)
    rho = torch.exp(target_lp - behaviour_lp)
    policy_loss = -torch.minimum(rho * adv, torch.clamp(rho, 1 - clipping_epsilon, 1 + clipping_epsilon) * adv).mean()
    v_loss = ((vs - baseline) ** 2).mean() * 0.5 * 0.5
    ent = (0.5 + 0.5 * math.log(2 * math.pi) + torch.log(scale) + ldj(loc + scale * c(batch["eps_ent"]))).sum(-1)
    entropy_loss = entropy_cost * -ent.mean()
    kl = kl_weight * (-0.5 * torch.mean(1 + zlv - zm ** 2 - torch.exp(zlv)))
    total = policy_loss + v_loss + entropy_loss + kl
    total.backward()
    f_ = lambda x: float(x.detach())
    metrics = dict(total_loss=f_(total), policy_loss=f_(policy_loss), v_loss=f_(v_loss), entropy_loss=f_(entropy_loss),
                   kl_loss_intention=f_(kl), mean_rho=f_(rho.mean()))
    aux = dict(logits=logits.detach(), baseline=baseline.detach(), vs=vs, adv=adv, target_lp=target_lp.detach(), dlogits=logits.grad,
               dbaseline=baseline.grad, rho=rho.detach(), pre=[x.detach() for x in pres])
    return total, metrics, {k: v.grad for k, v in Pp.items()}, {k: v.grad for k, v in Vp.items()}, aux


def reference_adam(p, g, m, v, step, lr, b1=0.9, b2=0.999, eps=1e-8):
    """optax.adam update restated (scale_by_adam + scale(-lr)); returns (p', m', v')."""
    m2, v2 = b1 * m + (1 - b1) * g, b2 * v + (1 - b2) * g * g
    return p - lr * (m2 / (1 - b1 ** step)) / ((v2 / (1 - b2 ** step)) ** 0.5 + eps), m2, v2
