"""Host side of the intention-network policy forward (SURVEY section 8 row f1; C ABI in include/vnl_policy.h).

Mirrors the reference's rollout policy (ppo_imitation/ppo_networks.py:45-83 `make_inference_fn(...).policy` over
ppo_imitation/intention_policy_network.py:20-105): same parameter tree (flax names), same call shape
`policy(traj, obs, key) -> (action, extras{log_prob, rand_log_prob, raw_action, logits})`, the random draws passed as
operands instead of a PRNG key.  The arithmetic runs in libvnl_b200.so (`vnl_policy_forward`, tcgen05 tensor cores);
there is no CPU or torch fallback on this path — `reference_forward` below is the fp32 torch restatement that the tests
compare against, never the product.
"""
from __future__ import annotations

import ctypes
from typing import Dict, Optional, Sequence

import numpy as np

from . import _lib
from . import learner as lrn
from . import train_kernels as tk

# flax parameter tree of IntentionNetwork, in the order vnl_policy_pack takes the arrays
PARAM_ORDER = (
    "encoder/hidden_0/kernel", "encoder/hidden_0/bias", "encoder/LayerNorm_0/scale", "encoder/LayerNorm_0/bias",
    "encoder/hidden_1/kernel", "encoder/hidden_1/bias", "encoder/LayerNorm_1/scale", "encoder/LayerNorm_1/bias",
    "encoder/fc2_mean/kernel", "encoder/fc2_mean/bias", "encoder/fc2_logvar/kernel", "encoder/fc2_logvar/bias",
    "decoder/hidden_0/kernel", "decoder/hidden_0/bias", "decoder/LayerNorm_0/scale", "decoder/LayerNorm_0/bias",
    "decoder/hidden_1/kernel", "decoder/hidden_1/bias", "decoder/LayerNorm_1/scale", "decoder/LayerNorm_1/bias",
    "decoder/hidden_2/kernel", "decoder/hidden_2/bias",
)


# the same entries as (module, layer, leaf) of the flax dict `params["params"]` (INTEGRATION.md)
PARAM_ORDER_TUPLES = tuple(tuple(k.split("/")) for k in PARAM_ORDER)


class VnlPolicyDims(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in ("traj", "obs", "latent", "e1", "e2", "d1", "d2", "nu")]


POLICY_EXPORTS = ("vnl_policy_check", "vnl_policy_blob_bytes", "vnl_policy_pack", "vnl_policy_forward", "vnl_policy_debug",
                  "vnl_xla_policy_forward")


def _bind(lib):
    P = ctypes.POINTER(VnlPolicyDims)
    v = ctypes.c_void_p
    lib.vnl_policy_check.argtypes = [P]
    lib.vnl_policy_blob_bytes.argtypes = [P]
    lib.vnl_policy_blob_bytes.restype = ctypes.c_size_t
    lib.vnl_policy_pack.argtypes = [P, ctypes.POINTER(v), v, ctypes.c_size_t]
    lib.vnl_policy_forward.argtypes = [v, P, ctypes.c_int] + [v] * 15
    lib.vnl_policy_debug.argtypes = [v, P, ctypes.c_int, v, v, v, v, v, ctypes.c_int, v, v]
    lib.vnl_xla_policy_forward.argtypes = [v, ctypes.POINTER(v), ctypes.c_char_p, ctypes.c_size_t, v]
    lib.vnl_xla_policy_forward.restype = None
    return lib


def param_shapes(traj_size: int, obs_size: int, action_size: int, latent: int = 64, encoder_layer_sizes: Sequence[int] = (256, 128),
                 decoder_layer_sizes: Sequence[int] = (128, 256)) -> Dict[str, tuple]:
    """Shapes of the flax tree of `make_intention_policy` (intention_policy_network.py:108-139; sizes from
    configs/train_config.yaml:15-17; the decoder's last layer has NormalTanhDistribution.param_size = 2 * action_size)."""
    (e1, e2), (d1, d2) = encoder_layer_sizes, decoder_layer_sizes
    dense = {"encoder/hidden_0": (traj_size, e1), "encoder/hidden_1": (e1, e2), "encoder/fc2_mean": (e2, latent),
             "encoder/fc2_logvar": (e2, latent), "decoder/hidden_0": (latent + obs_size, d1), "decoder/hidden_1": (d1, d2),
             "decoder/hidden_2": (d2, 2 * action_size)}
    shapes = {}
    for k, (i, o) in dense.items():
        shapes[k + "/kernel"], shapes[k + "/bias"] = (i, o), (o,)
    for k, n in (("encoder/LayerNorm_0", e1), ("encoder/LayerNorm_1", e2), ("decoder/LayerNorm_0", d1), ("decoder/LayerNorm_1", d2)):
        shapes[k + "/scale"], shapes[k + "/bias"] = (n,), (n,)
    return shapes


def init_params(rng: np.random.Generator, shapes: Dict[str, tuple], perturb: float = 0.0) -> Dict[str, np.ndarray]:
    """Random init in the reference's scheme: lecun_uniform kernels (intention_policy_network.py:26,54), zero biases, unit
    LayerNorm scales.  `perturb` > 0 additionally jitters biases / scales so that tests exercise them."""
    out = {}
    for k, s in shapes.items():
        if k.endswith("/kernel"):
            lim = np.sqrt(3.0 / s[0])
            out[k] = rng.uniform(-lim, lim, size=s).astype(np.float32)
        elif k.endswith("/scale"):
            out[k] = (1.0 + perturb * rng.standard_normal(s)).astype(np.float32)
        else:
            out[k] = (perturb * rng.standard_normal(s)).astype(np.float32)
    return out


def alloc_outputs(policy, B: int, heads: bool = False):
    """The output tensors of one call of `policy` (IntentionPolicy or PrecisePolicy: their `alloc_outputs` method) for B rows."""
    t, nu = policy.torch, policy.action_size
    f = lambda *s: t.empty(*s, dtype=t.float32, device=policy.device)
    out = {"action": f(B, nu), "raw_action": f(B, nu), "logits": f(B, 2 * nu), "log_prob": f(B), "rand_log_prob": f(B)}
    if heads:
        out["z_mean"], out["z_logvar"] = f(B, policy.latent), f(B, policy.latent)
    return out


class IntentionPolicy:
    """Device-resident packed parameters + the `policy(traj, obs, draws)` call of the rollout."""

    alloc_outputs = alloc_outputs

    def __init__(self, params: Dict[str, np.ndarray], device: str = "cuda:0", obs_mean=None, obs_std=None):
        import torch

        if not torch.cuda.is_available():
            raise RuntimeError("vnl_b200 policy needs a CUDA device (sm_100a); there is no CPU fallback")
        self.torch = torch
        self.lib = _bind(_lib.load_library())
        self.device = torch.device(device)
        w = lrn.policy_widths(params)
        self.dims = VnlPolicyDims(**w)
        rc = self.lib.vnl_policy_check(ctypes.byref(self.dims))
        if rc:
            raise ValueError(f"layer sizes not supported by the policy kernel ({rc})")
        self.traj_size, self.obs_size, self.latent, self.action_size = w["traj"], w["obs"], w["latent"], w["nu"]
        self.load_params(params)
        self.set_normalizer(obs_mean, obs_std)
        self.launches = 0

    def load_params(self, params: Dict[str, np.ndarray]) -> None:
        """Pack the flax tree (host, C: vnl_policy_pack) and upload it; call again after every PPO update."""
        arrs = [np.ascontiguousarray(params[k], dtype=np.float32) for k in PARAM_ORDER]
        ptrs = (ctypes.c_void_p * len(arrs))(*[a.ctypes.data for a in arrs])
        n = int(self.lib.vnl_policy_blob_bytes(ctypes.byref(self.dims)))
        host = np.zeros((n + 3) // 4, dtype=np.int32)
        rc = self.lib.vnl_policy_pack(ctypes.byref(self.dims), ptrs, host.ctypes.data, host.nbytes)
        if rc:
            raise RuntimeError(f"vnl_policy_pack failed ({rc})")
        self.blob_host = host
        # The device blob keeps ONE address for the life of the policy: `rollout.Rollout` captures `blob_dev.data_ptr()` into
        # its CUDA graph, so a re-upload after a PPO update must land in the same buffer (stream-ordered copy).
        if getattr(self, "blob_dev", None) is None:
            self.blob_dev = self.torch.from_numpy(host).to(self.device)
        else:
            self.blob_dev.copy_(self.torch.from_numpy(host), non_blocking=False)

    def set_normalizer(self, mean, std) -> None:
        """brax running_statistics.normalize parameters for obs (ppo_imitation/train.py:220-229); None = identity."""
        t = self.torch
        # like the blob, the mean / std operands keep their device addresses once they exist (captured by CUDA graphs);
        # switching between identity (None) and a real normaliser after a capture is refused instead of silently ignored
        for name, val in (("obs_mean", mean), ("obs_std", std)):
            cur = getattr(self, name, None)
            if val is None:
                if cur is not None and getattr(self, "_norm_pinned", False):
                    raise ValueError("the normaliser operands were captured; pass tensors (e.g. zeros / ones), not None")
                setattr(self, name, None)
                continue
            src = t.as_tensor(val, dtype=t.float32)
            if cur is None:
                if getattr(self, "_norm_pinned", False):
                    raise ValueError("the policy was captured without a normaliser; build it with obs_mean / obs_std instead")
                # a contiguous fp32 tensor already on the device is ADOPTED (shared with e.g. normalizer.RunningStatistics,
                # whose in-place updates then reach the next launch); anything else is uploaded once
                setattr(self, name, src.to(self.device).contiguous())
            elif isinstance(val, t.Tensor) and val.data_ptr() == cur.data_ptr():
                pass  # the shared tensor itself
            else:
                if tuple(src.shape) != tuple(cur.shape):
                    raise ValueError("normaliser shape changed")
                cur.copy_(src)

    def pin_operands(self) -> None:
        """Called by a capturer (rollout.Rollout) once the operand addresses are baked into a CUDA graph."""
        self._norm_pinned = True

    def __call__(self, traj, obs, eps_z, eps_a, rand_action=None, out: Optional[dict] = None, heads: bool = False):
        """One launch: (action [B,nu], extras) as `policy(trajectories, observations, key)` of ppo_networks.py:55-83.
        eps_z [B,latent], eps_a [B,nu]: standard-normal draws; rand_action [B,nu]: the uniform(-1,1) draw (optional).
        eps_a=None gives the deterministic policy of evaluation (`mode(logits)`; the latent is still sampled, as there)."""
        t = self.torch
        B = traj.shape[0]
        for x, w in ((traj, self.traj_size), (obs, self.obs_size), (eps_z, self.latent), (eps_a, self.action_size)):
            if x is None and w == self.action_size:
                continue  # eps_a=None: `deterministic=True` of make_policy (ppo_networks.py:63-64), action = mode = tanh(loc)
            if x.dtype != t.float32 or not x.is_contiguous() or x.shape != (B, w) or x.device != self.device:
                raise ValueError("policy operands must be contiguous fp32 [B, width] tensors on the policy's device")
        if out is None:
            out = self.alloc_outputs(B, heads)
        p = lambda x: None if x is None else x.data_ptr()
        stream = t.cuda.current_stream(self.device).cuda_stream
        with t.cuda.device(self.device):
            rc = self.lib.vnl_policy_forward(self.blob_dev.data_ptr(), ctypes.byref(self.dims), B, p(traj), p(obs), p(self.obs_mean),
                                             p(self.obs_std), p(eps_z), p(eps_a), p(rand_action), p(out["action"]),
                                             p(out["raw_action"]), p(out["logits"]), p(out["log_prob"]),
                                             p(out["rand_log_prob"]) if rand_action is not None else None,
                                             p(out.get("z_mean")), p(out.get("z_logvar")), stream)
        if rc:
            raise RuntimeError(f"vnl_policy_forward failed ({rc})")
        self.launches += 1
        return out["action"], out

    def debug_layer(self, traj, obs, eps_z, layer: int):
        """Raw tensor-core accumulators of layer 0..5 for the first 128 envs (test hook)."""
        t = self.torch
        n = (self.dims.e1, self.dims.e2, 2 * self.dims.latent, self.dims.d1, self.dims.d2, (2 * self.dims.nu + 31) // 32 * 32)[layer]
        dump = t.zeros(128, n, dtype=t.float32, device=self.device)
        p = lambda x: None if x is None else x.data_ptr()
        with t.cuda.device(self.device):
            rc = self.lib.vnl_policy_debug(self.blob_dev.data_ptr(), ctypes.byref(self.dims), traj.shape[0], p(traj), p(obs),
                                           p(self.obs_mean), p(self.obs_std), p(eps_z), layer, dump.data_ptr(),
                                           t.cuda.current_stream(self.device).cuda_stream)
        if rc:
            raise RuntimeError(f"vnl_policy_debug failed ({rc})")
        return dump


class PrecisePolicy:
    """The same `policy(traj, obs, draws)` call as IntentionPolicy at the REFERENCE's precision (fp32 network, VERDICT r1 / ADVICE r1:
    the bf16 kernel's behaviour log-probs are 0.05-0.35 away from the fp32 network the learner re-evaluates, the size of the PPO
    clip range).  Runs the learner's forward pass (learner.PolicyForward: `vnl_gemm_tf32` in `precision="3xtf32"`, the default,
    fp32-class: log-probs within ~1e-4 of an fp32 / float64 evaluation, or `"tf32"`, one pass as XLA runs the reference on a GPU), then
    `vnl_policy_sample`.  ~25 launches instead of one (0.25 ms at 8192 envs beside a 7.7 ms env step), all CUDA-graph capturable: the
    parameters are one flat buffer `blob_dev` laid out as the learner's policy bucket, refreshed in place with its 3xTF32 splits by
    `load_params`; the workspaces are allocated once per batch size.  Drop-in for IntentionPolicy in rollout.Rollout."""

    alloc_outputs = alloc_outputs

    def __init__(self, params: Dict[str, np.ndarray], device: str = "cuda:0", obs_mean=None, obs_std=None, precision: str = "3xtf32"):
        import torch

        if not torch.cuda.is_available():
            raise RuntimeError("vnl_b200 policy needs a CUDA device (sm_100a); there is no CPU fallback")
        if precision not in ("3xtf32", "tf32"):
            raise ValueError("precision must be '3xtf32' or 'tf32'")
        self.torch, self.x3 = torch, precision == "3xtf32"
        self.device = torch.device(device)
        self.widths = w = lrn.policy_widths(params)
        self.traj_size, self.obs_size, self.latent, self.action_size = w["traj"], w["obs"], w["latent"], w["nu"]
        lrn.PolicyForward.check(w)
        shapes = lrn.policy_tensor_shapes({k: v.shape for k, v in params.items()})
        # The parameters keep ONE address for the life of the policy: `rollout.Rollout` captures `blob_dev.data_ptr()` into its CUDA
        # graph, so `load_params` after a PPO update must land in the same buffer.
        self.blob_dev = torch.zeros(lrn.flat_layout(shapes)[2], dtype=torch.float32, device=self.device)
        self.p = lrn.flat_views(self.blob_dev, shapes)
        self.blob_split = (tk.like(self.blob_dev), tk.like(self.blob_dev))  # its 3xTF32 hi / lo
        self.splits = tuple(lrn.flat_views(x, shapes) for x in self.blob_split)
        self.obs_mean, self.obs_std = (torch.full((self.obs_size,), v, dtype=torch.float32, device=self.device) for v in (0.0, 1.0))
        self._identity = True
        self.bufs = {}
        self.launches = 0
        self.load_params(params)
        self.set_normalizer(obs_mean, obs_std)

    def load_params(self, params) -> None:
        lrn.pack_policy(self.p, params)
        if self.x3:
            tk.split_into(self.blob_dev, *self.blob_split)

    def set_normalizer(self, mean, std) -> None:
        """None = identity.  Tensors already on the device are ADOPTED when first given (shared with normalizer.RunningStatistics),
        later calls copy into the same storage."""
        t = self.torch
        for name, val, ident in (("obs_mean", mean, 0.0), ("obs_std", std, 1.0)):
            cur = getattr(self, name)
            if val is None:
                cur.fill_(ident)
            elif isinstance(val, t.Tensor) and val.is_cuda and val.dtype == t.float32 and val.is_contiguous() and self._identity and not getattr(self, "_norm_pinned", False):
                setattr(self, name, val)
            elif not (isinstance(val, t.Tensor) and val.data_ptr() == cur.data_ptr()):
                cur.copy_(t.as_tensor(val, dtype=t.float32))
        self._identity = mean is None and std is None and self._identity

    def pin_operands(self) -> None:
        self._norm_pinned = True

    def __call__(self, traj, obs, eps_z, eps_a, rand_action=None, out: Optional[dict] = None, heads: bool = False):
        """(action [B, nu], extras) as IntentionPolicy.__call__; rand_action: the reference's ONE uniform draw of shape (nu,)
        (a [B, nu] tensor is accepted for compatibility: its first row is used)."""
        t, L_, chk = self.torch, tk.lib(), tk.check
        B = traj.shape[0]
        for x, w in ((traj, self.traj_size), (obs, self.obs_size), (eps_z, self.latent)):
            if x.dtype != t.float32 or not x.is_contiguous() or x.shape != (B, w) or x.device != self.device:
                raise ValueError("policy operands must be contiguous fp32 [B, width] tensors on the policy's device")
        if out is None:
            out = self.alloc_outputs(B, heads)
        if B == 0:
            return out["action"], out
        if B not in self.bufs:  # the forward's workspaces, and traj rows padded to tk.ld4 floats (a TMA row stride)
            self.bufs[B] = dict(fwd=lrn.PolicyForward(self.widths, B, self.device, self.x3), idx=t.arange(B, dtype=t.int32, device=self.device),
                                traj=t.zeros(B, tk.ld4(self.traj_size), dtype=t.float32, device=self.device))
        b, st, ptr = self.bufs[B], tk.stream(traj), (lambda x: None if x is None else x.data_ptr())
        with t.cuda.device(self.device):
            chk(L_.vnl_gather_rows(ptr(traj), 1, B, self.traj_size, ptr(b["idx"]), B, ptr(b["traj"]), b["traj"].stride(0), st), "pad traj")
            b["fwd"](self.p, b["traj"], obs, self.obs_mean, self.obs_std, eps_z, out["logits"], self.splits)
            if rand_action is not None and rand_action.dim() == 2:
                rand_action = rand_action[0].contiguous()
            chk(L_.vnl_policy_sample(ptr(out["logits"]), out["logits"].stride(0), ptr(eps_a), ptr(rand_action), B, self.action_size, ptr(out["action"]),
                                     ptr(out["raw_action"]), ptr(out["log_prob"]), ptr(out["rand_log_prob"]) if rand_action is not None else None, st),
                "policy_sample")
            if heads:
                h = b["fwd"].ws["heads"]
                out["z_mean"].copy_(h[:, :self.latent]); out["z_logvar"].copy_(h[:, self.latent:])
        self.launches += 1
        return out["action"], out


def reference_forward(params, traj, obs, eps_z, eps_a, rand_action=None, obs_mean=None, obs_std=None, operand_dtype=None):
    """fp32 torch restatement of the reference policy (checker for tests / tools; works on CPU tensors too).
    `operand_dtype=torch.bfloat16` rounds the operands of every dense layer the way the kernel does (fp32 accumulation)."""
    import torch

    P = {k: torch.as_tensor(v, dtype=torch.float32, device=traj.device) for k, v in params.items()}
    rnd = (lambda x: x) if operand_dtype is None else (lambda x: x.to(operand_dtype).to(torch.float32))

    def dense(x, name):
        return torch.matmul(rnd(x).double(), rnd(P[name + "/kernel"]).double()).float() + P[name + "/bias"]

    def ln(x, name):  # flax LayerNorm: fast variance, eps 1e-6
        m = x.mean(-1, keepdim=True)
        var = torch.clamp((x * x).mean(-1, keepdim=True) - m * m, min=0.0)
        return (x - m) * torch.rsqrt(var + 1e-6) * P[name + "/scale"] + P[name + "/bias"]

    pre = {}
    h = traj
    for i in range(2):  # Encoder, intention_policy_network.py:31-41
        pre[i] = dense(h, f"encoder/hidden_{i}")
        h = ln(torch.relu(pre[i]), f"encoder/LayerNorm_{i}")
    mean, logvar = dense(h, "encoder/fc2_mean"), dense(h, "encoder/fc2_logvar")
    pre[2] = torch.cat([mean, logvar], -1)
    z = mean + eps_z * torch.exp(0.5 * logvar)  # reparameterize, :76-79
    o = obs if obs_mean is None else (obs - obs_mean) / obs_std  # the `apply` closure normalises obs only, :124-126
    h = torch.cat([z, o], -1)
    for i in range(2):  # Decoder, :58-73
        pre[3 + i] = dense(h, f"decoder/hidden_{i}")
        h = ln(torch.relu(pre[3 + i]), f"decoder/LayerNorm_{i}")
    logits = dense(h, "decoder/hidden_2")
    pre[5] = logits
    nu = logits.shape[-1] // 2
    loc, scale = logits[..., :nu], torch.nn.functional.softplus(logits[..., nu:]) + 1e-3  # brax NormalTanhDistribution
    raw = loc + scale * eps_a
    log_det = lambda x: 2.0 * (np.log(2.0) - x - torch.nn.functional.softplus(-2.0 * x))
    normal_lp = lambda x: -0.5 * ((x - loc) / scale) ** 2 - torch.log(scale) - 0.5 * np.log(2 * np.pi)
    out = {"action": torch.tanh(raw), "raw_action": raw, "logits": logits, "log_prob": (normal_lp(raw) - log_det(raw)).sum(-1),
           "z_mean": mean, "z_logvar": logvar, "pre": pre}
    if rand_action is not None:
        out["rand_log_prob"] = (normal_lp(rand_action) - log_det(rand_action)).sum(-1)
    return out
