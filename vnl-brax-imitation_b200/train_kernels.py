"""ctypes binding of the PPO-update kernels (include/vnl_train.h) over torch CUDA tensors (torch = device memory + streams)."""
from __future__ import annotations

import ctypes
from typing import Optional

from . import _lib

TRAIN_EXPORTS = ("vnl_gemm_tf32", "vnl_gemm_tf32_ex", "vnl_split_tf32", "vnl_gather_rows", "vnl_obs_normalize", "vnl_relu_ln_fwd", "vnl_relu_ln_bwd",
                 "vnl_swish_fwd", "vnl_swish_bwd", "vnl_reparam_fwd", "vnl_heads_bwd", "vnl_colsum", "vnl_rowdot", "vnl_outer", "vnl_outer_swish_bwd", "vnl_gather_scalars",
                 "vnl_ppo_rows", "vnl_ppo_loss_bwd", "vnl_adam_tick", "vnl_adam", "vnl_policy_sample", "vnl_eval_metrics",
                 "vnl_metrics_accumulate")
_bound = None


def lib():
    global _bound
    if _bound is None:
        L = _lib.load_library()
        v, i, f, sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_size_t
        PP = ctypes.POINTER(ctypes.c_void_p)
        L.vnl_gemm_tf32.argtypes = [i, i, i, i, PP, i, i, PP, i, i, v, i, v, i, v]
        L.vnl_gemm_tf32_ex.argtypes = [i, i, i, i, PP, i, i, PP, i, i, v, i, v, i, i, v, i, v]
        L.vnl_split_tf32.argtypes = [v, sz, v, v, v]
        L.vnl_gather_rows.argtypes = [v, i, i, i, v, i, v, i, v]
        L.vnl_obs_normalize.argtypes = [v, i, i, i, v, v, v, i, v]
        L.vnl_relu_ln_fwd.argtypes = [v, i, i, i, v, v, v, i, v, v]
        L.vnl_relu_ln_bwd.argtypes = [v, i, v, i, v, v, i, i, v, i, v, v, v, v]
        L.vnl_swish_fwd.argtypes = [v, sz, v, v]
        L.vnl_swish_bwd.argtypes = [v, v, sz, v, v]
        L.vnl_reparam_fwd.argtypes = [v, v, i, i, v, i, v]
        L.vnl_heads_bwd.argtypes = [v, i, v, v, i, i, f, v, v, v]
        L.vnl_colsum.argtypes = [v, i, i, i, v, v, v]
        L.vnl_rowdot.argtypes = [v, i, i, i, v, v, v, v]
        L.vnl_outer.argtypes = [v, i, v, i, v, i, v]
        L.vnl_outer_swish_bwd.argtypes = [v, i, v, i, v, v, v]
        L.vnl_gather_scalars.argtypes = [i, v, v, i, i, v, i, v]
        L.vnl_ppo_rows.argtypes = [v, i, v, v, i, i, v, v, v, f, v, v, v, v, v]
        L.vnl_ppo_loss_bwd.argtypes = [v, i, v, v, i, i, v, v, v, v, v, v, f, f, i, v, i, v, v, v, v]
        L.vnl_policy_sample.argtypes = [v, i, v, v, i, i, v, v, v, v, v]
        L.vnl_eval_metrics.argtypes = [i, i, i, v, v, v, v, v, v, v]
        L.vnl_adam_tick.argtypes = [v, f, f, v, v]
        L.vnl_adam.argtypes = [v, v, v, v, sz, f, f, f, f, i, f, v, v]
        L.vnl_metrics_accumulate.argtypes = [v, i, v, v]
        _bound = L
    return _bound


def stream(t) -> int:
    import torch
    return torch.cuda.current_stream(t.device).cuda_stream


def check(rc: int, what: str):
    if rc:
        raise RuntimeError(f"{what} failed with code {rc}")


def capture(device, warmup, *fns):
    """One CUDA graph per function in `fns`, for the rollout's unroll and the trainer's minibatch update.  `warmup()` runs first,
    eagerly on a side stream (lazy module loads, ctypes bindings and allocations happen outside the capture); then the device is
    synchronised and each fn is captured with capture_error_mode="thread_local", so calls from other threads -- NCCL's watchdog
    querying its events -- do not invalidate the capture.  No fn may issue a collective: an 8-GPU run hung when the gradient
    all-reduce was captured with the update (DESIGN §3d)."""
    import torch
    main = torch.cuda.current_stream(device)
    side = torch.cuda.Stream(device=device)
    side.wait_stream(main)
    with torch.cuda.stream(side):
        warmup()
    main.wait_stream(side)
    torch.cuda.synchronize(device)
    graphs = []
    for fn in fns:
        graphs.append(torch.cuda.CUDAGraph())
        with torch.cuda.graph(graphs[-1], capture_error_mode="thread_local"):
            fn()
    return graphs


def _ptrs(ts):
    return (ctypes.c_void_p * len(ts))(*[t.data_ptr() for t in ts])


# ---- row strides of GEMM operands --------------------------------------------------------------------------------------
# A TMA tensor map needs a row stride that is a multiple of 16 bytes, so every operand of `gemm` with a width n that is not a
# multiple of 4 floats lives in a zeroed [rows, ld4(n)] buffer and is passed as its [rows, n] view: the kernels take the row
# stride (`ld`) from `x.stride(0)`, and TMA never reads the padding columns (it fills out-of-range elements with zeros).  For
# widths that are multiples of 4 the rule is the identity.
def ld4(n: int) -> int:
    """Row stride in floats of an operand of width n (also the 16-byte alignment of a tensor in a flat buffer)."""
    return (int(n) + 3) // 4 * 4


def padded(rows: int, n: int, device, dtype=None):
    """Zeroed [rows, ld4(n)] buffer returned as its [rows, n] view (stride(0) == ld4(n))."""
    import torch
    return torch.zeros(int(rows), ld4(n), dtype=dtype or torch.float32, device=device)[:, :int(n)]


def like(x):
    """Uninitialised tensor with x's shape AND strides (torch.empty_like of a row-padded view would be dense)."""
    import torch
    return torch.empty_strided(x.size(), x.stride(), dtype=x.dtype, device=x.device)


def _extent(x) -> int:
    """Floats from x's first to its last element (the padding between rows of a row-padded view included)."""
    return 1 + sum((s - 1) * st for s, st in zip(x.shape, x.stride())) if x.numel() else 0


def split(x):
    """(hi, lo) of the 3xTF32 scheme, with x's row stride."""
    hi, lo = like(x), like(x)
    return split_into(x, hi, lo)


def split_into(x, hi, lo):
    """3xTF32 split into preallocated tensors of x's strides (no allocation: CUDA-graph capturable)."""
    assert hi.stride() == x.stride() and lo.stride() == x.stride()
    check(lib().vnl_split_tf32(x.data_ptr(), _extent(x), hi.data_ptr(), lo.data_ptr(), stream(x)), "vnl_split_tf32")
    return hi, lo


def gemm(A, a_mn: int, B, b_mn: int, C, M: int, N: int, K: int, bias=None, x3: bool = False, splitk: int = 1, parts=None, zero: bool = True,
         epilogue: int = 0, aux=None):
    """C[M, N] (+)= A . B^T (+ bias); operands are 2-D fp32 tensors whose row stride is their ld.  `x3`: 3xTF32 (the operands are
    split here unless `parts` = ((A_hi, A_lo), (B_hi, B_lo)) is given).  splitk > 1 accumulates into C (zeroed here unless the caller says it already is: `zero=False`).
    epilogue 1: aux = swish(C) written beside C; 2: C = (A . B^T) * swish'(aux)  (include/vnl_train.h: vnl_gemm_tf32_ex)."""
    for t in (A, B, C):
        assert t.dim() == 2 and t.stride(1) == 1 and t.dtype.is_floating_point and t.element_size() == 4
    if x3:
        (ah, al), (bh, bl) = parts if parts is not None else (split(A), split(B))
        As, Bs = [ah, ah, al], [bh, bl, bh]
    else:
        As, Bs = [A], [B]
    if splitk > 1 and zero:
        C.zero_()
    if epilogue:
        assert aux is not None and aux.dim() == 2 and aux.stride(1) == 1 and aux.shape[0] >= M
        rc = lib().vnl_gemm_tf32_ex(M, N, K, len(As), _ptrs(As), A.stride(0), int(a_mn), _ptrs(Bs), B.stride(0), int(b_mn), C.data_ptr(), C.stride(0),
                                    None if bias is None else bias.data_ptr(), int(splitk), int(epilogue), aux.data_ptr(), aux.stride(0), stream(C))
    else:
        rc = lib().vnl_gemm_tf32(M, N, K, len(As), _ptrs(As), A.stride(0), int(a_mn), _ptrs(Bs), B.stride(0), int(b_mn), C.data_ptr(), C.stride(0),
                                 None if bias is None else bias.data_ptr(), int(splitk), stream(C))
    check(rc, "vnl_gemm_tf32")
    return C
