"""Observation normaliser (include/vnl_normalizer.h): brax running_statistics.update restated in torch fp64 (two passes,
psum points marked) is the checker.  CPU: exported symbols, and — with a real 2-rank gloo group — that the single
all-reduce of [sum d | sum d^2 | rows] reproduces brax's three psums (the split the kernels rely on).  GPU: kernels vs the
restatement over several updates, ragged shapes, determinism."""
import os
import re
import subprocess
import sys
import textwrap

import numpy as np
import pytest
import torch

from conftest import ROOT, pkg

nz = pkg("normalizer")
libm = pkg("_lib")


def brax_update(state, batches, std_min=1e-6, std_max=1e6):
    """running_statistics.update with pmap_axis_name: `batches` = the per-device batches; psum = sum over the list."""
    count, mean, sv = state
    count = count + sum(b.shape[0] for b in batches)                                   # psum(step_increment)
    mean_update = sum((b - mean).sum(0) for b in batches) / count                      # psum(sum(diff_to_old_mean)) / count
    new_mean = mean + mean_update
    sv = sv + sum(((b - mean) * (b - new_mean)).sum(0) for b in batches)               # psum(variance_update)
    std = torch.clamp(torch.sqrt(torch.clamp(sv, min=0) / count), std_min, std_max)
    return (count, new_mean, sv), std


def test_header_and_binding_agree():
    txt = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "vnl_normalizer.h")).read(), flags=re.S)
    declared = sorted(set(re.findall(r"\b(vnl_(?:xla_)?obs_[a-z_0-9]+)\s*\(", txt)))
    assert set(declared) == set(nz.NORMALIZER_EXPORTS)
    if not os.path.exists(libm.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = nz._bind(libm.load_library())
    for n in declared:
        assert getattr(lib, n) is not None
    assert lib.vnl_obs_stats_workspace_bytes(232) == 148 * 2 * 232 * 4 + 16
    assert lib.vnl_obs_stats_workspace_bytes(0) == 0 and lib.vnl_obs_stats_workspace_bytes(1025) == 0


def test_normalizer_refuses_to_run_without_gpu(monkeypatch):
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)  # also on a GPU machine
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        nz.RunningStatistics(232)


WORKER = """
import sys, torch, torch.distributed as dist
sys.path.insert(0, {root!r}); sys.path.insert(0, {root!r} + "/tests")
import importlib
nz = importlib.import_module("vnl-brax-imitation_b200.normalizer")
from test_normalizer import brax_update
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=2)
rank = dist.get_rank()
g = torch.Generator().manual_seed(7)
full = [torch.randn(n, 5, generator=g, dtype=torch.float64) * 3 + 1 for n in (40, 24)]   # rank 0 / rank 1 batches
state = (torch.zeros((), dtype=torch.float64), torch.zeros(5, dtype=torch.float64), torch.zeros(5, dtype=torch.float64))
mine_state = [s.clone() for s in state]
for it in range(3):
    batches = [b + it for b in full]
    state, std = brax_update(state, batches)
    # the split: local one-pass sums against the OLD mean, one all-reduce, width-sized epilogue
    d = batches[rank] - mine_state[1]
    sums = torch.cat([d.sum(0), (d * d).sum(0), torch.tensor([float(d.shape[0])], dtype=torch.float64)])
    nz.all_reduce_sums(sums)
    cnt = mine_state[0] + sums[10]
    mu = sums[:5] / cnt
    mine_state = [cnt, mine_state[1] + mu, mine_state[2] + sums[5:10] - mu * sums[:5]]
    for a, b in zip(mine_state, state):
        assert torch.allclose(a, b, rtol=1e-12, atol=1e-12), (it, a, b)
dist.barrier(); dist.destroy_process_group()
print("ok", rank)
"""


def test_two_rank_gloo_single_allreduce_equals_brax_psums(tmp_path):
    import socket
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    script = tmp_path / "w.py"
    script.write_text(textwrap.dedent(WORKER.format(root=ROOT, port=port)))
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
             for r in range(2)]
    outs = [p.communicate(timeout=240)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    assert all("ok" in o for o in outs), outs


@pytest.mark.gpu
@pytest.mark.parametrize("width,rows", [(232, (4096, 20000, 7)), (55, (1000, 3, 8192)), (1, (17,)), (1024, (300,))])
def test_update_matches_brax_restatement(width, rows):
    st = nz.RunningStatistics(width, "cuda:0")
    ref = (torch.zeros((), dtype=torch.float64), torch.zeros(width, dtype=torch.float64), torch.zeros(width, dtype=torch.float64))
    assert float(st.std.min()) == 1.0 and float(st.count) == 0.0  # init_state
    g = torch.Generator().manual_seed(width)
    for i, n in enumerate(rows):
        x = (torch.randn(n, width, generator=g) * (1 + i) + 0.5 * i).float()
        st.update(x.cuda())
        ref, std = brax_update(ref, [x.double()])
        torch.cuda.synchronize()
        assert float(st.count) == float(ref[0])
        np.testing.assert_allclose(st.mean.cpu().numpy(), ref[1].numpy(), rtol=0, atol=2e-5)
        np.testing.assert_allclose(st.summed_variance.cpu().numpy(), ref[2].numpy(), rtol=2e-4)
        np.testing.assert_allclose(st.std.cpu().numpy(), std.numpy(), rtol=2e-4)


@pytest.mark.gpu
def test_update_is_deterministic_and_accepts_time_major_batches():
    x = torch.randn(6, 500, 232, generator=torch.Generator().manual_seed(1)).cuda()  # [T, B, obs] as the rollout stores it
    a, b = nz.RunningStatistics(232), nz.RunningStatistics(232)
    a.update(x); b.update(x.reshape(-1, 232))
    torch.cuda.synchronize()
    for k in ("count", "mean", "summed_variance", "std"):
        assert torch.equal(getattr(a, k), getattr(b, k)), k
    with pytest.raises(ValueError):
        a.update(x[:, :, :100])


@pytest.mark.gpu
def test_xla_custom_call_trampolines_equal_direct_calls():
    """Legacy XLA custom-call ABI: uninitialised scratch / result buffers, state passed functionally (operands -> results)."""
    import ctypes
    import struct
    W, n = 232, 5000
    x = torch.randn(n, W, generator=torch.Generator().manual_seed(2)).cuda() * 2 + 1
    st = nz.RunningStatistics(W)
    st.update(x[:2000].contiguous())
    old = {k: getattr(st, k).clone() for k in ("count", "mean", "summed_variance", "std")}
    st.update(x[2000:].contiguous())
    torch.cuda.synchronize()
    lib, stream = st.lib, torch.cuda.current_stream().cuda_stream
    garbage = lambda m: torch.full((m,), float("nan"), device="cuda")
    sums, work = garbage(2 * W + 1), garbage(st.workspace.numel())
    batch = x[2000:].contiguous()
    arr = (ctypes.c_void_p * 4)(batch.data_ptr(), old["mean"].data_ptr(), sums.data_ptr(), work.data_ptr())
    op = struct.pack("<qi", n - 2000, W)
    lib.vnl_xla_obs_stats_partial(stream, arr, op, len(op), None)
    new = {k: garbage(v.numel()) for k, v in old.items()}
    arr = (ctypes.c_void_p * 9)(sums.data_ptr(), *[old[k].data_ptr() for k in ("count", "mean", "summed_variance", "std")],
                                *[new[k].data_ptr() for k in ("count", "mean", "summed_variance", "std")])
    op = struct.pack("<iff", W, 1e-6, 1e6)
    lib.vnl_xla_obs_stats_finish(stream, arr, op, len(op), None)
    torch.cuda.synchronize()
    for k in new:
        assert torch.equal(new[k], getattr(st, k)), k


@pytest.mark.gpu
def test_empty_batches():
    """rows = 0 (a rank with no envs this step) contributes zeros to the exchange; an all-empty update keeps init_state."""
    st = nz.RunningStatistics(232)
    st.update(torch.zeros(0, 232, device="cuda"))
    torch.cuda.synchronize()
    assert float(st.count) == 0 and float(st.std.min()) == 1.0 and not torch.isnan(st.mean).any()
    x = torch.randn(100, 232, device="cuda")
    st.update(x)
    before = {k: getattr(st, k).clone() for k in ("count", "mean", "summed_variance", "std")}
    st.update(torch.zeros(0, 232, device="cuda"))
    torch.cuda.synchronize()
    for k, v in before.items():
        assert torch.equal(getattr(st, k), v), k
