"""vnl_gae == compute_gae of ppo_imitation/intention_losses.py:26-89, restated line by line in torch fp64 (the scan as a
python loop) as the checker."""
import os
import re
import struct

import numpy as np
import pytest
import torch

from conftest import ROOT, pkg

ppo = pkg("ppo")
libm = pkg("_lib")


def reference_gae(truncation, termination, rewards, values, bootstrap_value, lambda_=1.0, discount=0.99):
    truncation_mask = 1 - truncation
    values_t_plus_1 = torch.cat([values[1:], bootstrap_value[None]], 0)
    deltas = rewards + discount * (1 - termination) * values_t_plus_1 - values
    deltas = deltas * truncation_mask
    acc = torch.zeros_like(bootstrap_value)
    out = []
    for t in reversed(range(truncation.shape[0])):  # lax.scan(..., reverse=True)
        acc = deltas[t] + discount * (1 - termination[t]) * truncation_mask[t] * lambda_ * acc
        out.append(acc)
    vs_minus_v_xs = torch.stack(out[::-1], 0)
    vs = vs_minus_v_xs + values
    vs_t_plus_1 = torch.cat([vs[1:], bootstrap_value[None]], 0)
    advantages = (rewards + discount * (1 - termination) * vs_t_plus_1 - values) * truncation_mask
    return vs, advantages


def test_header_and_binding_agree():
    txt = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "vnl_ppo.h")).read(), flags=re.S)
    declared = sorted(set(re.findall(r"\b(vnl_[a-z_0-9]+)\s*\(", txt)))
    assert set(declared) == set(ppo.PPO_EXPORTS)
    if not os.path.exists(libm.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = ppo._bind(libm.load_library())
    for n in declared:
        assert getattr(lib, n) is not None


def test_gae_refuses_to_run_without_gpu(monkeypatch):
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)  # also on a GPU machine
    z = torch.zeros(2, 3)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ppo.compute_gae(z, z, z, z, torch.zeros(3))


def _case(T, B, seed):
    g = torch.Generator().manual_seed(seed)
    trunc = (torch.rand(T, B, generator=g) < 0.1).float()
    done = (torch.rand(T, B, generator=g) < 0.15).float()
    term = done * (1 - trunc)  # intention_losses.py:158: termination = (1 - discount) * (1 - truncation)
    return trunc, term, torch.randn(T, B, generator=g), torch.randn(T, B, generator=g) * 3, torch.randn(B, generator=g) * 3


@pytest.mark.gpu
@pytest.mark.parametrize("T,B,lam,disc", [(20, 8192, 0.95, 0.9), (1, 5, 1.0, 0.99), (7, 1, 0.0, 0.5), (150, 300, 0.95, 0.99)])
def test_gae_matches_restatement(T, B, lam, disc):
    c = _case(T, B, seed=T * 1000 + B)
    vs, adv = ppo.compute_gae(*[x.cuda() for x in c], lambda_=lam, discount=disc)
    rvs, radv = reference_gae(*[x.double() for x in c], lambda_=lam, discount=disc)
    torch.cuda.synchronize()
    np.testing.assert_allclose(vs.cpu().numpy(), rvs.numpy(), rtol=2e-5, atol=2e-5)
    np.testing.assert_allclose(adv.cpu().numpy(), radv.numpy(), rtol=2e-5, atol=2e-5)
    # truncated steps carry no advantage; an untruncated terminal step bootstraps nothing
    assert float(adv.cpu()[c[0] > 0].abs().max() if (c[0] > 0).any() else 0.0) == 0.0


@pytest.mark.gpu
def test_gae_xla_trampoline_and_argument_errors():
    import ctypes
    T, B = 6, 130
    c = [x.cuda() for x in _case(T, B, seed=3)]
    vs, adv = ppo.compute_gae(*c, lambda_=0.95, discount=0.9)
    vs2, adv2 = torch.full_like(vs, float("nan")), torch.full_like(adv, float("nan"))
    lib = ppo._bind(libm.load_library())
    arr = (ctypes.c_void_p * 7)(*[x.data_ptr() for x in c], vs2.data_ptr(), adv2.data_ptr())
    op = struct.pack("<iiff", T, B, 0.95, 0.9)
    lib.vnl_xla_gae(torch.cuda.current_stream().cuda_stream, arr, op, len(op), None)
    torch.cuda.synchronize()
    assert torch.equal(vs, vs2) and torch.equal(adv, adv2)
    with pytest.raises(ValueError):
        ppo.compute_gae(c[0][:, :5], *c[1:])
    assert lib.vnl_gae(T, B, None, None, None, None, None, 0.95, 0.9, None, None, None) < 0
    assert lib.vnl_gae(0, B, None, None, None, None, None, 0.95, 0.9, None, None, None) == 0
