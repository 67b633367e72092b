"""Gradient with respect to the memory items, on the CPU: the float64 oracle against torch's autograd of the
reference op chain, and the host-side argument checks of the two backward entry points."""
import numpy as np
import pytest
import torch

from oracle import ref_port as P
from keys_oracle import memory_keys_backward


def _memory_loss_torch(k):
    """model/Memory.py:52-59 restated with torch ops"""
    m = k.shape[0]
    return torch.sum(torch.abs(k @ k.t() / 2 + 0.5 - torch.eye(m, dtype=k.dtype))) / (m * (m - 1))


@pytest.mark.parametrize("train", [True, False])
@pytest.mark.parametrize("B,d,h,w,m", [(2, 32, 4, 4, 10), (1, 24, 3, 5, 7)])
def test_keys_oracle_matches_torch_autograd_of_reference_chain(B, d, h, w, m, train):
    rng = np.random.default_rng(B * 10 + m)
    query = rng.standard_normal((B, d, h, w))
    keys = rng.random((m, d)) * 0.4                         # not unit norm: no entry of S near 0
    W = rng.standard_normal((B, 2 * d, h, w))
    for cu, cs in [(1.0, 0.0), (0.0, 1.3), (1.0, 1.3)]:
        k = torch.tensor(keys, requires_grad=True)
        out = P.memory_forward(torch.tensor(query), k, train=train)
        loss = 0.7 * out[4] + cu * (out[0] * torch.tensor(W)).sum() + cs * _memory_loss_torch(k)
        if train:
            loss = loss + 0.3 * out[5]
        loss.backward()
        ref = memory_keys_backward(query, keys, W * cu if cu else None, cs if cs else None)
        np.testing.assert_allclose(k.grad.numpy(), ref, rtol=0, atol=1e-12 * max(np.abs(ref).max(), 1.0))


def test_keys_oracle_tie_band_zeroes_sign_noise():
    keys = np.eye(3)                                        # unit rows: S_ii = 0 exactly, off-diagonal S = 1/2
    ref0 = memory_keys_backward(np.zeros((1, 3, 1, 1)), keys, None, 1.0)
    ref1 = memory_keys_backward(np.zeros((1, 3, 1, 1)), keys, None, 1.0, tie=1e-5)
    np.testing.assert_allclose(ref0, ref1)                  # sgn(0) = 0 already
    keys = keys * (1 + 1e-9)
    refn = memory_keys_backward(np.zeros((1, 3, 1, 1)), keys, None, 1.0)
    reft = memory_keys_backward(np.zeros((1, 3, 1, 1)), keys, None, 1.0, tie=1e-5)
    assert np.abs(refn - reft).max() > 0.1 / 6 and np.allclose(reft, ref1, atol=1e-8)


def test_keys_backward_workspace_queries_are_pure_host_functions():
    import videoad_b200 as V
    l = V._lib.lib()
    assert l.vadc_memory_keys_bwd_workspace_bytes(64, 768, 1024, 2000) >= 2 * 65536 * 2000 * 2
    assert l.vadc_memory_keys_bwd_workspace_bytes(1, 96, 35, 33) > 0
    assert l.vadc_memory_separateness_bwd_workspace_bytes(2000, 768) >= 2000 * 2000 * 4


def test_keys_backward_argument_validation_happens_before_any_cuda_call():
    import videoad_b200 as V
    l = V._lib.lib()
    ws = 1 << 40
    fake = 16                                               # never dereferenced: every call below fails on the host
    # bad shapes
    assert l.vadc_memory_keys_bwd(fake, fake, 2, 0, 16, 10, fake, fake, ws, None) == -1
    assert l.vadc_memory_keys_bwd(fake, fake, 2, 32, 0, 10, fake, fake, ws, None) == -1
    assert l.vadc_memory_keys_bwd(fake, fake, 2, 32, 16, 0, fake, fake, ws, None) == -1
    assert l.vadc_memory_keys_bwd(fake, fake, -1, 32, 16, 10, fake, fake, ws, None) == -1
    assert l.vadc_memory_separateness_bwd(fake, fake, 1, 32, fake, fake, ws, None) == -1
    assert l.vadc_memory_separateness_bwd(fake, fake, 10, 0, fake, fake, ws, None) == -1
    # NULL pointers
    assert l.vadc_memory_keys_bwd(None, fake, 2, 32, 16, 10, fake, fake, ws, None) == -2
    assert l.vadc_memory_keys_bwd(fake, None, 2, 32, 16, 10, fake, fake, ws, None) == -2
    assert l.vadc_memory_keys_bwd(fake, fake, 2, 32, 16, 10, None, fake, ws, None) == -2
    assert l.vadc_memory_keys_bwd(fake, fake, 2, 32, 16, 10, fake, None, ws, None) == -2
    assert l.vadc_memory_separateness_bwd(None, fake, 10, 32, fake, fake, ws, None) == -2
    assert l.vadc_memory_separateness_bwd(fake, None, 10, 32, fake, fake, ws, None) == -2
    assert l.vadc_memory_separateness_bwd(fake, fake, 10, 32, None, fake, ws, None) == -2
    # outside what the tensor-core contraction takes, and too small a workspace
    assert l.vadc_memory_keys_bwd(fake, fake, 2, 4, 16, 10, fake, fake, ws, None) == -6
    assert l.vadc_memory_keys_bwd(fake, fake, 2, 32, 16, 10, fake, fake, 16, None) == -4
    assert l.vadc_memory_separateness_bwd(fake, fake, 10, 32, fake, fake, 16, None) == -4
