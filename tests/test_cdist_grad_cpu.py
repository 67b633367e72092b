"""Gradients of the stand-alone cdist on the CPU: the float64 oracle of vadc_cdist_bwd's math against torch's float64
autograd of torch.cdist (one problem, batched, broadcast, self, exact zeros of D), and the host-side argument checks
of the new entry point."""
import zlib

import numpy as np
import pytest
import torch

import cdist_grad_oracle as G


def _close(got, ref):
    got, ref = np.asarray(got), np.asarray(ref)
    assert got.shape == ref.shape
    np.testing.assert_allclose(got, ref, rtol=0, atol=1e-12 * max(float(np.abs(ref).max()), 1.0))


def _torch_grads(a, b, g, same=False):
    ta = torch.tensor(a, dtype=torch.float64, requires_grad=True)
    tb = ta if same else torch.tensor(b, dtype=torch.float64, requires_grad=True)
    D = torch.cdist(ta, tb, compute_mode="donot_use_mm_for_euclid_dist")     # the self diagonal exactly 0
    (D * torch.tensor(g, dtype=torch.float64)).sum().backward()
    return D.detach().numpy(), ta.grad.numpy(), None if same else tb.grad.numpy()


def _rng(*k):
    return np.random.default_rng(zlib.crc32(repr(k).encode()))


@pytest.mark.parametrize("ashape,bshape", [
    ((37, 24), (10, 24)),                 # one problem
    ((3, 33, 16), (3, 27, 16)),           # batched
    ((2, 40, 8), (12, 8)),                # 2-D b against 3-D a
    ((12, 8), (2, 40, 8)),                # 2-D a against 3-D b
    ((2, 1, 30, 8), (3, 26, 8)),          # [2, 1, R, C] against [3, P, C]
])
def test_oracle_matches_torch_autograd(ashape, bshape):
    rng = _rng(ashape, bshape)
    a, b = rng.standard_normal(ashape), rng.standard_normal(bshape)
    lead = torch.broadcast_shapes(ashape[:-2], bshape[:-2])
    g = rng.standard_normal(tuple(lead) + (ashape[-2], bshape[-2]))
    D, ga_ref, gb_ref = _torch_grads(a, b, g)
    ga, gb = G.broadcast_cdist_backward(a, b, D, g)
    _close(ga, ga_ref)
    _close(gb, gb_ref)


@pytest.mark.parametrize("shape", [(30, 16), (4, 24, 12)])
def test_self_oracle_matches_torch_autograd(shape):
    rng = _rng(shape)
    c = rng.random(shape)
    g = rng.standard_normal(shape[:-1] + (shape[-2],))
    D, gc_ref, _ = _torch_grads(c, None, g, same=True)
    _close(G.self_cdist_backward(c, D, g), gc_ref)


def test_exact_zero_distances():
    """a zero row on both sides: D == 0 there, the ratio is masked (ATen's rule), the gradients stay finite"""
    rng = _rng("zero")
    a, b = rng.standard_normal((2, 20, 8)), rng.standard_normal((2, 9, 8))
    a[:, 3] = 0.0
    b[:, 5] = 0.0
    g = rng.standard_normal((2, 20, 9))
    D, ga_ref, gb_ref = _torch_grads(a, b, g)
    assert (D[:, 3, 5] == 0).all()
    ga, gb = G.cdist_backward(a, b, D, g)
    assert np.isfinite(ga).all() and np.isfinite(gb).all()
    _close(ga, ga_ref)
    _close(gb, gb_ref)
    c = np.concatenate([a[0], np.zeros((1, 8))])          # a duplicate (zero) row: off-diagonal D == 0 in the self case
    gs = rng.standard_normal((21, 21))
    D, gc_ref, _ = _torch_grads(c, None, gs, same=True)
    _close(G.self_cdist_backward(c, D, gs), gc_ref)


def test_cdist_bwd_workspace_query_needs_no_device():
    """the size query allocates and launches nothing; like the other backward workspace queries it sizes the split-K
    partials from the device's SM count, which it reads when a device is present (148 without one)"""
    import videoad_b200 as V
    l = V._lib.lib()
    wb = l.vadc_cdist_bwd_workspace_bytes
    assert wb(1, 65536, 1024, 192) >= 65536 * 1024 * 4          # the ratio matrix
    assert wb(192, 16, 128, 784) >= 192 * 64 * 128 * 4           # batched: a batch's rows padded to 64
    assert wb(1, 37, 10, 20) > 0
    assert wb(0, 0, 0, 8) > 0
    assert wb(-1, 4, 4, 8) == 0


def test_cdist_bwd_argument_validation_happens_before_any_cuda_call():
    import videoad_b200 as V
    l = V._lib.lib()
    fb = l.vadc_cdist_bwd
    ws = 1 << 40
    f = 16                                                  # never dereferenced: every call below fails on the host
    #         a  b  dist g  nb  R   P   C  self ga gb ws bytes stream
    assert fb(f, f, f, f, -1, 32, 16, 8, 0, f, f, f, ws, None) == -1
    assert fb(f, f, f, f, 1, -32, 16, 8, 0, f, f, f, ws, None) == -1
    assert fb(f, f, f, f, 1, 32, -16, 8, 0, f, f, f, ws, None) == -1
    assert fb(f, f, f, f, 1, 32, 16, 0, 0, f, f, f, ws, None) == -1
    assert fb(f, f, f, f, 1, 32, 32, 8, 1, f, f, f, ws, None) == -1      # self: gb must be NULL
    assert fb(f, f, f, f, 1, 32, 16, 8, 1, f, None, f, ws, None) == -1   # self: R == P
    assert fb(f, f, None, f, 1, 32, 16, 8, 0, f, f, f, ws, None) == -2   # dist
    assert fb(f, f, f, None, 1, 32, 16, 8, 0, f, f, f, ws, None) == -2   # g
    assert fb(None, f, f, f, 1, 32, 16, 8, 0, f, f, f, ws, None) == -2
    assert fb(f, None, f, f, 1, 32, 16, 8, 0, f, f, f, ws, None) == -2
    assert fb(f, f, f, f, 1, 32, 16, 8, 0, f, f, None, ws, None) == -2   # workspace
    assert fb(f, f, f, f, 70000, 32, 16, 8, 0, f, f, f, ws, None) == -6
    assert fb(f, f, f, f, 1, 32, 16, 8, 0, f, f, f, 16, None) == -4      # short workspace
    assert fb(f, None, f, f, 1, 32, 32, 8, 1, f, None, f, 16, None) == -4
