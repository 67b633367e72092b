"""Gradients through the stand-alone cdist (euclid_dis, self_similarity) on the B200: every path of vadc_cdist_bwd —
SIMT, tensor-core one problem (transposed ga, split-K gb), batched (the space head's layout), torch.cdist's
leading-dimension broadcasting, the centroid self-distance — against float64 torch.cdist autograd."""
import os

import numpy as np
import pytest
import torch

import videoad_b200 as V
from gpu_util import N, T, dev, rel

pytestmark = pytest.mark.gpu

TOL = 3e-4          # the space head's gradients meet the same bar


def _ref(a, b, g, same=False, need=(True, True)):
    """float64 torch.cdist (exact distance form) autograd on the CPU -> (D, ga, gb)"""
    ta = torch.tensor(a, dtype=torch.float64, requires_grad=need[0])
    tb = ta if same else torch.tensor(b, dtype=torch.float64, requires_grad=need[1])
    D = torch.cdist(ta, tb, compute_mode="donot_use_mm_for_euclid_dist")
    (D * torch.tensor(g, dtype=torch.float64)).sum().backward()
    return D.detach().numpy(), ta.grad, None if same else tb.grad


def _run(a, b, g, need=(True, True)):
    ta, tb = T(a, grad=need[0]), T(b, grad=need[1])
    D = V.cdist(ta, tb)
    (D * T(g)).sum().backward()
    return D, ta.grad, tb.grad


def _check(a, b, need=(True, True), seed=0):
    g = _g(np.random.default_rng(seed), a, b)
    D64, ga64, gb64 = _ref(a, b, g, need=need)
    D, ga, gb = _run(a, b, g, need=need)
    assert tuple(D.shape) == D64.shape
    assert rel(N(D), D64) < 1e-5
    for got, want, n in ((ga, ga64, need[0]), (gb, gb64, need[1])):
        if n:
            assert torch.isfinite(got).all()
            assert rel(N(got), want.numpy()) < TOL
        else:
            assert got is None


def _g(rng, a, b):
    lead = torch.broadcast_shapes(np.shape(a)[:-2], np.shape(b)[:-2])
    return rng.standard_normal(tuple(lead) + (np.shape(a)[-2], np.shape(b)[-2])).astype(np.float32)


def _inputs(ashape, bshape, seed=1):
    rng = np.random.default_rng(seed)
    return rng.standard_normal(ashape).astype(np.float32), rng.standard_normal(bshape).astype(np.float32)


@pytest.mark.parametrize("R,P,C", [
    (37, 10, 24),          # SIMT: P % 8 != 0
    (37, 16, 20),          # SIMT: C % 8 != 0
    (8192, 1024, 192),     # tensor cores, ga transposed (C >= 128), split-K gb
    (20000, 64, 768),      # split-K gb with a ragged last k-block (20000 = 312 x 64 + 32)
    (4096, 256, 64),       # tensor cores, ga row per lane (C < 128)
])
def test_one_problem(R, P, C):
    a, b = _inputs((R, C), (P, C))
    _check(a, b)


@pytest.mark.parametrize("nb,R,P,C", [(24, 64, 128, 784), (192, 16, 128, 784), (6, 100, 40, 32),
                                       (4, 512, 40, 256), (4, 512, 72, 256)])
def test_batched(nb, R, P, C):
    """the space head's layout (a batch's rows padded to a k-block for the contraction over them), a SIMT shape, and
    tensor-core batches whose P is not a multiple of the 64-wide k-block: the batched ga contraction's last k-block
    reaches into the next batch's rows of b, which meet the zero-filled columns past P of r"""
    a, b = _inputs((nb, R, C), (nb, P, C))
    _check(a, b)


@pytest.mark.parametrize("ashape,bshape", [
    ((4, 512, 192), (256, 192)),      # 2-D b: a's leading dimensions fold into its rows (tensor cores)
    ((300, 64), (3, 200, 64)),        # 2-D a: b's leading dimensions fold into its rows
    ((2, 1, 96, 64), (3, 80, 64)),    # [2, 1, R, C] against [3, P, C]: expanded in torch
])
def test_broadcast(ashape, bshape):
    a, b = _inputs(ashape, bshape)
    _check(a, b)
    assert V.cdist(T(a), T(b)).shape == torch.cdist(torch.tensor(a), torch.tensor(b)).shape


def test_broadcast_mismatch_raises_torchs_error():
    a, b = torch.zeros(2, 5, 8, device=dev()), torch.zeros(3, 6, 8, device=dev())
    with pytest.raises(RuntimeError) as want:
        torch.cdist(a.cpu(), b.cpu())
    with pytest.raises(RuntimeError) as got:
        V.cdist(a, b)
    assert str(got.value) == str(want.value)


@pytest.mark.parametrize("need", [(True, False), (False, True), (True, True)])
def test_only_the_requested_gradients(need):
    a, b = _inputs((8192, 192), (1024, 192), seed=2)
    _check(a, b, need=need)
    a, b = _inputs((24, 64, 784), (24, 128, 784), seed=2)
    _check(a, b, need=need)


def test_zero_distances_give_finite_gradients():
    """exact zero rows on both sides: D == 0 there (the mm form gives 0 + 0 - 0), the ratio is masked as ATen masks it"""
    for ashape, bshape in (((37, 24), (10, 24)), ((4096, 192), (512, 192)), ((24, 64, 784), (24, 128, 784))):
        a, b = _inputs(ashape, bshape, seed=3)
        a[..., 5, :] = 0.0
        b[..., 3, :] = 0.0
        _check(a, b, seed=3)


def test_self_distance_of_the_native_head():
    """EuclidDistance_Assign_Module(192, 1024).self_similarity() (tensor cores) and a K = 30 head (SIMT) under a
    weighted-sum loss"""
    for C, K in ((192, 1024), (64, 30)):
        torch.manual_seed(K)
        m = V.EuclidDistance_Assign_Module(C, K).to(dev())
        S = m.self_similarity()
        w = torch.rand(K, K, device=dev())
        (S * w).sum().backward()
        _, gc64, _ = _ref(N(m.cluster_center), None, N(w), same=True)
        assert torch.isfinite(m.cluster_center.grad).all()
        assert rel(N(m.cluster_center.grad), gc64.numpy()) < TOL


def test_self_distance_batched_and_with_duplicate_rows():
    """the space head's live self-distance [192, 128, 784] (batched tensor cores), and two equal centroids (D == 0 off
    the diagonal)"""
    rng = np.random.default_rng(5)
    for shape in ((192, 128, 784), (40, 16)):
        c = rng.random(shape).astype(np.float32)
        c[..., 7, :] = c[..., 2, :]
        tc = T(c, grad=True)
        S = V.cdist(tc, tc)
        w = rng.random(S.shape).astype(np.float32)
        (S * T(w)).sum().backward()
        _, gc64, _ = _ref(c, None, w, same=True)
        assert torch.isfinite(tc.grad).all()
        assert rel(N(tc.grad), gc64.numpy()) < TOL


def test_bf16x3_mode():
    """VADC_TC_BF16X3=1 selects the three-term bf16 split of the operands"""
    from videoad_b200 import _lib
    os.environ["VADC_TC_BF16X3"] = "1"
    _lib.lib().vadc_refresh_env()
    try:
        _check(*_inputs((8192, 192), (1024, 192), seed=4))
        _check(*_inputs((24, 64, 784), (24, 128, 784), seed=4))
    finally:
        os.environ.pop("VADC_TC_BF16X3", None)
        _lib.lib().vadc_refresh_env()


def test_deterministic_and_graph_capturable():
    """two backward calls give bit-identical gradients; forward + backward captured in a CUDA graph on a side stream and
    replayed once equal the eager result"""
    for ashape, bshape in (((8192, 192), (1024, 192)), ((24, 64, 784), (24, 128, 784)), ((37, 24), (10, 24))):
        a, b = _inputs(ashape, bshape, seed=6)
        g = T(_g(np.random.default_rng(6), a, b))
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            ta, tb = T(a, grad=True), T(b, grad=True)

            def step():
                ta.grad = tb.grad = None
                (V.cdist(ta, tb) * g).sum().backward()
                return ta.grad, tb.grad

            e1 = [t.clone() for t in step()]
            e2 = [t.clone() for t in step()]
            for x, y in zip(e1, e2):
                assert torch.equal(x, y)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=side):
                cap = step()
            graph.replay()
            side.synchronize()
            for x, y in zip(cap, e1):
                assert torch.equal(x, y)
        torch.cuda.current_stream().wait_stream(side)


def test_empty_inputs_give_torchs_shapes_and_zero_gradients():
    """R == 0, P == 0, an empty leading dimension and an empty self-distance: torch.cdist's (empty) result, and
    gradients that are zero where the input is not empty"""
    cases = (((2, 0, 8), (2, 5, 8)), ((2, 4, 8), (2, 0, 8)), ((0, 4, 8), (0, 5, 8)), ((2, 0, 8), (5, 8)),
             ((4, 8), (2, 0, 8)), ((2, 1, 0, 8), (3, 5, 8)))
    for ashape, bshape in cases:
        ta, tb = torch.zeros(ashape, device=dev(), requires_grad=True), torch.ones(bshape, device=dev(), requires_grad=True)
        D = V.cdist(ta, tb)
        assert D.shape == torch.cdist(torch.zeros(ashape), torch.ones(bshape)).shape
        D.sum().backward()
        assert ta.grad.shape == ta.shape and tb.grad.shape == tb.shape
        assert (ta.grad == 0).all() and (tb.grad == 0).all()
    for shape in ((0, 8), (3, 0, 8)):            # self-distance with K == 0
        tc = torch.ones(shape, device=dev(), requires_grad=True)
        S = V.cdist(tc, tc)
        assert S.shape == torch.cdist(torch.ones(shape), torch.ones(shape)).shape
        S.sum().backward()
        assert tc.grad.shape == tc.shape
    m = V.EuclidDistance_Assign_Module(8, 0).to(dev())
    S = m.self_similarity()
    assert S.shape == (0, 0)
    S.sum().backward()
    assert m.cluster_center.grad.shape == (0, 8)
