"""Memory: gradient with respect to learnable memory items (keys) through read (Memory.py:255) and MemoryLoss
(:52-59), against the float64 oracle"""
import os
import threading

import numpy as np
import pytest
import torch

import videoad_b200 as V
from oracle import np_oracle as O
from oracle import ref_port as P
from conftest import load_golden
from gpu_util import T, N, rel, dev
from keys_oracle import memory_keys_backward, separateness_sign
from test_gpu_space_memory import _TwoRanks

pytestmark = pytest.mark.gpu

TIE = 1e-5


def _inputs(name_or_shape, seed=0):
    if isinstance(name_or_shape, str):
        g = load_golden(name_or_shape)
        query, keys = g["query"], g["keys"]
        W = g["g_updated_query"]
    else:
        B, d, h, w, m = name_or_shape
        rng = np.random.default_rng(seed + m + d)
        keys = rng.random((m, d)).astype(np.float32)
        keys /= np.linalg.norm(keys, axis=1, keepdims=True)
        query = rng.standard_normal((B, d, h, w)).astype(np.float32)
        W = rng.standard_normal((B, 2 * d, h, w)).astype(np.float32)
    return query, keys, W


def assert_keys_grad(got, query, keys, W, g_sep):
    """2e-5 of the largest entry against the oracle with sgn(S) = 0 inside the tie band |S| < 1e-5; a row with t tie
    entries may differ by t max|k| |g_sep| / (m (m-1)) more (the sign of a rounding-noise S is either)"""
    m = keys.shape[0]
    ref = memory_keys_backward(query, keys, W, g_sep, tie=TIE)
    err = np.abs(np.asarray(got, np.float64) - ref)
    slack = 0.0
    if g_sep is not None:
        k = np.asarray(keys, np.float64)
        S = k @ k.T / 2 + 0.5 - np.eye(m)
        ties = (np.abs(S) < TIE).sum(1)
        slack = ties * np.abs(k).max() * abs(g_sep) / (m * (m - 1))
    bound = 2e-5 * np.abs(ref).max() + slack
    assert (err.max(1) <= bound).all(), (err.max(), np.abs(ref).max(), float(np.max(slack)))


def _run(mem, query, keys, W, train, cu, cs):
    q = T(query).requires_grad_(True)
    k = T(keys).requires_grad_(True)
    o = mem(q, k, train=train)
    loss = 0.7 * o[4] + (0.3 * o[5] if train else 0)
    if cu:
        loss = loss + cu * (o[0] * T(W)).sum()
    if cs:
        loss = loss + cs * V.MemoryLoss(k)
    loss.backward()
    return q, k, o


SHAPES = ["memory_d32_m10", "memory_d64_m50", (2, 768, 32, 32, 2000), (1, 96, 7, 5, 33)]


@pytest.mark.parametrize("train", [True, False])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: s if isinstance(s, str) else "x".join(map(str, s)))
def test_keys_grad_vs_oracle(shape, train):
    """read alone, MemoryLoss alone, both; the query gradient is the one of the query-only path"""
    query, keys, W = _inputs(shape)
    m, d = keys.shape
    mem = V.Memory(m, d, d, 0.1, 0.1)
    f = O.memory_forward(query, keys, train=True, dtype=np.float64)
    for cu, cs in [(1.0, None), (0.0, 1.3), (1.0, 1.3)]:
        q, k, o = _run(mem, query, keys, W, train, cu, cs)
        assert_keys_grad(N(k.grad), query, keys, W * cu if cu else None, cs)
        qref = O.memory_query_backward(query, keys, f["top1"], f["top2"] if train else None, W * cu if cu else None,
                                       0.7, 0.3 if train else None)
        assert rel(N(q.grad), qref) < 2e-5, (cu, cs)


def test_keys_grad_three_term_mode():
    """VADC_MEMORY_TERMS=3 selects the bf16 x3 split for the keys contraction as for the forward"""
    from videoad_b200 import _lib
    os.environ["VADC_MEMORY_TERMS"] = "3"
    _lib.lib().vadc_refresh_env()
    try:
        for shape in [(2, 768, 32, 32, 2000), (1, 96, 7, 5, 33)]:
            query, keys, W = _inputs(shape)
            m, d = keys.shape
            _, k, _ = _run(V.Memory(m, d, d, 0.1, 0.1), query, keys, W, True, 1.0, 1.3)
            assert_keys_grad(N(k.grad), query, keys, W, 1.3)
    finally:
        os.environ.pop("VADC_MEMORY_TERMS", None)
        _lib.lib().vadc_refresh_env()


def test_memory_loss_ties_on_unit_norm_keys():
    """unit-norm keys put S_ii = (|k_i|^2 - 1)/2 at rounding noise, in the reference too: either sign is accepted there"""
    rng = np.random.default_rng(3)
    keys = O.l2_normalize(rng.standard_normal((300, 64)).astype(np.float32), 1)
    assert (np.abs(np.diag(separateness_sign(keys))) <= 1).all()
    k = T(keys).requires_grad_(True)
    V.MemoryLoss(k).backward()
    assert_keys_grad(N(k.grad), np.zeros((1, 64, 1, 1), np.float32), keys, None, 1.0)


def test_keys_grad_full_size():
    """N = 65536 tokens (B=64, 32x32), m = 2000, d = 768 against a float64 GEMM of the returned score_memory with W"""
    B, d, h, w, m = 64, 768, 32, 32, 2000
    g = torch.Generator(device="cuda").manual_seed(7)
    query = torch.randn(B, d, h, w, device=dev(), generator=g)
    keys = torch.nn.functional.normalize(torch.rand(m, d, device=dev(), generator=g), dim=1).requires_grad_(True)
    W = torch.randn(B, 2 * d, h, w, device=dev(), generator=g)
    mem = V.Memory(m, d, d, 0.1, 0.1)
    uq, um, sq, sm, gl, sl = mem(query, keys, train=True)
    (uq * W).sum().backward()
    gr = W[:, d:].permute(0, 2, 3, 1).reshape(-1, d).double()
    ref = sm.detach().double().t() @ gr
    assert float((keys.grad.double() - ref).abs().max() / ref.abs().max()) < 2e-4


def test_plain_keys_take_the_query_only_path():
    query, keys, W = _inputs((2, 96, 8, 8, 40))
    m, d = keys.shape
    mem = V.Memory(m, d, d, 0.1, 0.1)
    counts = []
    for learnable in (False, True):
        q = T(query).requires_grad_(True)
        k = T(keys).requires_grad_(learnable)
        o = mem(q, k, train=True)
        loss = (o[0] * T(W)).sum() + 0.7 * o[4] + 0.3 * o[5]
        torch.cuda.synchronize()
        c0 = V.launch_count()
        loss.backward()
        counts.append(V.launch_count() - c0)
        if not learnable:
            assert k.grad is None
    assert counts[0] == 1 and counts[1] > 1, counts                  # vadc_memory_query_bwd alone without learnable keys


def test_keys_grad_two_shards_sum_to_full_batch():
    """Memory.global_batch: each rank's g_keys is its tokens' share; the two shares sum to the full-batch g_keys"""
    d, h, w, m = 768, 16, 16, 2000
    rng = np.random.default_rng(m)
    keys = rng.random((m, d)).astype(np.float32)
    keys /= np.linalg.norm(keys, axis=1, keepdims=True)
    query = rng.standard_normal((2, d, h, w)).astype(np.float32)
    query[1] *= 1.7
    W = rng.standard_normal((2, 2 * d, h, w)).astype(np.float32)
    kf = T(keys).requires_grad_(True)
    of = V.Memory(m, d, d, 0.1, 0.1)(T(query), kf, train=True)
    ((of[0] * T(W)).sum() + 0.7 * of[4] + 0.3 * of[5]).backward()

    ranks, out = _TwoRanks(), [None, None]

    def run(rank):
        ranks.lock.acquire()
        try:
            mem = V.Memory(m, d, d, 0.1, 0.1)
            mem.global_batch, mem._reduce = True, ranks.reducer(rank)
            k = T(keys).requires_grad_(True)
            o = mem(T(query[rank:rank + 1]), k, train=True)
            ((o[0] * T(W[rank:rank + 1])).sum() + 0.7 * o[4] + 0.3 * o[5]).backward()
            out[rank] = k.grad
        finally:
            ranks.lock.release()

    th = [threading.Thread(target=run, args=(r,)) for r in range(2)]
    [t.start() for t in th]
    [t.join(timeout=120) for t in th]
    assert out[0] is not None and out[1] is not None
    assert rel(N(out[0] + out[1]), N(kf.grad)) < 2e-5


def test_keys_grad_is_bit_identical_across_backwards():
    query, keys, W = _inputs((2, 768, 32, 32, 2000))
    m, d = keys.shape
    mem = V.Memory(m, d, d, 0.1, 0.1)
    a = _run(mem, query, keys, W, True, 1.0, 1.3)[1].grad
    b = _run(mem, query, keys, W, True, 1.0, 1.3)[1].grad
    assert torch.equal(a, b)


def test_learnable_keys_sgd_matches_float64_chain():
    """three plain SGD steps on an nn.Parameter of memory items with MemoryLoss in the loss, against the same steps
    through the reference op chain in float64 (oracle/ref_port.py) with torch autograd"""
    g = load_golden("memory_d64_m50")
    query, W = g["query"], g["g_updated_query"]
    keys0 = g["keys"].astype(np.float64) * 0.8                 # off the unit sphere: no sign ties in MemoryLoss
    m, d = keys0.shape
    lr = 0.1
    mem = V.Memory(m, d, d, 0.1, 0.1)
    kp = torch.nn.Parameter(T(keys0))
    opt = torch.optim.SGD([kp], lr=lr)
    kr = torch.tensor(keys0, requires_grad=True)
    qr, Wr = torch.tensor(query, dtype=torch.float64), torch.tensor(W, dtype=torch.float64)
    for _ in range(3):
        opt.zero_grad()
        o = mem(T(query), kp, train=True)
        ((o[0] * T(W)).sum() + 0.7 * o[4] + 0.3 * o[5] + 2.0 * V.MemoryLoss(kp)).backward()
        opt.step()
        r = P.memory_forward(qr, kr, train=True)
        lr_ = (r[0] * Wr).sum() + 0.7 * r[4] + 0.3 * r[5]
        lr_ = lr_ + 2.0 * torch.sum(torch.abs(kr @ kr.t() / 2 + 0.5 - torch.eye(m, dtype=torch.float64))) / (m * (m - 1))
        gk, = torch.autograd.grad(lr_, kr)
        with torch.no_grad():
            kr = (kr - lr * gk).requires_grad_(True)
    got, want = N(kp).astype(np.float64), kr.detach().numpy()
    assert np.abs(got - want).max() < 1e-5 * np.abs(want).max()
