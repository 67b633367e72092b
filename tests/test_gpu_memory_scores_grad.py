"""Memory.differentiable_scores: gradients through the returned score_query / score_memory (get_score,
Memory.py:133-143) to the query and learnable memory items, against the float64 oracle"""
import os
import threading

import numpy as np
import pytest
import torch

import videoad_b200 as V
from oracle import ref_port as P
from conftest import load_golden
from gpu_util import T, N, rel, dev
from scores_oracle import memory_backward, entropy_grad, cancellation_scales
from test_gpu_space_memory import _TwoRanks

pytestmark = pytest.mark.gpu

TIE = 1e-5
# (Wq, Wm, entropy, with <updated_query, W>, gathering, spreading and MemoryLoss)
LOSSES = [(1, 1, 0, 0), (0, 0, 1, 0), (1, 0, 0, 0), (1, 1, 0, 1), (0, 0, 1, 1)]


def _inputs(name_or_shape, seed=0):
    if isinstance(name_or_shape, str):
        g = load_golden(name_or_shape)
        query, keys, W = g["query"], g["keys"], g["g_updated_query"]
    else:
        B, d, h, w, m = name_or_shape
        rng = np.random.default_rng(seed + m + d)
        keys = rng.random((m, d)).astype(np.float32)
        keys /= np.linalg.norm(keys, axis=1, keepdims=True)
        query = rng.standard_normal((B, d, h, w)).astype(np.float32)
        W = rng.standard_normal((B, 2 * d, h, w)).astype(np.float32)
    B, d, h, w = query.shape
    rng = np.random.default_rng(seed + 1)
    n, m = B * h * w, keys.shape[0]
    return query, keys, W, rng.standard_normal((n, m)).astype(np.float32), rng.standard_normal((n, m)).astype(np.float32)


def _memory(m, d):
    mem = V.Memory(m, d, d, 0.1, 0.1)
    mem.differentiable_scores = True
    return mem


def _loss(o, k, W, Wq, Wm, train, loss, learnable, n_all=None):
    lq, lm, ent, rest = loss
    sq, sm = o[2], o[3]
    L = 0
    if lq:
        L = L + (sq * T(Wq)).sum()
    if lm:
        L = L + (sm * T(Wm)).sum()
    if ent:
        L = L - (sm * torch.log(sm)).sum() / (n_all or sm.shape[0])
    if rest:
        L = L + (o[0] * T(W)).sum() + 0.7 * o[4] + (0.3 * o[5] if train else 0)
        if learnable:
            L = L + 1.3 * V.MemoryLoss(k)
    return L


def _run(mem, query, keys, W, Wq, Wm, train, loss, learnable=True):
    q = T(query).requires_grad_(True)
    k = T(keys).requires_grad_(learnable)
    o = mem(q, k, train=train)
    _loss(o, k, W, Wq, Wm, train, loss, learnable).backward()
    return q, k


def _reference(query, keys, W, Wq, Wm, train, loss):
    """(g_query, g_keys, S_q, S_k): the float64 gradients and the size of the score share's terms (cancellation_scales)"""
    lq, lm, ent, rest = loss
    g_sq = Wq if lq else None
    g_sm = ((Wm if lm else 0) + (entropy_grad(query, keys) if ent else 0)) if (lm or ent) else None
    gq, gk = memory_backward(query, keys, train, W if rest else None, 0.7 if rest else None, 0.3 if rest else None,
                             g_sq, g_sm, 1.3 if rest else None, tie=TIE)
    return (gq, gk) + cancellation_scales(query, keys, g_sq, g_sm)


def assert_query_grad(got, ref, scale, what=None):
    """2e-5 of the largest entry, or 2e-6 of the size of the score share's terms where they cancel to far less than
    that (an entropy loss alone: fp32 autograd of the reference chain misses the float64 result by 2e-3 of its max)"""
    err = np.abs(np.asarray(got, np.float64) - ref).max()
    assert err <= max(2e-5 * np.abs(ref).max(), 2e-6 * scale), (what, err, np.abs(ref).max(), scale)


def assert_keys_grad(got, ref, keys, g_sep, scale=0.0):
    """2e-5 of the largest entry (or 2e-6 of the size of the score share's terms, as for the query); a row with t
    MemoryLoss sign ties (|S| < 1e-5, e.g. the diagonal of unit-norm keys: either sign is the reference's too) may
    differ by t max|k| |g_sep| / (m (m-1)) more"""
    m = keys.shape[0]
    err = np.abs(np.asarray(got, np.float64) - ref)
    slack = 0.0
    if g_sep:
        k = np.asarray(keys, np.float64)
        ties = (np.abs(k @ k.T / 2 + 0.5 - np.eye(m)) < TIE).sum(1)
        slack = ties * np.abs(k).max() * g_sep / (m * (m - 1))
    bound = max(2e-5 * np.abs(ref).max(), 2e-6 * scale)
    assert (err.max(1) <= bound + slack).all(), (err.max(), np.abs(ref).max(), scale)


SHAPES = ["memory_d32_m10", "memory_d64_m50", (2, 768, 32, 32, 2000), (1, 96, 7, 5, 33), (3, 64, 8, 8, 2),
          (1, 20, 3, 3, 7)]


@pytest.mark.parametrize("train", [True, False])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: s if isinstance(s, str) else "x".join(map(str, s)))
def test_scores_grad_vs_oracle(shape, train):
    """each score loss alone and with every other loss, plain and learnable keys"""
    query, keys, W, Wq, Wm = _inputs(shape)
    m, d = keys.shape
    mem = _memory(m, d)
    for loss in LOSSES:
        gq_ref, gk_ref, sq_, sk_ = _reference(query, keys, W, Wq, Wm, train, loss)
        for learnable in (False, True):
            q, k = _run(mem, query, keys, W, Wq, Wm, train, loss, learnable)
            assert_query_grad(N(q.grad), gq_ref, sq_, (loss, learnable))
            if learnable:
                assert_keys_grad(N(k.grad), gk_ref, keys, 1.3 if loss[3] else None, sk_)
            else:
                assert k.grad is None


def test_scores_grad_three_term_mode():
    """VADC_MEMORY_TERMS=3 selects the bf16 x3 split for both contractions as for the forward"""
    from videoad_b200 import _lib
    os.environ["VADC_MEMORY_TERMS"] = "3"
    _lib.lib().vadc_refresh_env()
    try:
        for shape in [(2, 768, 32, 32, 2000), (1, 96, 7, 5, 33), (1, 20, 3, 3, 7)]:
            query, keys, W, Wq, Wm = _inputs(shape)
            m, d = keys.shape
            for loss in [(1, 1, 1, 1), (0, 0, 1, 0)]:
                gq_ref, gk_ref, sq_, sk_ = _reference(query, keys, W, Wq, Wm, True, loss)
                q, k = _run(_memory(m, d), query, keys, W, Wq, Wm, True, loss)
                assert_query_grad(N(q.grad), gq_ref, sq_, (shape, loss))
                assert_keys_grad(N(k.grad), gk_ref, keys, 1.3 if loss[3] else None, sk_)
    finally:
        os.environ.pop("VADC_MEMORY_TERMS", None)
        _lib.lib().vadc_refresh_env()


def test_scores_grad_full_size():
    """N = 65536 tokens (B=64, 32x32), m = 2000, d = 768: g_s, g_s K, the normalize backward and g_s^T q-hat in float64
    on the GPU from the returned score matrices"""
    B, d, h, w, m = 64, 768, 32, 32, 2000
    g = torch.Generator(device="cuda").manual_seed(11)
    query = torch.randn(B, d, h, w, device=dev(), generator=g)
    keys = torch.nn.functional.normalize(torch.rand(m, d, device=dev(), generator=g), dim=1).requires_grad_(True)
    Wq = torch.randn(B * h * w, m, device=dev(), generator=g)
    q = query.clone().requires_grad_(True)
    o = _memory(m, d)(q, keys, train=True)
    sq, sm = o[2], o[3]
    ((sq * Wq).sum() - (sm * torch.log(sm)).sum(1).mean()).backward()
    with torch.no_grad():
        sq, sm = sq.double(), sm.double()
        Gq, Gm = Wq.double(), -(torch.log(sm) + 1.0) / sm.shape[0]
        gs = sq * (Gq - (Gq * sq).sum(0, keepdim=True)) + sm * (Gm - (Gm * sm).sum(1, keepdim=True))
        del sq, sm, Gq, Gm
        x = query.double().permute(0, 2, 3, 1).reshape(-1, d)
        nrm = x.norm(dim=1, keepdim=True).clamp_min(1e-12)
        qh = x / nrm
        k64 = keys.detach().double()
        gk_ref = gs.t() @ qh
        gh = gs @ k64
        del gs
        gx = (gh - qh * (qh * gh).sum(1, keepdim=True)) / nrm
        gq_ref = gx.reshape(B, h, w, d).permute(0, 3, 1, 2)
    assert float((q.grad.double() - gq_ref).abs().max() / gq_ref.abs().max()) < 2e-4
    assert float((keys.grad.double() - gk_ref).abs().max() / gk_ref.abs().max()) < 2e-4


def _saved_and_launches(mem, query, keys, W, learnable, score_loss):
    """(tensors the forward saves, backward launches) of <updated_query, W> + gathering + spreading (+ a score loss)"""
    q = T(query).requires_grad_(True)
    k = T(keys).requires_grad_(learnable)
    packed = []
    with torch.autograd.graph.saved_tensors_hooks(lambda t: packed.append(t) or t, lambda t: t):
        o = mem(q, k, train=True)
    loss = (o[0] * T(W)).sum() + 0.7 * o[4] + 0.3 * o[5]
    if score_loss:
        loss = loss + o[3].sum()
    torch.cuda.synchronize()
    c0 = V.launch_count()
    loss.backward()
    return len(packed), V.launch_count() - c0, o


def test_attribute_off_and_unused_scores_change_nothing():
    query, keys, W, _, _ = _inputs((2, 96, 8, 8, 40))
    m, d = keys.shape
    off = V.Memory(m, d, d, 0.1, 0.1)
    assert off.differentiable_scores is False
    for learnable in (False, True):
        n_off, l_off, o = _saved_and_launches(off, query, keys, W, learnable, False)
        assert not o[2].requires_grad and not o[3].requires_grad and not o[1].requires_grad
        if not learnable:
            assert (n_off, l_off) == (4, 1)                   # qc, keys, top1, top2; vadc_memory_query_bwd alone
        n_on, l_on, o = _saved_and_launches(_memory(m, d), query, keys, W, learnable, False)
        assert o[2].requires_grad and o[3].requires_grad and not o[1].requires_grad
        assert l_on == l_off, (learnable, l_on, l_off)         # no loss on the scores: no extra launch
        assert n_on == 6                                       # ... and both score matrices are kept
    # a loss on score_memory with the attribute off is silently dropped exactly as before
    q = T(query).requires_grad_(True)
    o = off(q, T(keys), train=True)
    ((o[0] * T(W)).sum() + o[3].sum()).backward()
    ref = T(query).requires_grad_(True)
    (off(ref, T(keys), train=True)[0] * T(W)).sum().backward()
    assert torch.equal(q.grad, ref.grad)


def test_scores_grad_two_shards_equal_full_batch():
    """Memory.global_batch: each rank's q.grad is its shard of the full-batch q.grad, the two g_keys sum to the full one
    (the column dots of score_query are all-reduced in the backward)"""
    d, h, w, m = 768, 16, 16, 2000
    query, keys, W, Wq, Wm = _inputs((2, d, h, w, m), seed=5)
    query[1] *= 1.7
    n_all = 2 * h * w
    loss = (1, 1, 1, 1)
    qf = T(query).requires_grad_(True)
    kf = T(keys).requires_grad_(True)
    of = _memory(m, d)(qf, kf, train=True)
    _loss(of, kf, W, Wq, Wm, True, loss, False, n_all).backward()

    # The forwards run in two threads that exchange their reductions.  Both backwards would run on autograd's one
    # worker thread for the device, where a blocking exchange cannot happen, so each rank's backward first runs once
    # to record its column dots and then once more with the other rank's recorded dots added.
    ranks, phase, recorded = _TwoRanks(), ["fwd"], [None, None]

    def reducer(rank):
        fwd = ranks.reducer(rank)

        def reduce(t, op):
            if phase[0] == "fwd":
                return fwd(t, op)
            if phase[0] == "record":
                recorded[rank] = t.clone()
                return t
            return t + recorded[1 - rank]
        return reduce

    inp, losses = [None, None], [None, None]

    def run(rank):
        ranks.lock.acquire()
        try:
            mem = _memory(m, d)
            mem.global_batch, mem._reduce = True, reducer(rank)
            inp[rank] = (T(query[rank:rank + 1]).requires_grad_(True), T(keys).requires_grad_(True))
            o = mem(*inp[rank], train=True)
            rows = slice(rank * h * w, (rank + 1) * h * w)
            losses[rank] = _loss(o, inp[rank][1], W[rank:rank + 1], Wq[rows], Wm[rows], True, loss, False, n_all)
        finally:
            ranks.lock.release()

    th = [threading.Thread(target=run, args=(r,)) for r in range(2)]
    [t.start() for t in th]
    [t.join(timeout=120) for t in th]
    assert losses[0] is not None and losses[1] is not None
    phase[0] = "record"
    for r in range(2):
        losses[r].backward(retain_graph=True)
        inp[r][0].grad = inp[r][1].grad = None
    phase[0] = "replay"
    for r in range(2):
        losses[r].backward()
    for r in range(2):
        assert rel(N(inp[r][0].grad), N(qf.grad[r:r + 1])) < 2e-5, r
    assert rel(N(inp[0][1].grad + inp[1][1].grad), N(kf.grad)) < 2e-5


def test_scores_grad_is_bit_identical_across_backwards():
    query, keys, W, Wq, Wm = _inputs((2, 768, 32, 32, 2000))
    m, d = keys.shape
    mem = _memory(m, d)
    a = _run(mem, query, keys, W, Wq, Wm, True, (1, 1, 1, 1))
    b = _run(mem, query, keys, W, Wq, Wm, True, (1, 1, 1, 1))
    assert torch.equal(a[0].grad, b[0].grad) and torch.equal(a[1].grad, b[1].grad)


def test_learnable_keys_sgd_with_entropy_matches_float64_chain():
    """three plain SGD steps on an nn.Parameter of memory items with an entropy penalty on score_memory and MemoryLoss,
    against the same steps through the reference op chain in float64 (oracle/ref_port.py) with torch autograd"""
    g = load_golden("memory_d64_m50")
    query, W = g["query"], g["g_updated_query"]
    keys0 = g["keys"].astype(np.float64) * 0.8                 # off the unit sphere: no sign ties in MemoryLoss
    m, d = keys0.shape
    lr = 0.1
    mem = _memory(m, d)
    kp = torch.nn.Parameter(T(keys0))
    opt = torch.optim.SGD([kp], lr=lr)
    kr = torch.tensor(keys0, requires_grad=True)
    qr, Wr = torch.tensor(query, dtype=torch.float64), torch.tensor(W, dtype=torch.float64)
    for _ in range(3):
        opt.zero_grad()
        o = mem(T(query), kp, train=True)
        ent = -(o[3] * torch.log(o[3])).sum(1).mean()
        ((o[0] * T(W)).sum() + 0.7 * o[4] + 0.3 * o[5] + 5.0 * ent + 2.0 * V.MemoryLoss(kp)).backward()
        opt.step()
        r = P.memory_forward(qr, kr, train=True)
        lr_ = (r[0] * Wr).sum() + 0.7 * r[4] + 0.3 * r[5] - 5.0 * (r[3] * torch.log(r[3])).sum(1).mean()
        lr_ = lr_ + 2.0 * torch.sum(torch.abs(kr @ kr.t() / 2 + 0.5 - torch.eye(m, dtype=torch.float64))) / (m * (m - 1))
        gk, = torch.autograd.grad(lr_, kr)
        with torch.no_grad():
            kr = (kr - lr * gk).requires_grad_(True)
    got, want = N(kp).astype(np.float64), kr.detach().numpy()
    assert np.abs(got - want).max() < 1e-5 * np.abs(want).max()
