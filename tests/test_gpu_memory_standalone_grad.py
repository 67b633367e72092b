"""Gradients of Memory's stand-alone methods (get_score, read, gather_loss, spread_loss, prepare_query) against the
float64 oracle (standalone_oracle.py), the reference's forward composed from them, and what they launch."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import videoad_b200 as V
import standalone_oracle as S
from conftest import load_golden
from gpu_util import T, N, dev
from test_gpu_memory_scores_grad import TIE

pytestmark = pytest.mark.gpu

SHAPES = ["memory_d32_m10", "memory_d64_m50", (2, 768, 32, 32, 2000), (1, 96, 7, 5, 33), (3, 64, 8, 8, 2),
          (1, 20, 3, 3, 7)]
SHAPE_IDS = lambda s: s if isinstance(s, str) else "x".join(map(str, s))   # noqa: E731


def _inputs(shape, seed=0):
    if isinstance(shape, str):
        g = load_golden(shape)
        query, keys = g["query"], g["keys"]
    else:
        B, d, h, w, m = shape
        rng = np.random.default_rng(seed + m + d)
        keys = rng.random((m, d)).astype(np.float32)
        keys /= np.linalg.norm(keys, axis=1, keepdims=True)
        query = rng.standard_normal((B, d, h, w)).astype(np.float32)
    B, d, h, w = query.shape
    m = keys.shape[0]
    rng = np.random.default_rng(seed + 1)
    n = B * h * w
    W = rng.standard_normal((B, 2 * d, h, w)).astype(np.float32)
    Wq, Wm = rng.standard_normal((n, m)).astype(np.float32), rng.standard_normal((n, m)).astype(np.float32)
    return query, keys, W, Wq, Wm


def _terms(n):
    os.environ.pop("VADC_MEMORY_TERMS", None)
    if n == 3:
        os.environ["VADC_MEMORY_TERMS"] = "3"
    V._lib.lib().vadc_refresh_env()


@pytest.fixture
def terms():
    yield _terms
    _terms(2)


# every loss: (get_score <sq,Wq> + <sm,Wm>, entropy on sm, read <uq,W>, gathering, spreading)
LOSSES = {"get_score": (1, 0, 0, 0, 0), "entropy": (0, 1, 0, 0, 0), "read": (0, 0, 1, 0, 0),
          "gather": (0, 0, 0, 1, 0), "spread": (0, 0, 0, 0, 1), "all": (1, 1, 1, 1, 1)}


def _ours(mem, q4, k, W, Wq, Wm, loss):
    ls, ent, rd, ga, sp = loss
    L = 0
    if ls or ent:
        sq, sm = mem.get_score(k, q4)
        if ls:
            L = L + (sq * T(Wq)).sum() + (sm * T(Wm)).sum()
        if ent:
            L = L - (sm * torch.log(sm)).sum(1).mean()
    if rd:
        uq, sq, sm = mem.read(q4, k)
        L = L + (uq * T(W)).sum() + (((sq * T(Wq)).sum() + (sm * T(Wm)).sum()) if ls else 0)
    if ga:
        L = L + 0.7 * mem.gather_loss(q4, k, True)
    if sp:
        L = L + 0.3 * mem.spread_loss(q4, k, True)
    return L


def _oracle(qr, keys, W, Wq, Wm, loss, kernel_top, learnable):
    """(g_q [N,d], g_keys, S_q, S_k) in float64 for the loss of _ours (get_score's score losses count twice when the
    read also runs: once through get_score, once through read's own matrices)"""
    ls, ent, rd, ga, sp = loss
    m = keys.shape[0]
    g_sq = g_sm = None
    mult = 2.0 if (ls and rd) else 1.0
    if ls:
        g_sq, g_sm = mult * Wq, mult * Wm
    if ent:
        e = S.entropy_grad(S.scores(qr, keys)[1])
        g_sm = e if g_sm is None else g_sm + e
    gq, gk = S.read_backward(qr, keys, W if rd else None, g_sq, g_sm)
    top1, top2 = S.picks(qr, keys, kernel_top)
    if ga:
        gq = gq + S.gather_backward(qr, keys, 0.7, top1)
    if sp and m > 1:
        gq = gq + S.spread_backward(qr, keys, 0.3, top1, top2)
    if learnable and ga:                                     # _run adds MemoryLoss with the gathering loss
        gk = gk + S.memory_loss_backward(keys, 1.3, tie=TIE)
    sq_, sk_ = S.cancellation_scales(qr, keys, g_sq, g_sm)
    return gq, gk, sq_, sk_


def _check(got, ref, scale, what, slack=None):
    """2e-5 of the largest reference entry, or 2e-6 of the size of the score share's terms where they cancel (an
    entropy loss alone; the cancellation_scales rule of test_gpu_memory_scores_grad.py); ``slack`` per row: MemoryLoss
    sign ties of unit-norm keys"""
    err = (got.double() - ref).abs()
    bound = max(2e-5 * float(ref.abs().max()), 2e-6 * scale)
    if slack is None:
        assert float(err.max()) <= bound, (what, float(err.max()), float(ref.abs().max()), scale)
    else:
        assert bool((err.max(1).values <= bound + slack).all()), (what, float(err.max()), float(ref.abs().max()))


def _tie_slack(keys):
    m = keys.shape[0]
    ties = ((keys @ keys.t() / 2 + 0.5 - torch.eye(m, dtype=keys.dtype, device=keys.device)).abs() < TIE).sum(1)
    return ties * keys.abs().max() * 1.3 / max(m * (m - 1), 1)


def _run_case(mem, query, keys, W, Wq, Wm, name, learnable, view):
    """one loss, our methods against the oracle; view: the query is F.normalize(x, dim=1).permute(0,2,3,1) of a leaf
    x (as the reference's forward hands it over), else a contiguous channel-last leaf.  Where float64 sees a near-tie
    in top1 / top2 (a logit gap below 1e-6 relative), the oracle uses the picks the kernel returned (S.picks)."""
    loss = LOSSES[name]
    B, d, h, w = query.shape
    m = keys.shape[0]
    if loss[4] and m < 2:
        return
    x = T(query).requires_grad_(True)
    if view:
        q4 = F.normalize(x, dim=1).permute(0, 2, 3, 1)
    else:
        x = F.normalize(T(query), dim=1).permute(0, 2, 3, 1).contiguous().mul(1.3).requires_grad_(True)
        q4 = x
    k = T(keys).requires_grad_(learnable)
    L = _ours(mem, q4, k, W, Wq, Wm, loss)
    if learnable and loss[3]:
        L = L + 1.3 * V.MemoryLoss(k)
    L.backward()
    qr32 = q4.detach().reshape(-1, d).contiguous()
    kt = V.memory._compute_scores(qr32, T(keys), False)
    qr, k64 = qr32.double(), T(keys).double()
    gq, gk, sq_, sk_ = _oracle(qr, k64, T(W).double(), T(Wq).double(), T(Wm).double(), loss, (kt.top1, kt.top2),
                               learnable)
    if view:
        inv = 1.0 / x.detach().double().norm(dim=1).clamp_min(1e-12).max()
        gx = S.prepare_query_backward(x.detach().double(), gq.reshape(B, h, w, d))
        _check(x.grad, gx, sq_ * float(inv), (name, learnable, view))
    else:
        _check(x.grad.reshape(-1, d), gq, sq_, (name, learnable, view))
    if learnable and name != "spread":                       # spread_loss alone never reaches the (detached) keys
        _check(k.grad, gk, sk_, (name, "keys"), slack=_tie_slack(k64) if loss[3] else None)
    else:
        assert k.grad is None


@pytest.mark.parametrize("n_terms", [2, 3])
@pytest.mark.parametrize("view", [False, True], ids=["contiguous", "normalize_view"])
@pytest.mark.parametrize("shape", SHAPES, ids=SHAPE_IDS)
def test_standalone_grads_vs_oracle(shape, view, n_terms, terms):
    terms(n_terms)
    query, keys, W, Wq, Wm = _inputs(shape)
    m, d = keys.shape
    mem = V.Memory(m, d, d, 0.1, 0.1)
    for name in LOSSES:
        for learnable in (False, True):
            _run_case(mem, query, keys, W, Wq, Wm, name, learnable, view)


@pytest.mark.parametrize("train", [True, False])
@pytest.mark.parametrize("shape", ["memory_d64_m50", (2, 768, 32, 32, 2000), (1, 96, 7, 5, 33)], ids=SHAPE_IDS)
def test_composition_matches_fused_forward(shape, train):
    """the reference's forward written with our methods (Memory.py:145-175): prepare_query -> gather_loss +
    spread_loss + read; the query gradient of <uq, W> + 0.7 gathering + 0.3 spreading matches Memory.forward's"""
    query, keys, W, _, _ = _inputs(shape)
    m, d = keys.shape
    mem = V.Memory(m, d, d, 0.1, 0.1)
    k = T(keys)
    x = T(query, grad=True)
    q4 = mem.prepare_query(x)
    L = 0.7 * mem.gather_loss(q4, k, train) + (0.3 * mem.spread_loss(q4, k, train) if train else 0)
    L = L + (mem.read(q4, k)[0] * T(W)).sum()
    L.backward()
    x2 = T(query, grad=True)
    o = mem(x2, k, train=train)
    L2 = (o[0] * T(W)).sum() + 0.7 * o[4] + (0.3 * o[5] if train else 0)
    L2.backward()
    ref = x2.grad.double()
    err = float((x.grad.double() - ref).abs().max())
    assert err <= 2e-5 * float(ref.abs().max()), (err, float(ref.abs().max()))


def test_full_size_vs_float64_on_the_gpu():
    """N = 65 536, m = 2000, d = 768: g_keys in full, g_query on 4096 seeded rows, against float64 on the same GPU.
    2e-4 of the max, as the other full-size memory tests: the split-K contraction over 65 536 tokens (tcgen05
    accumulators round toward zero) leaves g_keys 6e-5 of its max from float64, the same for the read's share
    score_memory^T G_r through the unchanged vadc_memory_keys_bwd"""
    B, d, h, w, m = 64, 768, 32, 32, 2000
    g = torch.Generator(device=dev()).manual_seed(7)
    keys = torch.rand((m, d), device=dev(), generator=g)
    keys /= keys.norm(dim=1, keepdim=True)
    q4 = F.normalize(torch.randn((B, d, h, w), device=dev(), generator=g), dim=1).permute(0, 2, 3, 1).contiguous()
    n = B * h * w
    Wq = torch.randn((n, m), device=dev(), generator=g)
    Wm = torch.randn((n, m), device=dev(), generator=g)
    W = torch.randn((B, 2 * d, h, w), device=dev(), generator=g)
    mem = V.Memory(m, d, d, 0.1, 0.1)
    q = q4.clone().requires_grad_(True)
    k = keys.clone().requires_grad_(True)
    uq, sq, sm = mem.read(q, k)
    L = (uq * W).sum() + (sq * Wq).sum() + (sm * Wm).sum() + 0.7 * mem.gather_loss(q, k, True) + \
        0.3 * mem.spread_loss(q, k, True)
    L.backward()
    qr = q4.reshape(n, d)
    kt = V.memory._compute_scores(qr, keys, False)
    q64, k64 = qr.double(), keys.double()
    sq64, sm64 = S.scores(q64, k64)
    gs = S.g_s(sq64, sm64, Wq.double(), Wm.double())
    del sq64
    rows = W.double().permute(0, 2, 3, 1).reshape(n, 2 * d)
    gk = gs.t() @ q64 + sm64.t() @ rows[:, d:]
    del sm64
    err_k = float((k.grad.double() - gk).abs().max() / gk.abs().max())
    idx = torch.randperm(n, generator=torch.Generator().manual_seed(3))[:4096].to(dev())
    top1, top2 = S.picks(q64[idx], k64, (kt.top1[idx], kt.top2[idx]))
    gq = gs[idx] @ k64 + rows[idx, :d]
    gq = gq + 2.0 * 0.7 * (q64[idx] - k64[top1]) / (n * d)
    gq = gq + S.spread_backward(q64[idx], k64, 0.3, top1, top2) * idx.numel() / n
    err_q = float((q.grad.reshape(n, d)[idx].double() - gq).abs().max() / gq.abs().max())
    print(f"full size: g_keys {err_k:.2e}, g_query sample {err_q:.2e} of the max")
    assert err_k < 2e-4 and err_q < 2e-4, (err_k, err_q)


def _kernels(fn):
    """the set of CUDA kernel names fn launches, under torch.profiler.  A warm-up session comes first: CUDA activity
    records arrive asynchronously, and the first session of a process initialises the activity tracing."""
    from torch.profiler import profile, ProfilerActivity
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]):
        torch.ones(1, device=dev()).add_(1)
        torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "emcpy" not in e.name
            and "emset" not in e.name}


def _launches(fn):
    """(library launches, fn's result): the count of libvadc's own launch counter, exact and in launch order"""
    torch.cuda.synchronize()
    c0 = V.launch_count()
    out = fn()
    return V.launch_count() - c0, out


def test_no_grad_and_plain_inputs_launch_what_a_forward_only_call_launches():
    query, keys, _, _, _ = _inputs((1, 96, 7, 5, 33))
    mem = V.Memory(33, 96, 96, 0.1, 0.1)
    x = T(query)
    q4 = F.normalize(x, dim=1).permute(0, 2, 3, 1).contiguous()
    k = T(keys)

    def calls(q4, k, x):
        return [mem.prepare_query(x), *mem.get_score(k, q4), *mem.read(q4, k), mem.gather_loss(q4, k, True),
                mem.spread_loss(q4, k, True)]

    n_base, outs = _launches(lambda: calls(q4, k, x))
    assert all(o.grad_fn is None for o in outs)
    names = _kernels(lambda: calls(q4, k, x))
    assert not any("bwd" in n for n in names), names
    qg, kg, xg = q4.clone().requires_grad_(True), k.clone().requires_grad_(True), x.clone().requires_grad_(True)
    with torch.no_grad():
        n, outs = _launches(lambda: calls(qg, kg, xg))
        assert n == n_base and all(o.grad_fn is None for o in outs)
        assert _kernels(lambda: calls(qg, kg, xg)) == names
    # with gradients possible the forward launches the same kernels, and each output has its grad_fn
    n, outs = _launches(lambda: calls(qg, kg, xg))
    assert n == n_base and all(o.grad_fn is not None for o in outs)
    assert _kernels(lambda: calls(qg, kg, xg)) == names


def test_loss_on_updated_query_alone_launches_no_score_backward():
    query, keys, W, _, _ = _inputs((2, 768, 32, 32, 2000))
    mem = V.Memory(2000, 768, 768, 0.1, 0.1)
    for learnable in (False, True):
        q = F.normalize(T(query), dim=1).permute(0, 2, 3, 1).contiguous().requires_grad_(True)
        k = T(keys).requires_grad_(learnable)
        L = (mem.read(q, k)[0] * T(W)).sum()
        if not learnable:
            assert _launches(lambda: L.backward(retain_graph=True))[0] == 1      # memory_rows_bwd_kernel alone
        names = _kernels(L.backward)
        assert not any("scores_bwd" in n or "rows_transpose" in n for n in names), names
        assert sum("tc_gemm" in n for n in names) == (1 if learnable else 0), names   # the read's g_keys only
        assert any("memory_rows_bwd_kernel" in n for n in names)


@pytest.mark.parametrize("shape", SHAPES, ids=SHAPE_IDS)
def test_prepare_query_alone_vs_oracle(shape):
    """prepare_query's backward (vadc_memory_prepare_query_bwd) against the float64 closed form, with one all-zero
    token: there the clamp holds (|x| < 1e-12), q-hat . g is taken as 0 and g_x = g / 1e-12"""
    query, _, _, _, _ = _inputs(shape)
    B, d, h, w = query.shape
    query = query.copy()
    query[0, :, 0, 0] = 0.0
    G4 = np.random.default_rng(5).standard_normal((B, h, w, d)).astype(np.float32)
    mem = V.Memory(2, d, d, 0.1, 0.1)
    x = T(query, grad=True)
    q4 = mem.prepare_query(x)
    assert q4.grad_fn is not None and q4.is_contiguous()
    (q4 * T(G4)).sum().backward()
    ref = S.prepare_query_backward(T(query).double(), T(G4).double())
    got = x.grad.double()
    z = (slice(0, 1), slice(None), slice(0, 1), slice(0, 1))      # the zero token: g / 1e-12, about 1e12
    assert float((got[z] - ref[z]).abs().max()) <= 1e-6 * float(ref[z].abs().max())
    got[z] = 0.0
    ref[z] = 0.0
    err = float((got - ref).abs().max())
    assert err <= 2e-5 * float(ref.abs().max()), (err, float(ref.abs().max()))


def test_backward_is_bit_identical_when_repeated():
    query, keys, W, Wq, Wm = _inputs((2, 768, 32, 32, 2000))
    mem = V.Memory(2000, 768, 768, 0.1, 0.1)
    grads = []
    for _ in range(2):
        x = T(query, grad=True)
        k = T(keys).requires_grad_(True)
        q4 = mem.prepare_query(x)
        (_ours(mem, q4, k, W, Wq, Wm, LOSSES["all"]) + 1.3 * V.MemoryLoss(k)).backward()
        grads.append((x.grad.clone(), k.grad.clone()))
    for a, b in zip(*grads):
        assert torch.equal(a, b)


def test_errors():
    mem = V.Memory(10, 4, 4, 0.1, 0.1)
    q = torch.randn((1, 3, 3, 4), device=dev(), requires_grad=True)
    k = torch.randn((10, 4), device=dev())
    sq, _ = mem.get_score(k, q)
    with pytest.raises(RuntimeError, match="vadc_memory_scores_bwd_rows failed"):
        sq.sum().backward()
    mem1 = V.Memory(1, 32, 32, 0.1, 0.1)
    q = torch.randn((1, 3, 3, 32), device=dev(), requires_grad=True)
    with pytest.raises(RuntimeError, match="selected index k out of range"):
        mem1.spread_loss(q, torch.randn((1, 32), device=dev()), True)
