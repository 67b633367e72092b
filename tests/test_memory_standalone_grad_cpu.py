"""Gradients of Memory's stand-alone methods on the CPU: the float64 oracle against torch's autograd of the reference's
method bodies, and the host-side argument checks of the new entry points."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import standalone_oracle as S

SHAPES = [(2, 32, 4, 4, 10), (1, 24, 3, 5, 7)]


def _inputs(B, d, h, w, m, unit_keys):
    rng = np.random.default_rng(B * 100 + d + m)
    x = torch.tensor(rng.standard_normal((B, d, h, w)))
    keys = torch.tensor(rng.random((m, d)) * 0.4)            # not unit norm: no entry of K K^T/2 + 1/2 - I near 0
    if unit_keys:
        keys = keys / keys.norm(dim=1, keepdim=True) * 0.999
    N = B * h * w
    W = torch.tensor(rng.standard_normal((B, 2 * d, h, w)))
    Wq, Wm = torch.tensor(rng.standard_normal((N, m))), torch.tensor(rng.standard_normal((N, m)))
    G4 = torch.tensor(rng.standard_normal((B, h, w, d)))
    return x, keys, W, Wq, Wm, G4


def _close(got, ref):
    np.testing.assert_allclose(got.numpy(), ref.numpy(), rtol=0, atol=1e-12 * max(float(ref.abs().max()), 1.0))


@pytest.mark.parametrize("unit_keys", [False, True])
@pytest.mark.parametrize("B,d,h,w,m", SHAPES)
def test_each_method_alone_matches_torch_autograd(B, d, h, w, m, unit_keys):
    x, keys, W, Wq, Wm, G4 = _inputs(B, d, h, w, m, unit_keys)
    q4 = F.normalize(x, dim=1).permute(0, 2, 3, 1) * 1.7        # the query as passed is not re-normalised
    N = B * h * w
    qr = q4.reshape(N, d)
    top1, top2 = S.picks(qr, keys)

    # get_score, with a linear loss on each matrix and an entropy penalty on score_memory
    for lq, lm, ent in ((1, 0, 0), (0, 1, 0), (0, 0, 1), (1, 1, 1)):
        q = q4.clone().requires_grad_(True)
        k = keys.clone().requires_grad_(True)
        sq, sm = S.ref_get_score(k, q)
        L = lq * (sq * Wq).sum() + lm * (sm * Wm).sum() - ent * (sm * torch.log(sm)).sum(1).mean()
        L.backward()
        g_sm = (Wm if lm else 0) + (S.entropy_grad(S.scores(qr, keys)[1]) if ent else 0)
        gq, gk = S.get_score_backward(qr, keys, Wq if lq else None, g_sm if (lm or ent) else None)
        _close(q.grad.reshape(N, d), gq)
        _close(k.grad, gk)

    # read, with a loss on updated_query alone and on all three outputs
    for scores_too in (False, True):
        q = q4.clone().requires_grad_(True)
        k = keys.clone().requires_grad_(True)
        uq, sq, sm = S.ref_read(q, k)
        L = (uq * W).sum() + (((sq * Wq).sum() + (sm * Wm).sum()) if scores_too else 0)
        L.backward()
        gq, gk = S.read_backward(qr, keys, W, Wq if scores_too else None, Wm if scores_too else None)
        _close(q.grad.reshape(N, d), gq)
        _close(k.grad, gk)

    # gather_loss and spread_loss: the query only (the keys are detached)
    q = q4.clone().requires_grad_(True)
    (0.7 * S.ref_gather_loss(q, keys)).backward()
    _close(q.grad.reshape(N, d), S.gather_backward(qr, keys, 0.7, top1))
    q = q4.clone().requires_grad_(True)
    (0.3 * S.ref_spread_loss(q, keys)).backward()
    _close(q.grad.reshape(N, d), S.spread_backward(qr, keys, 0.3, top1, top2))

    # prepare_query
    xx = x.clone().requires_grad_(True)
    (F.normalize(xx, dim=1).permute(0, 2, 3, 1) * G4).sum().backward()
    _close(xx.grad, S.prepare_query_backward(x, G4))


@pytest.mark.parametrize("unit_keys", [False, True])
@pytest.mark.parametrize("B,d,h,w,m", SHAPES)
def test_all_methods_under_one_loss_match_torch_autograd(B, d, h, w, m, unit_keys):
    """the reference's forward composed from its methods (Memory.py:145-175), the score matrices of get_score and a
    learnable memory under one loss: linear losses on sq, sm and uq, an entropy penalty, gathering, spreading and
    MemoryLoss"""
    x, keys, W, Wq, Wm, _ = _inputs(B, d, h, w, m, unit_keys)
    N = B * h * w
    xx = x.clone().requires_grad_(True)
    k = keys.clone().requires_grad_(True)
    q4 = F.normalize(xx, dim=1).permute(0, 2, 3, 1)
    sq, sm = S.ref_get_score(k, q4)
    uq, _, _ = S.ref_read(q4, k)
    L = ((sq * Wq).sum() + (sm * Wm).sum() - (sm * torch.log(sm)).sum(1).mean() + (uq * W).sum()
         + 0.7 * S.ref_gather_loss(q4, k) + 0.3 * S.ref_spread_loss(q4, k) + 1.3 * S.ref_memory_loss(k))
    L.backward()

    qr = F.normalize(x, dim=1).permute(0, 2, 3, 1).reshape(N, d)
    top1, top2 = S.picks(qr, keys)
    g_sm = Wm + S.entropy_grad(S.scores(qr, keys)[1])
    gq1, gk1 = S.get_score_backward(qr, keys, Wq, g_sm)
    gq2, gk2 = S.read_backward(qr, keys, W)
    gq = gq1 + gq2 + S.gather_backward(qr, keys, 0.7, top1) + S.spread_backward(qr, keys, 0.3, top1, top2)
    gx = S.prepare_query_backward(x, gq.reshape(B, h, w, d))
    gk = gk1 + gk2 + S.memory_loss_backward(keys, 1.3)
    _close(xx.grad, gx)
    _close(k.grad, gk)


def test_standalone_backward_workspace_queries_are_pure_host_functions():
    import videoad_b200 as V
    l = V._lib.lib()
    assert l.vadc_memory_scores_bwd_rows_workspace_bytes(65536, 768, 2000) >= 2 * 65536 * 2000 * 2
    assert l.vadc_memory_scores_bwd_rows_workspace_bytes(65536, 768, 2000) == \
        l.vadc_memory_scores_bwd_workspace_bytes(1, 768, 65536, 2000)
    assert l.vadc_memory_scores_bwd_rows_workspace_bytes(1, 8, 2) > 0
    assert l.vadc_memory_scores_bwd_rows_workspace_bytes(0, 8, 2) > 0


def test_standalone_backward_argument_validation_happens_before_any_cuda_call():
    import videoad_b200 as V
    l = V._lib.lib()
    ws = 1 << 40
    f = 16                                                  # never dereferenced: every call below fails on the host
    sr, rb, pb = l.vadc_memory_scores_bwd_rows, l.vadc_memory_rows_bwd, l.vadc_memory_prepare_query_bwd
    #          q keys sq sm Gq Gm coldot N d m g_q g_keys ws bytes stream
    assert sr(f, f, f, f, f, f, f, -1, 32, 10, f, f, f, ws, None) == -1
    assert sr(f, f, f, f, f, f, f, 64, 0, 10, f, f, f, ws, None) == -1
    assert sr(f, f, f, f, f, f, f, 64, 32, 0, f, f, f, ws, None) == -1
    assert sr(None, f, f, f, f, f, f, 64, 32, 10, f, f, f, ws, None) == -2
    assert sr(f, None, f, f, f, f, f, 64, 32, 10, f, f, f, ws, None) == -2
    assert sr(f, f, f, f, None, None, f, 64, 32, 10, f, f, f, ws, None) == -2     # no incoming gradient
    assert sr(f, f, f, f, f, f, f, 64, 32, 10, None, None, f, ws, None) == -2     # nothing to compute
    assert sr(f, f, None, f, f, None, f, 64, 32, 10, f, f, f, ws, None) == -2     # Gq needs score_query
    assert sr(f, f, f, f, f, None, None, 64, 32, 10, f, f, f, ws, None) == -2     # ... and the column dots
    assert sr(f, f, f, None, None, f, None, 64, 32, 10, f, f, f, ws, None) == -2  # Gm needs score_memory
    assert sr(f, f, f, f, f, f, f, 64, 32, 10, f, f, None, ws, None) == -2
    assert sr(f, f, f, f, f, f, f, 64, 4, 10, f, f, f, ws, None) == -6            # d < 8
    assert sr(f, f, f, f, f, f, f, 64, 32, 10, f, f, f, 16, None) == -4
    #          q keys top1 top2 g_uq g_gather g_spread g_q_rows B d HW m g_query stream
    assert rb(f, f, f, f, f, f, f, f, -1, 32, 16, 10, f, None) == -1
    assert rb(f, f, f, f, f, f, f, f, 2, 0, 16, 10, f, None) == -1
    assert rb(f, f, f, f, f, f, f, f, 2, 32, 0, 10, f, None) == -1
    assert rb(f, f, f, f, f, f, f, f, 2, 32, 16, 0, f, None) == -1
    assert rb(None, f, f, f, f, f, f, f, 2, 32, 16, 10, f, None) == -2
    assert rb(f, f, f, f, f, f, f, f, 2, 32, 16, 10, None, None) == -2
    assert rb(f, f, f, f, None, None, None, None, 2, 32, 16, 10, f, None) == -2   # no term
    assert rb(f, f, None, f, None, f, None, None, 2, 32, 16, 10, f, None) == -2   # gathering needs top1
    assert rb(f, f, f, None, None, None, f, None, 2, 32, 16, 10, f, None) == -2   # spreading needs top2
    assert rb(f, f, f, f, f, f, f, f, 70000, 32, 16, 10, f, None) == -6
    #          g query B d HW g_x stream
    assert pb(f, f, -1, 32, 16, f, None) == -1
    assert pb(f, f, 2, 0, 16, f, None) == -1
    assert pb(f, f, 2, 32, 0, f, None) == -1
    assert pb(None, f, 2, 32, 16, f, None) == -2
    assert pb(f, None, 2, 32, 16, f, None) == -2
    assert pb(f, f, 2, 32, 16, None, None) == -2
    assert pb(f, f, 70000, 32, 16, f, None) == -6
