"""Gradient through the returned score matrices, on the CPU: the float64 oracle against torch's autograd of the
reference op chain, and the host-side argument checks of the new entry points."""
import numpy as np
import pytest
import torch

from oracle import ref_port as P
from scores_oracle import memory_backward, entropy_grad

# (Wq, Wm, entropy, with <updated_query, W>, gathering, spreading and MemoryLoss)
LOSSES = [(1, 1, 0, 0), (0, 0, 1, 0), (1, 0, 0, 0), (0, 1, 0, 0), (1, 1, 0, 1), (0, 0, 1, 1), (1, 1, 1, 1)]


def _memory_loss_torch(k):
    m = k.shape[0]
    return torch.sum(torch.abs(k @ k.t() / 2 + 0.5 - torch.eye(m, dtype=k.dtype))) / (m * (m - 1))


@pytest.mark.parametrize("train", [True, False])
@pytest.mark.parametrize("B,d,h,w,m", [(2, 32, 4, 4, 10), (1, 24, 3, 5, 7)])
def test_scores_oracle_matches_torch_autograd_of_reference_chain(B, d, h, w, m, train):
    rng = np.random.default_rng(B * 10 + m)
    query = rng.standard_normal((B, d, h, w))
    keys = rng.random((m, d)) * 0.4                         # not unit norm: no entry of S near 0
    W = rng.standard_normal((B, 2 * d, h, w))
    N = B * h * w
    Wq, Wm = rng.standard_normal((N, m)), rng.standard_normal((N, m))
    for lq, lm, ent, rest in LOSSES:
        q = torch.tensor(query, requires_grad=True)
        k = torch.tensor(keys, requires_grad=True)
        out = P.memory_forward(q, k, train=train)
        sq, sm = out[2], out[3]
        loss = lq * (sq * torch.tensor(Wq)).sum() + lm * (sm * torch.tensor(Wm)).sum()
        if ent:
            loss = loss - (sm * torch.log(sm)).sum(1).mean()
        if rest:
            loss = loss + (out[0] * torch.tensor(W)).sum() + 0.7 * out[4] + 1.3 * _memory_loss_torch(k)
            if train:
                loss = loss + 0.3 * out[5]
        loss.backward()
        g_sm = (Wm if lm else 0) + (entropy_grad(query, keys) if ent else 0)
        gq, gk = memory_backward(query, keys, train, W if rest else None, 0.7 if rest else None,
                                 0.3 if rest else None, Wq if lq else None,
                                 g_sm if (lm or ent) else None, 1.3 if rest else None)
        for got, ref in ((q.grad.numpy(), gq), (k.grad.numpy(), gk)):
            np.testing.assert_allclose(got, ref, rtol=0, atol=1e-12 * max(np.abs(ref).max(), 1.0))


def test_scores_backward_workspace_queries_are_pure_host_functions():
    import videoad_b200 as V
    l = V._lib.lib()
    assert l.vadc_memory_scores_bwd_workspace_bytes(64, 768, 1024, 2000) >= 2 * 65536 * 2000 * 2
    assert l.vadc_memory_scores_bwd_workspace_bytes(1, 96, 35, 33) > 0
    assert l.vadc_memory_score_coldot_workspace_bytes(65536, 2000) >= 2000 * 4
    assert l.vadc_memory_score_coldot_workspace_bytes(1, 2) > 0


def test_scores_backward_argument_validation_happens_before_any_cuda_call():
    import videoad_b200 as V
    l = V._lib.lib()
    ws = 1 << 40
    f = 16                                                  # never dereferenced: every call below fails on the host
    sb, cd = l.vadc_memory_scores_bwd, l.vadc_memory_score_coldot
    #          query keys sq sm Gq Gm coldot B d HW m g_qhat g_keys ws bytes stream
    # bad shapes
    assert sb(f, f, f, f, f, f, f, -1, 32, 16, 10, f, f, f, ws, None) == -1
    assert sb(f, f, f, f, f, f, f, 2, 0, 16, 10, f, f, f, ws, None) == -1
    assert sb(f, f, f, f, f, f, f, 2, 32, 0, 10, f, f, f, ws, None) == -1
    assert sb(f, f, f, f, f, f, f, 2, 32, 16, 0, f, f, f, ws, None) == -1
    assert cd(f, f, -1, 10, f, f, ws, None) == -1
    assert cd(f, f, 16, 0, f, f, ws, None) == -1
    # NULL pointers
    assert sb(None, f, f, f, f, f, f, 2, 32, 16, 10, f, f, f, ws, None) == -2
    assert sb(f, None, f, f, f, f, f, 2, 32, 16, 10, f, f, f, ws, None) == -2
    assert sb(f, f, f, f, None, None, f, 2, 32, 16, 10, f, f, f, ws, None) == -2     # no incoming gradient
    assert sb(f, f, f, f, f, f, f, 2, 32, 16, 10, None, None, f, ws, None) == -2     # nothing to compute
    assert sb(f, f, None, f, f, None, f, 2, 32, 16, 10, f, f, f, ws, None) == -2     # Gq needs score_query
    assert sb(f, f, f, f, f, None, None, 2, 32, 16, 10, f, f, f, ws, None) == -2     # ... and the column dots
    assert sb(f, f, f, None, None, f, None, 2, 32, 16, 10, f, f, f, ws, None) == -2  # Gm needs score_memory
    assert sb(f, f, f, f, f, f, f, 2, 32, 16, 10, f, f, None, ws, None) == -2
    assert cd(None, f, 16, 10, f, f, ws, None) == -2
    assert cd(f, None, 16, 10, f, f, ws, None) == -2
    assert cd(f, f, 16, 10, None, f, ws, None) == -2
    assert cd(f, f, 16, 10, f, None, ws, None) == -2
    # outside what the tensor-core contractions take, and too small a workspace
    assert sb(f, f, f, f, f, f, f, 2, 4, 16, 10, f, f, f, ws, None) == -6
    assert sb(f, f, f, f, f, f, f, 2, 32, 16, 10, f, f, f, 16, None) == -4
    assert cd(f, f, 16, 10, f, f, 16, None) == -4
    # the extended query backward keeps the checks of vadc_memory_query_bwd
    qb = l.vadc_memory_query_bwd_ex
    assert qb(f, f, f, None, None, None, None, f, 2, 0, 16, 10, f, None) == -1
    assert qb(None, f, f, None, None, None, None, f, 2, 32, 16, 10, f, None) == -2
    assert qb(f, f, f, None, None, None, None, f, 70000, 32, 16, 10, f, None) == -6
