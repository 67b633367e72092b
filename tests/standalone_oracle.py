"""float64 oracle of the gradients of Memory's stand-alone methods (model/Memory.py get_score :133-143, read :249-261,
gather_loss :233-247, spread_loss :214-231) and of prepare_query (F.normalize + permute, :148-149).

The methods take the query channel-last, [B,h,w,d] flattened to q [N,d], and do not normalise it.  Everything here is
closed form, written with torch float64 tensors so that it runs on the CPU and, at full size, on the GPU.  ``ref_*``
restate the reference's method bodies op for op (as oracle/ref_port.py::memory_forward does for forward) for torch's
autograd to differentiate."""
import numpy as np
import torch
import torch.nn.functional as F

from keys_oracle import memory_keys_backward


# -- the reference's methods, restated ----------------------------------------------------------------------------
def ref_get_score(mem, query):
    bs, h, w, d = query.size()
    m, d = mem.size()
    score = torch.matmul(query, torch.t(mem)).view(bs * h * w, m)
    return F.softmax(score, dim=0), F.softmax(score, dim=1)


def ref_read(query, updated_memory):
    bs, h, w, d = query.size()
    sq, sm = ref_get_score(updated_memory, query)
    query_reshape = query.contiguous().view(bs * h * w, d)
    concat_memory = torch.matmul(sm.detach(), updated_memory)
    updated_query = torch.cat((query_reshape, concat_memory), dim=1)
    return updated_query.view(bs, h, w, 2 * d).permute(0, 3, 1, 2), sq, sm


def ref_gather_loss(query, keys):
    bs, h, w, d = query.size()
    _, sm = ref_get_score(keys, query)
    query_reshape = query.contiguous().view(bs * h * w, d)
    _, idx = torch.topk(sm, 1, dim=1)
    return torch.nn.MSELoss()(query_reshape, keys[idx].squeeze(1).detach())


def ref_spread_loss(query, keys):
    bs, h, w, d = query.size()
    _, sm = ref_get_score(keys, query)
    query_reshape = query.contiguous().view(bs * h * w, d)
    _, idx = torch.topk(sm, 2, dim=1)
    pos, neg = keys[idx[:, 0]], keys[idx[:, 1]]
    return torch.nn.TripletMarginLoss(margin=1.0)(query_reshape, pos.detach(), neg.detach())


def ref_memory_loss(k):
    m = k.shape[0]
    return torch.sum(torch.abs(k @ k.t() / 2 + 0.5 - torch.eye(m, dtype=k.dtype, device=k.device))) / (m * (m - 1))


# -- closed forms ---------------------------------------------------------------------------------------------------
def scores(q, keys):
    s = q @ keys.t()
    return torch.softmax(s, 0), torch.softmax(s, 1)


def g_s(sq, sm, g_sq=None, g_sm=None):
    """g_s = sq (Gq - 1 c^T) + sm (Gm - r 1^T), c = sum_n Gq sq, r = sum_i Gm sm"""
    gs = torch.zeros_like(sm)
    if g_sq is not None:
        gs += sq * (g_sq - (g_sq * sq).sum(0, keepdim=True))
    if g_sm is not None:
        gs += sm * (g_sm - (g_sm * sm).sum(1, keepdim=True))
    return gs


def get_score_backward(q, keys, g_sq=None, g_sm=None):
    """(g_q [N,d], g_keys [m,d]) of <sq, Gq> + <sm, Gm>: g_q = g_s K, g_keys = g_s^T q"""
    sq, sm = scores(q, keys)
    gs = g_s(sq, sm, g_sq, g_sm)
    return gs @ keys, gs.t() @ q


def read_backward(q, keys, g_uq=None, g_sq=None, g_sm=None):
    """(g_q [N,d], g_keys [m,d]) of <uq, G_uq> + <sq, Gq> + <sm, Gm>; G_uq [B,2d,h,w].  uq = cat(q, sm.detach() K):
    g_q = G_uq[:, :d] (channel-last) + g_s K, g_keys = sm^T G_uq[:, d:] + g_s^T q"""
    d = q.shape[1]
    gq, gk = get_score_backward(q, keys, g_sq, g_sm)
    if g_uq is not None:
        rows = g_uq.permute(0, 2, 3, 1).reshape(-1, 2 * d)
        gq = gq + rows[:, :d]
        gk = gk + scores(q, keys)[1].t() @ rows[:, d:]
    return gq, gk


def picks(q, keys, kernel_top=None, rel_gap=1e-6):
    """(top1, top2) of score_memory, as torch.topk takes them.  Where float64 sees a near-tie (the gap between the
    first and second, or second and third, logits is below rel_gap of their size) the picks of ``kernel_top`` (the
    kernel's own (top1, top2)) are used instead: there the order is decided by rounding, not by the model."""
    s = q @ keys.t()
    v, idx = torch.sort(s, dim=1, descending=True, stable=True)
    top1, top2 = idx[:, 0].clone(), idx[:, min(1, s.shape[1] - 1)].clone()
    if kernel_top is not None:
        scale = v[:, 0].abs().clamp_min(1.0)
        tie = (v[:, 0] - v[:, min(1, s.shape[1] - 1)]) < rel_gap * scale
        if s.shape[1] > 2:
            tie |= (v[:, 1] - v[:, 2]) < rel_gap * scale
        top1 = torch.where(tie, kernel_top[0].to(top1), top1)
        top2 = torch.where(tie, kernel_top[1].to(top2), top2)
    return top1, top2


def gather_backward(q, keys, g, top1):
    """d/dq of g MSELoss(q, K[top1]): 2 g (q - K[top1]) / (N d)"""
    N, d = q.shape
    return 2.0 * g * (q - keys[top1]) / (N * d)


def spread_backward(q, keys, g, top1, top2):
    """d/dq of g TripletMarginLoss(margin=1, p=2, eps=1e-6)(q, K[top1], K[top2]), mean over the tokens"""
    N = q.shape[0]
    a, e = q - keys[top1] + 1e-6, q - keys[top2] + 1e-6
    dap, dan = a.norm(dim=1, keepdim=True), e.norm(dim=1, keepdim=True)
    active = (dap - dan + 1.0 >= 0).to(q.dtype)
    return g / N * active * (a / torch.where(dap > 0, dap, 1.0) - e / torch.where(dan > 0, dan, 1.0))


def prepare_query_backward(x, g):
    """d/dx of <F.normalize(x, dim=1).permute(0,2,3,1), g>: x [B,d,h,w], g [B,h,w,d] -> [B,d,h,w]
    g_x = (g - q-hat (q-hat . g)) / max(|x|, 1e-12), q-hat . g taken as 0 where the clamp holds"""
    gc = g.permute(0, 3, 1, 2)
    nrm = x.norm(dim=1, keepdim=True)
    den = nrm.clamp_min(1e-12)
    qh = x / den
    dot = torch.where(nrm < 1e-12, 0.0, (qh * gc).sum(1, keepdim=True))
    return (gc - qh * dot) / den


def memory_loss_backward(keys, g_sep, tie=0.0):
    """d/dkeys of g_sep MemoryLoss(keys) (keys_oracle; sign ties |S| < tie set to 0)"""
    k = keys.detach().cpu().numpy()
    gk = memory_keys_backward(np.zeros((1, k.shape[1], 1, 1)), k, None, g_sep, tie=tie)
    return torch.tensor(gk, dtype=keys.dtype, device=keys.device)


def cancellation_scales(q, keys, g_sq=None, g_sm=None):
    """(S_q, S_k): the size of the terms of the score share of g_q and g_keys before they cancel (the sums of
    |sq Gq| + |sq c| + |sm Gm| + |sm r| against |K| and |q|), as scores_oracle.cancellation_scales for the
    channel-last, unnormalised query.  Rounding errors of an fp32 computation scale with these."""
    sq, sm = scores(q, keys)
    t = torch.zeros_like(sm)
    if g_sq is not None:
        t += sq * (g_sq.abs() + (g_sq * sq).sum(0, keepdim=True).abs())
    if g_sm is not None:
        t += sm * (g_sm.abs() + (g_sm * sm).sum(1, keepdim=True).abs())
    return float((t @ keys.abs()).max()), float((t.t() @ q.abs()).max())


def entropy_grad(sm):
    """d/d score_memory of the entropy penalty -mean_n sum_i sm log sm: -(log sm + 1) / N"""
    return -(torch.log(sm) + 1.0) / sm.shape[0]
