"""float64 oracle of the gradient through the two score matrices Memory.forward returns (score_query, score_memory)"""
import numpy as np

from oracle import np_oracle as O
from keys_oracle import memory_keys_backward


def memory_scores_backward(query, keys, g_score_query=None, g_score_memory=None, dtype=np.float64):
    """get_score (model/Memory.py:133-143) backward: s = q-hat K^T, sq = softmax(s, dim=0), sm = softmax(s, dim=1).
    With Gq, Gm the gradients of sq, sm ([N,m], either may be None):
        c = sum_n Gq sq (per column),  r = sum_i Gm sm (per row),  g_s = sq (Gq - c) + sm (Gm - r)
    returns (g_qhat [B,d,h,w], the gradient with respect to the normalised query in the query's layout, which joins
    the first d channels of g_updated_query before F.normalize; g_keys [m,d] = g_s^T q-hat)"""
    query = np.asarray(query, dtype)
    keys = np.asarray(keys, dtype)
    B, d, h, w = query.shape
    q = O.memory_prepare_query(query, dtype)
    sq, sm = O.memory_get_score(keys, q, dtype)
    gs = np.zeros_like(sq)
    if g_score_query is not None:
        gq = np.asarray(g_score_query, dtype)
        gs += sq * (gq - (gq * sq).sum(0, keepdims=True))
    if g_score_memory is not None:
        gm = np.asarray(g_score_memory, dtype)
        gs += sm * (gm - (gm * sm).sum(1, keepdims=True))
    g_qhat = (gs @ keys).reshape(B, h, w, d).transpose(0, 3, 1, 2)
    return g_qhat, gs.T @ q


def cancellation_scales(query, keys, g_score_query=None, g_score_memory=None, dtype=np.float64):
    """(S_q, S_k): the size of the terms of the score share of g_query and g_keys before they cancel, i.e. the same
    sums over |sq Gq| + |sq c| + |sm Gm| + |sm r|, |K|, |q-hat| and 1/|x|.  Rounding errors of an fp32 computation
    scale with these, not with the result: with an entropy loss alone and nearly parallel keys the result is 1e-4 of
    them (torch's fp32 autograd of the reference chain then misses the float64 result by 2e-3 of its max)."""
    query = np.asarray(query, dtype)
    keys = np.asarray(keys, dtype)
    B, d, h, w = query.shape
    x = query.transpose(0, 2, 3, 1).reshape(B * h * w, d)
    q = O.memory_prepare_query(query, dtype)
    sq, sm = O.memory_get_score(keys, q, dtype)
    t = np.zeros_like(sq)
    if g_score_query is not None:
        gq = np.asarray(g_score_query, dtype)
        t += sq * (np.abs(gq) + np.abs((gq * sq).sum(0, keepdims=True)))
    if g_score_memory is not None:
        gm = np.asarray(g_score_memory, dtype)
        t += sm * (np.abs(gm) + np.abs((gm * sm).sum(1, keepdims=True)))
    nrm = np.maximum(np.sqrt((x * x).sum(1, keepdims=True)), 1e-12)
    return float(((t @ np.abs(keys)) / nrm).max()), float((t.T @ np.abs(q)).max())


def entropy_grad(query, keys, dtype=np.float64):
    """d/d score_memory of the entropy penalty -mean_n sum_i sm log sm: -(log sm + 1) / N"""
    sm = O.memory_get_score(keys, O.memory_prepare_query(query, dtype), dtype)[1]
    return -(np.log(sm) + 1.0) / sm.shape[0]


def memory_backward(query, keys, train, W=None, g_gather=None, g_spread=None, g_sq=None, g_sm=None, g_sep=None,
                    tie=0.0, dtype=np.float64):
    """(g_query, g_keys) of <updated_query, W> + g_gather gathering + g_spread spreading + <score_query, g_sq> +
    <score_memory, g_sm> + g_sep MemoryLoss(keys), with keys learnable"""
    query = np.asarray(query, dtype)
    B, d, h, w = query.shape
    f = O.memory_forward(query, keys, train=True, dtype=dtype)
    g_qhat, gk = memory_scores_backward(query, keys, g_sq, g_sm, dtype)
    g_uq = np.zeros((B, 2 * d, h, w), dtype) if W is None else np.array(W, dtype)
    g_uq[:, :d] += g_qhat
    gq = O.memory_query_backward(query, keys, f["top1"], f["top2"] if train else None, g_uq, g_gather,
                                 g_spread if train else None, dtype)
    return gq, gk + memory_keys_backward(query, keys, W, g_sep, tie=tie, dtype=dtype)
