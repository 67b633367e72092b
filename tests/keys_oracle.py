"""float64 oracle of the gradient of the memory module with respect to its memory items (keys)"""
import numpy as np

from oracle import np_oracle as O


def memory_keys_backward(query, keys, g_updated_query=None, g_sep=None, tie=0.0, dtype=np.float64):
    """d/d keys of ``<updated_query, g_updated_query> + g_sep * MemoryLoss(keys)`` (autograd of model/Memory.py:255
    and :52-59).  The read ``score_memory.detach() @ keys`` gives score_memory^T G_r, G_r = channels d..2d-1 of
    g_updated_query in token order; MemoryLoss gives g_sep / (m (m-1)) (G + G^T)/2 K with G = sgn(K K^T/2 + 1/2 - I),
    set to 0 wherever |S| < ``tie`` (entries whose sign is rounding noise, e.g. the diagonal of unit-norm keys).
    Nothing else reaches the keys: the losses use detached copies, updated_memory is detached.
    query [B,d,h,w], keys [m,d]; returns g_keys [m,d]."""
    query = np.asarray(query, dtype)
    keys = np.asarray(keys, dtype)
    B, d, h, w = query.shape
    m = keys.shape[0]
    g = np.zeros((m, d), dtype)
    if g_updated_query is not None:
        q = O.memory_prepare_query(query, dtype)
        sm = O.memory_get_score(keys, q, dtype)[1]
        gr = np.asarray(g_updated_query, dtype)[:, d:].transpose(0, 2, 3, 1).reshape(B * h * w, d)
        g += sm.T @ gr
    if g_sep is not None:
        G = separateness_sign(keys, tie)
        g += dtype(g_sep) / (m * (m - 1)) * (0.5 * (G + G.T)) @ keys
    return g


def separateness_sign(keys, tie=0.0):
    """sgn(K K^T/2 + 1/2 - I) in float64, 0 where |S| < tie"""
    k = np.asarray(keys, np.float64)
    S = k @ k.T / 2 + 0.5 - np.eye(k.shape[0])
    return np.where(np.abs(S) < tie, 0.0, np.sign(S))
