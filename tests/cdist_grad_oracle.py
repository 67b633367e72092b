"""float64 oracle of the stand-alone cdist backward (ATen's _euclidean_dist_backward), the math of vadc_cdist_bwd:
per batch, with D = cdist(a, b) and g = dL/dD,

    r = g / D (0 where D == 0),  ga = a rowsum(r) - r b,  gb = b colsum(r) - r^T a

and, for cdist(c, c), gc = c rowsum(r + r^T) - (r + r^T) c with the diagonal of r skipped (its exact contribution is
r_ii (c_i - c_i) = 0).

It lives next to the other gradient oracles of the suite (keys_oracle.py, scores_oracle.py, standalone_oracle.py) rather
than in oracle/np_oracle.py: the oracle/ package is the reference the existing tests are measured against and feature
work leaves it unchanged."""
import numpy as np


def ratio(D, g):
    D = np.asarray(D, np.float64)
    g = np.asarray(g, np.float64)
    return np.where(D == 0, 0.0, g / np.where(D == 0, 1.0, D))


def cdist_backward(a, b, D, g):
    """a [..., R, C], b [..., P, C], D and g [..., R, P] with equal leading dimensions -> (ga, gb)"""
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    r = ratio(D, g)
    rt = np.swapaxes(r, -1, -2)
    ga = a * r.sum(-1)[..., None] - r @ b
    gb = b * rt.sum(-1)[..., None] - rt @ a
    return ga, gb


def self_cdist_backward(c, D, g):
    """the whole gradient of cdist(c, c) with respect to c [..., K, C]"""
    c = np.asarray(c, np.float64)
    r = ratio(D, g)
    K = r.shape[-1]
    r[..., np.arange(K), np.arange(K)] = 0.0
    r = r + np.swapaxes(r, -1, -2)
    return c * r.sum(-1)[..., None] - r @ c


def broadcast_cdist_backward(a, b, D, g):
    """torch.cdist's leading-dimension broadcasting: both sides expanded to D's leading shape, each gradient summed
    back to its own side's shape"""
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    lead = np.shape(D)[:-2]
    ae = np.broadcast_to(a, lead + a.shape[-2:])
    be = np.broadcast_to(b, lead + b.shape[-2:])
    ga, gb = cdist_backward(ae, be, D, g)
    return _sum_to(ga, a.shape), _sum_to(gb, b.shape)


def _sum_to(x, shape):
    extra = x.ndim - len(shape)
    x = x.sum(axis=tuple(range(extra))) if extra else x
    keep = tuple(i for i, n in enumerate(shape) if n == 1 and x.shape[i] != 1)
    return x.sum(axis=keep, keepdims=True) if keep else x
