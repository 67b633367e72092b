"""Host-side mirror of the reference's cluster head (model/cluster.py) on top
of libvadc.so.  Class names, constructor / forward signatures, parameter names
and state_dict keys are the reference's (SURVEY.md §8b) so the classes drop into
``Mymodel`` (model/backbone.py:40-41) unchanged."""
import ctypes
import math

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from ._lib import check, f32c, ptr, stream, workspace


def cluster_alpha(max_n=40):
    """annealing schedule of model/cluster.py:15-24 (unused by the reference's drivers)"""
    alphas = np.zeros(max_n, dtype=float)
    alphas[0] = 0.1
    for i in range(1, max_n):
        alphas[i] = (2 ** (1 / (np.log(i + 1)) ** 2)) * alphas[i - 1]
    return alphas


# ---------------------------------------------------------------------------
# C1 / C2
# ---------------------------------------------------------------------------
class _ClusterAssign(torch.autograd.Function):
    """fused LN -> cdist -> argmin -> softmin -> A@centers (+ sum (D*A)^2) and its backward"""

    @staticmethod
    def forward(ctx, x, centers, ln_w, ln_b, alpha, eps, impl):
        _lib.require_cuda(x, centers, ln_w, ln_b)
        lead, C = x.shape[:-1], x.shape[-1]
        K = centers.shape[0]
        if centers.shape[1] != C:
            raise RuntimeError("X1 and X2 must have the same number of columns. X1: %d X2: %d"
                               % (C, centers.shape[1]))       # torch.cdist's message
        x2 = f32c(x).reshape(-1, C)
        cen, w, b = f32c(centers), f32c(ln_w), f32c(ln_b)
        N = x2.shape[0]
        dev = x2.device
        # any cluster_num (model/cluster.py:58-75): rows of K values are addressed with 128-bit accesses, so the
        # centroids are padded with zero rows to a multiple of 4 and the padding is excluded on the device
        # (vadc_cluster_fwd_padded: A is exactly 0 there); the outputs are cut back to K columns
        K_valid = K
        if K % 4:
            K = K + 4 - K % 4
            cen = torch.cat([cen, cen.new_zeros((K - K_valid, C))])
        D = torch.empty((N, K), device=dev, dtype=torch.float32)
        A = torch.empty((N, K), device=dev, dtype=torch.float32)
        R = torch.empty((N, C), device=dev, dtype=torch.float32)
        F = torch.empty((N, C), device=dev, dtype=torch.float32)
        label = torch.empty((N,), device=dev, dtype=torch.int64)
        mu = torch.empty((N,), device=dev, dtype=torch.float32)
        rstd = torch.empty((N,), device=dev, dtype=torch.float32)
        rowstats = torch.empty((N, 4), device=dev, dtype=torch.float32)
        loss_sq = torch.empty((1,), device=dev, dtype=torch.float32)
        l = _lib.lib()
        nb = l.vadc_cluster_fwd_workspace_bytes(N, C, K, impl)
        ws = workspace(nb, dev)
        if K_valid == K:
            check(l.vadc_cluster_fwd(ptr(x2), ptr(w), ptr(b), ptr(cen), N, C, K, float(alpha), float(eps),
                                     ptr(D), ptr(A), ptr(R), ptr(F), ptr(label), ptr(mu), ptr(rstd),
                                     ptr(rowstats), ptr(loss_sq), ptr(ws), ws.numel(), impl, stream()),
                  "vadc_cluster_fwd")
        else:
            check(l.vadc_cluster_fwd_padded(ptr(x2), ptr(w), ptr(b), ptr(cen), N, C, K, K_valid, float(alpha), float(eps),
                                            ptr(D), ptr(A), ptr(R), ptr(F), ptr(label), ptr(mu), ptr(rstd),
                                            ptr(rowstats), ptr(loss_sq), ptr(ws), ws.numel(), stream()),
                  "vadc_cluster_fwd_padded")
        ctx.save_for_backward(x2, cen, w, b, D, A, F, mu, rstd, rowstats)
        ctx.alpha, ctx.lead, ctx.K_valid = float(alpha), lead, K_valid
        ctx.mark_non_differentiable(label)
        ctx.set_materialize_grads(False)          # unused outputs arrive as None, not as zero tensors
        if K_valid != K:
            Dv, Av = D[:, :K_valid].contiguous(), A[:, :K_valid].contiguous()
            return (Dv.view(*lead, K_valid), Av.view(*lead, K_valid), R.view(*lead, C), F, label, loss_sq)
        return (D.view(*lead, K), A.view(*lead, K), R.view(*lead, C), F, label, loss_sq)

    @staticmethod
    def backward(ctx, gD, gA, gR, gF, _glabel, gLsq):
        x2, cen, w, b, D, A, F, mu, rstd, rowstats = ctx.saved_tensors
        N, C = x2.shape
        K = cen.shape[0]
        dev = x2.device

        Kv = ctx.K_valid

        def prep(g, cols):
            return None if g is None else f32c(g).reshape(-1, cols)

        def prep_k(g):                             # gradients of the K_valid real columns; the padding gets zeros
            if g is None:
                return None
            g = f32c(g).reshape(-1, Kv)
            return g if Kv == K else torch.nn.functional.pad(g, (0, K - Kv))

        gD, gA, gR, gF = prep_k(gD), prep_k(gA), prep(gR, C), prep(gF, C)
        gLsq = None if gLsq is None else f32c(gLsq)
        gx = torch.empty((N, C), device=dev, dtype=torch.float32)
        gc = torch.empty((K, C), device=dev, dtype=torch.float32)
        gw = torch.empty((C,), device=dev, dtype=torch.float32)
        gb = torch.empty((C,), device=dev, dtype=torch.float32)
        l = _lib.lib()
        nb = l.vadc_cluster_bwd_workspace_bytes(N, C, K)
        ws = workspace(nb, dev)
        check(l.vadc_cluster_bwd(ptr(x2), ptr(mu), ptr(rstd), ptr(rowstats), ptr(F), ptr(w), ptr(b), ptr(cen), ptr(D), ptr(A),
                                 ptr(gD), ptr(gA), ptr(gR), ptr(gF), ptr(gLsq), N, C, K, ctx.alpha,
                                 ptr(gx), ptr(gc), ptr(gw), ptr(gb), ptr(ws), ws.numel(), stream()),
              "vadc_cluster_bwd")
        return gx.view(*ctx.lead, C), (gc if Kv == K else gc[:Kv]), gw, gb, None, None, None


def _cdist_fwd(a3, b3):
    """vadc_cdist of a3 [nb,R,C] and b3 [nb,P,C] (fp32, contiguous) -> [nb,R,P]"""
    nbatch, R, C = a3.shape
    P = b3.shape[1]
    out = torch.empty((nbatch, R, P), device=a3.device, dtype=torch.float32)
    l = _lib.lib()
    nb = l.vadc_cdist_workspace_bytes(nbatch, R, P, C)
    ws = workspace(nb, a3.device)
    check(l.vadc_cdist(ptr(a3), ptr(b3), nbatch, R, P, C, ptr(out), ptr(ws), ws.numel(), stream()), "vadc_cdist")
    return out


def _cdist_bwd(a3, b3, D, g, need_a, need_b, self_mode=False):
    """(ga, gb) of cdist(a3, b3) for the upstream gradient g [nb,R,P] (vadc_cdist_bwd); an unrequested one is None.
    self_mode: b3 is a3, and ga is the whole gradient of cdist(a3, a3)."""
    nbatch, R, C = a3.shape
    P = b3.shape[1]
    g = f32c(g)
    ga = torch.empty_like(a3) if need_a else None
    gb = torch.empty_like(b3) if need_b and not self_mode else None
    l = _lib.lib()
    nb = l.vadc_cdist_bwd_workspace_bytes(nbatch, R, P, C)
    ws = workspace(nb, a3.device)
    check(l.vadc_cdist_bwd(ptr(a3), None if self_mode else ptr(b3), ptr(D), ptr(g), nbatch, R, P, C, int(self_mode),
                           ptr(ga), ptr(gb), ptr(ws), ws.numel(), stream()), "vadc_cdist_bwd")
    return ga, gb


class _CDist(torch.autograd.Function):
    """cdist(a [nb,R,C], b [nb,P,C]) -> [nb,R,P] and its backward on the vadc kernels"""

    @staticmethod
    def forward(ctx, a3, b3):
        D = _cdist_fwd(a3, b3)
        ctx.save_for_backward(a3, b3, D)
        ctx.set_materialize_grads(False)
        return D

    @staticmethod
    def backward(ctx, g):
        if g is None:
            return None, None
        a3, b3, D = ctx.saved_tensors
        return _cdist_bwd(a3, b3, D, g, ctx.needs_input_grad[0], ctx.needs_input_grad[1])


class _SelfDist(torch.autograd.Function):
    """cdist(c, c) of c [nb,K,C] -> [nb,K,K] (self_similarity(), model/cluster.py:77-79,124-125).  The reference never
    back-propagates through it (backbone.py:95-97 are commented out); the backward is vadc_cdist_bwd's self mode."""

    @staticmethod
    def forward(ctx, c3):
        S = _cdist_fwd(c3, c3)
        ctx.save_for_backward(c3, S)
        ctx.set_materialize_grads(False)
        return S

    @staticmethod
    def backward(ctx, gS):
        if gS is None:
            return None
        c3, S = ctx.saved_tensors
        return _cdist_bwd(c3, c3, S, gS, True, False, self_mode=True)[0]


def cdist(a, b):
    """``torch.cdist(a, b)`` (p=2, mm form) on the vadc kernels, differentiable in both arguments.
    a [..., R, C], b [..., P, C]; the leading dimensions broadcast as torch.cdist's do.  ``cdist(c, c)`` (the same
    tensor twice, as in self_similarity()) takes the self-distance path."""
    _lib.require_cuda(a, b)
    for name, t in (("X1", a), ("X2", b)):
        if t.dim() < 2:
            raise RuntimeError("cdist only supports at least 2D tensors, %s got: %dD" % (name, t.dim()))
    if a.shape[-1] != b.shape[-1]:
        raise RuntimeError("X1 and X2 must have the same number of columns. X1: %d X2: %d"
                           % (a.shape[-1], b.shape[-1]))
    R, P, C = a.shape[-2], b.shape[-2], a.shape[-1]
    # every reshape names its sizes: a -1 next to a zero-sized dimension is ambiguous to torch, and empty inputs (R, P
    # or a leading dimension 0) give torch.cdist's empty result and zero / empty gradients
    if a is b:
        lead = a.shape[:-2]
        return _SelfDist.apply(f32c(a).reshape(math.prod(lead), R, C)).view(*lead, R, P)
    if a.dim() == 2 and b.dim() == 2:
        return _CDist.apply(f32c(a)[None], f32c(b)[None]).view(R, P)      # a view: its backward copies nothing
    if b.dim() == 2:              # b's rows are shared by every batch of a: a's leading dimensions fold into its rows
        lead = a.shape[:-2]
        return _CDist.apply(f32c(a).reshape(1, math.prod(lead) * R, C), f32c(b)[None]).view(*lead, R, P)
    if a.dim() == 2:              # a's rows are shared: b's leading dimensions fold into its rows, D^T per batch
        lead = b.shape[:-2]
        Dt = _CDist.apply(f32c(b).reshape(1, math.prod(lead) * P, C), f32c(a)[None])          # [1, n P, R]
        return Dt.view(*lead, P, R).transpose(-1, -2).contiguous()
    lead = a.shape[:-2]
    if b.shape[:-2] != lead:      # the smaller side is expanded (autograd sums its gradient back); torch's error otherwise
        lead = torch.broadcast_tensors(torch.empty(lead, device="meta"), torch.empty(b.shape[:-2], device="meta"))[0].shape
    nbatch = math.prod(lead)
    a3 = f32c(a.expand(*lead, R, C)).reshape(nbatch, R, C)
    b3 = f32c(b.expand(*lead, P, C)).reshape(nbatch, P, C)
    return _CDist.apply(a3, b3).view(*lead, R, P)


class PosSoftAssign(nn.Module):
    """model/cluster.py:27-39"""

    def __init__(self, dims=1, alpha=1.0):
        super().__init__()
        self.dims = dims
        self.alpha = alpha

    def forward(self, x, alpha=None):
        if not alpha == None:  # noqa: E711  (reference semantics: persistently overwrites)
            self.alpha = alpha
        return soft_assign(x, self.dims, self.alpha)


class NegSoftAssign(nn.Module):
    """model/cluster.py:42-55"""

    def __init__(self, dims=1, alpha=32.0):
        super().__init__()
        self.dims = dims
        self.alpha = alpha

    def forward(self, x, alpha=None):
        if not alpha == None:  # noqa: E711
            self.alpha = alpha
        return soft_assign(x, self.dims, -self.alpha)


class _SoftAssign(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x2, signed_alpha):
        _lib.require_cuda(x2)
        rows, K = x2.shape
        out = torch.empty_like(x2)
        check(_lib.lib().vadc_soft_assign(ptr(x2), rows, K, float(signed_alpha), ptr(out), stream()),
              "vadc_soft_assign")
        ctx.save_for_backward(out)
        ctx.a = float(signed_alpha)
        return out

    @staticmethod
    def backward(ctx, g):
        (y,) = ctx.saved_tensors
        g = f32c(g)
        gx = torch.empty_like(y)
        check(_lib.lib().vadc_soft_assign_bwd(ptr(y), ptr(g), y.shape[0], y.shape[1], ctx.a, ptr(gx), stream()),
              "vadc_soft_assign_bwd")
        return gx, None


def soft_assign(x, dim, signed_alpha):
    """exp(a (x - ext)) / sum along ``dim`` (ext = max for a > 0, min for a < 0)"""
    xt = f32c(x.movedim(dim, -1))
    K = xt.shape[-1]
    y = _SoftAssign.apply(xt.reshape(-1, K), signed_alpha)
    return y.view(xt.shape).movedim(-1, dim)


class EuclidDistance_Assign_Module(nn.Module):
    """Drop-in for model/cluster.py:58-99.

    forward(x [B,D,H,W,C], alpha=None) ->
        (x_distance [B,D,H,W,K], x_distance_assign [B,D,H,W,K], cluster_dist [K,K],
         x_rec [B,D,H,W,C], feature [N,C], feature_label [N] int64)
    Extra (not in the reference): ``self.loss_sq`` holds sum (D*A)^2 of the last
    forward, connected to autograd; ``fused_cluster_loss()`` returns
    sqrt(loss_sq) == torch.norm(x_distance * x_distance_assign) (backbone.py:98)
    without two extra passes over [N,K].  ``impl`` selects the kernel family.
    """

    def __init__(self, feature_dim, cluster_num=256, maxpool=1, soft_assign_alpha=32.0):
        super().__init__()
        self.euclid_dis = cdist
        self.act = nn.Sigmoid()
        self.feature_dim = feature_dim
        self.cluster_num = cluster_num
        self.norm = nn.LayerNorm(feature_dim)
        self.assign_func = NegSoftAssign(-1, soft_assign_alpha)
        self.impl = _lib.IMPL_AUTO
        self.loss_sq = None
        self.register_param()

    def register_param(self):
        cluster_center = nn.Parameter(torch.rand(self.cluster_num, self.feature_dim), requires_grad=True)
        identity_matrix = nn.Parameter(torch.eye(self.cluster_num), requires_grad=False)
        self.register_parameter('cluster_center', cluster_center)
        self.register_parameter('identity_matrix', identity_matrix)
        return

    def self_similarity(self):
        return cdist(self.cluster_center, self.cluster_center)

    def forward(self, x, alpha=None):
        if not alpha == None:  # noqa: E711  (cluster.py:49-50: persists on assign_func)
            self.assign_func.alpha = alpha
        if x.dim() != 5:
            raise ValueError("not enough values to unpack (expected 5, got %d)" % x.dim())
        D, A, R, F, label, loss_sq = _ClusterAssign.apply(
            x, self.cluster_center, self.norm.weight, self.norm.bias,
            self.assign_func.alpha, self.norm.eps, self.impl)
        self.loss_sq = loss_sq
        cluster_dist = self.self_similarity()
        return D, A, cluster_dist, R, F, label

    def fused_cluster_loss(self):
        """== torch.norm(x_distance * x_distance_assign) of the last forward"""
        return torch.sqrt(self.loss_sq[0])


# ---------------------------------------------------------------------------
# C3
# ---------------------------------------------------------------------------
class _SpaceClusterAssign(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, centers, ln_w, ln_b, alpha, eps):
        _lib.require_cuda(x, centers, ln_w, ln_b)
        B, Dd, H, W, C = x.shape
        Cc, K, P = centers.shape
        if Cc != C:
            raise RuntimeError("Expected size for first two dimensions of batch2 tensor to be: "
                               f"[{C}, ...] but got: [{Cc}, ...].")
        if P != H * W:
            raise RuntimeError("X1 and X2 must have the same number of columns. X1: %d X2: %d" % (H * W, P))
        x2 = f32c(x).reshape(-1, C)
        cen, w, b = f32c(centers), f32c(ln_w), f32c(ln_b)
        M = B * Dd
        dev = x2.device
        K_valid = K
        if K % 4:                                  # any cluster_num: zero rows up to a multiple of 4, excluded on the device
            K = K + 4 - K % 4
            cen = torch.cat([cen, cen.new_zeros((C, K - K_valid, P))], dim=1)
        Ds = torch.empty((M, C, K), device=dev, dtype=torch.float32)
        As = torch.empty((M, C, K), device=dev, dtype=torch.float32)
        Sd = torch.empty((C, K, K), device=dev, dtype=torch.float32)      # cdist(centers, centers), model/cluster.py:134
        mu = torch.empty((M * P,), device=dev, dtype=torch.float32)
        rstd = torch.empty((M * P,), device=dev, dtype=torch.float32)
        loss_sq = torch.empty((1,), device=dev, dtype=torch.float32)
        l = _lib.lib()
        # LayerNorm output in the [C, M, P] cdist layout, kept for the backward: opaque (bf16 operand terms or fp32)
        zt = torch.empty((l.vadc_space_cluster_saved_bytes(M, P, C, K),), device=dev, dtype=torch.uint8)
        nb = l.vadc_space_cluster_fwd_workspace_bytes(M, P, C, K)
        ws = workspace(nb, dev)
        if K_valid == K:
            check(l.vadc_space_cluster_fwd(ptr(x2), ptr(w), ptr(b), ptr(cen), M, P, C, K, float(alpha),
                                           float(eps), ptr(Ds), ptr(As), ptr(Sd), ptr(zt), ptr(mu), ptr(rstd),
                                           ptr(loss_sq), ptr(ws), ws.numel(), stream()),
                  "vadc_space_cluster_fwd")
        else:
            check(l.vadc_space_cluster_fwd_padded(ptr(x2), ptr(w), ptr(b), ptr(cen), M, P, C, K, K_valid, float(alpha),
                                                  float(eps), ptr(Ds), ptr(As), ptr(Sd), ptr(zt), ptr(mu), ptr(rstd),
                                                  ptr(loss_sq), ptr(ws), ws.numel(), stream()),
                  "vadc_space_cluster_fwd_padded")
        if K_valid != K:
            Sd = Sd[:, :K_valid, :K_valid].contiguous()
        ctx.save_for_backward(x2, cen, w, b, Ds, As, zt, mu, rstd, Sd)
        ctx.alpha, ctx.shape, ctx.K_valid = float(alpha), (B, Dd, H, W, C), K_valid
        ctx.set_materialize_grads(False)
        if K_valid != K:
            return (Ds[:, :, :K_valid].contiguous().view(B, Dd, C, K_valid),
                    As[:, :, :K_valid].contiguous().view(B, Dd, C, K_valid), loss_sq, Sd)
        return Ds.view(B, Dd, C, K), As.view(B, Dd, C, K), loss_sq, Sd

    @staticmethod
    def backward(ctx, gD, gA, gLsq, gS=None):
        x2, cen, w, b, Ds, As, zt, mu, rstd, Sd = ctx.saved_tensors
        B, Dd, H, W, C = ctx.shape
        M, P, K = B * Dd, H * W, cen.shape[1]
        dev = x2.device
        Kv = ctx.K_valid

        def prep_k(g):
            if g is None:
                return None
            g = f32c(g).reshape(M, C, Kv)
            return g if Kv == K else torch.nn.functional.pad(g, (0, K - Kv))

        gD, gA = prep_k(gD), prep_k(gA)
        gLsq = None if gLsq is None else f32c(gLsq)
        gx = torch.empty((M * P, C), device=dev, dtype=torch.float32)
        gc = torch.empty_like(cen)
        gw = torch.empty((C,), device=dev, dtype=torch.float32)
        gb = torch.empty((C,), device=dev, dtype=torch.float32)
        l = _lib.lib()
        nb = l.vadc_space_cluster_bwd_workspace_bytes(M, P, C, K)
        ws = workspace(nb, dev)
        check(l.vadc_space_cluster_bwd(ptr(x2), ptr(mu), ptr(rstd), ptr(zt), ptr(w), ptr(b), ptr(cen), ptr(Ds),
                                       ptr(As), ptr(gD), ptr(gA), ptr(gLsq), M, P, C, K, ctx.alpha,
                                       ptr(gx), ptr(gc), ptr(gw), ptr(gb), ptr(ws), ws.numel(), stream()),
              "vadc_space_cluster_bwd")
        gc = gc if Kv == K else gc[:, :Kv].contiguous()
        if gS is not None:     # the reference never back-propagates through the self-distance (backbone.py:95-97 are comments)
            c3 = cen if Kv == K else cen[:, :Kv].contiguous()
            gc = gc + _cdist_bwd(c3, c3, Sd, gS, True, False, self_mode=True)[0]
        return gx.view(B, Dd, H, W, C), gc, gw, gb, None, None


class Space_EuclidDistance_Assign_Module(nn.Module):
    """Drop-in for model/cluster.py:102-149.  forward(x [B,D,H,W,C]) ->
    (x_distance [B,D,C,K], x_distance_assign [B,D,C,K], cluster_dist [C,K,K], [])
    — the last element is an empty Python list, as in the reference (:135)."""

    def __init__(self, feature_dim, cluster_num=128, space_size=28, maxpool=1, soft_assign_alpha=32.0):
        super().__init__()
        self.euclid_dis = cdist
        self.act = nn.Sigmoid()
        self.feature_dim = feature_dim
        self.cluster_num = cluster_num
        self.norm = nn.LayerNorm(feature_dim)
        self.space_size = space_size * space_size
        self.assign_func = NegSoftAssign(-1, soft_assign_alpha)
        self.loss_sq = None
        self.register_param()

    def register_param(self):
        cluster_center = nn.Parameter(torch.rand(self.feature_dim, self.cluster_num, self.space_size),
                                      requires_grad=True)
        identity_matrix = nn.Parameter(
            torch.eye(self.cluster_num).unsqueeze(0).repeat(self.feature_dim, 1, 1), requires_grad=False)
        self.register_parameter('cluster_center', cluster_center)
        self.register_parameter('identity_matrix', identity_matrix)
        return

    def self_similarity(self):
        return cdist(self.cluster_center, self.cluster_center)

    def forward(self, x, alpha=None):
        if not alpha == None:  # noqa: E711
            self.assign_func.alpha = alpha
        Ds, As, loss_sq, cluster_dist = _SpaceClusterAssign.apply(
            x, self.cluster_center, self.norm.weight, self.norm.bias,
            self.assign_func.alpha, self.norm.eps)       # cluster_dist = self_similarity(), from the same centroid terms
        self.loss_sq = loss_sq
        x_rec = []
        return Ds, As, cluster_dist, x_rec

    def fused_cluster_loss(self):
        """== torch.norm(xf_distance * xf_assign) (backbone.py:94) of the last forward"""
        return torch.sqrt(self.loss_sq[0])
