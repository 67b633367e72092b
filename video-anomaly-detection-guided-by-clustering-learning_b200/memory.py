"""Host-side mirror of the MNAD memory module (model/Memory.py:62-261) on top
of libvadc.so.  Same class / method names and return tuples; ``keys`` in,
``updated_memory`` out (stateless, detached) like the reference.

What changes underneath (SURVEY.md §3.3): ``get_score`` is computed ONCE per
forward instead of four times, and the python loop over memory slots with a
``nonzero()`` host sync per slot (Memory.py:100-113) is a stable counting sort
plus a segmented weighted sum on the device.
"""
import torch
import torch.nn as nn

from . import _lib
from ._lib import check, f32c, ptr, stream, workspace


class _MemoryLoss(torch.autograd.Function):
    """separateness of the memory items and its gradient: with S = K K^T/2 + 1/2 - I and G = sgn(S) (sgn(0) = 0, as
    torch's abs backward), d/dK = g / (m (m-1)) (G + G^T)/2 K"""

    @staticmethod
    def forward(ctx, memory):
        k = f32c(memory)
        m, d = k.shape
        out = torch.empty((), device=k.device, dtype=torch.float32)
        l = _lib.lib()
        ws = workspace(l.vadc_memory_separateness_workspace_bytes(m, d), k.device)
        check(l.vadc_memory_separateness(ptr(k), m, d, ptr(out), ptr(ws), ws.numel(), stream()),
              "vadc_memory_separateness")
        if ctx.needs_input_grad[0]:
            ctx.save_for_backward(k)
        return out

    @staticmethod
    def backward(ctx, g_out):
        (k,) = ctx.saved_tensors
        m, d = k.shape
        g = f32c(g_out).reshape(1)
        gk = torch.empty_like(k)
        l = _lib.lib()
        ws = workspace(l.vadc_memory_separateness_bwd_workspace_bytes(m, d), k.device)
        check(l.vadc_memory_separateness_bwd(ptr(k), ptr(g), m, d, ptr(gk), ptr(ws), ws.numel(), stream()),
              "vadc_memory_separateness_bwd")
        return gk


def MemoryLoss(memory):
    """model/Memory.py:52-59: separateness sum |K K^T/2 + 1/2 - I| / (m (m-1)); differentiable with respect to
    ``memory`` (the regulariser of learnable memory items)"""
    _lib.require_cuda(memory)
    return _MemoryLoss.apply(memory)


def _dist_reduce(t, op):
    """all-reduce over the default process group (NCCL over NVLink); identity when not distributed"""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM)
    return t


class _Scores:
    """everything ``get_score`` + the topk calls derive from one (query, keys) pair"""
    __slots__ = ("q", "score_query", "score_memory", "colmax", "colsum", "top1", "top2", "score_memory_terms")


def _compute_scores(q, keys, need_query_softmax=True, want_read_terms=False):
    N, d = q.shape
    m = keys.shape[0]
    dev = q.device
    s = _Scores()
    s.q = q
    s.score_memory = torch.empty((N, m), device=dev, dtype=torch.float32)
    s.score_query = torch.empty((N, m), device=dev, dtype=torch.float32) if need_query_softmax else None
    s.colmax = torch.empty((m,), device=dev, dtype=torch.float32)
    s.colsum = torch.empty((m,), device=dev, dtype=torch.float32)
    s.top1 = torch.empty((N,), device=dev, dtype=torch.int64)
    s.top2 = torch.empty((N,), device=dev, dtype=torch.int64)
    # operand terms of score_memory for the read contraction, written in the softmax pass (opaque: 4 bytes per element)
    s.score_memory_terms = torch.empty((N * m * 4 + 16,), device=dev, dtype=torch.uint8) if want_read_terms else None
    l = _lib.lib()
    ws = workspace(l.vadc_memory_score_workspace_bytes(N, m, d), dev)
    check(l.vadc_memory_score(ptr(q), ptr(keys), N, m, d, ptr(s.score_query), ptr(s.score_memory),
                              ptr(s.colmax), ptr(s.colsum), ptr(s.top1), ptr(s.top2), ptr(s.score_memory_terms),
                              ptr(ws), ws.numel(), stream()), "vadc_memory_score")
    return s


class _MemoryForward(torch.autograd.Function):
    """Memory.forward (Memory.py:145-175) as one autograd node.  Gradients flow to ``query`` exactly where
    the reference graph lets them: through the first half of ``updated_query`` (the read softmax is
    ``.detach()``ed, :255), ``gathering_loss`` (:245) and ``spreading_loss`` (:229), back through
    ``F.normalize`` (:148).  ``keys`` get a gradient only through the read product (:255, ``score_memory`` detached):
    g_keys = score_memory^T G_r, computed when ``keys`` requires grad (e.g. an ``nn.Parameter``; main.py:131 passes
    a plain tensor, and then nothing extra is saved or launched).  Every other use of ``keys`` is detached (:229,
    :245), ``updated_memory`` is detached (:204).  The two score matrices are not differentiable unless
    ``Memory.differentiable_scores`` is set: then, as in the reference graph (get_score, :133-143), their gradients
    reach the query through F.normalize and, when ``keys`` require grad, the keys (vadc_memory_score_coldot,
    vadc_memory_scores_bwd), and both matrices are kept for the backward.  Under ``Memory.global_batch`` the read
    softmax is per token and the column dots of score_query are all-reduced, so each rank's g_keys is the
    contribution of its own tokens: their sum over ranks is the full-batch gradient, and summing it is left to the
    caller (DDP's gradient all-reduce, or ``allreduce_sum_packed``)."""

    @staticmethod
    def forward(ctx, mod, query, keys, train):
        keys_c = f32c(keys)
        qc = f32c(query)
        q4 = mod.prepare_query(qc)
        q, shp = mod._flat(q4)
        s = _compute_scores(q, keys_c, want_read_terms=True)
        gathering_loss, spreading_loss = mod._losses(s, keys_c, train)
        gathering_loss = gathering_loss.clone()           # separate outputs, not two views of one buffer
        spreading_loss = None if spreading_loss is None else spreading_loss.clone()
        updated_query = mod._read(s, keys_c, shp)
        ctx.loss_scale = 1.0
        glob = mod.global_batch and mod._reduce is not None
        if glob:
            # tokens are sharded over ranks: column statistics, losses and update sums become those of the full batch
            n_all = mod._reduce(torch.tensor([float(q.shape[0])], device=q.device), "sum")
            ctx.loss_scale = float(q.shape[0]) / float(n_all)         # local mean -> this rank's share of the global mean
            cm_g, contrib, S = mod._dp_column_stats(s)
            mod._dp_rescale_scores(s, contrib, S)
            gathering_loss = mod._reduce(gathering_loss.reshape(1) * ctx.loss_scale, "sum")[0]
            if spreading_loss is not None:
                spreading_loss = mod._reduce(spreading_loss.reshape(1) * ctx.loss_scale, "sum")[0]
        # differentiable score matrices: both are kept for the backward (2 N m floats, as the reference's softmax nodes)
        ctx.scores = bool(mod.differentiable_scores) and any(ctx.needs_input_grad[1:3])
        ctx.reduce = mod._reduce if (ctx.scores and glob) else None
        if ctx.scores:
            ctx.save_for_backward(qc, keys_c, s.top1, s.top2, s.score_query, s.score_memory)
        elif ctx.needs_input_grad[2]:                     # learnable memory items: the read needs score_memory back
            ctx.save_for_backward(qc, keys_c, s.top1, s.top2, s.score_memory)
        else:
            ctx.save_for_backward(qc, keys_c, s.top1, s.top2)
        ctx.train = bool(train)
        ctx.set_materialize_grads(False)
        if train:
            updated_memory = mod._dp_update(s, keys_c, cm_g) if glob else mod._update(s, keys_c)
            if ctx.scores:
                ctx.mark_non_differentiable(updated_memory)
            else:
                ctx.mark_non_differentiable(updated_memory, s.score_query, s.score_memory)
            return (updated_query, updated_memory, s.score_query, s.score_memory,
                    gathering_loss, spreading_loss)
        if not ctx.scores:
            ctx.mark_non_differentiable(s.score_query, s.score_memory)
        return updated_query, s.score_query, s.score_memory, gathering_loss

    @staticmethod
    def backward(ctx, *grads):
        qc, keys_c, top1, top2 = ctx.saved_tensors[:4]
        if ctx.train:
            g_uq, _, g_sq, g_sm, g_gather, g_spread = grads
        else:
            (g_uq, g_sq, g_sm, g_gather), g_spread = grads, None
        if not ctx.scores:
            g_sq = g_sm = None
        if g_uq is None and g_gather is None and g_spread is None and g_sq is None and g_sm is None:
            return None, None, None, None
        B, d, h, w = qc.shape
        g_uq = None if g_uq is None else f32c(g_uq)                  # [B,2d,h,w]; the first d channels reach q
        # (global batch: the kernel divides by the local token count; loss_scale turns that into the global mean)
        g_gather = None if g_gather is None else f32c(g_gather).reshape(1) * ctx.loss_scale
        g_spread = None if g_spread is None else f32c(g_spread).reshape(1) * ctx.loss_scale
        l = _lib.lib()
        m = keys_c.shape[0]
        gq = gk = None
        if ctx.needs_input_grad[2] and g_uq is not None:   # the losses reach keys only through detached copies
            score_memory = ctx.saved_tensors[-1]
            gk = torch.empty_like(keys_c)
            ws = workspace(l.vadc_memory_keys_bwd_workspace_bytes(B, d, h * w, m), gk.device)
            check(l.vadc_memory_keys_bwd(ptr(score_memory), ptr(g_uq), B, d, h * w, m, ptr(gk), ptr(ws), ws.numel(),
                                         stream()), "vadc_memory_keys_bwd")
        g_qhat = None
        if g_sq is not None or g_sm is not None:
            g_qhat, gk = _scores_backward(ctx, qc, keys_c, f32c(g_sq), f32c(g_sm), gk)
        if ctx.needs_input_grad[1]:
            gq = torch.empty_like(qc)
            if g_qhat is None:
                check(l.vadc_memory_query_bwd(ptr(qc), ptr(keys_c), ptr(top1), ptr(top2) if ctx.train else None,
                                              ptr(g_uq), ptr(g_gather), ptr(g_spread), B, d, h * w,
                                              m, ptr(gq), stream()), "vadc_memory_query_bwd")
            else:
                check(l.vadc_memory_query_bwd_ex(ptr(qc), ptr(keys_c), ptr(top1), ptr(top2) if ctx.train else None,
                                                 ptr(g_uq), ptr(g_gather), ptr(g_spread), ptr(g_qhat), B, d, h * w,
                                                 m, ptr(gq), stream()), "vadc_memory_query_bwd_ex")
        return None, gq, gk, None


def _scores_backward(ctx, qc, keys_c, g_sq, g_sm, gk):
    """the share of the returned score matrices: (g_qhat [B,d,h,w] or None, g_keys) with g_keys = gk + g_s^T q-hat
    when the keys require grad (gk None: the read contributed nothing)"""
    sq, sm = ctx.saved_tensors[-2:]
    B, d, h, w = qc.shape
    N, m = sm.shape
    l = _lib.lib()
    coldot = None
    if g_sq is not None:
        coldot = torch.empty((m,), device=qc.device, dtype=torch.float32)
        ws = workspace(l.vadc_memory_score_coldot_workspace_bytes(N, m), qc.device)
        check(l.vadc_memory_score_coldot(ptr(sq), ptr(g_sq), N, m, ptr(coldot), ptr(ws), ws.numel(), stream()),
              "vadc_memory_score_coldot")
        if ctx.reduce is not None:                        # global batch: the column softmax spans every rank's tokens
            coldot = ctx.reduce(coldot, "sum")
    g_qhat = torch.empty_like(qc) if ctx.needs_input_grad[1] else None
    if ctx.needs_input_grad[2] and gk is None:
        gk = torch.zeros_like(keys_c)
    elif not ctx.needs_input_grad[2]:
        gk = None
    ws = workspace(l.vadc_memory_scores_bwd_workspace_bytes(B, d, h * w, m), qc.device)
    check(l.vadc_memory_scores_bwd(ptr(qc), ptr(keys_c), ptr(sq), ptr(sm), ptr(g_sq), ptr(g_sm), ptr(coldot),
                                   B, d, h * w, m, ptr(g_qhat), ptr(gk), ptr(ws), ws.numel(), stream()),
          "vadc_memory_scores_bwd")
    return g_qhat, gk


def _grad_possible(*tensors):
    """True when autograd would record a graph for a call on these tensors"""
    return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors)


def _prepare_query(qc):
    B, d, h, w = qc.shape
    out = torch.empty((B, h, w, d), device=qc.device, dtype=torch.float32)
    l = _lib.lib()
    ws = workspace(l.vadc_memory_prepare_query_workspace_bytes(B, h * w), qc.device)
    check(l.vadc_memory_prepare_query(ptr(qc), B, d, h * w, ptr(out), ptr(ws), ws.numel(), stream()),
          "vadc_memory_prepare_query")
    return out


class _PrepareQuery(torch.autograd.Function):
    """F.normalize(query, dim=1).permute(0, 2, 3, 1) (Memory.py:148-149) as an autograd node: per token,
    g_x = (g - q-hat (q-hat . g)) / max(|x|, 1e-12), with g channel-last and g_x channel-first"""

    @staticmethod
    def forward(ctx, query):
        qc = f32c(query)
        ctx.save_for_backward(qc)
        return _prepare_query(qc)

    @staticmethod
    def backward(ctx, g):
        (qc,) = ctx.saved_tensors
        B, d, h, w = qc.shape
        g = f32c(g)
        gx = torch.empty_like(qc)
        check(_lib.lib().vadc_memory_prepare_query_bwd(ptr(g), ptr(qc), B, d, h * w, ptr(gx), stream()),
              "vadc_memory_prepare_query_bwd")
        return gx


def _scores_rows_backward(q, keys_c, sq, sm, g_sq, g_sm, need_q, need_k, gk):
    """the share of get_score's two matrices for a channel-last, unnormalised q [N,d]: (g_q [N,d] or None, g_keys),
    g_keys = gk + g_s^T q when ``need_k`` (gk None: nothing else reached the keys).  Launches nothing when no score
    gradient arrived."""
    if (g_sq is None and g_sm is None) or not (need_q or need_k):
        return None, gk
    g_sq, g_sm = f32c(g_sq), f32c(g_sm)
    N, m = sm.shape
    d = q.shape[1]
    l = _lib.lib()
    coldot = None
    if g_sq is not None:
        coldot = torch.empty((m,), device=q.device, dtype=torch.float32)
        ws = workspace(l.vadc_memory_score_coldot_workspace_bytes(N, m), q.device)
        check(l.vadc_memory_score_coldot(ptr(sq), ptr(g_sq), N, m, ptr(coldot), ptr(ws), ws.numel(), stream()),
              "vadc_memory_score_coldot")
    g_rows = torch.empty_like(q) if need_q else None
    if need_k and gk is None:
        gk = torch.zeros_like(keys_c)
    ws = workspace(l.vadc_memory_scores_bwd_rows_workspace_bytes(N, d, m), q.device)
    check(l.vadc_memory_scores_bwd_rows(ptr(q), ptr(keys_c), ptr(sq), ptr(sm), ptr(g_sq), ptr(g_sm), ptr(coldot),
                                        N, d, m, ptr(g_rows), ptr(gk if need_k else None), ptr(ws), ws.numel(),
                                        stream()), "vadc_memory_scores_bwd_rows")
    return g_rows, gk


class _GetScore(torch.autograd.Function):
    """get_score (Memory.py:133-143) on a channel-last query as an autograd node, differentiable with respect to the
    query and the memory: g_s = sq (Gq - 1 c^T) + sm (Gm - r 1^T), g_q = g_s K, g_K = g_s^T q"""

    @staticmethod
    def forward(ctx, query, mem):
        q, _ = Memory._flat(query)
        keys_c = f32c(mem)
        s = _compute_scores(q, keys_c)
        ctx.save_for_backward(q, keys_c, s.score_query, s.score_memory)
        ctx.qshape = query.shape
        ctx.set_materialize_grads(False)
        return s.score_query, s.score_memory

    @staticmethod
    def backward(ctx, g_sq, g_sm):
        q, keys_c, sq, sm = ctx.saved_tensors
        gq, gk = _scores_rows_backward(q, keys_c, sq, sm, g_sq, g_sm, ctx.needs_input_grad[0],
                                       ctx.needs_input_grad[1], None)
        return (None if gq is None else gq.view(ctx.qshape)), gk


class _Read(torch.autograd.Function):
    """read (Memory.py:249-261) as an autograd node: updated_query = cat(q, score_memory.detach() K) permuted to
    [B,2d,h,w], plus the two score matrices.  The query gets the first d channels of G_uq (transposed to channel-last)
    and the score share g_s K; the memory gets score_memory^T G_r (vadc_memory_keys_bwd) and the score share g_s^T q."""

    @staticmethod
    def forward(ctx, mod, query, mem):
        q, shp = mod._flat(query)
        keys_c = f32c(mem)
        s = _compute_scores(q, keys_c, want_read_terms=True)
        uq = mod._read(s, keys_c, shp)
        ctx.save_for_backward(q, keys_c, s.score_query, s.score_memory)
        ctx.shp = shp
        ctx.set_materialize_grads(False)
        return uq, s.score_query, s.score_memory

    @staticmethod
    def backward(ctx, g_uq, g_sq, g_sm):
        q, keys_c, sq, sm = ctx.saved_tensors
        need_q, need_k = ctx.needs_input_grad[1], ctx.needs_input_grad[2]
        B, h, w, d = ctx.shp
        m = keys_c.shape[0]
        g_uq = None if g_uq is None else f32c(g_uq)                  # [B,2d,h,w]
        l = _lib.lib()
        gk = None
        if need_k and g_uq is not None:
            gk = torch.empty_like(keys_c)
            ws = workspace(l.vadc_memory_keys_bwd_workspace_bytes(B, d, h * w, m), gk.device)
            check(l.vadc_memory_keys_bwd(ptr(sm), ptr(g_uq), B, d, h * w, m, ptr(gk), ptr(ws), ws.numel(), stream()),
                  "vadc_memory_keys_bwd")
        gq, gk = _scores_rows_backward(q, keys_c, sq, sm, g_sq, g_sm, need_q, need_k, gk)
        if need_q and g_uq is not None:
            out = gq if gq is not None else torch.empty_like(q)
            check(l.vadc_memory_rows_bwd(ptr(q), ptr(keys_c), None, None, ptr(g_uq), None, None, ptr(gq), B, d,
                                         h * w, m, ptr(out), stream()), "vadc_memory_rows_bwd")
            gq = out
        return None, (None if gq is None else gq.view(B, h, w, d)), gk


class _MemoryLossTerm(torch.autograd.Function):
    """gather_loss (Memory.py:233-247) or spread_loss (:214-231) as an autograd node, differentiable with respect to
    the query only (the reference detaches the keys, :229, :245); keeps top1 (and top2), no [N, m] matrix"""

    @staticmethod
    def forward(ctx, mod, query, keys, spread):
        q, _ = mod._flat(query)
        keys_c = f32c(keys)
        s = _compute_scores(q, keys_c, False)
        gathering, spreading = mod._losses(s, keys_c, spread)
        ctx.save_for_backward(q, keys_c, s.top1, s.top2 if spread else None)
        ctx.qshape = query.shape
        return spreading if spread else gathering

    @staticmethod
    def backward(ctx, g):
        q, keys_c, top1, top2 = ctx.saved_tensors
        g = f32c(g).reshape(1)
        B, h, w, d = ctx.qshape
        gq = torch.empty_like(q)
        check(_lib.lib().vadc_memory_rows_bwd(ptr(q), ptr(keys_c), ptr(top1), ptr(top2), None,
                                              None if top2 is not None else ptr(g), ptr(g) if top2 is not None else None,
                                              None, B, d, h * w, keys_c.shape[0], ptr(gq), stream()),
              "vadc_memory_rows_bwd")
        return None, gq.view(ctx.qshape), None, None


class Memory(nn.Module):
    """Drop-in for model/Memory.py:62-261.  ``forward`` is differentiable with respect to ``query`` and, when they
    require grad, the memory items ``keys`` (``_MemoryForward``); with ``differentiable_scores`` set, also through
    the returned ``score_query`` / ``score_memory``.  The stand-alone public methods are differentiable where the
    reference's are: ``prepare_query`` (our helper for F.normalize + permute) to its query, ``get_score`` and ``read``
    to the query and the memory argument, ``gather_loss`` and ``spread_loss`` to the query (the keys are detached there,
    as in the reference).  They take the query channel-last, [B,h,w,d], as the reference's do, and do not normalise it.
    Under ``torch.no_grad()``, or when no tensor argument requires grad, they launch and return exactly what a
    forward-only call does, with no ``grad_fn``.  They stay per rank: ``global_batch`` applies to ``forward`` only.
    Not differentiable, by design: ``update`` (its result is detached in the reference, :204) and
    ``get_update_query`` (only ever called inside ``update``); ``updated_memory`` carries no gradient to ``keys``.
    ``pointwise_gather_loss`` is plain torch indexing and differentiable as such.  The reference module is not wired
    into ``Mymodel`` (SURVEY.md D5)."""

    def __init__(self, memory_size, feature_dim, key_dim, temp_update, temp_gather):
        super().__init__()
        self.memory_size = memory_size
        self.feature_dim = feature_dim
        self.key_dim = key_dim
        self.temp_update = temp_update
        self.temp_gather = temp_gather
        # data parallel, SURVEY 8e: False = every rank treats its shard as the batch (what the reference's DDP run
        # does); True = column softmax, update sums and loss means over the tokens of ALL ranks, i.e. the
        # single-process full-batch result: all-reduce MAX of the column maxima [m], SUM of the column sums [m],
        # SUM of the update sums [m,d] and of three scalars
        self.global_batch = False
        # True: score_query and score_memory returned by forward are differentiable, as in the reference (a loss on
        # the addressing weights, e.g. an entropy penalty, reaches the query and learnable keys).  False (default):
        # they are returned for inspection only, and nothing extra is kept for the backward.  When True, the two
        # [N, m] matrices stay alive until the backward (2 N m floats: 1 GB at N = 65536, m = 2000).
        self.differentiable_scores = False
        self._reduce = _dist_reduce

    # -- helpers ------------------------------------------------------------
    @staticmethod
    def _flat(query):
        """[B,h,w,d] (the layout every public method of the reference takes) -> [N,d]"""
        _lib.require_cuda(query)
        B, h, w, d = query.shape
        return f32c(query).reshape(B * h * w, d), (B, h, w, d)

    @staticmethod
    def prepare_query(query):
        """F.normalize(query, dim=1) + permute(0,2,3,1)  (Memory.py:148-149):
        [B,d,h,w] -> [B,h,w,d] contiguous; differentiable with respect to ``query``"""
        _lib.require_cuda(query)
        if _grad_possible(query):
            return _PrepareQuery.apply(query)
        return _prepare_query(f32c(query))

    # -- reference API --------------------------------------------------------
    def get_score(self, mem, query):
        """Memory.py:133-143 -> (softmax over tokens, softmax over slots), [N,m] each; differentiable with respect to
        ``query`` (channel-last, as passed) and ``mem``.  Per rank: ignores ``global_batch``."""
        if _grad_possible(query, mem):
            _lib.require_cuda(query, mem)
            return _GetScore.apply(query, mem)
        q, _ = self._flat(query)
        s = _compute_scores(q, f32c(mem))
        return s.score_query, s.score_memory

    def forward(self, query, keys, train=True):
        """Memory.py:145-175.  query [B,d,h,w], keys [m,d]."""
        _lib.require_cuda(query, keys)
        if train:
            return _MemoryForward.apply(self, query, keys, True)
        uq, sq, sm, gl = _MemoryForward.apply(self, query, keys, False)
        return uq, keys, sq, sm, gl

    def update(self, query, keys, train):
        """Memory.py:177-204 (forward-only: the reference detaches the result, :204)"""
        with torch.no_grad():
            q, _ = self._flat(query)
            keys_c = f32c(keys)
            return self._update(_compute_scores(q, keys_c), keys_c)

    def get_update_query(self, mem, max_indices, update_indices, score, query, train):
        """Memory.py:94-131: weighted sum of the queries assigned to each slot (forward-only: only ever called
        inside ``update``, whose result the reference detaches)"""
        with torch.no_grad():
            q = f32c(query)
            return self._segmented_update(q, f32c(mem), f32c(score),
                                          max_indices.reshape(-1).to(torch.int64).contiguous())[0]

    def pointwise_gather_loss(self, query_reshape, keys, gathering_indices, train):
        """Memory.py:206-212 (elementwise, not a hot path: plain indexing)"""
        return (query_reshape - keys[gathering_indices].squeeze(1).detach()) ** 2

    def spread_loss(self, query, keys, train):
        """Memory.py:214-231; differentiable with respect to ``query`` (the keys are detached, :229).  Per rank:
        ignores ``global_batch``."""
        if _grad_possible(query):
            _lib.require_cuda(query, keys)
            return _MemoryLossTerm.apply(self, query, keys.detach(), True)
        with torch.no_grad():
            q, _ = self._flat(query)
            keys_c = f32c(keys)
            return self._losses(_compute_scores(q, keys_c, False), keys_c, True)[1]

    def gather_loss(self, query, keys, train):
        """Memory.py:233-247; differentiable with respect to ``query`` (the keys are detached, :245).  Per rank:
        ignores ``global_batch``."""
        if _grad_possible(query):
            _lib.require_cuda(query, keys)
            return _MemoryLossTerm.apply(self, query, keys.detach(), False)
        with torch.no_grad():
            q, _ = self._flat(query)
            keys_c = f32c(keys)
            return self._losses(_compute_scores(q, keys_c, False), keys_c, False)[0]

    def read(self, query, updated_memory):
        """Memory.py:249-261 -> (updated_query [B,2d,h,w], score_query, score_memory); differentiable with respect to
        ``query`` and ``updated_memory`` (through the read product and the two score matrices).  Per rank: ignores
        ``global_batch``."""
        if _grad_possible(query, updated_memory):
            _lib.require_cuda(query, updated_memory)
            return _Read.apply(self, query, updated_memory)
        with torch.no_grad():
            q, shp = self._flat(query)
            keys_c = f32c(updated_memory)
            s = _compute_scores(q, keys_c, want_read_terms=True)
            return self._read(s, keys_c, shp), s.score_query, s.score_memory

    # -- kernels --------------------------------------------------------------
    def _losses(self, s, keys, with_spread):
        N, d = s.q.shape
        m = keys.shape[0]
        if with_spread and m < 2:
            raise RuntimeError("selected index k out of range")      # torch.topk(…, 2) on m < 2
        out = torch.empty((2,), device=s.q.device, dtype=torch.float32)
        l = _lib.lib()
        ws = workspace(l.vadc_memory_losses_workspace_bytes(N, d), s.q.device)
        check(l.vadc_memory_losses(ptr(s.q), ptr(keys), ptr(s.top1), ptr(s.top2) if with_spread else None,
                                   N, m, d, ptr(out), ptr(ws), ws.numel(), stream()), "vadc_memory_losses")
        return out[0], (out[1] if with_spread else None)

    def _read(self, s, keys, shp):
        B, h, w, d = shp
        N, m = s.q.shape[0], keys.shape[0]
        uq = torch.empty((N, 2 * d), device=s.q.device, dtype=torch.float32)
        l = _lib.lib()
        ws = workspace(l.vadc_memory_read_workspace_bytes(N, m, d), uq.device)
        check(l.vadc_memory_read(ptr(s.q), ptr(s.score_memory), ptr(s.score_memory_terms), ptr(keys),
                                 N, m, d, ptr(uq), ptr(ws), ws.numel(), stream()), "vadc_memory_read")
        return uq.view(B, h, w, 2 * d).permute(0, 3, 1, 2)          # Memory.py:258-259

    def _segmented_update(self, q, keys, score_query, top1):
        N, d = q.shape
        m = keys.shape[0]
        qu = torch.empty((m, d), device=q.device, dtype=torch.float32)
        um = torch.empty((m, d), device=q.device, dtype=torch.float32)
        l = _lib.lib()
        ws = workspace(l.vadc_memory_update_workspace_bytes(N, m, d), q.device)
        check(l.vadc_memory_update(ptr(q), ptr(keys), ptr(score_query), ptr(top1), N, m, d, ptr(qu), ptr(um),
                                   ptr(ws), ws.numel(), stream()), "vadc_memory_update")
        return qu, um

    def _update(self, s, keys):
        return self._segmented_update(s.q, keys, s.score_query, s.top1)[1].detach()

    # -- global batch over ranks (include/vadc.h: vadc_memory_dp_*) -------------
    def _dp_column_stats(self, s):
        """(global column maxima, this rank's share of the column sums, the global column sums)"""
        l = _lib.lib()
        m = s.colmax.numel()
        cm_g = self._reduce(s.colmax.clone(), "max")
        contrib = torch.empty_like(s.colsum)
        check(l.vadc_memory_dp_contrib(ptr(s.colmax), ptr(s.colsum), ptr(cm_g), m, ptr(contrib), stream()),
              "vadc_memory_dp_contrib")
        S = self._reduce(contrib.clone(), "sum")
        return cm_g, contrib, S

    def _dp_rescale_scores(self, s, contrib, S):
        """local softmax over this rank's tokens -> softmax over all ranks' tokens, in place"""
        N, m = s.score_query.shape
        check(_lib.lib().vadc_scale_columns(ptr(s.score_query), ptr(contrib), ptr(S), N, m, stream()),
              "vadc_scale_columns")

    def _dp_update(self, s, keys, cm_g):
        """update sums of this rank (their weights are invariant under the rescaling above), scaled to the global
        column maximum, summed over ranks, then normalize(u + keys) — identical on every rank"""
        l = _lib.lib()
        m, d = keys.shape
        qu = self._segmented_update(s.q, keys, s.score_query, s.top1)[0]
        check(l.vadc_memory_dp_scale_update(ptr(qu), ptr(s.colmax), ptr(cm_g), m, d, stream()),
              "vadc_memory_dp_scale_update")
        qu = self._reduce(qu, "sum")
        um = torch.empty_like(qu)
        check(l.vadc_memory_finish_update(ptr(qu), ptr(keys), m, d, ptr(um), stream()), "vadc_memory_finish_update")
        return um.detach()
