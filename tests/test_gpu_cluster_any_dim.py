"""EuclidDistance_Assign_Module at any feature_dim (1 <= C <= 4096): C % 4 != 0 and C > 1024 against the float64 oracle,
forward and backward, on every path that takes them (tcgen05 fp16 x2 / bf16 x3 for K % 8 == 0, SIMT, the padded-K
route); which kernels ran; misaligned and stand-alone layouts; the space head at ragged C; the full-size head against
float64 torch autograd on the device."""
import gc
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import videoad_b200 as V
from videoad_b200 import _lib
from videoad_b200.cluster import _ClusterAssign
from oracle import np_oracle as O
from gpu_util import T, N, rel, dev, assert_labels_match, assert_selfdist_close, make_cluster_module

pytestmark = pytest.mark.gpu


@pytest.fixture
def bf16x3():
    os.environ["VADC_TC_BF16X3"] = "1"
    _lib.lib().vadc_refresh_env()
    yield
    os.environ.pop("VADC_TC_BF16X3", None)
    _lib.lib().vadc_refresh_env()


def _cuda_kernels(fn, reps=2):
    """names of the CUDA kernels that ``fn()`` launches: one call before the capture (module loading, workspaces), then
    ``reps`` calls inside it, so that a kernel record the activity tracing misses around its start (seen for the first
    kernel of the window) still shows up from the next repetition"""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if e.device_type.name == "CUDA"}


def _vadc_kernels(names):
    """the library's kernels among ``names``, short enough for an assertion message"""
    return sorted({n.split("(")[0][-120:] for n in names if "vadc::" in n})


def _row_rel(a, b):
    """largest over rows of max |a - b| / max |b| within the row"""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float((np.abs(a - b).max(-1) / np.maximum(np.abs(b).max(-1), 1e-30)).max())


def _inputs(Ntok, C, K, seed):
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal((1, 1, 1, Ntok, C)) * 1.3 + 0.2).astype(np.float32)
    cen = rng.random((K, C)).astype(np.float32)
    if C == 1:
        # every token has the same z = beta, so the centroid gradient is the difference of two sums over all tokens,
        # sum r z and c sum r with r = g / D: a centroid within ~1e-3 of beta makes both ~1 / D times larger than their
        # difference, which no fp32 evaluation (ATen's backward forms the same two terms) keeps within 2e-4; keep D >= 0.2
        cen = (0.5 + 0.5 * cen).astype(np.float32)
    w = (1 + 0.2 * rng.standard_normal(C)).astype(np.float32)
    b = (0.1 * rng.standard_normal(C)).astype(np.float32)
    gR = rng.standard_normal((Ntok, C)).astype(np.float32)
    gF = (0.5 * rng.standard_normal((Ntok, C))).astype(np.float32)
    return x, cen, w, b, gR, gF


def _check_against_oracle(Ntok, C, K, impl, fused, seed, alpha=16.0):
    x, cen, w, b, gR, gF = _inputs(Ntok, C, K, seed)
    m = make_cluster_module(V, C, K, alpha, cen, w, b, impl)
    xt = T(x, grad=True)
    D, A, S, R, Fe, lab = m(xt)
    assert D.shape == (1, 1, 1, Ntok, K) and R.shape == (1, 1, 1, Ntok, C)
    o64 = O.cluster_forward(x, cen, w, b, alpha, dtype=np.float64)
    assert np.isfinite(N(D)).all() and np.isfinite(N(R)).all()
    assert rel(N(Fe).reshape(Ntok, C), o64["feature"].reshape(Ntok, C)) < 1e-5
    assert rel(N(D), o64["D"]) < 1e-5
    assert_labels_match(N(lab), o64["D"])
    np.testing.assert_allclose(N(A), o64["A"], rtol=2e-3, atol=1e-6)
    assert rel(N(R), o64["x_rec"]) < 1e-4
    lo = float(O.frobenius_loss(o64["D"], o64["A"], np.float64))
    closs = m.fused_cluster_loss() if fused else torch.norm(D * A)
    # 1e-5 relative, or the loss's own sensitivity to the (separately checked) error of D where that is larger: A moves
    # by alpha dD relative, so the loss by up to alpha max|dD| relative.  At C = 4096, D ~ 80 comes from fp32 sums over
    # 4096 channels (~1e-6 absolute) and alpha = 16 turns that into ~2e-5 of the loss.
    d_abs = float(np.abs(N(D).astype(np.float64) - o64["D"]).max())
    assert abs(float(closs.detach()) - lo) < max(1e-5, 2 * alpha * d_abs) * lo
    (1.3 * closs + (R * T(gR).view_as(R)).sum() + (Fe * T(gF).view_as(Fe)).sum()).backward()
    lD, lA = O.frobenius_loss_grads(o64["D"], o64["A"], 1.3, np.float64)
    gx, gc, gw, gb = O.cluster_backward(x, cen, w, b, alpha, gD=lD.reshape(Ntok, K), gA=lA.reshape(Ntok, K), gR=gR,
                                        gF=gF, dtype=np.float64)
    assert m.cluster_center.grad.shape == (K, C) and m.norm.weight.grad.shape == (C,) and m.norm.bias.grad.shape == (C,)
    gxd = N(xt.grad).reshape(Ntok, C)
    assert rel(gxd, gx) < 2e-4
    assert _row_rel(gxd, gx) < 2e-3
    assert rel(N(m.cluster_center.grad), gc) < 2e-4
    assert rel(N(m.norm.weight.grad), gw) < 2e-4
    assert rel(N(m.norm.bias.grad), gb) < 2e-4


# (C, K, tokens): every width class of the row kernels (one warp per row up to 512, 2 / 4 / 8 warps per row above), C = 1
# (LayerNorm of one element: z = beta), K on the tensor cores (32, 64, 1024) and on the padded-K route (1, 5)
CASES = [(1, 32, 301), (3, 5, 257), (6, 64, 300), (30, 1, 129), (30, 1024, 200), (190, 32, 333), (190, 1024, 300),
         (190, 5, 220), (770, 64, 211), (1026, 5, 150), (1026, 32, 170), (1536, 32, 190), (2048, 64, 130),
         (2048, 1, 90), (4096, 1024, 97), (4096, 32, 75)]


@pytest.mark.parametrize("fused", [True, False], ids=["fused_loss", "explicit_loss"])
@pytest.mark.parametrize("impl", [V.IMPL_AUTO, V.IMPL_SIMT], ids=["auto", "simt"])
@pytest.mark.parametrize("C,K,Ntok", CASES)
def test_any_feature_dim_forward_backward(C, K, Ntok, impl, fused):
    _check_against_oracle(Ntok, C, K, impl, fused, seed=C * 7 + K + Ntok)


@pytest.mark.parametrize("fused", [True, False], ids=["fused_loss", "explicit_loss"])
@pytest.mark.parametrize("C,K,Ntok", [(1, 32, 301), (6, 64, 300), (190, 32, 333), (190, 1024, 300), (770, 64, 211),
                                      (1536, 32, 190), (4096, 1024, 97)])
def test_any_feature_dim_bf16x3(C, K, Ntok, fused, bf16x3):
    _check_against_oracle(Ntok, C, K, V.IMPL_AUTO, fused, seed=C * 3 + K)


@pytest.mark.parametrize("C,K", [(190, 32), (1026, 64), (30, 1024)])
@pytest.mark.parametrize("mode", ["fp16x2", "bf16x3"])
def test_ragged_c_runs_on_the_tensor_cores(C, K, mode):
    """ragged C with K % 8 == 0: both contractions of the forward and all of the backward's on tc_gemm_persist_kernel,
    no SIMT GEMM, none of the fused fixed-shape kernels"""
    if mode == "bf16x3":
        os.environ["VADC_TC_BF16X3"] = "1"
        _lib.lib().vadc_refresh_env()
    try:
        x, cen, w, b, gR, _ = _inputs(600, C, K, 5)
        params = [T(cen, grad=True), T(w, grad=True), T(b, grad=True)]
        xt = T(x, grad=True)
        gRt = T(gR)

        def fwd_bwd():           # the head alone (the module's forward also runs the stand-alone centroid self-distance)
            D, A, R, Fe, lab, loss_sq = _ClusterAssign.apply(xt, *params, 16.0, 1e-5, V.IMPL_AUTO)
            (torch.sqrt(loss_sq[0]) + (R * gRt.view_as(R)).sum()).backward()

        names = _cuda_kernels(fwd_bwd)
    finally:
        os.environ.pop("VADC_TC_BF16X3", None)
        _lib.lib().vadc_refresh_env()
    vk = _vadc_kernels(names)
    for epi in ("TcDist", "TcPartialEpi", "TcGz"):
        assert any("tc_gemm_persist_kernel" in n and epi in n for n in names), (epi, vk)
    for row_kernel in ("ln_rows_any_kernel", "ln_bwd_any_kernel"):
        assert any(row_kernel in n for n in names), (row_kernel, vk)
    assert not any("sgemm_kernel" in n for n in names), vk
    for fused in ("cluster_fwd_ws_kernel", "cluster_fwd_tc_kernel", "cluster_bwd_tc2_kernel", "cluster_bwd_fused_kernel"):
        assert not any(fused in n for n in names), (fused, vk)


def test_c192_k32_keeps_the_fused_kernels():
    x, cen, w, b, gR, _ = _inputs(4096, 192, 32, 6)
    m = make_cluster_module(V, 192, 32, 16.0, cen, w, b)
    xt = T(x, grad=True)
    gRt = T(gR)

    def fwd_bwd():
        D, A, S, R, Fe, lab = m(xt)
        (m.fused_cluster_loss() + (R * gRt.view_as(R)).sum()).backward()

    names = _cuda_kernels(fwd_bwd)
    vk = _vadc_kernels(names)
    assert any("cluster_fwd_ws" in n for n in names), vk
    assert any("cluster_bwd_tc2" in n for n in names), vk
    assert not any("any_kernel" in n for n in names), vk


@pytest.mark.parametrize("C,K", [(190, 32), (30, 5), (1026, 64)])
def test_misaligned_view_and_self_similarity_at_ragged_c(C, K):
    """x as a contiguous view one float into its storage gives the same result as the aligned tensor; cluster_dist
    (self_similarity) and its gradient at ragged C against the oracle"""
    x, cen, w, b, gR, _ = _inputs(257, C, K, 9)
    m = make_cluster_module(V, C, K, 16.0, cen, w, b)
    flat = torch.empty(x.size + 1, device=dev())
    xv = flat[1:].view(x.shape)
    assert xv.data_ptr() % 16 != 0
    xv.copy_(T(x))
    xa = T(x)
    outs = []
    for inp in (xa, xv):
        t = inp.detach().requires_grad_(True)
        m.zero_grad()
        D, A, S, R, Fe, lab = m(t)
        (m.fused_cluster_loss() + (R * T(gR).view_as(R)).sum()).backward()
        outs.append((D, R, lab, t.grad, m.cluster_center.grad.clone()))
    for a, c in zip(*outs):
        assert torch.equal(a, c)
    ct = T(cen, grad=True)
    S = V.cdist(ct, ct)
    assert_selfdist_close(N(S), O.cdist_mm(cen, cen))
    g = np.random.default_rng(C).random((K, K)).astype(np.float32)
    (S * T(g)).sum().backward()
    c64 = cen.astype(np.float64)
    diff = c64[:, None, :] - c64[None, :, :]
    d = np.sqrt((diff * diff).sum(-1))
    r = np.divide(g + g.T, d, out=np.zeros_like(d), where=d > 0)
    np.fill_diagonal(r, 0.0)
    gc64 = (r[:, :, None] * diff).sum(1)             # d/dc_i of sum_ij g_ij |c_i - c_j|
    assert rel(N(ct.grad), gc64) < 2e-4
    mm = V.EuclidDistance_Assign_Module(C, K).to(dev())
    Sm = mm.self_similarity()
    assert Sm.shape == (K, K)
    Sm.sum().backward()
    assert mm.cluster_center.grad.shape == (K, C) and torch.isfinite(mm.cluster_center.grad).all()


@pytest.mark.parametrize("C", [6, 30, 190])
def test_space_head_at_ragged_c(C):
    B, Dd, side, K = 2, 3, 8, 16
    rng = np.random.default_rng(C)
    x = (rng.standard_normal((B, Dd, side, side, C)) * 1.3).astype(np.float32)
    cen = rng.random((C, K, side * side)).astype(np.float32)
    w = (1 + 0.2 * rng.standard_normal(C)).astype(np.float32)
    b = (0.1 * rng.standard_normal(C)).astype(np.float32)
    m = V.Space_EuclidDistance_Assign_Module(C, K, space_size=side, soft_assign_alpha=32.0).to(dev())
    with torch.no_grad():
        m.cluster_center.copy_(T(cen)); m.norm.weight.copy_(T(w)); m.norm.bias.copy_(T(b))
    xt = T(x, grad=True)
    Ds, As, S, rec = m(xt)
    o = O.space_cluster_forward(x, cen, w, b, 32.0, dtype=np.float64)
    assert rel(N(Ds), o["D"]) < 1e-5
    np.testing.assert_allclose(N(As), o["A"], rtol=3e-3, atol=1e-6)
    m.fused_cluster_loss().backward()
    gD, gA = O.frobenius_loss_grads(o["D"], o["A"], 1.0, np.float64)
    gx, gc, gw, gb = O.space_cluster_backward(x, cen, w, b, 32.0, gD=gD, gA=gA, dtype=np.float64)
    assert rel(N(xt.grad), gx) < 3e-4
    assert rel(N(m.cluster_center.grad), gc) < 3e-4
    assert rel(N(m.norm.weight.grad), gw) < 3e-4
    assert rel(N(m.norm.bias.grad), gb) < 3e-4


def test_c_above_4096_is_rejected():
    m = V.EuclidDistance_Assign_Module(4097, 32).to(dev())
    with pytest.raises(RuntimeError):
        m(torch.randn(1, 1, 1, 8, 4097, device=dev()))


# ---------------------------------------------------------------------------------------------------------------------
# full size: N = 65536 tokens, K = 1024, against float64 torch autograd of the reference op chain on the same GPU
# ---------------------------------------------------------------------------------------------------------------------
def _cdist_mm(a, b):
    d2 = (a * a).sum(-1, keepdim=True) + (b * b).sum(-1).unsqueeze(-2) - 2.0 * (a @ b.transpose(-1, -2))
    return d2.clamp_min(0).sqrt()


@pytest.mark.parametrize("C", [190, 2048])
def test_any_feature_dim_at_full_size(C):
    Ntok, K, alpha = 65536, 1024, 16.0
    torch.manual_seed(C)
    m = V.EuclidDistance_Assign_Module(C, K, soft_assign_alpha=alpha).to(dev())
    with torch.no_grad():
        m.norm.weight.copy_(1 + 0.2 * torch.randn(C, device=dev()))
        m.norm.bias.copy_(0.1 * torch.randn(C, device=dev()))
    x = torch.randn(1, 1, 1, Ntok, C, device=dev())

    def step():
        for p in m.parameters():
            p.grad = None
        xt = x.detach().requires_grad_(True)
        D, A, S, R, Fe, lab = m(xt)
        closs = m.fused_cluster_loss()
        (closs + V.e4_norm(R, xt.detach())).backward()
        return dict(D=D.detach().view(Ntok, K), A=A.detach().view(Ntok, K), R=R.detach().view(Ntok, C),
                    F=Fe.detach().view(Ntok, C), closs=closs.detach(), label=lab.view(Ntok), gx=xt.grad.view(Ntok, C),
                    gc=m.cluster_center.grad.clone(), gw=m.norm.weight.grad.clone(), gb=m.norm.bias.grad.clone())

    got = step()
    again = step()
    for k in got:
        assert torch.equal(got[k], again[k]), k
    del again
    # float64 reference: the whole graph (every parameter gradient), the per-token outputs on a 4096-row sample
    x64 = x.detach().double().view(Ntok, C).requires_grad_(True)
    c64, w64, b64 = [p.detach().double().requires_grad_(True) for p in (m.cluster_center, m.norm.weight, m.norm.bias)]
    z = F.layer_norm(x64, (C,), w64, b64, m.norm.eps)
    D = _cdist_mm(z, c64)
    A = torch.exp(-alpha * (D - D.min(-1, keepdim=True).values))
    A = A / A.sum(-1, keepdim=True)
    R = A @ c64
    closs = torch.norm(D * A)
    (closs + torch.norm((R - x64.detach()) ** 2)).backward()
    rows = torch.randperm(Ntok, generator=torch.Generator().manual_seed(C))[:4096].to(dev())

    def relmax(a, b):
        return float((a.double() - b).abs().max() / b.abs().max())

    errs = {"D": relmax(got["D"][rows], D[rows]), "F": relmax(got["F"][rows], z[rows]),
            "x_rec": relmax(got["R"][rows], R[rows]),
            "loss": abs(float(got["closs"]) - float(closs)) / float(closs),
            "gx": relmax(got["gx"][rows], x64.grad[rows]), "gc": relmax(got["gc"], c64.grad),
            "gw": relmax(got["gw"], w64.grad), "gb": relmax(got["gb"], b64.grad)}
    a_ratio = float(((got["A"][rows].double() - A[rows]).abs() / (1e-6 + 2e-3 * A[rows].abs())).max())
    gxr = got["gx"][rows].double()
    row_err = float(((gxr - x64.grad[rows]).abs().max(-1).values / x64.grad[rows].abs().max(-1).values.clamp_min(1e-30)).max())
    print(f"\nC={C}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()) + f", A/allowance {a_ratio:.2f}, gx_row {row_err:.2e}")
    assert_labels_match(N(got["label"][rows]), N(D[rows].detach()))
    tols = {"D": 1e-5, "F": 1e-5, "x_rec": 1e-4, "loss": 1e-5, "gx": 2e-4, "gc": 2e-4, "gw": 2e-4, "gb": 2e-4}
    for k, v in errs.items():
        assert v < tols[k], (k, v)
    assert a_ratio <= 1.0 and row_err < 2e-3
    del D, A, R, z, x64, c64, got
    gc.collect()
    torch.cuda.empty_cache()
