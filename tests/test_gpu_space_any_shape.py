"""Space_EuclidDistance_Assign_Module on the tensor cores at any cluster_num and any space_size: K not a multiple of 64
and P = space_size² not a multiple of 8, forward, backward and the centroid self-distance, in both operand-term modes
(fp16 x2 and VADC_SPACE_TERMS=3's bf16 x3).  The operand terms are then written at padded pitches (Pp = P rounded up to
8, Kp = K rounded up to 64) with zeros in the padding, and the epilogues stop at P and K.

Every case clears the tensor-core path's work threshold (M·P·K·C >= 2^28, asserted), is checked under torch.profiler
to run its three contractions on tc_gemm_persist_kernel and no SIMT GEMM, and is compared with the reference op chain
evaluated by torch autograd in float64 on the same GPU.  Run with ``-s`` to see the measured errors."""
import contextlib
import gc
import os

import pytest
import torch
import torch.nn.functional as F

import videoad_b200 as V
from videoad_b200 import _lib
from gpu_util import N, dev, assert_selfdist_close

pytestmark = pytest.mark.gpu

WORK_THRESHOLD = 1 << 28          # space_tc_ok in csrc/space_cluster.cu: M·P·K·C below this runs the SIMT path


@pytest.fixture(autouse=True)
def _release_device_memory():
    yield
    gc.collect()
    torch.cuda.empty_cache()


@contextlib.contextmanager
def _space_terms(terms):
    """operand terms of the space head's contractions: 2 (fp16 x2, the default) or 3 (bf16 x3)"""
    if terms == 3:
        os.environ["VADC_SPACE_TERMS"] = "3"
        _lib.lib().vadc_refresh_env()
    try:
        yield
    finally:
        os.environ.pop("VADC_SPACE_TERMS", None)
        _lib.lib().vadc_refresh_env()


def _padded_k(K):
    return K + (-K) % 4                                   # the module pads cluster_num to a multiple of 4 on the host


def _assert_clears_threshold(M, P, C, K):
    assert M * P * _padded_k(K) * C >= WORK_THRESHOLD, ("the case must take the tensor-core path", M, P, C, K)


def _relmax(a, b):
    return float((a.detach().double() - b).abs().max() / b.abs().max().clamp_min(1e-300))


def _row_relmax(a, b):
    a2, b2 = a.detach().reshape(-1, a.shape[-1]).double(), b.reshape(-1, b.shape[-1])
    return float(((a2 - b2).abs().max(-1).values / b2.abs().max(-1).values.clamp_min(1e-30)).max())


def _allclose_ratio(a, b, rtol, atol):
    return float(((a.detach().double() - b).abs() / (atol + rtol * b.abs())).max())


def _cdist_mm(a, b):
    d2 = (a * a).sum(-1, keepdim=True) + (b * b).sum(-1).unsqueeze(-2) - 2.0 * (a @ b.transpose(-1, -2))
    return d2.clamp_min(0).sqrt()


def _cuda_kernels(fn, reps=2):
    """kernel names of ``fn()``: one call before the capture, ``reps`` inside it"""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if e.device_type.name == "CUDA"}


def _space_module(C, K, side, seed):
    torch.manual_seed(seed)
    m = V.Space_EuclidDistance_Assign_Module(C, K, space_size=side).to(dev())
    with torch.no_grad():
        m.cluster_center.copy_(torch.rand(C, K, side * side, device=dev()))
        m.norm.weight.copy_(1 + 0.2 * torch.randn(C, device=dev()))
        m.norm.bias.copy_(0.1 * torch.randn(C, device=dev()))
    return m


def _reference(x, m, wS=None):
    """model/cluster.py:127-149 in float64: LayerNorm → 'B D H W C -> C (B D) (H W)' → cdist against centers [C, K, P] →
    softmin over K → 'C (B D) CN -> B D C CN'; S = cdist(centers, centers); objective torch.norm(Ds * As), plus
    sum(S * wS) when wS is given (a gradient through the self-distance)"""
    x64, c64, w64, b64 = [t.detach().double().requires_grad_(True) for t in
                          (x, m.cluster_center, m.norm.weight, m.norm.bias)]
    B, Dd, H, W, C = x.shape
    K = c64.shape[1]
    z = F.layer_norm(x64, (C,), w64, b64, m.norm.eps)
    zt = z.reshape(B * Dd, H * W, C).permute(2, 0, 1)
    Ds = _cdist_mm(zt, c64).reshape(C, B, Dd, K).permute(1, 2, 0, 3)
    e = torch.exp(-m.assign_func.alpha * (Ds - Ds.min(-1, keepdim=True).values))
    As = e / e.sum(-1, keepdim=True)
    S = torch.cdist(c64, c64, compute_mode="donot_use_mm_for_euclid_dist")
    loss = torch.norm(Ds * As)
    (loss if wS is None else loss + (S * wS.double()).sum()).backward()
    return dict(Ds=Ds.detach(), As=As.detach(), S=S.detach(), loss=loss.detach(), gx=x64.grad, gc=c64.grad,
                gw=w64.grad, gb=b64.grad)


def _step(m, x, loss_kind, wS=None):
    """forward + backward; loss_kind: 'fused' (fused_cluster_loss) or 'explicit' (torch.norm(Ds * As)); wS adds
    sum(cluster_dist * wS)"""
    for p in m.parameters():
        p.grad = None
    xt = x.detach().requires_grad_(True)
    Ds, As, S, rec = m(xt)
    loss = m.fused_cluster_loss() if loss_kind == "fused" else torch.norm(Ds * As)
    (loss if wS is None else loss + (S * wS).sum()).backward()
    return dict(Ds=Ds.detach(), As=As.detach(), S=S.detach(), loss=loss.detach(), gx=xt.grad,
                gc=m.cluster_center.grad, gw=m.norm.weight.grad, gb=m.norm.bias.grad)


def _check(got, ref, what):
    """Ds 1e-5, As rtol 3e-3 / atol 1e-6, loss 1e-5 relative, S as assert_selfdist_close; gx, gcenters, gγ, gβ 3e-4 of
    the largest entry and every token row of gx within 3e-3 of its own largest entry"""
    for k in ("Ds", "As", "S", "gx", "gc", "gw", "gb"):
        assert torch.isfinite(got[k]).all(), (what, k)
    errs = {"Ds": _relmax(got["Ds"], ref["Ds"]), "As/allowance": _allclose_ratio(got["As"], ref["As"], 3e-3, 1e-6),
            "loss": abs(float(got["loss"]) - float(ref["loss"])) / float(ref["loss"]),
            "gx": _relmax(got["gx"], ref["gx"]), "gx_row": _row_relmax(got["gx"], ref["gx"]),
            "gcenters": _relmax(got["gc"], ref["gc"]), "g_ln_w": _relmax(got["gw"], ref["gw"]),
            "g_ln_b": _relmax(got["gb"], ref["gb"])}
    print(f"\n{what}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    tols = {"Ds": 1e-5, "As/allowance": 1.0, "loss": 1e-5, "gx": 3e-4, "gx_row": 3e-3, "gcenters": 3e-4,
            "g_ln_w": 3e-4, "g_ln_b": 3e-4}
    for k, v in errs.items():
        assert v < tols[k], (what, k, v, errs)
    assert_selfdist_close(N(got["S"]), N(ref["S"]))


def _assert_tensor_core_kernels(names, P, C):
    vk = sorted({n.split("(")[0][-100:] for n in names if "vadc::" in n})
    for epi in ("TcBatchDistEpi", "TcSpaceGzEpi", "TcSpaceGcEpi"):
        assert any("tc_gemm_persist_kernel" in n and epi in n for n in names), (epi, vk)
    assert not any("sgemm_kernel" in n for n in names), vk
    if C > 256:
        assert any("ln_transpose_kernel" in n for n in names), vk          # the untiled LayerNorm kernels
    if C > 256 or P < 64:
        assert any("ln_bwd_transposed_kernel" in n for n in names), vk     # untiled backward, with rsum


# (B, D, side, C, K): M = B·D frames of P = side² positions, C channels, K = cluster_num
CASES = [
    (18, 8, 32, 64, 100),      # ragged K at P = 1024
    (18, 8, 32, 64, 130),      # Kp = 192
    (18, 8, 32, 64, 30),       # host-padded to 32, Kp = 64
    (18, 8, 32, 64, 32),       # the cluster head's cfg2 cluster_num
    (22, 8, 14, 64, 128),      # ragged P at K = 128: P = 196
    (5, 8, 30, 64, 128),       # P = 900 (a 240-pixel input)
    (52, 8, 9, 64, 128),       # P = 81
    (86, 8, 7, 64, 128),       # P = 49 < 64: the untiled LayerNorm backward with rsum
    (6, 8, 30, 64, 100),       # both ragged
    (7, 8, 14, 288, 100),      # C > 256: untiled LayerNorm kernels, bf16 x3 in both modes
    (15, 8, 30, 20, 130),      # few channels
    (64, 8, 32, 192, 100),     # the benchmarked size (M = 512, C = 192) with a ragged K
    (64, 8, 30, 192, 128),     # ... and with a ragged P
]
IDS = [f"M{b * d}_P{s * s}_C{c}_K{k}" for b, d, s, c, k in CASES]


@pytest.mark.parametrize("B,Dd,side,C,K", CASES, ids=IDS)
def test_space_head_any_shape(B, Dd, side, C, K):
    """both loss spellings in both term modes against float64; the backward run twice is bit-identical; the kernels"""
    M, P = B * Dd, side * side
    _assert_clears_threshold(M, P, C, K)
    m = _space_module(C, K, side, seed=M * 7 + P + C + K)
    x = torch.randn(B, Dd, side, side, C, device=dev()) * 1.3
    ref = _reference(x, m)
    for terms in (2, 3):
        with _space_terms(terms):
            for kind in ("fused", "explicit"):
                got = _step(m, x, kind)
                _check(got, ref, f"M={M} P={P} C={C} K={K} terms={terms} {kind}")
            again = _step(m, x, "explicit")
            for k in got:
                assert torch.equal(got[k], again[k]), (terms, k)
            del got, again
            _assert_tensor_core_kernels(_cuda_kernels(lambda: _step(m, x, "fused")), P, C)


@pytest.mark.parametrize("B,Dd,side,C,K", [(18, 8, 32, 64, 100), (6, 8, 30, 64, 100), (52, 8, 9, 64, 128)],
                         ids=["M144_P1024_K100", "M48_P900_K100", "M416_P81_K128"])
@pytest.mark.parametrize("terms", [2, 3])
def test_self_distance_gradient_any_shape(B, Dd, side, C, K, terms):
    """a loss on cluster_dist as well: its gradient reaches the centroids next to the head's own"""
    M, P = B * Dd, side * side
    _assert_clears_threshold(M, P, C, K)
    m = _space_module(C, K, side, seed=K + P)
    x = torch.randn(B, Dd, side, side, C, device=dev()) * 1.3
    wS = torch.rand(C, K, K, device=dev(), generator=torch.Generator(device=dev()).manual_seed(P))
    ref = _reference(x, m, wS)
    with _space_terms(terms):
        _check(_step(m, x, "fused", wS), ref, f"self-distance M={M} P={P} K={K} terms={terms}")


@pytest.mark.parametrize("B,Dd,side,C,K", [(6, 8, 30, 64, 100), (7, 8, 14, 288, 100)],
                         ids=["M48_P900_C64_K100", "M56_P196_C288_K100"])
def test_stale_memory_does_not_reach_the_results(B, Dd, side, C, K):
    """The saved state comes from torch.empty and the workspace is a grow-only cache: both are filled with NaN bytes
    before the forward, so a padding term that is assumed rather than written to be zero turns results into NaN."""
    M, P = B * Dd, side * side
    _assert_clears_threshold(M, P, C, K)
    Kh = _padded_k(K)
    m = _space_module(C, K, side, seed=3 * P + K)
    x = torch.randn(B, Dd, side, side, C, device=dev()) * 1.3
    ref = _reference(x, m)
    l = _lib.lib()
    saved = l.vadc_space_cluster_saved_bytes(M, P, C, Kh)
    ws = max(l.vadc_space_cluster_fwd_workspace_bytes(M, P, C, Kh), l.vadc_space_cluster_bwd_workspace_bytes(M, P, C, Kh))
    _lib.workspace(ws, dev())
    for buf in _lib._ws_cache.values():
        buf.fill_(255)                        # 0xFF bytes: NaN as fp32, bf16 and fp16
    # one NaN block for the saved state and the forward's other outputs, freed into a private pool of the caching
    # allocator in which it is the only free memory, so that the forward's allocations are carved from it
    pool = torch.cuda.MemPool()
    xt = x.detach().requires_grad_(True)
    with torch.cuda.use_mem_pool(pool):
        outputs = 4 * (2 * M * C * Kh + C * Kh * Kh + 2 * M * P + 64)
        block = torch.full((saved + outputs + (32 << 20),), 255, dtype=torch.uint8, device=dev())
        lo, hi = block.data_ptr(), block.data_ptr() + block.numel()
        del block
        Ds, As, S, _ = m(xt)
    zt_state = m.loss_sq.grad_fn.saved_tensors[6]
    assert zt_state.numel() == saved and lo <= zt_state.data_ptr() < hi, "the saved state must reuse the NaN block"
    del zt_state
    loss = m.fused_cluster_loss()
    loss.backward()
    got = dict(Ds=Ds.detach(), As=As.detach(), S=S.detach(), loss=loss.detach(), gx=xt.grad,
               gc=m.cluster_center.grad, gw=m.norm.weight.grad, gb=m.norm.bias.grad)
    _check(got, ref, f"stale memory M={M} P={P} C={C} K={K}")
