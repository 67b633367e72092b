"""The workloads bench.py times, checked at the sizes it times them (DESIGN §4): the space head (M = 512 frames × P = 1024,
C = 192, K = 128), the encoder tail ([64, 96, 8, 64, 64] → 524 288 tokens), the reference-native cluster head (K = 1024,
N = 65 536, forward and backward) and the decoder entry on the cfg2 token grid ([64, 8, 32, 32, 192]).

At these sizes the kernels take paths the oracle-sized tests never reach: LayerNorm-backward blocks that walk many tiles,
the persistent tcgen05 GEMM behind the encoder tail's forward and g_A, split-K slots 20–100× longer. Every case runs the
module on the GPU and compares every output and every gradient with the ORIGINAL module's op chain evaluated by torch
autograd in float64 on the same GPU (written out here, independently of the kernels' GEMM formulations); runs the
backward a second time on the same inputs, which must be bit-identical (split-K partials are summed in a fixed order);
asserts from the device's SM count that the shape reaches the multi-tile / persistent paths; and checks under
torch.profiler that the kernels it is written for were launched, so a change of dispatch cannot quietly turn it into a
small-size test. Run with ``-s`` to see the measured errors."""
import gc

import pytest
import torch
import torch.nn.functional as F

import videoad_b200 as V
from gpu_util import N, dev, assert_labels_match, assert_selfdist_close
from test_gpu_decoder_entry import _reference_chain

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _release_device_memory():
    """the float64 evaluations hold several GB: give them back before the next case"""
    yield
    gc.collect()
    torch.cuda.empty_cache()


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _relmax(a, b):
    """max |a - b| / max |b|, in float64 on the device"""
    return float((a.detach().double() - b).abs().max() / b.abs().max().clamp_min(1e-300))


def _row_relmax(a, b):
    """the largest over rows (last axis) of max |a - b| / max |b| within the row: an error local to a few rows hides
    under the global maximum"""
    a2, b2 = a.detach().reshape(-1, a.shape[-1]).double(), b.reshape(-1, b.shape[-1])
    return float(((a2 - b2).abs().max(-1).values / b2.abs().max(-1).values.clamp_min(1e-30)).max())


def _allclose_ratio(a, b, rtol, atol):
    """max of |a - b| / (atol + rtol |b|): at most 1 is numpy.testing.assert_allclose(a, b, rtol, atol)"""
    return float(((a.detach().double() - b).abs() / (atol + rtol * b.abs())).max())


def _cuda_kernels(fn):
    """names of the CUDA kernels that ``fn()`` launched"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if e.device_type.name == "CUDA"}


def _launched(names, *parts):
    return any(all(p in n for p in parts) for n in names)


def _kblocks_per_split_slot(tiles, contraction):
    """k-blocks (64 long) that each slot of a split-K GEMM contracts: the slots are chosen for about two work items per
    SM (bwd_tc_splits in csrc/cluster.cu, timedebd_splits in csrc/decoder_entry.cu), so their length depends on the
    device. At the oracle-sized tests it is 1-5."""
    nkb = (contraction + 63) // 64
    slots = min(max(1, (2 * _sms() + tiles - 1) // tiles), nkb)
    return (nkb + slots - 1) // slots


def _report(case, errs):
    print(f"\n{case}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))


def _check(errs, tols):
    for name, e in errs.items():
        assert e < tols[name], (name, e, tols[name], errs)


def _cdist_mm(a, b):
    """torch.cdist(a, b) as ATen evaluates it for more than 25 rows: sqrt(clamp_min(|a|² + |b|² − 2 a·bᵀ, 0))"""
    d2 = (a * a).sum(-1, keepdim=True) + (b * b).sum(-1).unsqueeze(-2) - 2.0 * (a @ b.transpose(-1, -2))
    return d2.clamp_min(0).sqrt()


def _neg_soft_assign(d, alpha):
    """NegSoftAssign over the last axis: exp(−α (d − min d)) / sum"""
    e = torch.exp(-alpha * (d - d.min(-1, keepdim=True).values))
    return e / e.sum(-1, keepdim=True)


def _leaf64(*ts):
    return [t.detach().double().requires_grad_(True) for t in ts]


# ---------------------------------------------------------------------------------------------------------------------
# space head (C3): bench lines space_fwd_bwd_M512_P1024_C192_K128 and space_fwd_M64_P1024_C192_K128
# ---------------------------------------------------------------------------------------------------------------------
def _space_module(C, K, side, seed):
    torch.manual_seed(seed)
    m = V.Space_EuclidDistance_Assign_Module(C, K, space_size=side).to(dev())
    with torch.no_grad():
        m.cluster_center.copy_(torch.rand(C, K, side * side, device=dev()))
        m.norm.weight.copy_(1 + 0.2 * torch.randn(C, device=dev()))
        m.norm.bias.copy_(0.1 * torch.randn(C, device=dev()))
    return m


def _space_fp64(x, m, backward):
    """Space_EuclidDistance_Assign_Module.forward (model/cluster.py:127-149) in float64: LayerNorm →
    'B D H W C -> C (B D) (H W)' → cdist against centers [C, K, P] → softmin over K → 'C (B D) CN -> B D C CN';
    S = cdist(centers, centers); objective torch.norm(Ds * As) (backbone.py:94)"""
    x64, c64, w64, b64 = _leaf64(x, m.cluster_center, m.norm.weight, m.norm.bias)
    B, Dd, H, W, C = x.shape
    K = c64.shape[1]
    z = F.layer_norm(x64, (C,), w64, b64, m.norm.eps)
    zt = z.reshape(B * Dd, H * W, C).permute(2, 0, 1)
    Ds = _cdist_mm(zt, c64).reshape(C, B, Dd, K).permute(1, 2, 0, 3)
    As = _neg_soft_assign(Ds, m.assign_func.alpha)
    with torch.no_grad():
        S = _cdist_mm(c64, c64)
    loss = torch.norm(Ds * As)
    out = dict(Ds=Ds.detach(), As=As.detach(), S=S, loss=loss.detach())
    if backward:
        loss.backward()
        out.update(gx=x64.grad, gc=c64.grad, gw=w64.grad, gb=b64.grad)
    return out


def _space_step(m, x, fused):
    for p in m.parameters():
        p.grad = None
    xt = x.detach().requires_grad_(True)
    Ds, As, S, rec = m(xt)
    loss = m.fused_cluster_loss() if fused else torch.norm(Ds * As)   # torch.norm: gD and gA arrive as tensors
    loss.backward()
    return dict(Ds=Ds.detach(), As=As.detach(), S=S.detach(), loss=loss.detach(), gx=xt.grad,
                gc=m.cluster_center.grad, gw=m.norm.weight.grad, gb=m.norm.bias.grad)


def _space_forward_errors(got, ref):
    errs = {"Ds": _relmax(got["Ds"], ref["Ds"]),
            "As/allowance": _allclose_ratio(got["As"], ref["As"], 3e-3, 1e-6),
            "loss": abs(float(got["loss"]) - float(ref["loss"])) / float(ref["loss"])}
    assert_selfdist_close(N(got["S"]), N(ref["S"]))
    return errs


SPACE_FWD_TOLS = {"Ds": 1e-5, "As/allowance": 1.0, "loss": 1e-5}


@pytest.mark.parametrize("B,side,fused", [
    (64, 32, True),     # the bench line: M = 512 frames x P = 1024, fused loss
    (64, 32, False),    # the same with the drop-in spelling torch.norm(Ds * As)
    (61, 32, True),     # ragged at scale: M = 488, blocks walk 13 or 14 tiles
    (64, 28, False),    # P = 784: tiles that straddle two frames, inside multi-tile blocks
], ids=["M512_P1024_fused", "M512_P1024_explicit", "M488_P1024_fused", "M512_P784_explicit"])
def test_space_head_at_bench_size(B, side, fused):
    """Ds 1e-5, As rtol 3e-3 / atol 1e-6, S as assert_selfdist_close, loss 1e-5 relative; gx, gcenters, gγ, gβ 3e-4 of the
    largest entry (test_space_vs_oracle's tolerances), every token row of gx within 3e-3 of that row's largest entry"""
    C, K, Dd = 192, 128, 8
    P, M = side * side, B * Dd
    tiles = (M * P + 63) // 64
    assert tiles > 4 * _sms(), ("the LayerNorm backward's blocks must walk several 64-token tiles", tiles, _sms())
    m = _space_module(C, K, side, seed=B * 100 + side + fused)
    x = torch.randn(B, Dd, side, side, C, device=dev()) * 1.3
    got = _space_step(m, x, fused)
    ref = _space_fp64(x, m, backward=True)
    errs = _space_forward_errors(got, ref)
    errs.update(gx=_relmax(got["gx"], ref["gx"]), gx_row=_row_relmax(got["gx"], ref["gx"]),
                gcenters=_relmax(got["gc"], ref["gc"]), g_ln_w=_relmax(got["gw"], ref["gw"]),
                g_ln_b=_relmax(got["gb"], ref["gb"]))
    del ref
    _report(f"space B={B} side={side} {'fused' if fused else 'explicit'}", errs)
    _check(errs, dict(SPACE_FWD_TOLS, gx=3e-4, gx_row=3e-3, gcenters=3e-4, g_ln_w=3e-4, g_ln_b=3e-4))
    again = {}
    names = _cuda_kernels(lambda: again.update(_space_step(m, x, fused)))
    assert _launched(names, "ln_bwd_transposed_tile_kernel"), sorted(names)
    for k in got:
        assert torch.equal(got[k], again[k]), k


def test_space_head_forward_M64():
    """the bench line space_fwd_M64_P1024_C192_K128 (x [8, 8, 32, 32, 192], forward only), same bars as above"""
    C, K, side = 192, 128, 32
    m = _space_module(C, K, side, seed=64)
    x = torch.randn(8, 8, side, side, C, device=dev()) * 1.3
    with torch.no_grad():
        Ds, As, S, _ = m(x)
        got = dict(Ds=Ds, As=As, S=S, loss=m.fused_cluster_loss())
        ref = _space_fp64(x, m, backward=False)
        errs = _space_forward_errors(got, ref)
        _report("space forward M=64", errs)
        _check(errs, SPACE_FWD_TOLS)
        Ds2, As2, S2, _ = m(x)
    assert torch.equal(Ds, Ds2) and torch.equal(As, As2) and torch.equal(S, S2)


# ---------------------------------------------------------------------------------------------------------------------
# encoder tail: bench line encoder_tail_fwd_bwd_524288tokens
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,W2", [(64, 64), (63, 62)], ids=["bench_524288tokens", "ragged_31columns"])
def test_encoder_tail_at_bench_size(B, W2):
    """Conv3d(96, 192, (1,2,2), stride (1,2,2)) + exact GELU → channel-last tokens against F.conv3d + GELU in float64 and
    the permute to channel-last: out 1e-5 of the largest entry (every token row within 1e-4 of its own), gx, g_weight,
    g_bias 2e-4 (test_downsample_gelu_forward_backward's tolerances). W2 = 62 gives 31 output columns, so the last
    32-token block of every row is short."""
    Cin, Cout, D, H2 = 96, 192, 8, 64
    NT = B * D * (H2 // 2) * (W2 // 2)
    tiles_fwd = ((Cout + 127) // 128) * ((NT + 127) // 128)        # out: rows = output channels, columns = tokens
    tiles_ga = ((4 * Cin + 127) // 128) * ((NT + 127) // 128)      # g_A: rows = patch entries, columns = tokens
    assert min(tiles_fwd, tiles_ga) > _sms(), ("the forward and g_A GEMMs must run persistent", tiles_fwd, tiles_ga)
    assert NT > 1024 * 256, "the bias gradient's column sum must run at its cap of 1024 row chunks"
    torch.manual_seed(B * 1000 + W2)
    seq = torch.nn.Sequential(torch.nn.Conv3d(Cin, Cout, (1, 2, 2), stride=(1, 2, 2)), torch.nn.GELU()).to(dev())
    x = torch.randn(B, Cin, D, H2, W2, device=dev()) * 1.3
    gy = torch.randn(B, D, H2 // 2, W2 // 2, Cout, device=dev())

    def step():
        for p in seq.parameters():
            p.grad = None
        xt = x.detach().requires_grad_(True)
        y = V.downsample_gelu_tokens(xt, seq[0], seq[1])
        y.backward(gy)
        return dict(out=y.detach(), gx=xt.grad, g_weight=seq[0].weight.grad, g_bias=seq[0].bias.grad)

    got = step()
    w64, b64 = _leaf64(seq[0].weight, seq[0].bias)
    x64, = _leaf64(x)
    y64 = F.gelu(F.conv3d(x64, w64, b64, stride=(1, 2, 2))).permute(0, 2, 3, 4, 1)     # 'n c d h w -> n d h w c'
    y64.backward(gy.double())
    ref = dict(out=y64.detach(), gx=x64.grad, g_weight=w64.grad, g_bias=b64.grad)
    del y64
    errs = {k: _relmax(got[k], ref[k]) for k in ref}
    errs["out_row"] = _row_relmax(got["out"], ref["out"])
    del ref, x64, w64, b64
    _report(f"encoder tail x [{B}, 96, 8, 64, {W2}]", errs)
    _check(errs, dict(out=1e-5, out_row=1e-4, gx=2e-4, g_weight=2e-4, g_bias=2e-4))
    # inference keeps no pre-activation; the g_W contraction cannot account for a persistent launch here
    inf, again = {}, {}
    with torch.no_grad():
        names = _cuda_kernels(lambda: inf.update(out=V.downsample_gelu_tokens(x, seq[0], seq[1])))
    assert _launched(names, "tc_gemm_persist_kernel", "TcBiasGeluTEpi"), sorted(names)
    assert torch.equal(inf["out"], got["out"])
    names = _cuda_kernels(lambda: again.update(step()))
    assert _launched(names, "tc_gemm_persist_kernel", "TcStoreTEpi"), sorted(names)      # g_A
    for k in got:
        assert torch.equal(got[k], again[k]), k


# ---------------------------------------------------------------------------------------------------------------------
# reference-native cluster head (C = 192, K = 1024): bench lines cluster_fwd_bwd_C192_K1024_N65536_{fused,explicit}_loss
# ---------------------------------------------------------------------------------------------------------------------
def _cluster_fp64(x, m):
    """EuclidDistance_Assign_Module.forward (model/cluster.py:81-99) in float64: LayerNorm → cdist → softmin →
    x_rec = A @ centers; objective torch.norm(D * A) + torch.norm(MSELoss(reduction='none')(x_rec, x.detach()))
    (bench.py native_step; main_predict.py:273-275)"""
    x64, c64, w64, b64 = _leaf64(x, m.cluster_center, m.norm.weight, m.norm.bias)
    z = F.layer_norm(x64, (x64.shape[-1],), w64, b64, m.norm.eps)
    D = _cdist_mm(z, c64)
    A = _neg_soft_assign(D, m.assign_func.alpha)
    R = A @ c64
    with torch.no_grad():
        S = _cdist_mm(c64, c64)
    closs = torch.norm(D * A)
    loss = closs + torch.norm((R - x64.detach()) ** 2)
    loss.backward()
    return dict(D=D.detach(), A=A.detach(), R=R.detach(), F=z.detach(), S=S, closs=closs.detach(),
                gx=x64.grad, gc=c64.grad, gw=w64.grad, gb=b64.grad)


@pytest.mark.parametrize("Ntok", [65536, 65536 - 37])
@pytest.mark.parametrize("fused", [True, False], ids=["fused_loss", "explicit_loss"])
def test_cluster_k1024_at_bench_size(Ntok, fused):
    """forward in full — D, feature 1e-5, A rtol 2e-3 / atol 1e-6, x_rec 1e-4, S as assert_selfdist_close, the cluster
    loss 1e-5 relative, labels bit-exact up to float64-adjudicated ties — and gx, gcenters, gγ, gβ 2e-4 of the largest
    entry, every row of gx within 2e-3 of its own (test_forward_vs_oracle / test_full_size_training_graph_backward)"""
    C, K, alpha = 192, 1024, 16.0
    per_slot = _kblocks_per_split_slot(((K + 127) // 128) * ((C + 127) // 128), Ntok)
    assert per_slot > 16, ("the centroid gradient's split-K slots must be long", per_slot)
    torch.manual_seed(Ntok + fused)
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
        closs = m.fused_cluster_loss() if fused else torch.norm(D * A)
        (closs + V.e4_norm(R, xt.detach())).backward()
        return dict(D=D.detach(), A=A.detach(), R=R.detach(), F=Fe.detach(), S=S.detach(), closs=closs.detach(),
                    label=lab, gx=xt.grad, gc=m.cluster_center.grad, gw=m.norm.weight.grad, gb=m.norm.bias.grad)

    got = step()
    ref = _cluster_fp64(x, m)
    errs = {"D": _relmax(got["D"].view(Ntok, K), ref["D"].view(Ntok, K)),
            "A/allowance": _allclose_ratio(got["A"].view(Ntok, K), ref["A"].view(Ntok, K), 2e-3, 1e-6),
            "x_rec": _relmax(got["R"], ref["R"]), "feature": _relmax(got["F"].view(Ntok, C), ref["F"].view(Ntok, C)),
            "loss": abs(float(got["closs"]) - float(ref["closs"])) / float(ref["closs"]),
            "gx": _relmax(got["gx"], ref["gx"]), "gx_row": _row_relmax(got["gx"], ref["gx"]),
            "gcenters": _relmax(got["gc"], ref["gc"]), "g_ln_w": _relmax(got["gw"], ref["gw"]),
            "g_ln_b": _relmax(got["gb"], ref["gb"])}
    assert float((got["A"].view(Ntok, K).double().sum(-1) - 1).abs().max()) < 1e-5
    assert_selfdist_close(N(got["S"]), N(ref["S"]))
    assert_labels_match(N(got["label"]), N(ref["D"].view(Ntok, K)))
    del ref
    _report(f"cluster K=1024 N={Ntok} {'fused' if fused else 'explicit'}", errs)
    _check(errs, {"D": 1e-5, "A/allowance": 1.0, "x_rec": 1e-4, "feature": 1e-5, "loss": 1e-5, "gx": 2e-4,
                  "gx_row": 2e-3, "gcenters": 2e-4, "g_ln_w": 2e-4, "g_ln_b": 2e-4})
    again = {}
    names = _cuda_kernels(lambda: again.update(step()))
    assert _launched(names, "tc_gemm_persist_kernel", "TcPartialEpi"), sorted(names)     # split-K on the persistent GEMM
    for k in got:
        assert torch.equal(got[k], again[k]), k


# ---------------------------------------------------------------------------------------------------------------------
# decoder entry (LayerNorm + ConvTranspose3d / predict-mode Conv3d) on the cfg2 token grid
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("predict", [False, True], ids=["conv_transpose", "predict_conv"])
def test_decoder_entry_at_cfg2_grid(predict):
    """norm_timedebd on x [64, 8, 32, 32, 192] against the reference chain (test_gpu_decoder_entry._reference_chain) in
    float64: out 1e-5, gx, gγ, gβ, g_weight, g_bias 2e-4 of the largest entry (that file's tolerances)"""
    B, D, H, W, C = 64, 8, 32, 32, 192
    rows = B * D * H * W // (2 if predict else 1)                  # the weight gradient contracts over these rows
    per_slot = _kblocks_per_split_slot(((C + 127) // 128) * ((2 * C + 127) // 128), rows)
    assert per_slot > 16, ("the weight gradient's split-K slots must be long", per_slot)
    torch.manual_seed(17 + predict)
    conv = torch.nn.Conv3d if predict else torch.nn.ConvTranspose3d
    norm = torch.nn.LayerNorm(C).to(dev())
    td = conv(C, C, kernel_size=(2, 1, 1), stride=(2, 1, 1)).to(dev())
    with torch.no_grad():
        norm.weight.copy_(1 + 0.2 * torch.randn(C, device=dev())); norm.bias.copy_(0.1 * torch.randn(C, device=dev()))
    x = torch.randn(B, D, H, W, C, device=dev()) * 1.4 + 0.3
    gy = torch.randn(B, D // 2 if predict else 2 * D, H, W, C, device=dev())

    def step():
        for p in list(norm.parameters()) + list(td.parameters()):
            p.grad = None
        xt = x.detach().requires_grad_(True)
        y = V.norm_timedebd(xt, norm, td)
        y.backward(gy)
        return dict(out=y.detach(), gx=xt.grad, g_ln_w=norm.weight.grad, g_ln_b=norm.bias.grad,
                    g_weight=td.weight.grad, g_bias=td.bias.grad)

    got = step()
    n64 = torch.nn.LayerNorm(C).to(dev()).double()
    t64 = conv(C, C, (2, 1, 1), stride=(2, 1, 1)).to(dev()).double()
    n64.load_state_dict({k: v.double() for k, v in norm.state_dict().items()})
    t64.load_state_dict({k: v.double() for k, v in td.state_dict().items()})
    x64, = _leaf64(x)
    y64 = _reference_chain(x64, n64, t64)
    y64.backward(gy.double())
    ref = dict(out=y64.detach(), gx=x64.grad, g_ln_w=n64.weight.grad, g_ln_b=n64.bias.grad, g_weight=t64.weight.grad,
               g_bias=t64.bias.grad)
    errs = {k: _relmax(got[k], ref[k]) for k in ref}
    del ref, y64, x64, n64, t64
    _report(f"decoder entry {'predict Conv3d' if predict else 'ConvTranspose3d'}", errs)
    _check(errs, dict(out=1e-5, gx=2e-4, g_ln_w=2e-4, g_ln_b=2e-4, g_weight=2e-4, g_bias=2e-4))
    again = {}
    names = _cuda_kernels(lambda: again.update(step()))
    assert _launched(names, "tc_gemm_persist_kernel", "TcPartialEpi"), sorted(names)     # split-K on the persistent GEMM
    for k in got:
        assert torch.equal(got[k], again[k]), k
