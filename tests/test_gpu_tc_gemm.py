"""TMA-fed tcgen05 GEMM (csrc/tc_gemm.cu): three-term bf16 split, six products -> fp32-faithful.
Checked against float64 numpy on shapes of the path: distance GEMM (N tokens x K centroids over C),
x_rec GEMM (MN-major B), memory score (m = 2000, d = 768) and read; ragged M / N / Kd tails."""
import numpy as np
import pytest
import torch

from videoad_b200 import _lib
from gpu_util import T, N as to_np, dev

pytestmark = pytest.mark.gpu


def run(A, B, b_mn):
    M, Kd = A.shape
    Nn = B.shape[1] if b_mn else B.shape[0]
    l = _lib.lib()
    # guard rows before and after the output: a tile epilogue that ignores the ragged edge would overwrite them
    big = torch.full((M + 16, Nn), float("nan"), device=dev(), dtype=torch.float32)
    out = big[8:8 + M]
    ws = torch.empty(l.vadc_debug_tc_gemm_workspace_bytes(M, Nn, Kd), device=dev(), dtype=torch.uint8)
    At, Bt = T(A), T(B)
    _lib.check(l.vadc_debug_tc_gemm(_lib.ptr(At), _lib.ptr(Bt), M, Nn, Kd, int(b_mn), _lib.ptr(out), _lib.ptr(ws),
                                    ws.numel(), _lib.stream()), "vadc_debug_tc_gemm")
    torch.cuda.synchronize()
    assert bool(torch.isnan(big[:8]).all()) and bool(torch.isnan(big[8 + M:]).all()), "write outside the output rows"
    return to_np(out)


@pytest.mark.parametrize("M,Nn,Kd", [(128, 128, 64), (300, 32, 192), (1000, 256, 768), (515, 1024, 192),
                                     (77, 16, 768), (129, 136, 200), (4096, 64, 768),   # fewer tiles than SMs: grid < SMs
                                     (2048, 2000, 768),        # 256 tiles: CTAs walk several tiles each
                                     (3001, 1096, 200),        # more tiles than SMs, ragged M / N / Kd
                                     (20000, 136, 64)])        # more tiles than SMs, one k-block per tile, 157 x 2 tiles
@pytest.mark.parametrize("b_mn", [0, 1])
def test_tc_gemm_vs_float64(M, Nn, Kd, b_mn):
    rng = np.random.default_rng(M + Nn + Kd + b_mn)
    A = rng.standard_normal((M, Kd)).astype(np.float32)
    B = rng.standard_normal((Nn, Kd)).astype(np.float32)
    got = run(A, np.ascontiguousarray(B.T) if b_mn else B, b_mn)
    ref = A.astype(np.float64) @ B.astype(np.float64).T
    err = np.abs(got - ref).max() / np.abs(ref).max()
    # fp32 TMEM accumulation over 6 Kd products (measured 5.7e-6 at Kd = 768; an fp32 SGEMM is ~2e-6)
    assert err < 1e-5, err


def test_tc_gemm_wide_dynamic_range():
    """the bf16 terms keep fp32's exponent range: scaling an operand by 2^±60 scales the result exactly"""
    rng = np.random.default_rng(3)
    A = rng.standard_normal((256, 192)).astype(np.float32)
    B = rng.standard_normal((64, 192)).astype(np.float32)
    base = run(A, B, 0)
    for s in (2.0 ** 60, 2.0 ** -60):
        got = run((A * np.float32(s)).astype(np.float32), B, 0)
        assert np.array_equal(got, (base * np.float32(s)).astype(np.float32))
