// decoder_entry.cu — SURVEY.md 8f-2: the immediate consumer of the cluster head's x_rec.
//
//   model/backbone.py:120-123        x = self.norm(x)                 LayerNorm(192) over the channel-last tokens
//   model/swin_decoder_predict.py:599-602  rearrange -> self.timedebd(x) -> rearrange
//       timedebd = ConvTranspose3d(192, 192, kernel (2,1,1), stride (2,1,1))   (non-predict decoder, :593-594):
//       out[b, co, 2d+j, h, w] = bias[co] + sum_ci z[b, ci, d, h, w] W[ci, co, j]
//
// In the reference that is a LayerNorm pass, a channel-last -> channel-first copy (cuDNN wants NCDHW), the transposed
// convolution, and a copy back.  On channel-last tokens it is one GEMM [N, C] x [C, 2C] whose epilogue scatters the two
// column halves to the output frames 2d and 2d+1 — x_rec is read once, the up-sampled tokens are written once,
// channel-last, nothing is transposed.  LayerNorm and the three-term bf16 split of its output are one row kernel, the
// contraction runs on the tcgen05 GEMM (fp32-faithful).  The backward is built from the same pieces:
//   gZ = gYm Wk^T,  gW = Z^T gYm (split over the tokens),  gbias = colsum(gY),  then the LayerNorm backward.
#include "common.cuh"
#include "rows.cuh"
#include "cluster.h"
#include "tc_gemm.cuh"
#include <algorithm>
#include <cuda_bf16.h>

namespace vadc {

// gY [2N, C] channel-last (frames 2f, 2f+1 of token frame f) -> the three bf16 terms of gYm [N, 2C]:
// gYm[n, j*C + c] = gY[((f*2 + j)*HW + hw), c],  n = f*HW + hw
__global__ void __launch_bounds__(256)
split3_frames_kernel(const float* __restrict__ gy, long long N, int C, long long HW, void* __restrict__ t0) {
  const long long total4 = N * 2 * (C / 4);
  const long long term = N * 2 * C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += (long long)gridDim.x * blockDim.x) {
    const long long row2 = i / (C / 4);                  // row of gY
    const int c4 = (int)(i - row2 * (C / 4));
    const long long fj = row2 / HW, hw = row2 - fj * HW;
    const long long f = fj >> 1;
    const int j = (int)(fj & 1);
    const float4 v = __ldg(reinterpret_cast<const float4*>(gy) + i);
    const float a[4] = {v.x, v.y, v.z, v.w};
    store_terms<3, 4>(t0, term, (f * HW + hw) * 2 * C + (long long)j * C + c4 * 4, a);
  }
}

__global__ void __launch_bounds__(256)
sum_partials_kernel(const float* __restrict__ q, int splits, long long n, float* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float s = 0.f;
  for (int sp = 0; sp < splits; ++sp) s += q[sp * n + i];       // fixed order: deterministic
  out[i] = s;
}

// column sums of a [R, C] matrix: one block per 32 columns, fixed-order tree (deterministic)
__global__ void __launch_bounds__(256)
colsum32_kernel(const float* __restrict__ a, long long R, int C, float* __restrict__ out) {
  __shared__ float red[8][32];
  const int c = blockIdx.x * 32 + (threadIdx.x & 31), w = threadIdx.x >> 5;
  float s = 0.f;
  if (c < C)
    for (long long r = w; r < R; r += 8) s += a[r * C + c];
  red[w][threadIdx.x & 31] = s;
  __syncthreads();
  if (w == 0 && c < C) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += red[i][threadIdx.x];
    out[c] = t;
  }
}

static int timedebd_splits(long long N) {
  long long s = (2ll * sm_count() + 5) / 6;               // [C, 2C] = 2 x 3 output tiles of 128 x 128 at C = 192
  const long long nkb = (N + 63) / 64;
  if (s > nkb) s = nkb;
  if (s < 1) s = 1;
  return (int)s;
}

}  // namespace vadc

using namespace vadc;

extern "C" size_t vadc_norm_timedebd_workspace_bytes(int64_t N, int C) {
  const size_t n = (size_t)(N > 0 ? N : 1);
  size_t b = 0;
  b += tc_terms_bytes(3, (long long)n, C);              // z terms
  b += tc_terms_bytes(3, 2 * C, C);                     // weight terms (either arrangement)
  b += tc_terms_bytes(3, (long long)n, 2 * C);          // gYm terms (backward)
  b += align_up(n * C * sizeof(float), 256);              // gZ (backward)
  b += align_up((size_t)timedebd_splits(N) * C * 2 * C * sizeof(float), 256);
  b += align_up((size_t)ln_bwd_blocks(N) * 2 * C * sizeof(float), 256);
  b += align_up(n * sizeof(float), 256) * 2;
  b += align_up(n * C * sizeof(float), 256);              // z in fp32 (predict-mode entry: gathered pairwise afterwards)
  return b + 256;
}

extern "C" int vadc_norm_timedebd_fwd(const float* x, const float* ln_w, const float* ln_b, const float* wt,
                                      const float* bias, int64_t N, int C, int64_t HW, float eps, float* out,
                                      float* mu, float* rstd, void* workspace, size_t workspace_bytes, void* stream) {
  VADC_REQUIRE(N >= 0 && C > 0 && HW > 0 && (C % 32) == 0 && C <= 1024, VADC_ERR_BAD_SHAPE);
  VADC_REQUIRE(N % HW == 0, VADC_ERR_BAD_SHAPE);
  if (N == 0) return VADC_OK;
  VADC_REQUIRE(x && ln_w && ln_b && wt && bias && out && mu && rstd && workspace, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(aligned16(x) && aligned16(out) && aligned16(wt), VADC_ERR_MISALIGNED);
  VADC_REQUIRE(workspace_bytes >= vadc_norm_timedebd_workspace_bytes(N, C), VADC_ERR_WORKSPACE);
  VADC_REQUIRE(tc_gemm_shape_ok(N, 2 * C, C, false), VADC_ERR_UNSUPPORTED);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Carver ws(workspace, workspace_bytes);
  void* zs = ws.take<uint8_t>(tc_terms_bytes(3, N, C));
  void* wsplit = ws.take<uint8_t>(tc_terms_bytes(3, 2 * C, C));
  int rc;
  if ((rc = launch_ln_rows(x, ln_w, ln_b, N, C, eps, nullptr, mu, rstd, nullptr, st, nullptr, zs))) return rc;
  if ((rc = tc_split<3>(wt, 2 * C, C, nullptr, wsplit, st))) return rc;
  return tc_gemm<3, false, false>({zs, wsplit, N, 2 * C, C}, TcTimeDebedEpi{out, bias, HW, C}, st);
}

extern "C" int vadc_norm_timedebd_bwd(const float* x, const float* mu, const float* rstd, const float* ln_w,
                                      const float* ln_b, const float* wk, const float* gout, int64_t N, int C,
                                      int64_t HW, float eps, float* gx, float* g_ln_w, float* g_ln_b, float* gwk,
                                      float* gbias, void* workspace, size_t workspace_bytes, void* stream) {
  VADC_REQUIRE(N >= 0 && C > 0 && HW > 0 && (C % 32) == 0 && C <= 1024, VADC_ERR_BAD_SHAPE);
  VADC_REQUIRE(N % HW == 0, VADC_ERR_BAD_SHAPE);
  VADC_REQUIRE(g_ln_w && g_ln_b && gwk && gbias && workspace, VADC_ERR_NULL_POINTER);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (N == 0) {
    VADC_CUDA(cudaMemsetAsync(gwk, 0, sizeof(float) * C * 2 * C, st));
    VADC_CUDA(cudaMemsetAsync(gbias, 0, sizeof(float) * C, st));
    VADC_CUDA(cudaMemsetAsync(g_ln_w, 0, sizeof(float) * C, st));
    VADC_CUDA(cudaMemsetAsync(g_ln_b, 0, sizeof(float) * C, st));
    return VADC_OK;
  }
  VADC_REQUIRE(x && mu && rstd && ln_w && ln_b && wk && gout && gx, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(aligned16(x) && aligned16(gout) && aligned16(wk) && aligned16(gx), VADC_ERR_MISALIGNED);
  VADC_REQUIRE(workspace_bytes >= vadc_norm_timedebd_workspace_bytes(N, C), VADC_ERR_WORKSPACE);
  Carver ws(workspace, workspace_bytes);
  void* zs = ws.take<uint8_t>(tc_terms_bytes(3, N, C));
  void* wsplit = ws.take<uint8_t>(tc_terms_bytes(3, 2 * C, C));
  void* gys = ws.take<uint8_t>(tc_terms_bytes(3, N, 2 * C));
  float* gz = ws.take<float>((size_t)N * C);
  const int sk = timedebd_splits(N);
  float* q = ws.take<float>((size_t)sk * C * 2 * C);
  float* lnpart = ws.take<float>((size_t)ln_bwd_blocks(N) * 2 * C);
  float* mu2 = ws.take<float>((size_t)N);
  float* rstd2 = ws.take<float>((size_t)N);
  int rc;
  // gYm terms (frames of a token side by side) and gbias = column sums of gY
  {
    const long long total4 = (long long)N * 2 * (C / 4);
    const int grid = (int)std::min<long long>((total4 + 255) / 256, (long long)sm_count() * 8);
    split3_frames_kernel<<<grid, 256, 0, st>>>(gout, N, C, HW, gys);
    VADC_CHECK_LAUNCH("split3_frames_kernel");
    colsum32_kernel<<<(C + 31) / 32, 256, 0, st>>>(gout, 2 * (long long)N, C, gbias);
    VADC_CHECK_LAUNCH("colsum32_kernel");
  }
  // gZ [N, C] = gYm [N, 2C] . Wk^T,  Wk [C rows = ci, 2C cols = j*C + co] is the K-major B operand
  if ((rc = tc_split<3>(wk, C, 2 * C, nullptr, wsplit, st))) return rc;
  if ((rc = tc_gemm<3, false, false>({gys, wsplit, N, C, 2 * C}, TcStoreEpi{gz, C}, st))) return rc;
  // z again (LayerNorm of x: its terms are the A operand of the weight-gradient contraction)
  if ((rc = launch_ln_rows(x, ln_w, ln_b, N, C, eps, nullptr, mu2, rstd2, nullptr, st, nullptr, zs))) return rc;
  // gWk [C, 2C] = Z^T gYm: both operands given as [tokens, .] (MN-major), split over the tokens
  if ((rc = tc_gemm<3, true, true>({zs, gys, C, 2 * C, N, nullptr, sk}, TcPartialEpi{q, 2 * C, (long long)C * 2 * C}, st))) return rc;
  {
    const long long n = (long long)C * 2 * C;
    sum_partials_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(q, sk, n, gwk);
    VADC_CHECK_LAUNCH("sum_partials_kernel");
  }
  return launch_ln_bwd(gz, x, mu, rstd, ln_w, N, C, gx, lnpart, g_ln_w, g_ln_b, st);
}

// ---------------------------------------------------------------------------------------------------------------------
// predict mode (model/swin_decoder_predict.py:591-592): timedebd = Conv3d(C, C, kernel (2,1,1), stride (2,1,1)) — two
// consecutive frames of a token position, side by side, are ONE row of a [N/2, 2C] matrix Zp (the same pair gather the
// non-predict backward applies to gY), and
//   out [N/2, C] = Zp . Wk^T + bias,        Wk [co, j*C + ci] = weight[co, ci, j]
// backward: gZp [N/2, 2C] = gY . Wk scattered back to the rows of the two frames (the ConvTranspose entry's forward
// scatter without its bias), gWk = gY^T . Zp split over the tokens, gbias = column sums of gY, LayerNorm backward.
// x [N, C] channel-last tokens of B * D frames (D even), HW tokens per frame; workspace: vadc_norm_timedebd_workspace_bytes.
// ---------------------------------------------------------------------------------------------------------------------
static int pair_terms(const float* x, const float* ln_w, const float* ln_b, int64_t N, int C, int64_t HW, float eps, float* z,
                      float* mu, float* rstd, void* zp, cudaStream_t st) {
  int rc;
  if ((rc = launch_ln_rows(x, ln_w, ln_b, N, C, eps, z, mu, rstd, nullptr, st))) return rc;
  const long long total4 = (long long)N * (C / 4);
  const int grid = (int)std::min<long long>((total4 + 255) / 256, (long long)sm_count() * 8);
  split3_frames_kernel<<<grid, 256, 0, st>>>(z, N / 2, C, HW, zp);
  VADC_CHECK_LAUNCH("split3_frames_kernel");
  return VADC_OK;
}

extern "C" int vadc_norm_timeconv_fwd(const float* x, const float* ln_w, const float* ln_b, const float* wk,
                                      const float* bias, int64_t N, int C, int64_t HW, float eps, float* out,
                                      float* mu, float* rstd, void* workspace, size_t workspace_bytes, void* stream) {
  VADC_REQUIRE(N >= 0 && C > 0 && HW > 0 && (C % 32) == 0 && C <= 1024, VADC_ERR_BAD_SHAPE);
  VADC_REQUIRE(N % (2 * HW) == 0, VADC_ERR_BAD_SHAPE);                       // an even number of frames
  if (N == 0) return VADC_OK;
  VADC_REQUIRE(x && ln_w && ln_b && wk && bias && out && mu && rstd && workspace, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(aligned16(x) && aligned16(out) && aligned16(wk), VADC_ERR_MISALIGNED);
  VADC_REQUIRE(workspace_bytes >= vadc_norm_timedebd_workspace_bytes(N, C), VADC_ERR_WORKSPACE);
  VADC_REQUIRE(tc_gemm_shape_ok(N / 2, C, 2 * C, false), VADC_ERR_UNSUPPORTED);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Carver ws(workspace, workspace_bytes);
  void* zp = ws.take<uint8_t>(tc_terms_bytes(3, N, C));
  void* wsplit = ws.take<uint8_t>(tc_terms_bytes(3, 2 * C, C));
  (void)ws.take<uint8_t>(tc_terms_bytes(3, N, 2 * C));
  float* z = ws.take<float>((size_t)N * C);                                  // the gZ slot of the backward
  int rc;
  if ((rc = pair_terms(x, ln_w, ln_b, N, C, HW, eps, z, mu, rstd, zp, st))) return rc;
  if ((rc = tc_split<3>(wk, C, 2 * C, nullptr, wsplit, st))) return rc;
  // rows = output channels, columns = (frame pair, position): coalesced channel-last stores (a handful of rows: row form)
  if (N / 2 >= 128) return tc_gemm<3, false, false>({wsplit, zp, C, N / 2, 2 * C}, TcBiasTEpi{out, bias, C}, st);
  return tc_gemm<3, false, false>({zp, wsplit, N / 2, C, 2 * C}, TcBiasEpi{out, bias, C}, st);
}

extern "C" int vadc_norm_timeconv_bwd(const float* x, const float* mu, const float* rstd, const float* ln_w,
                                      const float* ln_b, const float* wk, const float* gout, int64_t N, int C,
                                      int64_t HW, float eps, float* gx, float* g_ln_w, float* g_ln_b, float* gwk,
                                      float* gbias, void* workspace, size_t workspace_bytes, void* stream) {
  VADC_REQUIRE(N >= 0 && C > 0 && HW > 0 && (C % 32) == 0 && C <= 1024, VADC_ERR_BAD_SHAPE);
  VADC_REQUIRE(N % (2 * HW) == 0, VADC_ERR_BAD_SHAPE);
  VADC_REQUIRE(g_ln_w && g_ln_b && gwk && gbias && workspace, VADC_ERR_NULL_POINTER);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (N == 0) {
    VADC_CUDA(cudaMemsetAsync(gwk, 0, sizeof(float) * C * 2 * C, st));
    VADC_CUDA(cudaMemsetAsync(gbias, 0, sizeof(float) * C, st));
    VADC_CUDA(cudaMemsetAsync(g_ln_w, 0, sizeof(float) * C, st));
    VADC_CUDA(cudaMemsetAsync(g_ln_b, 0, sizeof(float) * C, st));
    return VADC_OK;
  }
  VADC_REQUIRE(x && mu && rstd && ln_w && ln_b && wk && gout && gx, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(aligned16(x) && aligned16(gout) && aligned16(wk) && aligned16(gx), VADC_ERR_MISALIGNED);
  VADC_REQUIRE(workspace_bytes >= vadc_norm_timedebd_workspace_bytes(N, C), VADC_ERR_WORKSPACE);
  Carver ws(workspace, workspace_bytes);
  void* zp = ws.take<uint8_t>(tc_terms_bytes(3, N, C));
  void* wsplit = ws.take<uint8_t>(tc_terms_bytes(3, 2 * C, C));
  void* gys = ws.take<uint8_t>(tc_terms_bytes(3, N, 2 * C));
  float* gz = ws.take<float>((size_t)N * C);
  const int sk = timedebd_splits(N);
  float* q = ws.take<float>((size_t)sk * C * 2 * C);
  float* lnpart = ws.take<float>((size_t)ln_bwd_blocks(N) * 2 * C);
  float* mu2 = ws.take<float>((size_t)N);
  float* rstd2 = ws.take<float>((size_t)N);
  float* z = ws.take<float>((size_t)N * C);
  const long long Nh = N / 2;
  int rc;
  if ((rc = tc_split<3>(gout, Nh, C, nullptr, gys, st))) return rc;
  colsum32_kernel<<<(C + 31) / 32, 256, 0, st>>>(gout, Nh, C, gbias);
  VADC_CHECK_LAUNCH("colsum32_kernel");
  // gZp [N/2, 2C] = gY [N/2, C] . Wk (Wk [co rows, 2C cols] read MN-major), column half j -> the rows of frame 2f + j
  if ((rc = tc_split<3>(wk, C, 2 * C, nullptr, wsplit, st))) return rc;
  if ((rc = tc_gemm<3, false, true>({gys, wsplit, Nh, 2 * C, C}, TcTimeDebedEpi{gz, nullptr, HW, C}, st))) return rc;
  // Zp again: gWk [C, 2C] = gY^T Zp, both operands given as [pair rows, .] (MN-major), split over the rows
  if ((rc = pair_terms(x, ln_w, ln_b, N, C, HW, eps, z, mu2, rstd2, zp, st))) return rc;
  if ((rc = tc_gemm<3, true, true>({gys, zp, C, 2 * C, Nh, nullptr, sk}, TcPartialEpi{q, 2 * C, (long long)C * 2 * C}, st))) return rc;
  {
    const long long n = (long long)C * 2 * C;
    sum_partials_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(q, sk, n, gwk);
    VADC_CHECK_LAUNCH("sum_partials_kernel");
  }
  return launch_ln_bwd(gz, x, mu, rstd, ln_w, N, C, gx, lnpart, g_ln_w, g_ln_b, st);
}
