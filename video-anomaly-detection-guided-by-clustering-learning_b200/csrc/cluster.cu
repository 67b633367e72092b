// cluster.cu — EuclidDistance_Assign_Module forward / backward (C1, C2, L1),
// SIMT fp32 path (VADC_IMPL_SIMT): valid for every shape; the tcgen05 kernel in
// cluster_tc.cu takes over when the shape fits (VADC_IMPL_AUTO).
#include <string.h>
#include "common.cuh"
#include "sgemm.cuh"
#include "rows.cuh"
#include "cluster.h"
#include "tc_gemm.cuh"
#include <algorithm>
#include <stdlib.h>

namespace vadc {

// D = sqrt(max(0, |a|^2 + |b|^2 - 2 a.b))   torch.cdist mm form (SURVEY.md D2)
struct DistEpilogue {
  float* out; const float* aa; const float* bb;
  long long ldo;            // row stride of out
  long long batch_out, batch_aa, batch_bb, col_stride;
  __device__ __forceinline__ void operator()(int batch, int, int m, int n, float v) const {
    float sq = aa[batch * batch_aa + m] + bb[batch * batch_bb + n] - 2.0f * v;
    out[batch * batch_out + (long long)m * ldo + (long long)n * col_stride] = sqrtf(fmaxf(sq, 0.f));
  }
};

struct StoreEpilogue {
  float* out; long long ldo;
  __device__ __forceinline__ void operator()(int, int, int m, int n, float v) const {
    out[(long long)m * ldo + n] = v;
  }
};

// gz = feature * rsum - acc + gF
struct GzEpilogue {
  float* out; const float* feature; const float* rsum; const float* gF; long long ld;
  __device__ __forceinline__ void operator()(int, int, int m, int n, float v) const {
    long long i = (long long)m * ld + n;
    float o = feature[i] * rsum[m] - v;
    if (gF) o += gF[i];
    out[i] = o;
  }
};

// split-K partial store: out[split][m][n]
struct PartialEpilogue {
  float* out; long long ld, split_stride;
  __device__ __forceinline__ void operator()(int, int split, int m, int n, float v) const {
    out[split * split_stride + (long long)m * ld + n] = v;
  }
};

// gcenters[k,c] = sum_s (P1 - P2)[s,k,c] + centers[k,c] * rcol[k]
__global__ void __launch_bounds__(256)
gcenters_finalize_kernel(const float* __restrict__ p1, const float* __restrict__ p2, int splits,
                         const float* __restrict__ centers, const float* __restrict__ rcol,
                         int K, int C, float* __restrict__ out) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long n = (long long)K * C;
  if (i >= n) return;
  float s = 0.f;
  for (int sp = 0; sp < splits; ++sp) {
    float a = p1 ? p1[sp * n + i] : 0.f;
    s += a - p2[sp * n + i];
  }
  out[i] = s + centers[i] * rcol[i / C];
}

// partial [nblocks, 2C] -> gw, gb: a block owns 32 columns, eight row groups stride the blocks (fixed order: deterministic)
__global__ void __launch_bounds__(256)
ln_bwd_finalize_kernel(const float* __restrict__ partial, int nblocks, int C,
                       float* __restrict__ gw, float* __restrict__ gb) {
  __shared__ float red[8][33];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + lane;
  float s = 0.f;
  if (c < 2 * C)
    for (int b = wid; b < nblocks; b += 8) s += partial[(size_t)b * 2 * C + c];
  red[wid][lane] = s;
  __syncthreads();
  if (wid == 0 && c < 2 * C) {
    float t = 0.f;
#pragma unroll
    for (int ww = 0; ww < 8; ++ww) t += red[ww][lane];
    if (c < C) gw[c] = t; else gb[c - C] = t;
  }
}

__global__ void zero_kernel(float* p, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = 0.f;
}

// ---------------------------------------------------------------------------
// launch helpers shared with space_cluster.cu / memory.cu
// ---------------------------------------------------------------------------
int launch_ln_rows(const float* x, const float* w, const float* b, long long N, int C, float eps,
                   float* z, float* mu, float* rstd, float* zz, cudaStream_t st, float* rowstats, void* split3,
                   const float* hscale) {
  if (N == 0) return VADC_OK;
  const int wpb = 8;
  dim3 grid((unsigned)((N + wpb - 1) / wpb));
#define LN_CASE(V) ln_rows_kernel<V><<<grid, wpb * 32, 0, st>>>(x, w, b, N, C, eps, z, mu, rstd, zz, rowstats, \
                                                              static_cast<__nv_bfloat16*>(split3), hscale)
  if (C <= 128) LN_CASE(1);
  else if (C <= 256) LN_CASE(2);
  else if (C <= 512) LN_CASE(4);
  else if (C <= 768) LN_CASE(6);
  else if (C <= 1024) LN_CASE(8);
  else return VADC_ERR_UNSUPPORTED;
#undef LN_CASE
  VADC_CHECK_LAUNCH("ln_rows_kernel");
  return VADC_OK;
}

int launch_row_sqnorm(const float* a, long long R, int C, float* out, cudaStream_t st) {
  if (R == 0) return VADC_OK;
  row_sqnorm_kernel<<<(unsigned)((R + 7) / 8), 256, 0, st>>>(a, R, C, out);
  VADC_CHECK_LAUNCH("row_sqnorm_kernel");
  return VADC_OK;
}

static inline int group_for(int K) {
  int nv = K / 4;
  if (nv <= 4) return 4;
  if (nv <= 8) return 8;
  if (nv <= 16) return 16;
  return 32;
}

int softmin_blocks(long long R, int K) {
  int G = group_for(K);
  return (int)((R + (256 / G) - 1) / (256 / G));
}

// A, label, loss_sq from D.  partial: softmin_blocks(R,K) doubles.
int launch_softmin_rows(const float* D, long long R, int K, float alpha, float* A, long long* label,
                        double* partial, float* loss_sq, cudaStream_t st, int k_valid, void* terms_h2, float sa) {
  __half* th = static_cast<__half*>(terms_h2);
  if (k_valid < 0 || k_valid > K) k_valid = K;
  if (R == 0) {
    zero_kernel<<<1, 32, 0, st>>>(loss_sq, 1);
    VADC_CHECK_LAUNCH("zero_kernel");
    return VADC_OK;
  }
  int G = group_for(K);
  int nb = softmin_blocks(R, K);
  switch (G) {
    case 4: softmin_rows_kernel<4><<<nb, 256, 0, st>>>(D, R, K, k_valid, alpha, A, label, partial, th, sa); break;
    case 8: softmin_rows_kernel<8><<<nb, 256, 0, st>>>(D, R, K, k_valid, alpha, A, label, partial, th, sa); break;
    case 16: softmin_rows_kernel<16><<<nb, 256, 0, st>>>(D, R, K, k_valid, alpha, A, label, partial, th, sa); break;
    default: softmin_rows_kernel<32><<<nb, 256, 0, st>>>(D, R, K, k_valid, alpha, A, label, partial, th, sa); break;
  }
  VADC_CHECK_LAUNCH("softmin_rows_kernel");
  finalize_sum_kernel<<<1, 1024, 0, st>>>(partial, nb, loss_sq);
  VADC_CHECK_LAUNCH("finalize_sum_kernel");
  return VADC_OK;
}

int launch_bwd_rows(const float* D, const float* A, const float* gemm, const float* gD,
                    const float* gA, const float* g_loss_sq, long long R, int K,
                    float alpha, float* r, float* rsum, cudaStream_t st, unsigned* absmax_bits) {
  if (R == 0) return VADC_OK;
  int G = group_for(K);
  int nb = (int)((R + (256 / G) - 1) / (256 / G));
  if (absmax_bits) VADC_CUDA(cudaMemsetAsync(absmax_bits, 0, sizeof(unsigned), st));
#define BR_CASE(GG) bwd_rows_kernel<GG><<<nb, 256, 0, st>>>(D, A, gemm, gD, gA, g_loss_sq, R, K, alpha, r, rsum, absmax_bits)
  switch (G) {
    case 4: BR_CASE(4); break;
    case 8: BR_CASE(8); break;
    case 16: BR_CASE(16); break;
    default: BR_CASE(32); break;
  }
#undef BR_CASE
  VADC_CHECK_LAUNCH("bwd_rows_kernel");
  return VADC_OK;
}

int ln_bwd_blocks(long long N) {
  long long b = (N + 63) / 64;          // >= 8 rows per warp before another block is worth it
  long long cap = (long long)sm_count() * 4;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

// gx, g_ln_w, g_ln_b from gz (row-major).  partial: ln_bwd_blocks(N)*2C floats.
int launch_ln_bwd(const float* gz, const float* x, const float* mu, const float* rstd,
                  const float* w, long long N, int C, float* gx, float* partial, float* gw,
                  float* gb, cudaStream_t st) {
  int nb = ln_bwd_blocks(N);
  size_t smem = (size_t)8 * 2 * C * sizeof(float);
#define LB_CASE(V)                                                                              \
  do {                                                                                          \
    if (smem > 48 * 1024)                                                                       \
      VADC_CUDA(cudaFuncSetAttribute(ln_bwd_rows_kernel<V>,                                     \
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));  \
    ln_bwd_rows_kernel<V><<<nb, 256, smem, st>>>(gz, x, mu, rstd, w, N, C, gx, partial);        \
  } while (0)
  if (C <= 128) LB_CASE(1);
  else if (C <= 256) LB_CASE(2);
  else if (C <= 512) LB_CASE(4);
  else if (C <= 768) LB_CASE(6);
  else if (C <= 1024) LB_CASE(8);
  else return VADC_ERR_UNSUPPORTED;
#undef LB_CASE
  VADC_CHECK_LAUNCH("ln_bwd_rows_kernel");
  ln_bwd_finalize_kernel<<<(2 * C + 31) / 32, 256, 0, st>>>(partial, nb, C, gw, gb);
  VADC_CHECK_LAUNCH("ln_bwd_finalize_kernel");
  return VADC_OK;
}

// batched cdist on precomputed norms
int launch_dist(const float* a, const float* b, const float* aa, const float* bb, int nb,
                long long R, long long P, int C, float* out, cudaStream_t st) {
  if (R == 0 || P == 0 || nb == 0) return VADC_OK;
  Operand A{a, C, 1};
  Operand B{b, 1, C};          // opB[k=c, n=p] = b[p*C + c]
  DistEpilogue epi{out, aa, bb, P, R * P, R, P, 1};
  cudaError_t e = sgemm_auto((int)R, (int)P, C, A, B, R * C, P * C, nb, 1, epi, st);
  if (e != cudaSuccess) return record_cuda_error(e, "dist sgemm");
  return VADC_OK;
}

int split_count(long long Ntok, int tiles) {
  long long want = ((long long)sm_count() * 2 + tiles - 1) / tiles;
  long long maxs = (Ntok + 511) / 512;
  if (want > maxs) want = maxs;
  if (want > 256) want = 256;
  if (want < 1) want = 1;
  return (int)want;
}

}  // namespace vadc

using namespace vadc;

// ---------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------
namespace vadc {
// rowstats for the forward paths that do not fuse them: one warp per token,
// {|f|^2, sum f gamma, sum f gamma xhat, 0} with f = feature row, xhat = (x - mu) rstd
__global__ void __launch_bounds__(256)
rowstats_kernel(const float* __restrict__ x, const float* __restrict__ feature, const float* __restrict__ mu,
                const float* __restrict__ rstd, const float* __restrict__ ln_w, long long N, int C,
                float* __restrict__ rowstats) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= N) return;
  const float m = mu[row], rs = rstd[row];
  float zz = 0.f, p1 = 0.f, p2 = 0.f;
  for (int c = lane; c < C; c += 32) {
    const float f = feature[row * C + c], xh = (x[row * C + c] - m) * rs, fg = f * ln_w[c];
    zz = fmaf(f, f, zz); p1 += fg; p2 = fmaf(fg, xh, p2);
  }
  zz = warp_sum(zz); p1 = warp_sum(p1); p2 = warp_sum(p2);
  if (lane == 0) reinterpret_cast<float4*>(rowstats)[row] = make_float4(zz, p1, p2, 0.f);
}
static int launch_rowstats(const float* x, const float* feature, const float* mu, const float* rstd,
                           const float* ln_w, long long N, int C, float* rowstats, cudaStream_t st) {
  if (!rowstats || N == 0) return VADC_OK;
  rowstats_kernel<<<(unsigned)((N + 7) / 8), 256, 0, st>>>(x, feature, mu, rstd, ln_w, N, C, rowstats);
  VADC_CHECK_LAUNCH("rowstats_kernel");
  return VADC_OK;
}
}  // namespace vadc

extern "C" size_t vadc_cluster_fwd_workspace_bytes(int64_t N, int C, int K, int impl) {
  (void)impl;
  size_t b = 0;
  b += align_up((size_t)(N > 0 ? N : 1) * sizeof(float), 256);           // |z|^2
  b += align_up((size_t)K * sizeof(float), 256);                         // |c|^2
  b += align_up((size_t)(softmin_blocks(N, K) + 1) * sizeof(double), 256);
  b += std::max(vadc_cluster_tc_extra_workspace_bytes(N, C, K), vadc_cluster_ws_extra_workspace_bytes(N, C, K));
  if (impl != VADC_IMPL_SIMT && N > 0)                                   // term copies for the tcgen05 GEMMs + scales
    b += tc_gemm_split_bytes(N, C) + tc_gemm_split_bytes(K, C) + tc_gemm_split_bytes(N, K) + 256;
  return b + 256;
}

static int cluster_fwd_impl(const float* x, const float* ln_w, const float* ln_b,
                            const float* centers, int64_t N, int C, int K, int k_valid, float alpha,
                            float eps, float* D, float* A, float* x_rec, float* feature,
                            int64_t* label, float* mu, float* rstd, float* rowstats, float* loss_sq,
                            void* workspace, size_t workspace_bytes, int impl, void* stream) {
  VADC_REQUIRE(N >= 0 && C > 0 && K > 0 && (C % 4) == 0 && (K % 4) == 0, VADC_ERR_BAD_SHAPE);
  VADC_REQUIRE(N < (1ll << 31) && C <= 1024, VADC_ERR_UNSUPPORTED);
  VADC_REQUIRE(ln_w && ln_b && centers && loss_sq && workspace, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(N == 0 || (x && D && A && x_rec && feature && label && mu && rstd), VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(aligned16(rowstats), VADC_ERR_MISALIGNED);
  VADC_REQUIRE(aligned16(x) && aligned16(ln_w) && aligned16(ln_b) && aligned16(centers) &&
               aligned16(D) && aligned16(A) && aligned16(x_rec) && aligned16(feature) &&
               aligned16(workspace), VADC_ERR_MISALIGNED);
  VADC_REQUIRE(workspace_bytes >= vadc_cluster_fwd_workspace_bytes(N, C, K, impl), VADC_ERR_WORKSPACE);
  cudaStream_t st = static_cast<cudaStream_t>(stream);

  if (impl != VADC_IMPL_SIMT) {
    int rc = vadc_cluster_fwd_ws(x, ln_w, ln_b, centers, N, C, K, alpha, eps, D, A, x_rec, feature,
                                 label, mu, rstd, rowstats, loss_sq, workspace, workspace_bytes, st);
    if (rc != VADC_ERR_UNSUPPORTED) return rc;
    rc = vadc_cluster_fwd_tc(x, ln_w, ln_b, centers, N, C, K, alpha, eps, D, A, x_rec, feature,
                             label, mu, rstd, loss_sq, workspace, workspace_bytes, st);
    if (rc == VADC_OK) return launch_rowstats(x, feature, mu, rstd, ln_w, N, C, rowstats, st);
    if (rc != VADC_ERR_UNSUPPORTED || impl == VADC_IMPL_TCGEN05) return rc;
  }
  Carver ws(workspace, workspace_bytes);
  float* zz = ws.take<float>(N > 0 ? N : 1);
  float* cc = ws.take<float>(K);
  double* partial = ws.take<double>(softmin_blocks(N, K) + 1);
  int rc;
  // shapes outside the fused kernels (C = 768, K = 16 / 64 / 256 / 1024): the two contractions run on the
  // tcgen05 GEMM (three-term bf16 split: fp32-faithful); LayerNorm (+ rowstats + the split of z) and softmin
  // stay row kernels
  const bool use_tc = impl != VADC_IMPL_SIMT && N > 0 && !env_on("VADC_NO_TC_GEMM") &&
                      tc_gemm_shape_ok(N, K, C, false) && tc_gemm_shape_ok(N, C, K, true);
  if (use_tc && !env_on("VADC_TC_BF16X3")) {
    // every operand of the forward is bounded (LayerNorm output, centroids, softmin weights in [0, 1]): two fp16
    // terms after a power-of-two scaling carry 22 significant bits (the fused K = 32 kernel's recipe): 2/3 of the
    // operand bytes and half the MMAs of the three-term bf16 split; the scales stay in device memory (no host sync)
    void* fs = ws.take<uint8_t>(tc_gemm_split2_bytes(N, C));
    void* cs = ws.take<uint8_t>(tc_gemm_split2_bytes(K, C));
    void* as = ws.take<uint8_t>(tc_gemm_split2_bytes(N, K));
    float* sc = ws.take<float>(8);
    if ((rc = tc_fwd_scales(centers, ln_w, ln_b, (long long)K * C, C, sc, st))) return rc;
    if ((rc = launch_ln_rows(x, ln_w, ln_b, N, C, eps, feature, mu, rstd, zz, st, rowstats, fs, sc + 0))) return rc;
    if ((rc = launch_row_sqnorm(centers, K, C, cc, st))) return rc;
    if ((rc = tc_split2h(centers, K, C, sc + 1, cs, st))) return rc;
    // from K = 128 up the distance GEMM runs with the operands swapped (rows = centroids): coalesced stores of D
    if (K >= 128) {
      if ((rc = launch_tc_gemm_h2<false>(cs, fs, K, N, C, sc + 2, TcDistTEpi{D, cc, zz, K}, st))) return rc;
    } else if ((rc = launch_tc_gemm_h2<false>(fs, cs, N, K, C, sc + 2, TcDistEpi{D, zz, cc, K}, st))) return rc;
    // softmin writes A and, in the same pass, its two fp16 terms scaled by s_a = 2^13 (the value fwd_scales_kernel puts in sc[3])
    if ((rc = launch_softmin_rows(D, N, K, alpha, A, (long long*)label, partial, loss_sq, st, k_valid, as, 8192.0f))) return rc;
    if (C >= 128)   // rows = channels (centers [K,C] as the MN-major A operand): coalesced x_rec
      return launch_tc_gemm_ex_h2<true, false>(cs, as, C, N, K, 1, sc + 4, TcStoreTEpi{x_rec, C}, st);
    return launch_tc_gemm_h2<true>(as, cs, N, C, K, sc + 4, TcStoreEpi{x_rec, C}, st);    // centers [K,C] read MN-major
  }
  if (use_tc) {
    void* fs = ws.take<uint8_t>(tc_gemm_split_bytes(N, C));
    void* cs = ws.take<uint8_t>(tc_gemm_split_bytes(K, C));
    void* as = ws.take<uint8_t>(tc_gemm_split_bytes(N, K));
    if ((rc = launch_ln_rows(x, ln_w, ln_b, N, C, eps, feature, mu, rstd, zz, st, rowstats, fs))) return rc;
    if ((rc = launch_row_sqnorm(centers, K, C, cc, st))) return rc;
    if ((rc = tc_split3(centers, K, C, cs, st))) return rc;
    if ((rc = launch_tc_gemm<false>(fs, cs, N, K, C, TcDistEpi{D, zz, cc, K}, st))) return rc;
    if ((rc = launch_softmin_rows(D, N, K, alpha, A, (long long*)label, partial, loss_sq, st, k_valid))) return rc;
    if ((rc = tc_split3(A, N, K, as, st))) return rc;
    return launch_tc_gemm<true>(as, cs, N, C, K, TcStoreEpi{x_rec, C}, st);    // centers [K,C] read MN-major
  }
  if ((rc = launch_ln_rows(x, ln_w, ln_b, N, C, eps, feature, mu, rstd, zz, st, rowstats))) return rc;
  if ((rc = launch_row_sqnorm(centers, K, C, cc, st))) return rc;
  if ((rc = launch_dist(feature, centers, zz, cc, 1, N, K, C, D, st))) return rc;
  if ((rc = launch_softmin_rows(D, N, K, alpha, A, (long long*)label, partial, loss_sq, st, k_valid))) return rc;
  if (N > 0) {
    Operand Aop{A, K, 1}, Bop{centers, C, 1};
    StoreEpilogue epi{x_rec, C};
    cudaError_t e = sgemm_auto((int)N, C, K, Aop, Bop, 0, 0, 1, 1, epi, st);
    if (e != cudaSuccess) return record_cuda_error(e, "x_rec sgemm");
  }
  return VADC_OK;
}

extern "C" int vadc_cluster_fwd(const float* x, const float* ln_w, const float* ln_b,
                                const float* centers, int64_t N, int C, int K, float alpha,
                                float eps, float* D, float* A, float* x_rec, float* feature,
                                int64_t* label, float* mu, float* rstd, float* rowstats, float* loss_sq,
                                void* workspace, size_t workspace_bytes, int impl, void* stream) {
  return cluster_fwd_impl(x, ln_w, ln_b, centers, N, C, K, K, alpha, eps, D, A, x_rec, feature, label, mu, rstd, rowstats,
                          loss_sq, workspace, workspace_bytes, impl, stream);
}

// any cluster_num: the host pads the centroids to K % 4 == 0 rows; the trailing K - K_valid rows are excluded
extern "C" int vadc_cluster_fwd_padded(const float* x, const float* ln_w, const float* ln_b,
                                       const float* centers, int64_t N, int C, int K, int K_valid, float alpha,
                                       float eps, float* D, float* A, float* x_rec, float* feature,
                                       int64_t* label, float* mu, float* rstd, float* rowstats, float* loss_sq,
                                       void* workspace, size_t workspace_bytes, void* stream) {
  VADC_REQUIRE(K_valid >= 1 && K_valid <= K, VADC_ERR_BAD_SHAPE);
  return cluster_fwd_impl(x, ln_w, ln_b, centers, N, C, K, K_valid, alpha, eps, D, A, x_rec, feature, label, mu, rstd,
                          rowstats, loss_sq, workspace, workspace_bytes, K_valid == K ? VADC_IMPL_AUTO : VADC_IMPL_SIMT, stream);
}

namespace vadc {
// cdist of a small problem (the [K,K] centroid self-distance of model/cluster.py:77-79 is 32 x 32 x 192) in ONE
// launch instead of two norm kernels + a tile GEMM: one block per output row i, 8 lanes per column j, the mm form
// sqrt(max(0, |a|^2 + |b|^2 - 2 a.b)) with fp32 accumulation
__global__ void __launch_bounds__(256)
cdist_small_kernel(const float* __restrict__ a, const float* __restrict__ b, int R, int P, int C,
                   float* __restrict__ out) {
  // block = one row i of one batch; 8 lanes per output column j (lane part p sums the float4 chunks p, p+8, ...)
  const int i = blockIdx.x, nbat = blockIdx.y, part = threadIdx.x & 7;
  const float4* ar = reinterpret_cast<const float4*>(a + ((size_t)nbat * R + i) * C);
  const int nv = C >> 2;
  for (int j = threadIdx.x >> 3; j < ((P + 31) & ~31); j += 32) {       // whole warps stay in the loop for the shuffles
    float aa = 0.f, bb = 0.f, ab = 0.f;
    if (j < P) {
      const float4* br = reinterpret_cast<const float4*>(b + ((size_t)nbat * P + j) * C);
      for (int c = part; c < nv; c += 8) {
        const float4 x = __ldg(ar + c), y = __ldg(br + c);
        aa += (x.x * x.x + x.y * x.y) + (x.z * x.z + x.w * x.w);
        bb += (y.x * y.x + y.y * y.y) + (y.z * y.z + y.w * y.w);
        ab += (x.x * y.x + x.y * y.y) + (x.z * y.z + x.w * y.w);
      }
    }
#pragma unroll
    for (int o = 1; o < 8; o <<= 1) {
      aa += __shfl_xor_sync(0xffffffffu, aa, o);
      bb += __shfl_xor_sync(0xffffffffu, bb, o);
      ab += __shfl_xor_sync(0xffffffffu, ab, o);
    }
    if (part == 0 && j < P) out[((size_t)nbat * R + i) * P + j] = sqrtf(fmaxf(aa + bb - 2.f * ab, 0.f));
  }
}
}  // namespace vadc

namespace vadc {
// batched cdist on the tcgen05 GEMM: tensor-bound sizes only (the split pass costs 10 bytes per operand element)
static bool cdist_tc_ok(int nb, long long R, long long P, int C) {
  return nb >= 1 && nb <= 65535 && (C % 8) == 0 && P >= 8 && (long long)nb * R < (1ll << 31) &&
         (long long)nb * P < (1ll << 31) && (double)nb * R * P * C >= (double)(1ll << 28) &&
         tc_gemm_shape_ok(R, P, C, false) && !env_on("VADC_NO_TC_GEMM");
}
}  // namespace vadc

extern "C" size_t vadc_cdist_workspace_bytes(int nb, int64_t R, int64_t P, int C) {
  size_t b = align_up((size_t)nb * R * sizeof(float), 256) + align_up((size_t)nb * P * sizeof(float), 256) + 256;
  if (nb > 0 && R > 0 && P > 0 && C > 0 && (C % 8) == 0)
    b += tc_gemm_split_bytes((long long)nb * R, C) + tc_gemm_split_bytes((long long)nb * P, C);
  return b;
}

extern "C" int vadc_cdist(const float* a, const float* b, int nb, int64_t R, int64_t P, int C,
                          float* out, void* workspace, size_t workspace_bytes, void* stream) {
  VADC_REQUIRE(nb >= 0 && R >= 0 && P >= 0 && C > 0, VADC_ERR_BAD_SHAPE);
  if (nb == 0 || R == 0 || P == 0) return VADC_OK;
  VADC_REQUIRE(a && b && out && workspace, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(R < (1ll << 31) && P < (1ll << 31), VADC_ERR_UNSUPPORTED);
  VADC_REQUIRE(workspace_bytes >= vadc_cdist_workspace_bytes(nb, R, P, C), VADC_ERR_WORKSPACE);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // launch-latency-bound sizes, and single problems too small to fill the GPU with GEMM tiles (the [K,K] centroid
  // self-distance at K = 256, C = 768 is 16 tiles: 135 us on the tile GEMM, one row per block does it in ~15 us)
  const long long macs = (long long)nb * R * P * C;
  const long long tiles = ((R + 127) / 128) * ((P + 127) / 128);       // 32 tiles and more keep the tile GEMM busy enough
  if ((macs <= (1ll << 21) || (nb == 1 && macs <= (1ll << 28) && tiles < 32)) && nb <= 65535 && (C % 4) == 0 && aligned16(a) &&
      aligned16(b)) {
    cdist_small_kernel<<<dim3((unsigned)R, (unsigned)nb), 256, 0, st>>>(a, b, (int)R, (int)P, C, out);
    VADC_CHECK_LAUNCH("cdist_small_kernel");
    return VADC_OK;
  }
  Carver ws(workspace, workspace_bytes);
  float* aa = ws.take<float>((size_t)nb * R);
  float* bb = ws.take<float>((size_t)nb * P);
  int rc;
  const bool self = a == b && R == P;          // centroid self-distance (model/cluster.py:82, :134): one norm pass, one split
  if (self) bb = aa;
  if ((rc = launch_row_sqnorm(a, (long long)nb * R, C, aa, st))) return rc;
  if (!self && (rc = launch_row_sqnorm(b, (long long)nb * P, C, bb, st))) return rc;
  if (cdist_tc_ok(nb, R, P, C)) {
    // one launch for all batches: A = a as [nb R, C], B = b as [nb P, C], batch z starts z R / z P rows further
    void* as = ws.take<uint8_t>(tc_gemm_split_bytes((long long)nb * R, C));
    void* bs = self ? as : ws.take<uint8_t>(tc_gemm_split_bytes((long long)nb * P, C));
    if ((rc = tc_split3(a, (long long)nb * R, C, as, st))) return rc;
    if (!self && (rc = tc_split3(b, (long long)nb * P, C, bs, st))) return rc;
    TcBatchDistEpi epi{out, aa, bb, P, R * P, R, P};
    return launch_tc_gemm_batched<false, false>(as, (long long)nb * R, C, bs, (long long)nb * P, C, R, P, C, nb,
                                                TcBatchOffsets{(int)R, 0, (int)P, 0}, epi, st);
  }
  return launch_dist(a, b, aa, bb, nb, R, P, C, out, st);
}

namespace vadc {
// split-K factor of the centroid-gradient GEMMs ([K,C] outputs, contraction over the tokens): ~2 CTAs per SM
static int bwd_tc_splits(long long N, int C, int K) {
  const long long tiles = (long long)((K + 127) / 128) * ((C + 127) / 128);
  const long long nkb = (N + 63) / 64;
  long long s = (2ll * sm_count() + tiles - 1) / tiles;
  if (s > nkb) s = nkb;
  if (s < 1) s = 1;
  return (int)s;
}
}  // namespace vadc

extern "C" size_t vadc_cluster_bwd_workspace_bytes(int64_t N, int C, int K) {
  size_t n = (size_t)(N > 0 ? N : 1);
  int tiles = ((K + 63) / 64) * ((C + 63) / 64);
  int splits = split_count(N, tiles);
  size_t b = 0;
  b += align_up(n * K * sizeof(float), 256);                 // gR.c^T
  b += align_up(n * K * sizeof(float), 256);                 // r
  b += align_up(n * sizeof(float), 256);                     // rsum
  b += align_up(n * C * sizeof(float), 256);                 // gz
  b += 2 * align_up((size_t)splits * K * C * sizeof(float), 256);   // split-K partials
  b += align_up((size_t)colsum_chunks(N) * K * sizeof(float), 256); // colsum partial
  b += align_up((size_t)K * sizeof(float), 256);             // rcol
  b += align_up((size_t)ln_bwd_blocks(N) * 2 * C * sizeof(float), 256);
  // generic path on the tcgen05 GEMM: bf16 term copies of gR, feature, A, r and the centroids + split-K partials
  b += 2 * tc_gemm_split_bytes((long long)n, C) + 2 * tc_gemm_split_bytes((long long)n, K) + tc_gemm_split_bytes(K, C) + 1024;
  b += 2 * align_up((size_t)bwd_tc_splits(N, C, K) * K * C * sizeof(float), 256);
  return std::max(std::max(b + 256, bwd_fused_workspace_bytes(N, C, K)), bwd_tc2_workspace_bytes(N, C, K));
}

extern "C" int vadc_cluster_bwd(const float* x, const float* mu, const float* rstd, const float* rowstats,
                                const float* feature, const float* ln_w, const float* ln_b,
                                const float* centers,
                                const float* D, const float* A, const float* gD, const float* gA,
                                const float* gR, const float* gF, const float* g_loss_sq,
                                int64_t N, int C, int K, float alpha,
                                float* gx, float* gcenters, float* g_ln_w, float* g_ln_b,
                                void* workspace, size_t workspace_bytes, void* stream) {
  VADC_REQUIRE(N >= 0 && C > 0 && K > 0 && (C % 4) == 0 && (K % 4) == 0, VADC_ERR_BAD_SHAPE);
  VADC_REQUIRE(N < (1ll << 31) && C <= 1024, VADC_ERR_UNSUPPORTED);
  VADC_REQUIRE(ln_w && centers && gcenters && g_ln_w && g_ln_b && workspace, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(N == 0 || (x && mu && rstd && feature && D && A && gx), VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(workspace_bytes >= vadc_cluster_bwd_workspace_bytes(N, C, K), VADC_ERR_WORKSPACE);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long KC = (long long)K * C;
  if (N == 0) {
    zero_kernel<<<(unsigned)((KC + 255) / 256), 256, 0, st>>>(gcenters, KC);
    zero_kernel<<<(C + 255) / 256, 256, 0, st>>>(g_ln_w, C);
    zero_kernel<<<(C + 255) / 256, 256, 0, st>>>(g_ln_b, C);
    VADC_CHECK_LAUNCH("zero_kernel");
    return VADC_OK;
  }
  const char* bimpl = env_str("VADC_BWD_IMPL");            // debugging / A-B runs: tc | fused | generic
  const bool want_tc = !bimpl || !strcmp(bimpl, "tc");
  if (want_tc && rowstats && ln_b && gR && !gD && !gA && !gF && bwd_tc2_shape_ok(N, C, K))
    return launch_cluster_bwd_tc2(x, mu, rstd, rowstats, ln_w, ln_b, centers, D, A, gR, g_loss_sq, N, C, K, alpha, gx,
                                  gcenters, g_ln_w, g_ln_b, workspace, workspace_bytes, st);
  if (bwd_fused_shape_ok(N, C, K) && !(bimpl && !strcmp(bimpl, "generic")))
    return launch_cluster_bwd_fused(x, mu, rstd, feature, ln_w, centers, D, A, gD, gA, gR, gF, g_loss_sq,
                                    N, C, K, alpha, gx, gcenters, g_ln_w, g_ln_b, workspace,
                                    workspace_bytes, st);
  int tiles = ((K + 63) / 64) * ((C + 63) / 64);
  int splits = split_count(N, tiles);
  Carver ws(workspace, workspace_bytes);
  float* gemm = ws.take<float>((size_t)N * K);
  float* r = ws.take<float>((size_t)N * K);
  float* rsum = ws.take<float>(N);
  float* gz = ws.take<float>((size_t)N * C);
  float* p1 = ws.take<float>((size_t)splits * KC);
  float* p2 = ws.take<float>((size_t)splits * KC);
  float* cpart = ws.take<float>((size_t)colsum_chunks(N) * K);
  float* rcol = ws.take<float>(K);
  float* lnpart = ws.take<float>((size_t)ln_bwd_blocks(N) * 2 * C);
  if (!env_on("VADC_NO_TC_GEMM") && vadc_device_ok() && (K % 8) == 0 && (C % 8) == 0 && K >= 8 && C >= 8) {
    // ---- the five contractions on the tcgen05 GEMM (three-term bf16 split): G1 = gR c^T; gz = z rsum - r c + gF;
    //      gcenters = A^T gR - r^T z + c colsum(r) with the token matrices read MN-major and split-K over the tokens
    const int sk = bwd_tc_splits(N, C, K);
    void* gRs = ws.take<uint8_t>(tc_gemm_split_bytes(N, C));
    void* fs = ws.take<uint8_t>(tc_gemm_split_bytes(N, C));
    void* as = ws.take<uint8_t>(tc_gemm_split_bytes(N, K));
    void* rs = ws.take<uint8_t>(tc_gemm_split_bytes(N, K));
    void* cs = ws.take<uint8_t>(tc_gemm_split_bytes(K, C));
    float* q1 = ws.take<float>((size_t)sk * KC);
    float* q2 = ws.take<float>((size_t)sk * KC);
    int rc;
    if (!env_on("VADC_TC_BF16X3")) {
      // two fp16 terms per operand, each scaled by the power of two of its measured bound (A: 2^13): 22 significant bits,
      // 2/3 of the operand bytes and half the MMAs of the bf16 x3 split (VADC_TC_BF16X3 keeps that one)
      unsigned* bits = ws.take<unsigned>(64);
      float* sc = ws.take<float>(64);
      VADC_CUDA(cudaMemsetAsync(bits, 0, 4 * sizeof(unsigned), st));
      if (gR && (rc = tc_absmax_bits(gR, (long long)N * C, bits + 0, st))) return rc;
      if ((rc = tc_absmax_bits(centers, (long long)K * C, bits + 1, st))) return rc;
      if ((rc = tc_absmax_bits(feature, (long long)N * C, bits + 2, st))) return rc;
      if ((rc = tc_cluster_bwd_scales(bits, 0, sc, st))) return rc;
      if ((rc = tc_split2h(centers, K, C, sc + 1, cs, st))) return rc;
      if (gR) {
        if ((rc = tc_split2h(gR, N, C, sc + 0, gRs, st))) return rc;
        if (K >= 128) {   // operands swapped: rows = centroids, coalesced stores
          if ((rc = launch_tc_gemm_h2<false>(cs, gRs, K, N, C, sc + 5, TcStoreTEpi{gemm, K}, st))) return rc;
        } else if ((rc = launch_tc_gemm_h2<false>(gRs, cs, N, K, C, sc + 5, TcStoreEpi{gemm, K}, st))) return rc;
      }
      // (max |r| for the fp16 scale of r comes out of the row pass itself)
      if ((rc = launch_bwd_rows(D, A, gR ? gemm : nullptr, gD, gA, g_loss_sq, N, K, alpha, r, rsum, st, bits + 3))) return rc;
      if ((rc = tc_cluster_bwd_scales(bits, 1, sc, st))) return rc;
      if ((rc = tc_split2h(r, N, K, sc + 4, rs, st))) return rc;
      if (C >= 128) {   // rows = channels: coalesced loads of feature / gF and stores of gz
        if ((rc = launch_tc_gemm_ex_h2<true, false>(cs, rs, C, N, K, 1, sc + 7, TcGzTEpi{gz, feature, rsum, gF, C}, st))) return rc;
      } else if ((rc = launch_tc_gemm_h2<true>(rs, cs, N, C, K, sc + 7, TcGzEpi{gz, feature, rsum, gF, C}, st))) return rc;
      if (gR) {
        if ((rc = tc_split2h(A, N, K, sc + 3, as, st))) return rc;
        if ((rc = launch_tc_gemm_ex_h2<true, true>(as, gRs, K, C, N, sk, sc + 6, TcPartialEpi{q1, C, KC}, st))) return rc;
      }
      if ((rc = tc_split2h(feature, N, C, sc + 2, fs, st))) return rc;
      if ((rc = launch_tc_gemm_ex_h2<true, true>(rs, fs, K, C, N, sk, sc + 8, TcPartialEpi{q2, C, KC}, st))) return rc;
      cudaError_t e2 = launch_colsum(r, N, K, cpart, rcol, st);
      if (e2 != cudaSuccess) return record_cuda_error(e2, "colsum r");
      gcenters_finalize_kernel<<<(unsigned)((KC + 255) / 256), 256, 0, st>>>(gR ? q1 : nullptr, q2, sk, centers, rcol, K, C, gcenters);
      VADC_CHECK_LAUNCH("gcenters_finalize_kernel");
      return launch_ln_bwd(gz, x, mu, rstd, ln_w, N, C, gx, lnpart, g_ln_w, g_ln_b, st);
    }
    if ((rc = tc_split3(centers, K, C, cs, st))) return rc;
    if (gR) {
      if ((rc = tc_split3(gR, N, C, gRs, st))) return rc;
      if ((rc = launch_tc_gemm<false>(gRs, cs, N, K, C, TcStoreEpi{gemm, K}, st))) return rc;
    }
    if ((rc = launch_bwd_rows(D, A, gR ? gemm : nullptr, gD, gA, g_loss_sq, N, K, alpha, r, rsum, st))) return rc;
    if ((rc = tc_split3(r, N, K, rs, st))) return rc;
    if ((rc = launch_tc_gemm<true>(rs, cs, N, C, K, TcGzEpi{gz, feature, rsum, gF, C}, st))) return rc;
    if (gR) {
      if ((rc = tc_split3(A, N, K, as, st))) return rc;
      if ((rc = launch_tc_gemm_ex<true, true>(as, gRs, K, C, N, sk, TcPartialEpi{q1, C, KC}, st))) return rc;
    }
    if ((rc = tc_split3(feature, N, C, fs, st))) return rc;
    if ((rc = launch_tc_gemm_ex<true, true>(rs, fs, K, C, N, sk, TcPartialEpi{q2, C, KC}, st))) return rc;
    cudaError_t e2 = launch_colsum(r, N, K, cpart, rcol, st);
    if (e2 != cudaSuccess) return record_cuda_error(e2, "colsum r");
    gcenters_finalize_kernel<<<(unsigned)((KC + 255) / 256), 256, 0, st>>>(gR ? q1 : nullptr, q2, sk, centers, rcol, K, C, gcenters);
    VADC_CHECK_LAUNCH("gcenters_finalize_kernel");
    return launch_ln_bwd(gz, x, mu, rstd, ln_w, N, C, gx, lnpart, g_ln_w, g_ln_b, st);
  }
  cudaError_t e;
  int rc;
  // (1) gR . centers^T  -> gemm [N,K]
  if (gR) {
    Operand Aop{gR, C, 1}, Bop{centers, 1, C};
    StoreEpilogue epi{gemm, K};
    e = sgemm_auto((int)N, K, C, Aop, Bop, 0, 0, 1, 1, epi, st);
    if (e != cudaSuccess) return record_cuda_error(e, "bwd sgemm gR.cT");
  }
  // (2) softmin backward + cdist ratio
  if ((rc = launch_bwd_rows(D, A, gR ? gemm : nullptr, gD, gA, g_loss_sq, N, K, alpha, r, rsum, st))) return rc;
  // (3) gz = feature * rsum - r @ centers + gF
  {
    Operand Aop{r, K, 1}, Bop{centers, C, 1};
    GzEpilogue epi{gz, feature, rsum, gF, C};
    e = sgemm_auto((int)N, C, K, Aop, Bop, 0, 0, 1, 1, epi, st);
    if (e != cudaSuccess) return record_cuda_error(e, "bwd sgemm r.c");
  }
  // (4) gcenters = A^T gR - r^T feature + centers * colsum(r)   (split over tokens)
  {
    PartialEpilogue e1{p1, C, KC}, e2{p2, C, KC};
    if (gR) {
      Operand Aop{A, 1, K}, Bop{gR, C, 1};
      e = launch_sgemm<64, 64>(K, C, (int)N, Aop, Bop, 0, 0, 1, splits, e1, st);
      if (e != cudaSuccess) return record_cuda_error(e, "bwd sgemm AT.gR");
    }
    Operand Aop{r, 1, K}, Bop{feature, C, 1};
    e = launch_sgemm<64, 64>(K, C, (int)N, Aop, Bop, 0, 0, 1, splits, e2, st);
    if (e != cudaSuccess) return record_cuda_error(e, "bwd sgemm rT.z");
    e = launch_colsum(r, N, K, cpart, rcol, st);
    if (e != cudaSuccess) return record_cuda_error(e, "colsum r");
    gcenters_finalize_kernel<<<(unsigned)((KC + 255) / 256), 256, 0, st>>>(gR ? p1 : nullptr, p2, splits, centers, rcol, K, C, gcenters);
    VADC_CHECK_LAUNCH("gcenters_finalize_kernel");
  }
  // (5) LayerNorm backward
  return launch_ln_bwd(gz, x, mu, rstd, ln_w, N, C, gx, lnpart, g_ln_w, g_ln_b, st);
}

// ---------------------------------------------------------------------------
// stand-alone PosSoftAssign / NegSoftAssign (model/cluster.py:27-55) over the
// last axis of a [rows, K] matrix, any K; one warp per row.
// y = exp(a (x - ext)) / sum, ext = max x for a > 0 and min x for a < 0.
// ---------------------------------------------------------------------------
namespace vadc {
__global__ void __launch_bounds__(256)
soft_assign_kernel(const float* __restrict__ x, long long rows, int K, float a, float* __restrict__ y) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= rows) return;
  const float* xr = x + row * K;
  float ext = (a >= 0.f) ? -INFINITY : INFINITY;
  for (int i = lane; i < K; i += 32) ext = (a >= 0.f) ? fmaxf(ext, xr[i]) : fminf(ext, xr[i]);
  ext = (a >= 0.f) ? warp_max(ext) : warp_min(ext);
  float s = 0.f;
  for (int i = lane; i < K; i += 32) s += expf(a * (xr[i] - ext));
  s = warp_sum(s);
  for (int i = lane; i < K; i += 32) y[row * K + i] = expf(a * (xr[i] - ext)) / s;
}

// gx = a * y * (g - sum_k g*y)
__global__ void __launch_bounds__(256)
soft_assign_bwd_kernel(const float* __restrict__ y, const float* __restrict__ g, long long rows,
                       int K, float a, float* __restrict__ gx) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= rows) return;
  float dot = 0.f;
  for (int i = lane; i < K; i += 32) dot += y[row * K + i] * g[row * K + i];
  dot = warp_sum(dot);
  for (int i = lane; i < K; i += 32) gx[row * K + i] = a * y[row * K + i] * (g[row * K + i] - dot);
}
}  // namespace vadc

extern "C" int vadc_soft_assign(const float* x, int64_t rows, int K, float signed_alpha, float* y,
                                void* stream) {
  VADC_REQUIRE(rows >= 0 && K > 0, VADC_ERR_BAD_SHAPE);
  if (rows == 0) return VADC_OK;
  VADC_REQUIRE(x && y, VADC_ERR_NULL_POINTER);
  soft_assign_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, rows, K, signed_alpha, y);
  VADC_CHECK_LAUNCH("soft_assign_kernel");
  return VADC_OK;
}

extern "C" int vadc_soft_assign_bwd(const float* y, const float* g, int64_t rows, int K,
                                    float signed_alpha, float* gx, void* stream) {
  VADC_REQUIRE(rows >= 0 && K > 0, VADC_ERR_BAD_SHAPE);
  if (rows == 0) return VADC_OK;
  VADC_REQUIRE(y && g && gx, VADC_ERR_NULL_POINTER);
  soft_assign_bwd_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(y, g, rows, K, signed_alpha, gx);
  VADC_CHECK_LAUNCH("soft_assign_bwd_kernel");
  return VADC_OK;
}
