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

// gz = feature * rsum - acc + gF   (batch z: out / feature / gF batch_out, rsum batch_rsum further)
struct GzEpilogue {
  float* out; const float* feature; const float* rsum; const float* gF; long long ld;
  long long batch_out = 0, batch_rsum = 0;
  __device__ __forceinline__ void operator()(int batch, int, int m, int n, float v) const {
    long long i = batch * batch_out + (long long)m * ld + n;
    float o = feature[i] * rsum[batch * batch_rsum + m] - v;
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
  if (ln_any_width(C)) {
    if (C > 4096) return VADC_ERR_UNSUPPORTED;
#define LA_CASE(E, WPR)                                                                                      \
  ln_rows_any_kernel<E, WPR><<<(unsigned)((N + 8 / WPR - 1) / (8 / WPR)), 256, 0, st>>>(                     \
      x, w, b, N, C, eps, z, mu, rstd, zz, rowstats, static_cast<__nv_bfloat16*>(split3), hscale, tc_pitch(C))
    if (C <= 128) LA_CASE(4, 1);
    else if (C <= 256) LA_CASE(8, 1);
    else if (C <= 512) LA_CASE(16, 1);
    else if (C <= 1024) LA_CASE(16, 2);
    else if (C <= 2048) LA_CASE(16, 4);
    else LA_CASE(16, 8);
#undef LA_CASE
    VADC_CHECK_LAUNCH("ln_rows_any_kernel");
    return VADC_OK;
  }
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
  if (ln_any_width(C)) {
    if (C > 4096) return VADC_ERR_UNSUPPORTED;
#define LA_CASE(E, WPR) ln_bwd_any_kernel<E, WPR><<<nb, 256, 0, st>>>(gz, x, mu, rstd, w, N, C, gx, partial)
    if (C <= 128) LA_CASE(4, 1);
    else if (C <= 256) LA_CASE(8, 1);
    else if (C <= 512) LA_CASE(16, 1);
    else if (C <= 1024) LA_CASE(16, 2);
    else if (C <= 2048) LA_CASE(16, 4);
    else LA_CASE(16, 8);
#undef LA_CASE
    VADC_CHECK_LAUNCH("ln_bwd_any_kernel");
    ln_bwd_finalize_kernel<<<(2 * C + 31) / 32, 256, 0, st>>>(partial, nb, C, gw, gb);
    VADC_CHECK_LAUNCH("ln_bwd_finalize_kernel");
    return VADC_OK;
  }
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
    b += tc_terms_bytes(3, N, tc_pitch(C)) + tc_terms_bytes(3, K, tc_pitch(C)) + tc_terms_bytes(3, N, K) + 256;
  return b + 256;
}

// the generic forward's two contractions on the tcgen05 GEMM.  TERMS = 3: bf16 x3 (fp32-faithful).  TERMS = 2: every
// operand is bounded (LayerNorm output, centroids, softmin weights in [0, 1]), so two fp16 terms after a power-of-two
// scaling carry 22 significant bits (the fused K = 32 kernel's recipe): 2/3 of the operand bytes and half the MMAs; the
// scales stay in device memory (no host sync).  The [., C] operands' terms have row pitch Cp = tc_pitch(C) (C rounded up to
// 8 for the any-width shapes, zero padding): the contractions over C run over Cp, the x_rec GEMM's C dimension reads the
// centroid terms at pitch Cp and its epilogue stops at C.
template <int TERMS>
static int cluster_fwd_tc(const float* x, const float* ln_w, const float* ln_b, const float* centers, int64_t N, int C,
                          int K, int k_valid, float alpha, float eps, float* D, float* A, float* x_rec, float* feature,
                          int64_t* label, float* mu, float* rstd, float* rowstats, float* loss_sq, float* zz, float* cc,
                          double* partial, Carver& ws, cudaStream_t st) {
  const long long Cp = tc_pitch(C);
  void* fs = ws.take<uint8_t>(tc_terms_bytes(TERMS, N, Cp));
  void* cs = ws.take<uint8_t>(tc_terms_bytes(TERMS, K, Cp));
  void* as = ws.take<uint8_t>(tc_terms_bytes(TERMS, N, K));
  float* sc = nullptr;
  int rc;
  if constexpr (TERMS == 2) {
    sc = ws.take<float>(8);
    if ((rc = tc_fwd_scales(centers, ln_w, ln_b, (long long)K * C, C, sc, st))) return rc;
  }
  if ((rc = launch_ln_rows(x, ln_w, ln_b, N, C, eps, feature, mu, rstd, zz, st, rowstats, fs, sc))) return rc;
  if ((rc = launch_row_sqnorm(centers, K, C, cc, st))) return rc;
  if ((rc = tc_split<TERMS>(centers, K, C, sc ? sc + 1 : nullptr, cs, st, Cp))) return rc;
  const float* sc2 = sc ? sc + 2 : nullptr;
  if constexpr (TERMS == 2) {
    // fp16 x2 only: from K = 128 up the distance GEMM runs with the operands swapped (rows = centroids): coalesced stores of D
    if (K >= 128) {
      if ((rc = tc_gemm<2, false, false>({cs, fs, K, N, Cp, sc2}, TcDistTEpi{D, cc, zz, K}, st))) return rc;
    } else if ((rc = tc_gemm<2, false, false>({fs, cs, N, K, Cp, sc2}, TcDistEpi{D, zz, cc, K}, st))) return rc;
    // softmin writes A and, in the same pass, its two fp16 terms scaled by s_a = 2^13 (the value fwd_scales_kernel puts in sc[3])
    if ((rc = launch_softmin_rows(D, N, K, alpha, A, (long long*)label, partial, loss_sq, st, k_valid, as, 8192.0f))) return rc;
    if (C >= 128)   // rows = channels (centers [K,C] as the MN-major A operand): coalesced x_rec
      return tc_gemm<2, true, false>({cs, as, C, N, K, sc + 4, 1, 1, {0, 0, 0, 0}, K, Cp}, TcStoreTEpi{x_rec, C}, st);
  } else {
    if ((rc = tc_gemm<3, false, false>({fs, cs, N, K, Cp}, TcDistEpi{D, zz, cc, K}, st))) return rc;
    if ((rc = launch_softmin_rows(D, N, K, alpha, A, (long long*)label, partial, loss_sq, st, k_valid))) return rc;
    if ((rc = tc_split<3>(A, N, K, nullptr, as, st))) return rc;
  }
  return tc_gemm<TERMS, false, true>({as, cs, N, C, K, sc ? sc + 4 : nullptr, 1, 1, {0, 0, 0, 0}, 0, 0, K, Cp},
                                     TcStoreEpi{x_rec, C}, st);    // centers [K,C] read MN-major
}

static int cluster_fwd_impl(const float* x, const float* ln_w, const float* ln_b,
                            const float* centers, int64_t N, int C, int K, int k_valid, float alpha,
                            float eps, float* D, float* A, float* x_rec, float* feature,
                            int64_t* label, float* mu, float* rstd, float* rowstats, float* loss_sq,
                            void* workspace, size_t workspace_bytes, int impl, void* stream) {
  VADC_REQUIRE(N >= 0 && C > 0 && K > 0 && (K % 4) == 0, VADC_ERR_BAD_SHAPE);
  VADC_REQUIRE(N < (1ll << 31) && C <= 4096, VADC_ERR_UNSUPPORTED);
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
  // stay row kernels.  Any-width C (C % 4 != 0, C > 1024) contracts over its padded pitch tc_pitch(C).
  const int Cp = tc_pitch(C);
  const bool use_tc = impl != VADC_IMPL_SIMT && N > 0 && !env_on("VADC_NO_TC_GEMM") &&
                      tc_gemm_shape_ok(N, K, Cp, false) && tc_gemm_shape_ok(N, Cp, K, true);
  if (use_tc)
    return env_on("VADC_TC_BF16X3")
               ? cluster_fwd_tc<3>(x, ln_w, ln_b, centers, N, C, K, k_valid, alpha, eps, D, A, x_rec, feature, label, mu,
                                   rstd, rowstats, loss_sq, zz, cc, partial, ws, st)
               : cluster_fwd_tc<2>(x, ln_w, ln_b, centers, N, C, K, k_valid, alpha, eps, D, A, x_rec, feature, label, mu,
                                   rstd, rowstats, loss_sq, zz, cc, partial, ws, st);
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
    b += tc_terms_bytes(3, (long long)nb * R, C) + tc_terms_bytes(3, (long long)nb * P, C);
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
    void* as = ws.take<uint8_t>(tc_terms_bytes(3, (long long)nb * R, C));
    void* bs = self ? as : ws.take<uint8_t>(tc_terms_bytes(3, (long long)nb * P, C));
    if ((rc = tc_split<3>(a, (long long)nb * R, C, nullptr, as, st))) return rc;
    if (!self && (rc = tc_split<3>(b, (long long)nb * P, C, nullptr, bs, st))) return rc;
    TcBatchDistEpi epi{out, aa, bb, P, R * P, R, P};
    return tc_gemm<3, false, false>({as, bs, R, P, C, nullptr, 1, nb, {(int)R, 0, (int)P, 0}, (long long)nb * R, C, (long long)nb * P, C},
                                    epi, st);
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

namespace vadc {
// the generic backward's five contractions on the tcgen05 GEMM: G1 = gR c^T; gz = z rsum - r c + gF;
// gcenters = A^T gR - r^T z + c colsum(r) with the token matrices read MN-major and split-K over the tokens.
// TERMS = 2: two fp16 terms per operand, each scaled by the power of two of its measured bound (A: 2^13): 22 significant
// bits, 2/3 of the operand bytes and half the MMAs of the bf16 x3 split (TERMS = 3)
template <int TERMS>
static int cluster_bwd_tc(const float* x, const float* mu, const float* rstd, const float* feature, const float* ln_w,
                          const float* centers, const float* D, const float* A, const float* gD, const float* gA,
                          const float* gR, const float* gF, const float* g_loss_sq, int64_t N, int C, int K, float alpha,
                          float* gx, float* gcenters, float* g_ln_w, float* g_ln_b, float* gemm, float* r, float* rsum,
                          float* gz, float* cpart, float* rcol, float* lnpart, Carver& ws, cudaStream_t st) {
  const long long KC = (long long)K * C, Cp = tc_pitch(C);     // terms of gR, feature, centers at row pitch Cp
  const int sk = bwd_tc_splits(N, C, K);
  void* gRs = ws.take<uint8_t>(tc_terms_bytes(3, N, Cp));
  void* fs = ws.take<uint8_t>(tc_terms_bytes(3, N, Cp));
  void* as = ws.take<uint8_t>(tc_terms_bytes(3, N, K));
  void* rs = ws.take<uint8_t>(tc_terms_bytes(3, N, K));
  void* cs = ws.take<uint8_t>(tc_terms_bytes(3, K, Cp));
  float* q1 = ws.take<float>((size_t)sk * KC);
  float* q2 = ws.take<float>((size_t)sk * KC);
  unsigned* bits = nullptr;
  float* sc = nullptr;
  // the scales' slots (tc_cluster_bwd_scales): inputs s_g, s_c, s_f, s_a, s_r; accumulators 1/(s_g s_c), 1/(s_a s_g),
  // 1/(s_r s_c), 1/(s_r s_f) — all NULL in bf16 x3
  auto at = [&](int i) -> const float* { return sc ? sc + i : nullptr; };
  int rc;
  if constexpr (TERMS == 2) {
    bits = ws.take<unsigned>(64);
    sc = ws.take<float>(64);
    VADC_CUDA(cudaMemsetAsync(bits, 0, 4 * sizeof(unsigned), st));
    if (gR && (rc = tc_absmax_bits(gR, (long long)N * C, bits + 0, st))) return rc;
    if ((rc = tc_absmax_bits(centers, (long long)K * C, bits + 1, st))) return rc;
    if ((rc = tc_absmax_bits(feature, (long long)N * C, bits + 2, st))) return rc;
    if ((rc = tc_cluster_bwd_scales(bits, 0, sc, st))) return rc;
  }
  if ((rc = tc_split<TERMS>(centers, K, C, at(1), cs, st, Cp))) return rc;
  if (gR) {
    if ((rc = tc_split<TERMS>(gR, N, C, at(0), gRs, st, Cp))) return rc;
    // fp16 x2 only: from K = 128 up the operands are swapped (rows = centroids): coalesced stores
    if constexpr (TERMS == 2) {
      if (K >= 128) rc = tc_gemm<2, false, false>({cs, gRs, K, N, Cp, at(5)}, TcStoreTEpi{gemm, K}, st);
      else rc = tc_gemm<2, false, false>({gRs, cs, N, K, Cp, at(5)}, TcStoreEpi{gemm, K}, st);
    } else {
      rc = tc_gemm<3, false, false>({gRs, cs, N, K, Cp}, TcStoreEpi{gemm, K}, st);
    }
    if (rc) return rc;
  }
  // (fp16 x2: max |r| for the scale of r comes out of the row pass itself)
  if ((rc = launch_bwd_rows(D, A, gR ? gemm : nullptr, gD, gA, g_loss_sq, N, K, alpha, r, rsum, st, bits ? bits + 3 : nullptr)))
    return rc;
  if constexpr (TERMS == 2)
    if ((rc = tc_cluster_bwd_scales(bits, 1, sc, st))) return rc;
  if ((rc = tc_split<TERMS>(r, N, K, at(4), rs, st))) return rc;
  // fp16 x2 only: from C = 128 up rows = channels, coalesced loads of feature / gF and stores of gz
  if constexpr (TERMS == 2) {
    if (C >= 128)
      rc = tc_gemm<2, true, false>({cs, rs, C, N, K, at(7), 1, 1, {0, 0, 0, 0}, K, Cp}, TcGzTEpi{gz, feature, rsum, gF, C}, st);
    else
      rc = tc_gemm<2, false, true>({rs, cs, N, C, K, at(7), 1, 1, {0, 0, 0, 0}, 0, 0, K, Cp}, TcGzEpi{gz, feature, rsum, gF, C}, st);
  } else {
    rc = tc_gemm<3, false, true>({rs, cs, N, C, K, nullptr, 1, 1, {0, 0, 0, 0}, 0, 0, K, Cp}, TcGzEpi{gz, feature, rsum, gF, C}, st);
  }
  if (rc) return rc;
  if (gR) {
    if ((rc = tc_split<TERMS>(A, N, K, at(3), as, st))) return rc;
    if ((rc = tc_gemm<TERMS, true, true>({as, gRs, K, C, N, at(6), sk, 1, {0, 0, 0, 0}, 0, 0, N, Cp}, TcPartialEpi{q1, C, KC}, st)))
      return rc;
  }
  if ((rc = tc_split<TERMS>(feature, N, C, at(2), fs, st, Cp))) return rc;
  if ((rc = tc_gemm<TERMS, true, true>({rs, fs, K, C, N, at(8), sk, 1, {0, 0, 0, 0}, 0, 0, N, Cp}, TcPartialEpi{q2, C, KC}, st)))
    return rc;
  cudaError_t e2 = launch_colsum(r, N, K, cpart, rcol, st);
  if (e2 != cudaSuccess) return record_cuda_error(e2, "colsum r");
  gcenters_finalize_kernel<<<(unsigned)((KC + 255) / 256), 256, 0, st>>>(gR ? q1 : nullptr, q2, sk, centers, rcol, K, C, gcenters);
  VADC_CHECK_LAUNCH("gcenters_finalize_kernel");
  return launch_ln_bwd(gz, x, mu, rstd, ln_w, N, C, gx, lnpart, g_ln_w, g_ln_b, st);
}
}  // namespace vadc

namespace vadc {
// split-K partials of the backward: [splits, K, C] for each of the two centroid-gradient contractions, SIMT and tcgen05.
// The slot count falls as C adds tiles, so for the any-width shapes this is the maximum over every width up to C (the
// product is largest at the end of a 64-wide tile band): a workspace sized for one head also serves every narrower one.
static size_t bwd_partial_bytes(long long N, int C, int K) {
  auto at = [&](int c) {
    const int tiles = ((K + 63) / 64) * ((c + 63) / 64);
    return 2 * align_up((size_t)split_count(N, tiles) * K * c * sizeof(float), 256) +
           2 * align_up((size_t)bwd_tc_splits(N, c, K) * K * c * sizeof(float), 256);
  };
  size_t b = at(C);
  if (ln_any_width(C))
    for (int c = 64; c < C; c += 64) b = std::max(b, at(c));
  return b;
}
}  // namespace vadc

extern "C" size_t vadc_cluster_bwd_workspace_bytes(int64_t N, int C, int K) {
  size_t n = (size_t)(N > 0 ? N : 1);
  size_t b = 0;
  b += align_up(n * K * sizeof(float), 256);                 // gR.c^T
  b += align_up(n * K * sizeof(float), 256);                 // r
  b += align_up(n * sizeof(float), 256);                     // rsum
  b += align_up(n * C * sizeof(float), 256);                 // gz
  b += align_up((size_t)colsum_chunks(N) * K * sizeof(float), 256); // colsum partial
  b += align_up((size_t)K * sizeof(float), 256);             // rcol
  b += align_up((size_t)ln_bwd_blocks(N) * 2 * C * sizeof(float), 256);
  // generic path on the tcgen05 GEMM: bf16 term copies of gR, feature, A, r and the centroids + split-K partials
  b += 2 * tc_terms_bytes(3, (long long)n, tc_pitch(C)) + 2 * tc_terms_bytes(3, (long long)n, K) + tc_terms_bytes(3, K, tc_pitch(C)) + 1024;
  b += bwd_partial_bytes(N, C, K);                           // split-K partials
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
  VADC_REQUIRE(N >= 0 && C > 0 && K > 0 && (K % 4) == 0, VADC_ERR_BAD_SHAPE);
  VADC_REQUIRE(N < (1ll << 31) && C <= 4096, VADC_ERR_UNSUPPORTED);
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
  // any-width C (C % 4 != 0, C > 1024) contracts over its padded pitch tc_pitch(C); C % 8 == 4 up to 1024 stays SIMT
  if (!env_on("VADC_NO_TC_GEMM") && vadc_device_ok() && (K % 8) == 0 && K >= 8 &&
      (((C % 8) == 0 && C >= 8) || ln_any_width(C))) {
    return env_on("VADC_TC_BF16X3")
               ? cluster_bwd_tc<3>(x, mu, rstd, feature, ln_w, centers, D, A, gD, gA, gR, gF, g_loss_sq, N, C, K, alpha,
                                   gx, gcenters, g_ln_w, g_ln_b, gemm, r, rsum, gz, cpart, rcol, lnpart, ws, st)
               : cluster_bwd_tc<2>(x, mu, rstd, feature, ln_w, centers, D, A, gD, gA, gR, gF, g_loss_sq, N, C, K, alpha,
                                   gx, gcenters, g_ln_w, g_ln_b, gemm, r, rsum, gz, cpart, rcol, lnpart, ws, st);
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
// backward of the stand-alone batched cdist (ATen's _euclidean_dist_backward), per batch z:
//   r = g / D (0 where D == 0),  rho_a = rowsum(r),  rho_b = colsum(r)
//   ga = a rho_a - r b,  gb = b rho_b - r^T a
// self (cdist(c, c)): r + r^T with the diagonal zeroed, gc = c rowsum(r + r^T) - (r + r^T) c — one contraction.
// Both sums of r come out of the pass that writes r, as per-block partials reduced in a fixed order, rather than from
// launch_colsum / launch_space_colsum over r afterwards: that would read r (4 nb R P bytes, 256 MB for 65536 tokens
// against 1024 centroids) a second time, and launch_space_colsum sums the space head's [M, C K] layout (a batch = a
// K-column window), not [nb, R, P] (a batch = R rows).
// ---------------------------------------------------------------------------
namespace vadc {
// Ratio pass: one block = 32 S rows of one batch (blockIdx.z) by a range of `tpc` 32-wide column tiles (blockIdx.y;
// warp = rows, lanes = columns: coalesced).  Writes r (batch stride Rp P; rows R..Rp-1 zero, so that a contraction over
// a batch's rows never reaches the next batch), the row sums (to rho with one column range, else the range's partials
// rowpart[blockIdx.y, z R + i]), the block's column partials colpart[blockIdx.x, z P + j] (optional) and max |r| as
// float bits.  SYM (R == P): r + r^T, the transposed tile through shared memory; the diagonal is skipped — its exact
// contribution is r_ii (c_i - c_i) = 0, and the mm-form D_ii is fp32 cancellation noise, not 0.
template <bool SYM, int S>
__global__ void __launch_bounds__(256, 2)      // (256) alone left SYM at 64 registers and a spill
cdist_ratio_kernel(const float* __restrict__ g, const float* __restrict__ D, long long R, long long P, long long Rp,
                   int tpc, float* __restrict__ r, float* __restrict__ rho, float* __restrict__ rowpart,
                   float* __restrict__ colpart, unsigned* __restrict__ absmax_bits) {
  __shared__ float tile[32][33];
  __shared__ float csum[8][33];
  __shared__ float bmax[8];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const long long z = blockIdx.z, i0 = (long long)blockIdx.x * 32 * S, nbt = gridDim.z;
  const float* gz = g + z * R * P;
  const float* dz = D + z * R * P;
  float* rz = r + z * Rp * P;
  float rs[4 * S];
#pragma unroll
  for (int q = 0; q < 4 * S; ++q) rs[q] = 0.f;
  float amax = 0.f;
  const long long jend = min(P, (long long)(blockIdx.y + 1) * tpc * 32);
  for (long long j0 = (long long)blockIdx.y * tpc * 32; j0 < jend; j0 += 32) {
    const long long j = j0 + tx;
    float cs = 0.f;
#pragma unroll
    for (int s = 0; s < S; ++s) {
      const long long ib = i0 + 32 * s;
      if (SYM) {                  // tile[jj][ii] = ratio at (row j0 + jj, column ib + ii)
        float dv[4], gv[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const long long jr = j0 + ty + 8 * q, ic = ib + tx;
          const bool in = jr < P && ic < R;
          dv[q] = in ? dz[jr * P + ic] : 0.f;
          gv[q] = in ? gz[jr * P + ic] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < 4; ++q) tile[ty + 8 * q][tx] = dv[q] != 0.f ? gv[q] / dv[q] : 0.f;
        __syncthreads();
      }
      float dv[4], gv[4];         // every load of the tile issued before the first use
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const long long i = ib + ty + 8 * q;
        const bool in = i < R && j < P;
        dv[q] = in ? dz[i * P + j] : 0.f;
        gv[q] = in ? gz[i * P + j] : 0.f;
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int ii = ty + 8 * q;
        const long long i = ib + ii;
        float v = dv[q] != 0.f ? gv[q] / dv[q] : 0.f;
        if (SYM) v = i == j ? 0.f : v + tile[tx][ii];
        if (i < Rp && j < P) rz[i * P + j] = v;
        rs[4 * s + q] += v;
        cs += v;
        amax = fmaxf(amax, fabsf(v));
      }
    }
    if (colpart) {               // the block's column sums, fixed order (deterministic)
      csum[ty][tx] = cs;
      __syncthreads();
      if (ty == 0 && j < P) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) t += csum[w][tx];
        colpart[(long long)blockIdx.x * nbt * P + z * P + j] = t;
      }
      __syncthreads();
    }
  }
  float* rout = gridDim.y == 1 ? rho : rowpart + (long long)blockIdx.y * nbt * R;
#pragma unroll
  for (int s = 0; s < S; ++s)
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float t = warp_sum(rs[4 * s + q]);
      const long long i = i0 + 32 * s + ty + 8 * q;
      if (tx == 0 && i < R) rout[z * R + i] = t;
    }
  amax = warp_max(amax);
  if (tx == 0) bmax[ty] = amax;
  __syncthreads();
  if (threadIdx.x == 0) {
    float m = bmax[0];
#pragma unroll
    for (int w = 1; w < 8; ++w) m = fmaxf(m, bmax[w]);
    if (m > 0.f && isfinite(m)) atomicMax(absmax_bits, __float_as_uint(m));
  }
}

// out[w] = sum_c partial[c, w] over nchunks rows, fixed order: a block owns 32 columns, its eight warps take every
// eighth chunk.  (colsum_stage2_kernel runs one thread per column through all chunks: with the ratio pass's ~1000
// chunks of 1024 columns that is four blocks of 1000 dependent loads each; ln_bwd_finalize_kernel has this shape but
// writes two fixed outputs.)
__global__ void __launch_bounds__(256)
colsum_chunks_kernel(const float* __restrict__ partial, int nchunks, long long W, float* __restrict__ out) {
  __shared__ float red[8][33];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const long long w = (long long)blockIdx.x * 32 + lane;
  float s = 0.f;
  if (w < W)
    for (int c = wid; c < nchunks; c += 8) s += partial[(long long)c * W + w];
  red[wid][lane] = s;
  __syncthreads();
  if (wid == 0 && w < W) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += red[k][lane];
    out[w] = t;
  }
}

// rows of one batch of r: batches of a batched launch start on a k-block boundary of the contraction over the rows
static long long cdist_bwd_rows(int nb, long long R) { return nb > 1 ? (R + 63) / 64 * 64 : R; }
// rows per ratio-pass block / 32: tall blocks for many rows keep the column partials few
static int cdist_ratio_s(bool self, long long R) { return !self && R >= 1024 ? 2 : 1; }
static long long cdist_ratio_chunks(long long Rp, int S) { return (Rp + 32ll * S - 1) / (32ll * S); }
// column ranges of the ratio pass: ~1024 blocks in all (a [K, K] self-distance alone is K / 32 row strips)
static int cdist_ratio_colchunks(int nb, long long Rp, long long P, int S) {
  const long long tiles = (P + 31) / 32, blocks = cdist_ratio_chunks(Rp, S) * nb;
  return (int)std::max<long long>(1, std::min<long long>(tiles, (1024 + blocks - 1) / blocks));
}
static int cdist_ratio_colchunks_max(int nb, long long Rp, long long P) {
  return std::max(cdist_ratio_colchunks(nb, Rp, P, 1), cdist_ratio_colchunks(nb, Rp, P, 2));
}
// split-K slots of the one-problem gb contraction (over the R rows): the larger of the tensor-core and SIMT counts
static int cdist_bwd_sk_tc(long long R, long long P, int C) { return bwd_tc_splits(R, C, (int)P); }
static int cdist_bwd_sk_simt(long long R, long long P, int C) {
  return split_count(R, (int)(((P + 63) / 64) * ((C + 63) / 64)));
}

// the two contractions on the tcgen05 GEMM: tensor-bound sizes (the operand splits cost a pass each), TMA row pitches
// (C, P multiples of 8) and every launch's shape predicate
static bool cdist_bwd_tc_ok(int nb, long long R, long long P, int C, const float* a, const float* b) {
  const long long Rp = cdist_bwd_rows(nb, R);
  return !env_on("VADC_NO_TC_GEMM") && (C % 8) == 0 && (P % 8) == 0 && (long long)nb * Rp < (1ll << 31) &&
         (long long)nb * P < (1ll << 31) && (double)nb * R * P * C >= (double)(1ll << 24) && aligned16(a) && aligned16(b) &&
         tc_gemm_shape_ok(R, C, P, true) && tc_gemm_shape_ok(C, R, P, false) && tc_gemm_shape_ok(P, C, Rp, true);
}
}  // namespace vadc

extern "C" size_t vadc_cdist_bwd_workspace_bytes(int nb, int64_t R, int64_t P, int C) {
  if (nb < 0 || R < 0 || P < 0 || C <= 0) return 0;
  const size_t n = nb > 0 ? (size_t)nb : 1, r1 = R > 0 ? (size_t)R : 1, p1 = P > 0 ? (size_t)P : 1;
  const size_t Rp = (size_t)cdist_bwd_rows((int)n, (long long)r1);
  size_t b = 0;
  b += align_up(n * Rp * p1 * sizeof(float), 256);                                             // r
  b += align_up(n * r1 * sizeof(float), 256) + align_up(n * p1 * sizeof(float), 256);          // rho_a, rho_b
  b += align_up((size_t)cdist_ratio_colchunks_max((int)n, (long long)Rp, (long long)p1) * n * r1 * sizeof(float), 256);  // row partials
  b += align_up((size_t)cdist_ratio_chunks((long long)Rp, 1) * n * p1 * sizeof(float), 256);  // column partials
  b += 2 * 256;                                                                                  // max bits, scales
  if (n == 1)                                                                                    // split-K partials
    b += align_up((size_t)std::max(cdist_bwd_sk_tc(r1, p1, C), cdist_bwd_sk_simt(r1, p1, C)) * p1 * C * sizeof(float), 256);
  if ((C % 8) == 0 && (p1 % 8) == 0)                                                             // operand terms
    b += tc_terms_bytes(3, (long long)(n * Rp), p1) + tc_terms_bytes(3, (long long)(n * r1), C) +
         tc_terms_bytes(3, (long long)(n * p1), C);
  return b + 256;
}

namespace vadc {
// (2) of cdist_bwd_impl: ga = a rho_a - r b  and  gb = b rho_b - r^T a  on the tcgen05 GEMM.  r as [nb Rp, P], a as
//     [nb R, C], b as [nb P, C]; gb: contraction over the rows, split-K for one problem, one batched launch otherwise.
// TERMS = 2: two fp16 terms of power-of-two-scaled operands; r has no a-priori bound, its scale comes from the measured
// max: sc[0..2] = {s_r, s_b, 1 / (s_r s_b)} (ga; self: s_b = s_a), sc[4..6] = {s_r, s_a, 1 / (s_r s_a)} (gb); no host sync.
// TERMS = 3: three bf16 terms per operand (fp32-faithful for any data, no scales)
template <int TERMS>
static int cdist_bwd_tc(const float* a, const float* b, const float* r, const float* rho_a, const float* rho_b, float* q,
                        unsigned* bits, float* sc, int nb, long long R, long long P, int C, bool self, float* ga, float* gb,
                        Carver& ws, cudaStream_t st) {
  const long long Rp = cdist_bwd_rows(nb, R), PC = P * C;
  const float* bb = self ? a : b;              // self: the one contraction is the ga form with b = a
  const int sk = cdist_bwd_sk_tc(R, P, C);
  void* rs = ws.take<uint8_t>(tc_terms_bytes(3, (long long)nb * Rp, P));
  void* as = ws.take<uint8_t>(tc_terms_bytes(3, (long long)nb * R, C));
  void* bs = self ? as : ws.take<uint8_t>(tc_terms_bytes(3, (long long)nb * P, C));
  const TcBatchOffsets oga{0, (int)P, (int)Rp, 0}, ogb{0, (int)Rp, 0, (int)R};
  const TcGzEpi ega{ga, a, rho_a, nullptr, C};
  auto at = [&](int i) -> const float* { return TERMS == 2 ? sc + i : nullptr; };
  int rc;
  if constexpr (TERMS == 2) {
    if ((gb || self) && (rc = tc_absmax_bits(a, (long long)nb * R * C, bits + 1, st))) return rc;
    if (ga && !self && (rc = tc_absmax_bits(b, (long long)nb * P * C, bits + 2, st))) return rc;
    if (ga && (rc = tc_pair_scales(bits, 0.f, self ? bits + 1 : bits + 2, 0.f, sc, st))) return rc;
    if (gb && (rc = tc_pair_scales(bits, 0.f, bits + 1, 0.f, sc + 4, st))) return rc;
  }
  if ((rc = tc_split<TERMS>(r, (long long)nb * Rp, P, at(ga ? 0 : 4), rs, st))) return rc;
  // bf16 x3 splits a once for both contractions; fp16 x2 splits each operand with the scale of its contraction
  if constexpr (TERMS == 3)
    if ((gb || self) && (rc = tc_split<3>(a, (long long)nb * R, C, nullptr, as, st))) return rc;
  if (ga) {
    if ((TERMS == 2 || !self) && (rc = tc_split<TERMS>(bb, (long long)nb * P, C, at(1), bs, st))) return rc;
    if (nb > 1) {
      rc = tc_gemm<TERMS, true, false>({bs, rs, C, R, P, at(2), 1, nb, oga, (long long)nb * P, C, (long long)nb * Rp, P},
                                       TcCdistGaTEpi{ga, a, rho_a, R, C}, st);
    } else if constexpr (TERMS == 2) {   // fp16 x2 only: one problem with C >= 128 runs transposed (coalesced stores)
      rc = C >= 128 ? tc_gemm<2, true, false>({bs, rs, C, R, P, sc + 2}, TcGzTEpi{ga, a, rho_a, nullptr, C}, st)
                    : tc_gemm<2, false, true>({rs, bs, R, C, P, sc + 2}, ega, st);
    } else {
      rc = tc_gemm<3, false, true>({rs, bs, R, C, P}, ega, st);
    }
    if (rc) return rc;
  }
  if (gb) {
    if constexpr (TERMS == 2)
      if ((rc = tc_split<2>(a, (long long)nb * R, C, sc + 5, as, st))) return rc;
    if (nb > 1)
      return tc_gemm<TERMS, true, true>({rs, as, P, C, Rp, at(6), 1, nb, ogb, (long long)nb * Rp, P, (long long)nb * R, C},
                                        TcSpaceGcEpi{gb, b, rho_b, PC, C, (int)P}, st);
    if ((rc = tc_gemm<TERMS, true, true>({rs, as, P, C, R, at(6), sk}, TcPartialEpi{q, C, PC}, st))) return rc;
    // one problem: gb = b rho_b - sum of the split-K partials
    gcenters_finalize_kernel<<<(unsigned)((PC + 255) / 256), 256, 0, st>>>(nullptr, q, sk, b, rho_b, (int)P, C, gb);
    VADC_CHECK_LAUNCH("gcenters_finalize_kernel");
  }
  return VADC_OK;
}

static int cdist_bwd_impl(const float* a, const float* b, const float* dist, const float* g, int nb, long long R,
                          long long P, int C, bool self, float* ga, float* gb, void* workspace, size_t workspace_bytes,
                          cudaStream_t st) {
  const long long Rp = cdist_bwd_rows(nb, R), PC = P * C;
  const int S = cdist_ratio_s(self, R);
  const long long chunks = cdist_ratio_chunks(Rp, S);
  Carver ws(workspace, workspace_bytes);
  float* r = ws.take<float>((size_t)nb * Rp * P);
  float* rho_a = ws.take<float>((size_t)nb * R);
  float* rho_b = ws.take<float>((size_t)nb * P);
  float* colpart = ws.take<float>((size_t)cdist_ratio_chunks(Rp, 1) * nb * P);
  float* rowpart = ws.take<float>((size_t)cdist_ratio_colchunks_max(nb, Rp, P) * nb * R);
  unsigned* bits = ws.take<unsigned>(64);
  float* sc = ws.take<float>(64);
  float* q = nb == 1 ? ws.take<float>((size_t)std::max(cdist_bwd_sk_tc(R, P, C), cdist_bwd_sk_simt(R, P, C)) * PC) : nullptr;
  // (1) r, rho_a, max |r| in one pass over g and D; rho_b from the column partials
  VADC_CUDA(cudaMemsetAsync(bits, 0, 4 * sizeof(unsigned), st));
  float* cp = gb ? colpart : nullptr;
  const int cch = cdist_ratio_colchunks(nb, Rp, P, S), tpc = (int)(((P + 31) / 32 + cch - 1) / cch);
  const dim3 grid((unsigned)chunks, (unsigned)cch, (unsigned)nb);
  if (self) cdist_ratio_kernel<true, 1><<<grid, 256, 0, st>>>(g, dist, R, P, Rp, tpc, r, rho_a, rowpart, nullptr, bits);
  else if (S == 2) cdist_ratio_kernel<false, 2><<<grid, 256, 0, st>>>(g, dist, R, P, Rp, tpc, r, rho_a, rowpart, cp, bits);
  else cdist_ratio_kernel<false, 1><<<grid, 256, 0, st>>>(g, dist, R, P, Rp, tpc, r, rho_a, rowpart, cp, bits);
  VADC_CHECK_LAUNCH("cdist_ratio_kernel");
  if (cch > 1) {
    colsum_chunks_kernel<<<(unsigned)((nb * R + 31) / 32), 256, 0, st>>>(rowpart, cch, (long long)nb * R, rho_a);
    VADC_CHECK_LAUNCH("colsum_chunks_kernel");
  }
  if (gb) {
    colsum_chunks_kernel<<<(unsigned)((nb * P + 31) / 32), 256, 0, st>>>(colpart, (int)chunks, (long long)nb * P, rho_b);
    VADC_CHECK_LAUNCH("colsum_chunks_kernel");
  }
  const float* bb = self ? a : b;              // self: the one contraction is the ga form with b = a
  if (cdist_bwd_tc_ok(nb, R, P, C, a, bb))
    return env_on("VADC_TC_BF16X3")
               ? cdist_bwd_tc<3>(a, b, r, rho_a, rho_b, q, bits, sc, nb, R, P, C, self, ga, gb, ws, st)
               : cdist_bwd_tc<2>(a, b, r, rho_a, rho_b, q, bits, sc, nb, R, P, C, self, ga, gb, ws, st);
  // (2') fp32 SIMT GEMM: shapes the tensor-core path does not take, and launch-bound sizes
  cudaError_t e;
  if (ga) {
    Operand Aop{r, P, 1}, Bop{bb, C, 1};
    GzEpilogue epi{ga, a, rho_a, nullptr, C, R * C, R};
    e = sgemm_auto((int)R, C, (int)P, Aop, Bop, Rp * P, PC, nb, 1, epi, st);
    if (e != cudaSuccess) return record_cuda_error(e, "cdist bwd sgemm r.b");
  }
  if (gb) {
    Operand Aop{r, 1, P}, Bop{a, C, 1};
    if (nb > 1) {
      e = sgemm_auto((int)P, C, (int)R, Aop, Bop, Rp * P, R * C, nb, 1, SpaceGcEpilogue{gb, b, rho_b, PC, C, (int)P}, st);
      if (e != cudaSuccess) return record_cuda_error(e, "cdist bwd sgemm rT.a");
      return VADC_OK;
    }
    const int sks = cdist_bwd_sk_simt(R, P, C);
    e = launch_sgemm<64, 64>((int)P, C, (int)R, Aop, Bop, 0, 0, 1, sks, PartialEpilogue{q, C, PC}, st);
    if (e != cudaSuccess) return record_cuda_error(e, "cdist bwd sgemm rT.a");
    gcenters_finalize_kernel<<<(unsigned)((PC + 255) / 256), 256, 0, st>>>(nullptr, q, sks, b, rho_b, (int)P, C, gb);
    VADC_CHECK_LAUNCH("gcenters_finalize_kernel");
  }
  return VADC_OK;
}
}  // namespace vadc

extern "C" int vadc_cdist_bwd(const float* a, const float* b, const float* dist, const float* g, int nb, int64_t R, int64_t P,
                              int C, int self, float* ga, float* gb, void* workspace, size_t workspace_bytes, void* stream) {
  VADC_REQUIRE(nb >= 0 && R >= 0 && P >= 0 && C > 0, VADC_ERR_BAD_SHAPE);
  VADC_REQUIRE(!self || (gb == nullptr && R == P && (b == nullptr || b == a)), VADC_ERR_BAD_SHAPE);
  VADC_REQUIRE(nb <= 65535 && R < (1ll << 31) && P < (1ll << 31), VADC_ERR_UNSUPPORTED);
  if (!ga && !gb) return VADC_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (nb == 0 || R == 0 || P == 0) {           // empty distance matrix: zero gradients
    if (ga && (long long)nb * R > 0) VADC_CUDA(cudaMemsetAsync(ga, 0, (size_t)nb * R * C * sizeof(float), st));
    if (gb && (long long)nb * P > 0) VADC_CUDA(cudaMemsetAsync(gb, 0, (size_t)nb * P * C * sizeof(float), st));
    return VADC_OK;
  }
  VADC_REQUIRE(a && g && dist && workspace && (self || b), VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(workspace_bytes >= vadc_cdist_bwd_workspace_bytes(nb, R, P, C), VADC_ERR_WORKSPACE);
  return cdist_bwd_impl(a, self ? a : b, dist, g, nb, R, P, C, self != 0, ga, gb, workspace, workspace_bytes, st);
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
