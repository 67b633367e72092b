// cluster.h — internal launch helpers shared between translation units.
#pragma once
#include "common.cuh"

namespace vadc {
int launch_ln_rows(const float* x, const float* w, const float* b, long long N, int C, float eps,
                   float* z, float* mu, float* rstd, float* zz, cudaStream_t st,
                   float* rowstats = nullptr, void* split3 = nullptr,    // optional fused outputs (rows.cuh)
                   const float* hscale = nullptr);                       // split3 then holds two fp16 terms of z * hscale[0]
int launch_row_sqnorm(const float* a, long long R, int C, float* out, cudaStream_t st);
int softmin_blocks(long long R, int K);
int launch_softmin_rows(const float* D, long long R, int K, float alpha, float* A, long long* label,
                        double* partial, float* loss_sq, cudaStream_t st, int k_valid = -1,
                        void* terms_h2 = nullptr, float sa = 0.f);     // optional: two fp16 terms of A * sa, [2][R*K]
int launch_bwd_rows(const float* D, const float* A, const float* gemm, const float* gD,
                    const float* gA, const float* g_loss_sq, long long R, int K,
                    float alpha, float* r, float* rsum, cudaStream_t st,
                    unsigned* absmax_bits = nullptr);     // optional: max |r| as float bits (zeroed here, atomicMax per block)
int ln_bwd_blocks(long long N);
int launch_ln_bwd(const float* gz, const float* x, const float* mu, const float* rstd,
                  const float* w, long long N, int C, float* gx, float* partial, float* gw,
                  float* gb, cudaStream_t st);
int launch_dist(const float* a, const float* b, const float* aa, const float* bb, int nb,
                long long R, long long P, int C, float* out, cudaStream_t st);
int split_count(long long Ntok, int tiles);
// gcenters[c,k,p] = centers[c,k,p] * rcol[c,k] - acc   (SIMT epilogue of the space head and the batched cdist backward)
struct SpaceGcEpilogue {
  float* out; const float* centers; const float* rcol; long long KP; int P, K;
  __device__ __forceinline__ void operator()(int batch, int, int m, int n, float v) const {
    long long i = (long long)batch * KP + (long long)m * P + n;
    out[i] = centers[i] * rcol[(long long)batch * K + m] - v;
  }
};
// fused small-K backward (cluster_bwd_fused.cu)
bool bwd_fused_shape_ok(long long N, int C, int K);
size_t bwd_fused_workspace_bytes(long long N, int C, int K);
int launch_cluster_bwd_fused(const float* x, const float* mu, const float* rstd, const float* feature,
                             const float* ln_w, const float* centers, const float* D, const float* A,
                             const float* gD, const float* gA, const float* gR, const float* gF,
                             const float* g_loss_sq, long long N, int C, int K, float alpha, float* gx,
                             float* gcenters, float* g_ln_w, float* g_ln_b, void* workspace,
                             size_t workspace_bytes, cudaStream_t st);
// tcgen05 warp-specialised backward, K == 32, training-graph case (cluster_bwd_tc2.cu): x through TMA into the epilogue
// warps, gR through register sets of the producer warps
bool bwd_tc2_shape_ok(long long N, int C, int K);
size_t bwd_tc2_workspace_bytes(long long N, int C, int K);
int launch_cluster_bwd_tc2(const float* x, const float* mu, const float* rstd, const float* rowstats, const float* ln_w,
                           const float* ln_b, const float* centers, const float* D, const float* A,
                           const float* gR, const float* g_loss_sq, long long N, int C, int K, float alpha,
                           float* gx, float* gcenters, float* g_ln_w, float* g_ln_b, void* workspace,
                           size_t workspace_bytes, cudaStream_t st);
}  // namespace vadc

// tcgen05 path (cluster_tc.cu)
extern "C" size_t vadc_cluster_tc_extra_workspace_bytes(int64_t N, int C, int K);
int vadc_cluster_fwd_tc(const float* x, const float* ln_w, const float* ln_b, const float* centers,
                        int64_t N, int C, int K, float alpha, float eps, float* D, float* A,
                        float* x_rec, float* feature, int64_t* label, float* mu, float* rstd,
                        float* loss_sq, void* workspace, size_t workspace_bytes, cudaStream_t st);
// warp-specialised tcgen05 path, K == 32 (cluster_fwd_ws.cu)
size_t vadc_cluster_ws_extra_workspace_bytes(int64_t N, int C, int K);
int vadc_cluster_fwd_ws(const float* x, const float* ln_w, const float* ln_b, const float* centers,
                        int64_t N, int C, int K, float alpha, float eps, float* D, float* A,
                        float* x_rec, float* feature, int64_t* label, float* mu, float* rstd,
                        float* rowstats, float* loss_sq, void* workspace, size_t workspace_bytes, cudaStream_t st);
