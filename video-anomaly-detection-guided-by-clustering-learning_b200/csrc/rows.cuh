// rows.cuh — row-wise kernels shared by the cluster head, the space head and
// the memory module: LayerNorm rows, squared row norms, the softmin / argmin /
// loss row pass, the backward row pass, and deterministic column reductions.
#pragma once
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include "common.cuh"
#include "tc_terms.cuh"

namespace vadc {

// ---------------------------------------------------------------------------
// LayerNorm over the last axis, one warp per row (model/cluster.py:84,129).
// Two-pass statistics (mean, then variance about the mean) held in registers.
// Writes z (row-major), mu, rstd and optionally |z|^2 per row.
// VPL = float4 per lane (C <= 128*VPL).  C % 4 == 0.
// ---------------------------------------------------------------------------
template <int VPL>
__global__ void __launch_bounds__(256)
ln_rows_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ b,
               long long N, int C, float eps, float* __restrict__ z, float* __restrict__ mu,
               float* __restrict__ rstd, float* __restrict__ zz, float* __restrict__ rowstats,
               __nv_bfloat16* __restrict__ split, const float* __restrict__ hscale) {
  // optional fused outputs: rowstats [N,4] = {|z|^2, sum z gamma, sum z gamma xhat, 0} (what the tcgen05 backward
  // uses) and the three bf16 terms of z ([3][N,C], the tcgen05 GEMM's A operand) - saves two more passes over z;
  // with hscale the split is two fp16 terms of z * hscale[0] instead ([2][N,C]: tc_gemm's two-term mode)
  const float hs = hscale ? __ldg(hscale) : 1.0f;
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= N) return;
  const int nv = C >> 2;
  const float4* xr = reinterpret_cast<const float4*>(x + row * C);
  float4 v[VPL];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    int c4 = lane + 32 * i;
    v[i] = (c4 < nv) ? ld_stream(xr + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
    s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  }
  const float mean = warp_sum(s) / (float)C;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    int c4 = lane + 32 * i;
    if (c4 < nv) {
      float a = v[i].x - mean, b2 = v[i].y - mean, c2 = v[i].z - mean, d = v[i].w - mean;
      q += (a * a + b2 * b2) + (c2 * c2 + d * d);
    }
  }
  const float var = warp_sum(q) / (float)C;
  const float rs = 1.0f / sqrtf(var + eps);
  float nz = 0.f, p1 = 0.f, p2 = 0.f;
  const long long term = N * (long long)C;
  float4* zr = reinterpret_cast<float4*>(z + row * C);
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    int c4 = lane + 32 * i;
    if (c4 < nv) {
      float4 g = __ldg(reinterpret_cast<const float4*>(w) + c4);
      float4 be = __ldg(reinterpret_cast<const float4*>(b) + c4);
      float4 o;
      o.x = (v[i].x - mean) * rs * g.x + be.x;
      o.y = (v[i].y - mean) * rs * g.y + be.y;
      o.z = (v[i].z - mean) * rs * g.z + be.z;
      o.w = (v[i].w - mean) * rs * g.w + be.w;
      if (z) zr[c4] = o;
      nz += (o.x * o.x + o.y * o.y) + (o.z * o.z + o.w * o.w);
      if (rowstats) {
        const float gx = o.x * g.x, gy = o.y * g.y, gz = o.z * g.z, gw = o.w * g.w;
        p1 += (gx + gy) + (gz + gw);
        p2 += (gx * ((v[i].x - mean) * rs) + gy * ((v[i].y - mean) * rs)) + (gz * ((v[i].z - mean) * rs) + gw * ((v[i].w - mean) * rs));
      }
      if (split && hscale) {
        const float a[4] = {o.x * hs, o.y * hs, o.z * hs, o.w * hs};
        store_terms<2, 4>(split, term, row * C + 4 * c4, a);
      } else if (split) {
        const float a[4] = {o.x, o.y, o.z, o.w};
        store_terms<3, 4>(split, term, row * C + 4 * c4, a);
      }
    }
  }
  nz = warp_sum(nz);
  if (rowstats) { p1 = warp_sum(p1); p2 = warp_sum(p2); }
  if (lane == 0) {
    mu[row] = mean;
    rstd[row] = rs;
    if (zz) zz[row] = nz;
    if (rowstats) reinterpret_cast<float4*>(rowstats)[row] = make_float4(nz, p1, p2, 0.f);
  }
}

// ---------------------------------------------------------------------------
// Rows of any width (the cluster head at C % 4 != 0 or C > 1024; ln_rows_kernel / ln_bwd_rows_kernel keep the rest).
// WPR warps share a row (one block = 8 / WPR rows), each lane holds E elements c = t + 32 WPR i (t = lane index within
// the row), loaded one float at a time: a row of pitch C % 4 != 0 is not 16-byte aligned.  Row sums go through the warp
// shuffles and, for WPR > 1, through shared memory in fixed warp order (deterministic).
// ---------------------------------------------------------------------------
inline bool ln_any_width(int C) { return (C % 4) != 0 || C > 1024; }
// row pitch of the operand terms of a [rows, C] matrix: C, or for the any-width shapes C rounded up to 8 (tc_gemm's TMA
// row pitch is a multiple of 16 bytes); the padding columns hold zeros, so a contraction over the padded pitch is exact
inline int tc_pitch(int C) { return ln_any_width(C) ? (C + 7) & ~7 : C; }

// sums NV values over the WPR warps of a row; red: 32 floats of shared memory.  Every thread of the block calls it.
template <int WPR, int NV>
__device__ __forceinline__ void row_sums(float (&v)[NV], float* red) {
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = warp_sum(v[i]);
  if constexpr (WPR > 1) {
    const int wid = threadIdx.x >> 5, w0 = wid - wid % WPR;
    if ((threadIdx.x & 31) == 0)
#pragma unroll
      for (int i = 0; i < NV; ++i) red[wid * 4 + i] = v[i];
    __syncthreads();
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      float s = 0.f;
#pragma unroll
      for (int k = 0; k < WPR; ++k) s += red[(w0 + k) * 4 + i];
      v[i] = s;
    }
    __syncthreads();
  }
}

// LayerNorm rows of any width: ln_rows_kernel's outputs (two-pass statistics from the E values a lane holds); the
// operand terms of z go to pitch ldt = tc_pitch(C) with zeros in columns C..ldt-1
template <int E, int WPR>
__global__ void __launch_bounds__(256)
ln_rows_any_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ b,
                   long long N, int C, float eps, float* __restrict__ z, float* __restrict__ mu,
                   float* __restrict__ rstd, float* __restrict__ zz, float* __restrict__ rowstats,
                   __nv_bfloat16* __restrict__ split, const float* __restrict__ hscale, int ldt) {
  __shared__ float red[32];
  const float hs = hscale ? __ldg(hscale) : 1.0f;
  const int t = (threadIdx.x >> 5) % WPR * 32 + (threadIdx.x & 31);
  const long long row = (long long)blockIdx.x * (8 / WPR) + (threadIdx.x >> 5) / WPR;
  const bool live = row < N;
  if (WPR == 1 && !live) return;
  const float* xr = x + row * C;
  float v[E];
  float s[1] = {0.f};
#pragma unroll
  for (int i = 0; i < E; ++i) {
    const int c = t + 32 * WPR * i;
    v[i] = (live && c < C) ? __ldcs(xr + c) : 0.f;
    s[0] += v[i];
  }
  row_sums<WPR, 1>(s, red);
  const float mean = s[0] / (float)C;
  float q[1] = {0.f};
#pragma unroll
  for (int i = 0; i < E; ++i) {
    const float d = v[i] - mean;
    if (t + 32 * WPR * i < C) q[0] = fmaf(d, d, q[0]);
  }
  row_sums<WPR, 1>(q, red);
  const float rs = 1.0f / sqrtf(q[0] / (float)C + eps);
  float st[3] = {0.f, 0.f, 0.f};                  // |z|^2, sum z gamma, sum z gamma xhat
  const long long plane = N * (long long)ldt;
#pragma unroll
  for (int i = 0; i < E; ++i) {
    const int c = t + 32 * WPR * i;
    if (live && c < C) {
      const float g = __ldg(w + c), xh = (v[i] - mean) * rs;
      const float o = xh * g + __ldg(b + c);
      if (z) z[row * C + c] = o;
      st[0] = fmaf(o, o, st[0]);
      st[1] += o * g;
      st[2] = fmaf(o * g, xh, st[2]);
      if (split && hscale) store_terms<2>(split, plane, row * ldt + c, o * hs);
      else if (split) store_terms<3>(split, plane, row * ldt + c, o);
    }
  }
  if (split && live && t < ldt - C) {
    if (hscale) store_terms<2>(split, plane, row * ldt + C + t, 0.f);
    else store_terms<3>(split, plane, row * ldt + C + t, 0.f);
  }
  row_sums<WPR, 3>(st, red);
  if (live && t == 0) {
    mu[row] = mean;
    rstd[row] = rs;
    if (zz) zz[row] = st[0];
    if (rowstats) reinterpret_cast<float4*>(rowstats)[row] = make_float4(st[0], st[1], st[2], 0.f);
  }
}

// |row|^2 for a [R, C] matrix, one warp per row (any C).
static __global__ void __launch_bounds__(256)
row_sqnorm_kernel(const float* __restrict__ a, long long R, int C, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= R) return;
  const float* p = a + row * C;
  float s = 0.f;
  if ((C & 3) == 0) {
    const float4* p4 = reinterpret_cast<const float4*>(p);
    for (int i = lane; i < (C >> 2); i += 32) {
      float4 v = __ldg(p4 + i);
      s += (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
    }
  } else {
    for (int i = lane; i < C; i += 32) { float v = __ldg(p + i); s += v * v; }
  }
  s = warp_sum(s);
  if (lane == 0) out[row] = s;
}

// ---------------------------------------------------------------------------
// softmin / argmin / loss row pass (model/cluster.py:88,92 + backbone.py:94,98).
// G lanes cooperate on one row of K distances (G in {4,8,16,32}; K % 4 == 0).
//   label = first argmin, A = exp(-alpha (d - dmin)) / sum, part += (d*A)^2.
// Block partial sums of (d*A)^2 go to `partial[blockIdx.x]` (double).
// ---------------------------------------------------------------------------
// columns >= k_valid are padding (the host pads cluster_num to a multiple of 4): excluded from argmin / softmin / loss,
// their A is exactly 0 (exp(-inf)); D keeps the finite distance to the padding row
__device__ __forceinline__ float4 mask_pad(float4 v, int k, int k_valid) {
  if (k + 3 >= k_valid) {
    if (k >= k_valid) v.x = INFINITY;
    if (k + 1 >= k_valid) v.y = INFINITY;
    if (k + 2 >= k_valid) v.z = INFINITY;
    if (k + 3 >= k_valid) v.w = INFINITY;
  }
  return v;
}
__device__ __forceinline__ float da_sq(float d, float a) { const float p = a == 0.f ? 0.f : d * a; return p * p; }

template <int G>
__global__ void __launch_bounds__(256)
softmin_rows_kernel(const float* __restrict__ D, long long R, int K, int k_valid, float alpha,
                    float* __restrict__ A, long long* __restrict__ label,
                    double* __restrict__ partial,
                    __half* __restrict__ terms /* optional: two fp16 terms of A * sa, [2][R*K] */, float sa) {
  __shared__ double red[32];
  const int tid = threadIdx.x;
  const int g = tid / G, gl = tid % G;
  const long long row = (long long)blockIdx.x * (blockDim.x / G) + g;
  const unsigned gmask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << ((tid & 31) / G * G));
  double lsum = 0.0;
  if (row < R) {
    const float4* dr = reinterpret_cast<const float4*>(D + row * K);
    const int nv = K >> 2;
    float best = INFINITY;
    int bidx = 0x7fffffff;
    for (int i = gl; i < nv; i += G) {
      int k = i * 4;
      float4 v = mask_pad(dr[i], k, k_valid);
      if (v.x < best) { best = v.x; bidx = k; }
      if (v.y < best) { best = v.y; bidx = k + 1; }
      if (v.z < best) { best = v.z; bidx = k + 2; }
      if (v.w < best) { best = v.w; bidx = k + 3; }
    }
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) {
      float ob = __shfl_xor_sync(gmask, best, o, G);
      int oi = __shfl_xor_sync(gmask, bidx, o, G);
      if (ob < best || (ob == best && oi < bidx)) { best = ob; bidx = oi; }
    }
    float s = 0.f;
    for (int i = gl; i < nv; i += G) {
      float4 v = mask_pad(dr[i], i * 4, k_valid);
      s += (expf(-alpha * (v.x - best)) + expf(-alpha * (v.y - best))) +
           (expf(-alpha * (v.z - best)) + expf(-alpha * (v.w - best)));
    }
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) s += __shfl_xor_sync(gmask, s, o, G);
    float4* ar = reinterpret_cast<float4*>(A + row * K);
    float l = 0.f;
    for (int i = gl; i < nv; i += G) {
      float4 v = mask_pad(dr[i], i * 4, k_valid), a;
      a.x = expf(-alpha * (v.x - best)) / s;
      a.y = expf(-alpha * (v.y - best)) / s;
      a.z = expf(-alpha * (v.z - best)) / s;
      a.w = expf(-alpha * (v.w - best)) / s;
      ar[i] = a;
      if (terms) {                          // the operand split of the x_rec GEMM, written in the same pass
        const float b[4] = {a.x * sa, a.y * sa, a.z * sa, a.w * sa};
        store_terms<2, 4>(terms, R * K, row * K + 4 * i, b);
      }
      l += (da_sq(v.x, a.x) + da_sq(v.y, a.y)) + (da_sq(v.z, a.z) + da_sq(v.w, a.w));
    }
    lsum = (double)l;
    if (gl == 0 && label) label[row] = bidx;
  }
  double tot = block_sum<double>(lsum, red);
  if (tid == 0) partial[blockIdx.x] = tot;
}

// sum `n` doubles (one block, 1024 threads: the softmin pass leaves one partial per 256-thread block, 65k of them at
// cfg2 sizes), write float out[0]; fixed summation order
static __global__ void __launch_bounds__(1024)
finalize_sum_kernel(const double* __restrict__ partial, int n, float* __restrict__ out) {
  __shared__ double red[32];
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  int i = threadIdx.x;
  for (; i + 3 * (int)blockDim.x < n; i += 4 * blockDim.x) {           // four independent loads in flight
    s0 += partial[i]; s1 += partial[i + blockDim.x]; s2 += partial[i + 2 * blockDim.x]; s3 += partial[i + 3 * blockDim.x];
  }
  for (; i < n; i += blockDim.x) s0 += partial[i];
  double s = (s0 + s1) + (s2 + s3);
  s = block_sum<double>(s, red);
  if (threadIdx.x == 0) out[0] = (float)s;
}

// ---------------------------------------------------------------------------
// backward row pass (softmin backward + cdist ratio), G lanes per row:
//   gA_tot = gemm + gA + 2 g D^2 A                (x_rec path, explicit grad, fused loss grad;
//                                                  g = d objective / d sum (D*A)^2)
//   gD_tot = gD + 2 g D A^2 - alpha*A*(gA_tot - sum_k gA_tot*A)
//   r      = gD_tot / D   (0 where D == 0; ATen _euclidean_dist_backward)
//   rsum   = sum_k r
// ---------------------------------------------------------------------------
template <int G>
__global__ void __launch_bounds__(256)
bwd_rows_kernel(const float* __restrict__ D, const float* __restrict__ A,
                const float* __restrict__ gemm, const float* __restrict__ gD,
                const float* __restrict__ gA, const float* __restrict__ g_loss_sq,
                long long R, int K, float alpha,
                float* __restrict__ r, float* __restrict__ rsum,
                unsigned* __restrict__ absmax_bits /* optional: max |r| as float bits (atomicMax; zeroed by the caller) */) {
  __shared__ float bmax[8];
  const int tid = threadIdx.x;
  const int g = tid / G, gl = tid % G;
  const long long row = (long long)blockIdx.x * (blockDim.x / G) + g;
  const unsigned gmask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << ((tid & 31) / G * G));
  float amax = 0.f;
  if (row < R) {
  const float sc = g_loss_sq ? 2.0f * __ldg(g_loss_sq) : 0.f;
  const int nv = K >> 2;
  const long long base = row * K;
  float dot = 0.f;
  for (int i = gl; i < nv; i += G) {
    float4 d = reinterpret_cast<const float4*>(D + base)[i];
    float4 a = reinterpret_cast<const float4*>(A + base)[i];
    float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
    if (gemm) t = reinterpret_cast<const float4*>(gemm + base)[i];
    if (gA) { float4 u = reinterpret_cast<const float4*>(gA + base)[i]; t.x += u.x; t.y += u.y; t.z += u.z; t.w += u.w; }
    t.x += sc * d.x * d.x * a.x; t.y += sc * d.y * d.y * a.y;
    t.z += sc * d.z * d.z * a.z; t.w += sc * d.w * d.w * a.w;
    dot += (t.x * a.x + t.y * a.y) + (t.z * a.z + t.w * a.w);
  }
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) dot += __shfl_xor_sync(gmask, dot, o, G);
  float rs = 0.f;
  for (int i = gl; i < nv; i += G) {
    float4 d = reinterpret_cast<const float4*>(D + base)[i];
    float4 a = reinterpret_cast<const float4*>(A + base)[i];
    float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
    if (gemm) t = reinterpret_cast<const float4*>(gemm + base)[i];
    if (gA) { float4 u = reinterpret_cast<const float4*>(gA + base)[i]; t.x += u.x; t.y += u.y; t.z += u.z; t.w += u.w; }
    t.x += sc * d.x * d.x * a.x; t.y += sc * d.y * d.y * a.y;
    t.z += sc * d.z * d.z * a.z; t.w += sc * d.w * d.w * a.w;
    float4 gd = make_float4(0.f, 0.f, 0.f, 0.f);
    if (gD) gd = reinterpret_cast<const float4*>(gD + base)[i];
    gd.x += sc * d.x * a.x * a.x - alpha * a.x * (t.x - dot);
    gd.y += sc * d.y * a.y * a.y - alpha * a.y * (t.y - dot);
    gd.z += sc * d.z * a.z * a.z - alpha * a.z * (t.z - dot);
    gd.w += sc * d.w * a.w * a.w - alpha * a.w * (t.w - dot);
    float4 o;
    o.x = (d.x == 0.f) ? 0.f : gd.x / d.x;
    o.y = (d.y == 0.f) ? 0.f : gd.y / d.y;
    o.z = (d.z == 0.f) ? 0.f : gd.z / d.z;
    o.w = (d.w == 0.f) ? 0.f : gd.w / d.w;
    reinterpret_cast<float4*>(r + base)[i] = o;
    rs += (o.x + o.y) + (o.z + o.w);
    amax = fmaxf(fmaxf(amax, fmaxf(fabsf(o.x), fabsf(o.y))), fmaxf(fabsf(o.z), fabsf(o.w)));
  }
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) rs += __shfl_xor_sync(gmask, rs, o, G);
  if (gl == 0) rsum[row] = rs;
  }
  if (absmax_bits) {                         // block maximum -> one atomic per block (max is order-independent: deterministic)
    amax = warp_max(amax);
    if ((tid & 31) == 0) bmax[tid >> 5] = amax;
    __syncthreads();
    if (tid == 0) {
      float m = bmax[0];
#pragma unroll
      for (int w = 1; w < 8; ++w) m = fmaxf(m, bmax[w]);
      if (m > 0.f && isfinite(m)) atomicMax(absmax_bits, __float_as_uint(m));
    }
  }
}

// ---------------------------------------------------------------------------
// deterministic column sums of a [R, W] matrix: stage 1 writes
// partial[blockIdx.y][col] over a row chunk, stage 2 adds the chunks in order.
// ---------------------------------------------------------------------------
static __global__ void __launch_bounds__(256)
colsum_stage1_kernel(const float* __restrict__ a, long long R, int W, long long rows_per_block,
                     float* __restrict__ partial) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= W) return;
  long long r0 = (long long)blockIdx.y * rows_per_block;
  long long r1 = min(R, r0 + rows_per_block);
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  long long r = r0;
  for (; r + 3 < r1; r += 4) {
    s0 += __ldg(a + r * W + col);
    s1 += __ldg(a + (r + 1) * W + col);
    s2 += __ldg(a + (r + 2) * W + col);
    s3 += __ldg(a + (r + 3) * W + col);
  }
  for (; r < r1; ++r) s0 += __ldg(a + r * W + col);
  partial[(long long)blockIdx.y * W + col] = (s0 + s1) + (s2 + s3);
}

static __global__ void __launch_bounds__(256)
colsum_stage2_kernel(const float* __restrict__ partial, int nchunks, int W, float* __restrict__ out) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= W) return;
  float s = 0.f;
  for (int c = 0; c < nchunks; ++c) s += partial[(long long)c * W + col];
  out[col] = s;
}

inline int colsum_chunks(long long R) {
  long long c = (R + 255) / 256;          // 256 rows per block: enough blocks to fill the SMs at a few thousand rows
  if (c > 1024) c = 1024;
  if (c < 1) c = 1;
  return (int)c;
}

// out[col] = sum_r a[r, col]; `partial` holds colsum_chunks(R) * W floats.
inline cudaError_t launch_colsum(const float* a, long long R, int W, float* partial, float* out,
                                 cudaStream_t st) {
  int chunks = colsum_chunks(R);
  long long rpb = (R + chunks - 1) / chunks;
  if (rpb < 1) rpb = 1;
  dim3 g1((W + 255) / 256, chunks);
  colsum_stage1_kernel<<<g1, 256, 0, st>>>(a, R, W, rpb, partial);
  colsum_stage2_kernel<<<(W + 255) / 256, 256, 0, st>>>(partial, chunks, W, out);
  count_launch(2);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// LayerNorm backward, one warp per row, warps loop over rows so gamma/beta
// partials stay in registers; block partials -> [gridDim.x, 2C] -> stage 2.
// gz row-major [N,C].  gx = rstd*(g - mean(g) - xhat*mean(g*xhat)), g = gz*w.
// ---------------------------------------------------------------------------
template <int VPL>
__global__ void __launch_bounds__(256)
ln_bwd_rows_kernel(const float* __restrict__ gz, const float* __restrict__ x,
                   const float* __restrict__ mu, const float* __restrict__ rstd,
                   const float* __restrict__ w, long long N, int C,
                   float* __restrict__ gx, float* __restrict__ partial /*[grid,2C]*/) {
  extern __shared__ float sm[];   // [nwarps][2C]
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int nv = C >> 2;
  float4 gw[VPL], gb[VPL], wv[VPL];
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    gw[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    gb[i] = gw[i];
    int c4 = lane + 32 * i;
    wv[i] = (c4 < nv) ? __ldg(reinterpret_cast<const float4*>(w) + c4) : gw[i];
  }
  for (long long row = (long long)blockIdx.x * nw + wid; row < N; row += (long long)gridDim.x * nw) {
    const float m = __ldg(mu + row), rs = __ldg(rstd + row);
    float4 g[VPL], xh[VPL];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      int c4 = lane + 32 * i;
      if (c4 < nv) {
        float4 gv = ld_stream(reinterpret_cast<const float4*>(gz + row * C) + c4);
        float4 xv = ld_stream(reinterpret_cast<const float4*>(x + row * C) + c4);
        xh[i].x = (xv.x - m) * rs; xh[i].y = (xv.y - m) * rs;
        xh[i].z = (xv.z - m) * rs; xh[i].w = (xv.w - m) * rs;
        gw[i].x += gv.x * xh[i].x; gw[i].y += gv.y * xh[i].y;
        gw[i].z += gv.z * xh[i].z; gw[i].w += gv.w * xh[i].w;
        gb[i].x += gv.x; gb[i].y += gv.y; gb[i].z += gv.z; gb[i].w += gv.w;
        g[i].x = gv.x * wv[i].x; g[i].y = gv.y * wv[i].y;
        g[i].z = gv.z * wv[i].z; g[i].w = gv.w * wv[i].w;
        s1 += (g[i].x + g[i].y) + (g[i].z + g[i].w);
        s2 += (g[i].x * xh[i].x + g[i].y * xh[i].y) + (g[i].z * xh[i].z + g[i].w * xh[i].w);
      }
    }
    s1 = warp_sum(s1) / (float)C;
    s2 = warp_sum(s2) / (float)C;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      int c4 = lane + 32 * i;
      if (c4 < nv) {
        float4 o;
        o.x = (g[i].x - s1 - xh[i].x * s2) * rs;
        o.y = (g[i].y - s1 - xh[i].y * s2) * rs;
        o.z = (g[i].z - s1 - xh[i].z * s2) * rs;
        o.w = (g[i].w - s1 - xh[i].w * s2) * rs;
        reinterpret_cast<float4*>(gx + row * C)[c4] = o;
      }
    }
  }
  // block reduce of the gamma / beta partials in fixed warp order
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    int c4 = lane + 32 * i;
    if (c4 < nv) {
      reinterpret_cast<float4*>(sm + (size_t)wid * 2 * C)[c4] = gw[i];
      reinterpret_cast<float4*>(sm + (size_t)wid * 2 * C + C)[c4] = gb[i];
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < 2 * C; c += blockDim.x) {
    float s = 0.f;
    for (int ww = 0; ww < nw; ++ww) s += sm[(size_t)ww * 2 * C + c];
    partial[(size_t)blockIdx.x * 2 * C + c] = s;
  }
}

// LayerNorm backward of any width (layout as ln_rows_any_kernel): a block's row groups walk the rows together, every
// lane carries the gamma / beta partials of its E columns in registers; at the end the block's 8 / WPR row groups are
// summed column slice by column slice through 2 KB of shared memory (not [8][2C] floats: 256 KB at C = 4096) into the
// same partial [grid, 2C] ln_bwd_finalize_kernel reduces
template <int E, int WPR>
__global__ void __launch_bounds__(256)
ln_bwd_any_kernel(const float* __restrict__ gz, const float* __restrict__ x, const float* __restrict__ mu,
                  const float* __restrict__ rstd, const float* __restrict__ w, long long N, int C,
                  float* __restrict__ gx, float* __restrict__ partial /*[grid,2C]*/) {
  constexpr int G = 8 / WPR, RT = 32 * WPR;      // row groups per block, threads per row
  __shared__ float red[32];
  __shared__ float cs[2][256];
  const int t = (threadIdx.x >> 5) % WPR * 32 + (threadIdx.x & 31), grp = (threadIdx.x >> 5) / WPR;
  float gw[E], gb[E], wv[E];
#pragma unroll
  for (int i = 0; i < E; ++i) {
    const int c = t + RT * i;
    gw[i] = 0.f; gb[i] = 0.f;
    wv[i] = c < C ? __ldg(w + c) : 0.f;
  }
  for (long long r0 = (long long)blockIdx.x * G; r0 < N; r0 += (long long)gridDim.x * G) {   // uniform over the block
    const long long row = r0 + grp;
    const bool live = row < N;
    const float m = live ? __ldg(mu + row) : 0.f, rs = live ? __ldg(rstd + row) : 0.f;
    float g[E], xh[E];
    float s[2] = {0.f, 0.f};
#pragma unroll
    for (int i = 0; i < E; ++i) {
      const int c = t + RT * i;
      g[i] = 0.f; xh[i] = 0.f;
      if (live && c < C) {
        const float gv = __ldcs(gz + row * C + c), xv = __ldcs(x + row * C + c);
        xh[i] = (xv - m) * rs;
        gw[i] = fmaf(gv, xh[i], gw[i]);
        gb[i] += gv;
        g[i] = gv * wv[i];
        s[0] += g[i];
        s[1] = fmaf(g[i], xh[i], s[1]);
      }
    }
    row_sums<WPR, 2>(s, red);
    const float s1 = s[0] / (float)C, s2 = s[1] / (float)C;
#pragma unroll
    for (int i = 0; i < E; ++i) {
      const int c = t + RT * i;
      if (live && c < C) gx[row * C + c] = (g[i] - s1 - xh[i] * s2) * rs;
    }
  }
#pragma unroll
  for (int i = 0; i < E; ++i) {
    if (RT * i >= C) break;                      // uniform
    cs[0][grp * RT + t] = gw[i];
    cs[1][grp * RT + t] = gb[i];
    __syncthreads();
    const int c = (int)threadIdx.x + RT * i;
    if ((int)threadIdx.x < RT && c < C) {
      float a = 0.f, e = 0.f;
#pragma unroll
      for (int k = 0; k < G; ++k) { a += cs[0][k * RT + threadIdx.x]; e += cs[1][k * RT + threadIdx.x]; }
      partial[(size_t)blockIdx.x * 2 * C + c] = a;
      partial[(size_t)blockIdx.x * 2 * C + C + c] = e;
    }
    __syncthreads();
  }
}

}  // namespace vadc
