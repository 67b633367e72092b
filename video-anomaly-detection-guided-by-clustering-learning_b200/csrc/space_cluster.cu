// space_cluster.cu — Space_EuclidDistance_Assign_Module forward / backward (C3)
// model/cluster.py:127-149.  Per-channel spatial-map clustering: for every
// channel c the M = B*D frames are P-vectors (P = H*W) compared with K
// centroids of that channel: a batched [M,P] x [P,K] contraction over C
// batches.
#include <algorithm>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include "common.cuh"
#include "sgemm.cuh"
#include "tc_gemm.cuh"
#include "rows.cuh"
#include "cluster.h"

namespace vadc {

// Operand terms of the tensor-core path, for any P and any K (a multiple of 4): zt [C, M, Pp], centroids [C, Kp, Pp]
// (channel c's rows from c Kp), r [M, C Kp] (channel c's columns from c Kp).  Pp = P rounded up to 8: the TMA row pitch
// is a multiple of 16 bytes.  Kp = K rounded up to 64: channel c's window of the r·centers contraction ends on a k-block,
// so no column of channel c + 1 enters its sum.  The padding is written as zeros; the epilogues stop at P and K.
__host__ __device__ __forceinline__ int space_pp(int P) { return (P + 7) & ~7; }
static int space_kp(int K) { return (K + 63) & ~63; }

// LayerNorm + transpose: x [T, C] tokens -> zt [C, T].  A block normalises 32
// tokens (one warp per 4 tokens), parks them in shared memory and writes 32
// consecutive tokens per channel (128-byte segments) so both sides coalesce.
// terms (instead of zt): the three bf16 terms of zt [C, T / P, Pp], the frame's last token also writing the zero columns
__global__ void __launch_bounds__(256)
ln_transpose_kernel(const float* __restrict__ x, const float* __restrict__ w,
                    const float* __restrict__ b, long long T, int P, int C, float eps,
                    float* __restrict__ zt, float* __restrict__ mu, float* __restrict__ rstd,
                    __nv_bfloat16* __restrict__ terms) {
  extern __shared__ float tile[];            // [32][C+1]
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const long long t0 = (long long)blockIdx.x * 32;
  const int ld = C + 1;
  for (int rr = wid; rr < 32; rr += 8) {
    long long row = t0 + rr;
    if (row >= T) break;
    const float* xr = x + row * C;
    float s = 0.f;
    for (int c = lane; c < C; c += 32) { float v = __ldg(xr + c); tile[rr * ld + c] = v; s += v; }
    const float mean = warp_sum(s) / (float)C;
    float q = 0.f;
    for (int c = lane; c < C; c += 32) { float d = tile[rr * ld + c] - mean; q += d * d; }
    const float rs = 1.0f / sqrtf(warp_sum(q) / (float)C + eps);
    for (int c = lane; c < C; c += 32)
      tile[rr * ld + c] = (tile[rr * ld + c] - mean) * rs * __ldg(w + c) + __ldg(b + c);
    if (lane == 0) { mu[row] = mean; rstd[row] = rs; }
  }
  __syncthreads();
  const long long row = t0 + lane;
  if (row < T) {
    if (zt) {
      for (int c = wid; c < C; c += 8) zt[(long long)c * T + row] = tile[lane * ld + c];
    } else {                                   // the operand split of the batched tcgen05 GEMM, written in the same pass
      const int Pp = space_pp(P);
      const long long f = row / P, p = row - f * P, Tp = T / P * Pp, n = (long long)C * Tp;
      for (int c = wid; c < C; c += 8) {
        const long long i = (long long)c * Tp + f * Pp + p;
        store_terms<3>(terms, n, i, tile[lane * ld + c]);
        if (p == P - 1)
          for (int j = 1; j <= Pp - P; ++j) store_terms<3>(terms, n, i + j, 0.f);
      }
    }
  }
}

// LayerNorm backward from a transposed upstream gradient gzt [C, T]:
// stage a 32-token tile of gzt into shared memory, then one warp per token.
__global__ void __launch_bounds__(256)
ln_bwd_transposed_kernel(const float* __restrict__ gzt, const float* __restrict__ x,
                         const float* __restrict__ mu, const float* __restrict__ rstd,
                         const float* __restrict__ w, const float* __restrict__ bias,
                         const float* __restrict__ rsum /* [T/P, C] or null */, int P, long long T, int C,
                         float* __restrict__ gx, float* __restrict__ partial /*[grid,2C]*/) {
  extern __shared__ float sm[];              // tile [32][C+1] + acc [8][2C]
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int ld = C + 1;
  float* tile = sm;
  float* acc = sm + 32 * ld;                 // per-warp gamma/beta partials
  for (int i = threadIdx.x; i < 8 * 2 * C; i += 256) acc[i] = 0.f;
  for (long long t0 = (long long)blockIdx.x * 32; t0 < T; t0 += (long long)gridDim.x * 32) {
    __syncthreads();
    {
      const long long row = t0 + lane;
      if (row < T) {
#pragma unroll 8
        for (int c = wid; c < C; c += 8) tile[lane * ld + c] = __ldg(gzt + (long long)c * T + row);
      }
    }
    __syncthreads();
    for (int rr = wid; rr < 32; rr += 8) {
      long long row = t0 + rr;
      if (row >= T) break;
      const float m = mu[row], rs = rstd[row];
      const float* xr = x + row * C;
      const float* rsr = rsum ? rsum + (row / P) * C : nullptr;
      float s1 = 0.f, s2 = 0.f;
      for (int c = lane; c < C; c += 32) {
        float xh = (__ldg(xr + c) - m) * rs;
        float gv = tile[rr * ld + c];
        if (rsr) { gv = (xh * __ldg(w + c) + __ldg(bias + c)) * __ldg(rsr + c) - gv; tile[rr * ld + c] = gv; }
        float g = gv * __ldg(w + c);
        s1 += g; s2 += g * xh;
        acc[wid * 2 * C + c] += gv * xh;
        acc[wid * 2 * C + C + c] += gv;
      }
      s1 = warp_sum(s1) / (float)C;
      s2 = warp_sum(s2) / (float)C;
      for (int c = lane; c < C; c += 32) {
        float xh = (__ldg(xr + c) - m) * rs;
        float g = tile[rr * ld + c] * __ldg(w + c);
        gx[row * C + c] = (g - s1 - xh * s2) * rs;
      }
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < 2 * C; c += 256) {
    float s = 0.f;
    for (int ww = 0; ww < 8; ++ww) s += acc[ww * 2 * C + c];
    partial[(size_t)blockIdx.x * 2 * C + c] = s;
  }
}

// partial [nblocks, 2C] -> gw, gb: a block owns 32 columns, eight row groups stride the blocks
__global__ void __launch_bounds__(256)
ln_bwd_finalize2_kernel(const float* __restrict__ partial, int nblocks, int C,
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

// ---- tiled variants for C <= 256 (a lane keeps its channels of a token in registers) ----------------------------
constexpr int kTileTok = 64, kTileLd = kTileTok + 1, kMaxCpl = 8, kTokPerWarp = kTileTok / 8;

// LayerNorm + transpose of one (frame m, 64-token chunk j) tile.  Phase 1: a warp owns eight tokens and issues ALL
// their loads before the first reduction (the whole 48 KB tile of a block is in flight at once), normalises them in
// registers and parks them in the transposed shared tile [C][65].  Phase 2 writes a channel's 64 tokens per warp
// instruction — either fp32 zt (SIMT contraction path) or the operand terms of the batched tcgen05 GEMM at row pitch Pp
// (the frame's last chunk also writes the zero columns P..Pp-1, from tile columns it zeroes first) plus the chunk's
// share of |zt[c,m,:]|^2 (sqpart [C*M, chunks]; fp32 zt is then never materialised).
// CPL = channels per lane (C <= 32 CPL).
// NT = 0: fp32 zt; 3: three bf16 terms; 2: two fp16 terms of zt * *scale (a power of two from the LayerNorm bound).
// FULL: C == 32 CPL, no per-channel predicates.
template <int NT, int CPL, bool FULL>
__global__ void __launch_bounds__(256)
ln_transpose_tile_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ b,
                         int M, int P, int C, float eps, float* __restrict__ zt, float* __restrict__ mu,
                         float* __restrict__ rstd, void* __restrict__ terms_, const float* __restrict__ scale,
                         float* __restrict__ sqpart) {
  extern __shared__ float tile[];            // [C][65]
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int chunks = (P + kTileTok - 1) / kTileTok;
  const int m = blockIdx.x / chunks, j = blockIdx.x - m * chunks;
  const int p0 = j * kTileTok, np = min(kTileTok, P - p0);
  const long long T = (long long)M * P, t0 = (long long)m * P + p0;
  float v[kTokPerWarp][CPL];
#pragma unroll
  for (int i = 0; i < kTokPerWarp; ++i) {
    const float* xr = x + (t0 + min(wid + 8 * i, np - 1)) * C;       // rows past the chunk: a valid row, result unused
#pragma unroll
    for (int q = 0; q < CPL; ++q) v[i][q] = (FULL || lane + 32 * q < C) ? __ldg(xr + lane + 32 * q) : 0.f;
  }
  float wv[CPL], bv[CPL];
#pragma unroll
  for (int q = 0; q < CPL; ++q) {
    const int c = lane + 32 * q;
    wv[q] = (FULL || c < C) ? __ldg(w + c) : 0.f; bv[q] = (FULL || c < C) ? __ldg(b + c) : 0.f;
  }
  const float invC = 1.0f / (float)C;        // one division per thread instead of two per token (each a branchy subroutine)
#pragma unroll
  for (int i = 0; i < kTokPerWarp; ++i) {
    const int rr = wid + 8 * i;
    float s = 0.f;
#pragma unroll
    for (int q = 0; q < CPL; ++q) s += v[i][q];
    const float mean = warp_sum(s) * invC;
    float qq = 0.f;
#pragma unroll
    for (int q = 0; q < CPL; ++q)
      if (FULL || lane + 32 * q < C) { const float d = v[i][q] - mean; qq += d * d; }
    const float rs = rsqrtf(warp_sum(qq) * invC + eps);       // as torch's CUDA LayerNorm (rsqrt)
    if (rr < np) {
#pragma unroll
      for (int q = 0; q < CPL; ++q) {
        const int c = lane + 32 * q;
        if (FULL || c < C) tile[c * kTileLd + rr] = (v[i][q] - mean) * rs * wv[q] + bv[q];
      }
      if (lane == 0) { mu[t0 + rr] = mean; rstd[t0 + rr] = rs; }
    }
  }
  const int Pp = space_pp(P), npp = min(kTileTok, Pp - p0);       // npp > np: the frame's last chunk, P % 8 != 0
  if (NT != 0 && npp > np)
    for (int c = wid; c < C; c += 8) if (lane < npp - np) tile[c * kTileLd + np + lane] = 0.f;
  __syncthreads();
  if constexpr (NT != 0) {
    // half a warp per channel, four tokens per lane (the padded pitch Pp is a multiple of 8): 8-byte stores
    const long long Tp = (long long)M * Pp, n = (long long)C * Tp;
    const int half = lane >> 4, l16 = lane & 15;
    const bool tok = 4 * l16 < npp;
    uint16_t* const tbase = static_cast<uint16_t*>(terms_) + (long long)m * Pp + p0 + 4 * l16;
    const float sc = NT == 2 ? __ldg(scale) : 1.0f;
    // pointers advance by 16 channels per iteration (no per-iteration 64-bit multiplies)
    uint16_t* d = tbase + (long long)(2 * wid + half) * Tp;
    float* sp = sqpart + ((long long)(2 * wid + half) * M + m) * chunks + j;
    const float* tp = tile + (2 * wid + half) * kTileLd + 4 * l16;
    const long long dstep = 16 * Tp, sstep = 16ll * M * chunks;
#pragma unroll 2
    for (int cc = 2 * wid; cc < C; cc += 16, d += dstep, sp += sstep, tp += 16 * kTileLd) {
      const int c = cc + half;
      const bool ok = tok && (FULL || c < C);
      float v[4] = {0.f, 0.f, 0.f, 0.f};
      if (ok) { v[0] = tp[0]; v[1] = tp[1]; v[2] = tp[2]; v[3] = tp[3]; }
      if constexpr (NT == 3) {
        __nv_bfloat162 h[3][2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          h[0][e] = __floats2bfloat162_rn(v[2 * e], v[2 * e + 1]);
          const float r0 = v[2 * e] - __low2float(h[0][e]), r1 = v[2 * e + 1] - __high2float(h[0][e]);
          h[1][e] = __floats2bfloat162_rn(r0, r1);
          h[2][e] = __floats2bfloat162_rn(r0 - __low2float(h[1][e]), r1 - __high2float(h[1][e]));
        }
        if (ok) {
          *reinterpret_cast<uint2*>(d) = *reinterpret_cast<uint2*>(h[0]);
          *reinterpret_cast<uint2*>(d + n) = *reinterpret_cast<uint2*>(h[1]);
          *reinterpret_cast<uint2*>(d + 2 * n) = *reinterpret_cast<uint2*>(h[2]);
        }
      } else {
        __half2 h[2][2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const float a0 = v[2 * e] * sc, a1 = v[2 * e + 1] * sc;
          h[0][e] = __floats2half2_rn(a0, a1);
          h[1][e] = __floats2half2_rn(a0 - __low2float(h[0][e]), a1 - __high2float(h[0][e]));
        }
        if (ok) {
          *reinterpret_cast<uint2*>(d) = *reinterpret_cast<uint2*>(h[0]);
          *reinterpret_cast<uint2*>(d + n) = *reinterpret_cast<uint2*>(h[1]);
        }
      }
      float sq = (v[0] * v[0] + v[1] * v[1]) + (v[2] * v[2] + v[3] * v[3]);
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
      if (l16 == 0 && (FULL || c < C)) *sp = sq;
    }
  } else {
    for (int c = wid; c < C; c += 8) {
      if (lane < np) zt[(long long)c * T + t0 + lane] = tile[c * kTileLd + lane];
      if (lane + 32 < np) zt[(long long)c * T + t0 + lane + 32] = tile[c * kTileLd + lane + 32];
    }
  }
}

__global__ void __launch_bounds__(256)
sqpart_reduce_kernel(const float* __restrict__ sqpart, long long rows, int chunks, float* __restrict__ out) {
  const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  float s = 0.f;
  for (int j = 0; j < chunks; ++j) s += sqpart[r * chunks + j];
  out[r] = s;
}

// the three bf16 terms of an operand element back to fp32 (exact: the split is)
__device__ __forceinline__ float terms_value(const __nv_bfloat16* t, long long n, long long i) {
  return (__bfloat162float(t[2 * n + i]) + __bfloat162float(t[n + i])) + __bfloat162float(t[i]);
}

__device__ __forceinline__ void cp_async4(float* smem_dst, const float* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(src) : "memory");
}

// LayerNorm backward from the transposed upstream gradient gzt [C, T], 64-token tiles: the tile's C rows of gzt go to
// shared [C][65] through cp.async (32 consecutive tokens per warp instruction) while the block's x rows — eight tokens
// per warp, all issued up front — travel to registers; then a warp finishes a token at a time from registers and the
// conflict-free transposed tile.  The gamma / beta partials stay in registers across a block's tiles.
// RSUM: the tile holds acc = r centers and the upstream gradient is zt rsum - acc with zt = x-hat gamma + beta (the
// tensor-core path; needs P >= 64 so that a tile touches two frames at most: their rsum rows ride along into shared
// memory).  FULL: C == 32 CPL, no per-channel predicates.
template <int CPL, bool RSUM, bool FULL>
__global__ void __launch_bounds__(256)
ln_bwd_transposed_tile_kernel(const float* __restrict__ gzt, const float* __restrict__ x,
                              const float* __restrict__ mu, const float* __restrict__ rstd,
                              const float* __restrict__ w, const float* __restrict__ bias,
                              const float* __restrict__ rsum /* [T/P, C] */, int P, long long T, int C,
                              float* __restrict__ gx, float* __restrict__ partial /*[grid,2C]*/) {
  extern __shared__ float tile[];            // [32 CPL][65] (rows >= C stay zero) + rsum rows [2][32 CPL]
  constexpr int CP = 32 * CPL;
  float* const rs_s = tile + CP * kTileLd;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  float aw[CPL], ab[CPL], wv[CPL], bv[CPL];
#pragma unroll
  for (int q = 0; q < CPL; ++q) {
    const bool in = FULL || lane + 32 * q < C;
    aw[q] = 0.f; ab[q] = 0.f; wv[q] = in ? __ldg(w + lane + 32 * q) : 0.f; bv[q] = (in && RSUM) ? __ldg(bias + lane + 32 * q) : 0.f;
  }
  if (!FULL) for (int i = C * kTileLd + threadIdx.x; i < CP * kTileLd + 2 * CP; i += 256) tile[i] = 0.f;
  const long long ntiles = (T + kTileTok - 1) / kTileTok;
  const float invC = 1.0f / (float)C;        // one division per thread, not two branchy ones per token
  for (long long tl = blockIdx.x; tl < ntiles; tl += gridDim.x) {
    const long long t0 = tl * kTileTok;
    const int np = (int)min((long long)kTileTok, T - t0);
    __syncthreads();                         // the previous tile has been consumed
    {
      const int k = threadIdx.x & 63;
      if (k < np) {
        const float* src = gzt + t0 + k;
        float* dst = tile + k;
        for (int c = threadIdx.x >> 6; c < C; c += 4) cp_async4(dst + c * kTileLd, src + (long long)c * T);
      }
    }
    int rem0 = 0;
    if constexpr (RSUM) {
      const long long f0 = t0 / P;
      const int nfr = (int)((t0 + np - 1) / P - f0) + 1;            // 1 or 2
      rem0 = (int)(t0 - f0 * P);                                     // position of the tile's first token inside frame f0
      for (int idx = threadIdx.x; idx < nfr * C; idx += 256) {
        const int f = idx >= C ? 1 : 0;
        cp_async4(rs_s + f * CP + (idx - f * C), rsum + f0 * C + idx);
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    float xh[kTokPerWarp][CPL], mr[kTokPerWarp], rr_[kTokPerWarp];
#pragma unroll
    for (int i = 0; i < kTokPerWarp; ++i) {
      const long long row = t0 + min(wid + 8 * i, np - 1);
      const float* xr = x + row * C;
#pragma unroll
      for (int q = 0; q < CPL; ++q) xh[i][q] = (FULL || lane + 32 * q < C) ? __ldg(xr + lane + 32 * q) : 0.f;
      mr[i] = __ldg(mu + row); rr_[i] = __ldg(rstd + row);
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
#pragma unroll
    for (int i = 0; i < kTokPerWarp; ++i) {
      const int rr = wid + 8 * i;
      const bool on = rr < np;
      const float m = mr[i], rs = rr_[i];
      const float* tp = tile + lane * kTileLd + (on ? rr : 0);
      const float* rss = rs_s + ((RSUM && rem0 + rr >= P) ? CP : 0) + lane;
      float g[CPL], s1 = 0.f, s2 = 0.f;
#pragma unroll
      for (int q = 0; q < CPL; ++q) {
        float gv = tp[32 * q * kTileLd];
        xh[i][q] = (xh[i][q] - m) * rs;
        if constexpr (RSUM) gv = (xh[i][q] * wv[q] + bv[q]) * rss[32 * q] - gv;
        gv = on ? gv : 0.f;
        g[q] = gv * wv[q];
        s1 += g[q]; s2 += g[q] * xh[i][q];
        aw[q] += gv * xh[i][q]; ab[q] += gv;
      }
      s1 = warp_sum(s1) * invC; s2 = warp_sum(s2) * invC;
      if (on) {
        float* go = gx + (t0 + rr) * C + lane;
#pragma unroll
        for (int q = 0; q < CPL; ++q)
          if (FULL || lane + 32 * q < C) go[32 * q] = (g[q] - s1 - xh[i][q] * s2) * rs;
      }
    }
  }
  __syncthreads();
#pragma unroll
  for (int q = 0; q < CPL; ++q) {
    const int c = lane + 32 * q;
    if (FULL || c < C) { tile[wid * 2 * C + c] = aw[q]; tile[wid * 2 * C + C + c] = ab[q]; }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < 2 * C; c += 256) {
    float s = 0.f;
    for (int ww = 0; ww < 8; ++ww) s += tile[ww * 2 * C + c];
    partial[(size_t)blockIdx.x * 2 * C + c] = s;
  }
}

// Ds[m,c,k] = sqrt(max(0, |zt[c,m]|^2 + |centers[c,k]|^2 - 2 acc))   ('C (B D) CN -> B D C CN')
struct SpaceDistEpilogue {
  float* out; const float* aa; const float* bb; long long CK; int K, M;
  __device__ __forceinline__ void operator()(int batch, int, int m, int n, float v) const {
    float sq = aa[(long long)batch * M + m] + bb[(long long)batch * K + n] - 2.0f * v;
    out[(long long)m * CK + (long long)batch * K + n] = sqrtf(fmaxf(sq, 0.f));
  }
};

// gzt[c,m,p] = zt[c,m,p] * rsum[m,c] - acc
struct SpaceGzEpilogue {
  float* out; const float* zt; const float* rsum; long long MP; int P, C;
  __device__ __forceinline__ void operator()(int batch, int, int m, int n, float v) const {
    long long i = (long long)batch * MP + (long long)m * P + n;
    out[i] = zt[i] * rsum[(long long)m * C + batch] - v;
  }
};


// The three contractions of the head as batched tcgen05 GEMMs: worth it from a few GFLOP up, for any P and K (the
// operand terms are padded to Pp, Kp: space_pp, space_kp); the batch offsets of the launches fit in int.
static bool space_tc_ok(long long M, int P, int C, int K) {
  return M >= 1 && C <= 65535 && (long long)C * M < (1ll << 31) && (long long)C * space_kp(K) < (1ll << 31) &&
         (double)M * P * K * C >= (double)(1ll << 28) && vadc_device_ok() != 0 && !env_on("VADC_NO_TC_GEMM");
}

static int space_ln_bwd_blocks(long long T, int C, bool tiled) {
  // tiled kernel: 64-token tiles, ~50 KB of shared memory per block at C = 192; otherwise 32-token tiles
  long long b = tiled ? (T + kTileTok - 1) / kTileTok : (T + 31) / 32;
  long long cap = (long long)sm_count() * (tiled ? 4 : 6);
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

// |zt[c,m,:]|^2 from the three operand terms (C > 256, where the tiled kernel does not apply): one warp per row
__global__ void __launch_bounds__(256)
row_sqnorm_terms_kernel(const __nv_bfloat16* __restrict__ t, long long n, long long R, int P, float* __restrict__ out) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= R) return;
  const long long base = row * space_pp(P);
  float s = 0.f;
  for (int p = threadIdx.x & 31; p < P; p += 32) { const float v = terms_value(t, n, base + p); s += v * v; }
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) out[row] = s;
}

static int space_chunks(int P) { return (P + kTileTok - 1) / kTileTok; }

// operand terms of the tensor-core path: two fp16 terms of power-of-two-scaled operands (22 significant bits: 2/3 of
// the bytes, half the MMAs) unless VADC_SPACE_TERMS=3 asks for the fp32-faithful three bf16 terms; the untiled
// LayerNorm kernels (C > 256) only write the latter
static int space_nt(int C) { return (C > 32 * kMaxCpl || env_int("VADC_SPACE_TERMS", 2) == 3) ? 3 : 2; }
// saved state of the tensor-core path: [ zt terms [C, M, Pp] | centroid terms [C, Kp, Pp] | forward scales (256 bytes) ]
static size_t space_zt_bytes(long long M, int P, int C) {
  return align_up((size_t)C * M * space_pp(P) * space_nt(C) * 2, 256);
}
static size_t space_cen_bytes(int P, int C, int K) {
  return align_up((size_t)C * space_kp(K) * space_pp(P) * space_nt(C) * 2, 256);
}

// column sums of r [M, C K]: few rows, many columns — split the rows so that the grid covers the SMs a few times
static int space_colsum_chunks(long long R, long long W) {
  long long want = (4ll * sm_count() + (W + 255) / 256 - 1) / ((W + 255) / 256);
  long long cap = R / 32 > 1 ? R / 32 : 1;
  long long c = std::max<long long>(colsum_chunks(R), std::min(want, cap));
  return (int)std::min<long long>(c, 1024);
}

static cudaError_t launch_space_colsum(const float* a, long long R, int W, float* partial, float* out, cudaStream_t st) {
  const int chunks = space_colsum_chunks(R, W);
  const long long rpb = std::max<long long>((R + chunks - 1) / chunks, 1);
  colsum_stage1_kernel<<<dim3((W + 255) / 256, chunks), 256, 0, st>>>(a, R, W, rpb, partial);
  colsum_stage2_kernel<<<(W + 255) / 256, 256, 0, st>>>(partial, chunks, W, out);
  count_launch(2);
  return cudaGetLastError();
}

template <int NT, int CPL>
static int launch_ln_transpose_tile_cpl(const float* x, const float* w, const float* b, int M, int P, int C, float eps,
                                        float* zt, float* mu, float* rstd, void* terms, const float* scale, float* sqpart,
                                        cudaStream_t st) {
  const size_t smem = (size_t)C * kTileLd * sizeof(float);
  auto kern = C == 32 * CPL ? ln_transpose_tile_kernel<NT, CPL, true> : ln_transpose_tile_kernel<NT, CPL, false>;
  if (smem > 48 * 1024) VADC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<(unsigned)((long long)M * space_chunks(P)), 256, smem, st>>>(x, w, b, M, P, C, eps, zt, mu, rstd, terms, scale, sqpart);
  VADC_CHECK_LAUNCH("ln_transpose_tile_kernel");
  return VADC_OK;
}

// nt = 0: fp32 zt; 3: bf16 x3 terms + sqpart; 2: fp16 x2 terms of zt * *scale + sqpart
static int launch_ln_transpose_tile(const float* x, const float* w, const float* b, int M, int P, int C, float eps,
                                    float* zt, float* mu, float* rstd, int nt, void* terms, const float* scale,
                                    float* sqpart, cudaStream_t st) {
  const int cpl = (C + 31) / 32;
#define VADC_LT(CPL)                                                                                                   \
  return nt == 3 ? launch_ln_transpose_tile_cpl<3, CPL>(x, w, b, M, P, C, eps, nullptr, mu, rstd, terms, nullptr, sqpart, st) \
       : nt == 2 ? launch_ln_transpose_tile_cpl<2, CPL>(x, w, b, M, P, C, eps, nullptr, mu, rstd, terms, scale, sqpart, st)   \
                 : launch_ln_transpose_tile_cpl<0, CPL>(x, w, b, M, P, C, eps, zt, mu, rstd, nullptr, nullptr, nullptr, st)
  if (cpl <= 2) { VADC_LT(2); }
  if (cpl <= 4) { VADC_LT(4); }
  if (cpl <= 6) { VADC_LT(6); }
  VADC_LT(8);
#undef VADC_LT
}

template <int CPL>
static int launch_ln_bwd_tile_cpl(const float* gzt, const float* x, const float* mu, const float* rstd, const float* w,
                                  const float* bias, const float* rsum, int P,
                                  long long T, int C, float* gx, float* partial, int nb, cudaStream_t st) {
  const size_t smem = ((size_t)32 * CPL * kTileLd + 2 * 32 * CPL) * sizeof(float);      // >= 16 C floats for the final reduction
  const bool full = C == 32 * CPL;
#define VADC_LB(RS, FU)                                                                                       \
  {                                                                                                           \
    auto kern = ln_bwd_transposed_tile_kernel<CPL, RS, FU>;                                                   \
    if (smem > 48 * 1024) VADC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    kern<<<nb, 256, smem, st>>>(gzt, x, mu, rstd, w, bias, rsum, P, T, C, gx, partial);                     \
  }
  if (rsum) { if (full) VADC_LB(true, true) else VADC_LB(true, false) }
  else { if (full) VADC_LB(false, true) else VADC_LB(false, false) }
#undef VADC_LB
  VADC_CHECK_LAUNCH("ln_bwd_transposed_tile_kernel");
  return VADC_OK;
}

// tiled LayerNorm backward: C <= 256, and with rsum (tensor-core path) P >= 64
static bool ln_bwd_tile_ok(int C, int P, bool with_rsum) { return C <= 32 * kMaxCpl && (!with_rsum || P >= kTileTok); }

static int launch_ln_bwd_tile(const float* gzt, const float* x, const float* mu, const float* rstd, const float* w,
                              const float* bias, const float* rsum, int P,
                              long long T, int C, float* gx, float* partial, int nb, cudaStream_t st) {
  const int cpl = (C + 31) / 32;
  if (cpl <= 2) return launch_ln_bwd_tile_cpl<2>(gzt, x, mu, rstd, w, bias, rsum, P, T, C, gx, partial, nb, st);
  if (cpl <= 4) return launch_ln_bwd_tile_cpl<4>(gzt, x, mu, rstd, w, bias, rsum, P, T, C, gx, partial, nb, st);
  if (cpl <= 6) return launch_ln_bwd_tile_cpl<6>(gzt, x, mu, rstd, w, bias, rsum, P, T, C, gx, partial, nb, st);
  return launch_ln_bwd_tile_cpl<8>(gzt, x, mu, rstd, w, bias, rsum, P, T, C, gx, partial, nb, st);
}

}  // namespace vadc

using namespace vadc;

// The LayerNorm output in the batched-cdist layout [C, M, P], kept from the forward for the backward: the operand
// terms of the tcgen05 GEMMs when those run (at the padded pitches of space_pp / space_kp; fp32 zt = their exact sum is
// never written) followed by the terms of the centroids, fp32 zt otherwise.  Opaque to the caller; forward and backward must
// see the same environment.
extern "C" size_t vadc_space_cluster_saved_bytes(int64_t M, int P, int C, int K) {
  const size_t n = (size_t)C * (size_t)(M > 0 ? M : 1) * P;
  if (!space_tc_ok(M, P, C, K)) return align_up(n * sizeof(float), 256);
  return space_zt_bytes(M > 0 ? M : 1, P, C) + space_cen_bytes(P, C, K) + 256;
}

extern "C" size_t vadc_space_cluster_fwd_workspace_bytes(int64_t M, int P, int C, int K) {
  size_t m = (size_t)(M > 0 ? M : 1);
  size_t b = 0;
  b += align_up((size_t)C * m * sizeof(float), 256);                  // |zt row|^2
  b += align_up((size_t)C * K * sizeof(float), 256);                  // |center row|^2
  b += align_up((size_t)(softmin_blocks(M * C, K) + 1) * sizeof(double), 256);
  b += align_up((size_t)C * m * space_chunks(P) * sizeof(float), 256); // per-chunk shares of |zt row|^2
  b += vadc_cdist_workspace_bytes(C, K, K, P);                        // centroid self-distance off the tensor-core path
  return b + 256;
}

// the forward's batched distance GEMM (batch c: A = zt[c] [M,P], B = centers[c]^T; out Ds[m, c, k]) and, from the same
// terms and norms, cdist(centers, centers) (model/cluster.py:134); fp16 x2 scales in sc (tc_fwd_scales_from_bits)
template <int TERMS>
static int space_dist_tc(const void* zs, const float* centers, void* cs, const float* sc, int64_t M, int P, int C, int K,
                         const float* zz, const float* cc, float* Ds, float* selfdist, cudaStream_t st) {
  const int Pp = space_pp(P), Kp = space_kp(K);
  const long long CM = (long long)C * M, CK = (long long)C * K, CKp = (long long)C * Kp;
  int rc;
  if ((rc = tc_split<TERMS>(centers, CK, P, TERMS == 2 ? sc + 1 : nullptr, cs, st, Pp, K, Kp))) return rc;
  if ((rc = tc_gemm<TERMS, false, false>({zs, cs, M, K, P, TERMS == 2 ? sc + 2 : nullptr, 1, C, {(int)M, 0, Kp, 0}, CM, Pp, CKp, Pp},
                                         TcBatchDistEpi{Ds, zz, cc, CK, K, M, K}, st))) return rc;
  if (!selfdist) return VADC_OK;
  return tc_gemm<TERMS, false, false>({cs, cs, K, K, P, TERMS == 2 ? sc + 5 : nullptr, 1, C, {Kp, 0, Kp, 0}, CKp, Pp, CKp, Pp},
                                      TcBatchDistEpi{selfdist, cc, cc, K, (long long)K * K, K, K}, st);
}

static int space_cluster_fwd_impl(const float* x, const float* ln_w, const float* ln_b,
                                  const float* centers, int64_t M, int P, int C, int K, int k_valid,
                                  float alpha, float eps, float* Ds, float* As, float* selfdist, void* zt_state,
                                  float* mu, float* rstd, float* loss_sq, void* workspace,
                                  size_t workspace_bytes, void* stream) {
  VADC_REQUIRE(M >= 0 && P > 0 && C > 0 && K > 0 && (K % 4) == 0, VADC_ERR_BAD_SHAPE);
  VADC_REQUIRE(M * (int64_t)P < (1ll << 31) && M * (int64_t)C < (1ll << 31), VADC_ERR_UNSUPPORTED);
  VADC_REQUIRE(ln_w && ln_b && centers && loss_sq && workspace, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(M == 0 || (x && Ds && As && zt_state && mu && rstd), VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(aligned16(Ds) && aligned16(As) && aligned16(zt_state), VADC_ERR_MISALIGNED);
  VADC_REQUIRE(workspace_bytes >= vadc_space_cluster_fwd_workspace_bytes(M, P, C, K), VADC_ERR_WORKSPACE);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Carver ws(workspace, workspace_bytes);
  float* zz = ws.take<float>((size_t)C * (M > 0 ? M : 1));
  float* cc = ws.take<float>((size_t)C * K);
  double* partial = ws.take<double>(softmin_blocks(M * C, K) + 1);
  float* sqpart = ws.take<float>((size_t)C * (M > 0 ? M : 1) * space_chunks(P));
  const long long T = (long long)M * P;
  int rc;
  bool selfdist_done = selfdist == nullptr;
  if (M > 0) {
    const bool tc = space_tc_ok(M, P, C, K);
    const bool tiled = C <= 32 * kMaxCpl;
    const int nt = tc ? space_nt(C) : 0;
    float* zt = tc ? nullptr : static_cast<float*>(zt_state);
    __nv_bfloat16* zs = tc ? static_cast<__nv_bfloat16*>(zt_state) : nullptr;
    uint8_t* cs = tc ? static_cast<uint8_t*>(zt_state) + space_zt_bytes(M, P, C) : nullptr;     // the backward reuses both
    float* sc = tc ? reinterpret_cast<float*>(cs + space_cen_bytes(P, C, K)) : nullptr;
    if (nt == 2) {                                   // scales: LayerNorm bound, measured max |centers| (device-side)
      unsigned* bits = reinterpret_cast<unsigned*>(sc + 32);
      if ((rc = tc_absmax_bits(centers, (long long)C * K * P, bits, st))) return rc;
      if ((rc = tc_fwd_scales_from_bits(bits, ln_w, ln_b, C, sc, st))) return rc;
    }
    if (tiled) {
      const long long rows = (long long)C * M;
      if ((rc = launch_ln_transpose_tile(x, ln_w, ln_b, (int)M, P, C, eps, zt, mu, rstd, nt, zs, sc, sqpart, st))) return rc;
      if (tc) {
        sqpart_reduce_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, st>>>(sqpart, rows, space_chunks(P), zz);
        VADC_CHECK_LAUNCH("sqpart_reduce_kernel");
      } else if ((rc = launch_row_sqnorm(zt, rows, P, zz, st))) return rc;
    } else {
      size_t smem = (size_t)32 * (C + 1) * sizeof(float);
      if (smem > 48 * 1024)
        VADC_CUDA(cudaFuncSetAttribute(ln_transpose_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      ln_transpose_kernel<<<(unsigned)((T + 31) / 32), 256, smem, st>>>(x, ln_w, ln_b, T, P, C, eps, zt, mu, rstd, zs);
      VADC_CHECK_LAUNCH("ln_transpose_kernel");
      if (tc) {
        const long long rows = (long long)C * M;
        row_sqnorm_terms_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, st>>>(zs, rows * space_pp(P), rows, P, zz);
        VADC_CHECK_LAUNCH("row_sqnorm_terms_kernel");
      } else if ((rc = launch_row_sqnorm(zt, (long long)C * M, P, zz, st))) return rc;
    }
    if ((rc = launch_row_sqnorm(centers, (long long)C * K, P, cc, st))) return rc;
    // batch c: A = zt[c] [M,P], B = centers[c]^T; out Ds[m, c, k]
    if (tc) {
      if ((rc = nt == 2 ? space_dist_tc<2>(zs, centers, cs, sc, M, P, C, K, zz, cc, Ds, selfdist, st)
                        : space_dist_tc<3>(zs, centers, cs, sc, M, P, C, K, zz, cc, Ds, selfdist, st))) return rc;
      selfdist_done = true;
    } else {
      Operand Aop{zt, P, 1}, Bop{centers, 1, P};
      SpaceDistEpilogue epi{Ds, zz, cc, (long long)C * K, K, (int)M};
      cudaError_t e = sgemm_auto((int)M, K, P, Aop, Bop, (long long)M * P, (long long)K * P, C, 1, epi, st);
      if (e != cudaSuccess) return record_cuda_error(e, "space dist sgemm");
    }
  }
  if (!selfdist_done) {
    const size_t nb = vadc_cdist_workspace_bytes(C, K, K, P);
    if ((rc = vadc_cdist(centers, centers, C, K, K, P, selfdist, ws.take<uint8_t>(nb), nb, stream))) return rc;
  }
  return launch_softmin_rows(Ds, M * (long long)C, K, alpha, As, nullptr, partial, loss_sq, st, k_valid);
}

extern "C" int vadc_space_cluster_fwd(const float* x, const float* ln_w, const float* ln_b,
                                      const float* centers, int64_t M, int P, int C, int K,
                                      float alpha, float eps, float* Ds, float* As, float* selfdist, void* zt_state,
                                      float* mu, float* rstd, float* loss_sq, void* workspace,
                                      size_t workspace_bytes, void* stream) {
  return space_cluster_fwd_impl(x, ln_w, ln_b, centers, M, P, C, K, K, alpha, eps, Ds, As, selfdist, zt_state, mu, rstd, loss_sq, workspace,
                                workspace_bytes, stream);
}

// any cluster_num: centers [C, K, P] padded by the host to K % 4 == 0; the trailing K - K_valid rows of every channel are excluded
extern "C" int vadc_space_cluster_fwd_padded(const float* x, const float* ln_w, const float* ln_b,
                                             const float* centers, int64_t M, int P, int C, int K, int K_valid,
                                             float alpha, float eps, float* Ds, float* As, float* selfdist, void* zt_state,
                                             float* mu, float* rstd, float* loss_sq, void* workspace,
                                             size_t workspace_bytes, void* stream) {
  VADC_REQUIRE(K_valid >= 1 && K_valid <= K, VADC_ERR_BAD_SHAPE);
  return space_cluster_fwd_impl(x, ln_w, ln_b, centers, M, P, C, K, K_valid, alpha, eps, Ds, As, selfdist, zt_state, mu, rstd, loss_sq,
                                workspace, workspace_bytes, stream);
}

extern "C" size_t vadc_space_cluster_bwd_workspace_bytes(int64_t M, int P, int C, int K) {
  size_t m = (size_t)(M > 0 ? M : 1);
  size_t b = 0;
  b += align_up(m * C * K * sizeof(float), 256);                       // r
  b += align_up(m * C * sizeof(float), 256);                           // rsum
  b += align_up((size_t)C * m * P * sizeof(float), 256);               // gzt
  b += align_up((size_t)space_colsum_chunks(M, (long long)C * K) * C * K * sizeof(float), 256);
  b += align_up((size_t)C * K * sizeof(float), 256);                   // rcol
  b += align_up((size_t)std::max(space_ln_bwd_blocks(M * (int64_t)P, C, true), space_ln_bwd_blocks(M * (int64_t)P, C, false)) * 2 * C * sizeof(float), 256);
  b += tc_terms_bytes(3, (long long)m, (long long)C * space_kp(K)) + 512;     // r terms [M, C Kp], scales
  return b + 512;
}

namespace vadc {
// the backward's two batched contractions on the tcgen05 GEMM (terms of zt and centers from the forward, r split here);
// fp16 x2: r has no a-priori bound, its scale comes from its measured max (device-side, no host sync)
template <int TERMS>
static int space_bwd_tc(const float* r, void* rs, const unsigned* rbits, const float* fsc, const void* zs, const void* cs,
                        const float* centers, int64_t M, int P, int C, int K, float* gzt, const float* rcol, float* gcenters,
                        Carver& ws, cudaStream_t st) {
  const float* bsc = nullptr;
  int rc;
  if constexpr (TERMS == 2) {
    float* s = ws.take<float>(64);
    if ((rc = tc_space_bwd_scales(rbits, fsc, s, st))) return rc;
    bsc = s;
  }
  const int Pp = space_pp(P), Kp = space_kp(K);
  const long long CKp = (long long)C * Kp;
  // r [M, C, K] as M C rows of K columns: its terms [M, C Kp], channel c's columns from c Kp
  if ((rc = tc_split<TERMS>(r, M * (long long)C, K, bsc, rs, st, Kp))) return rc;
  // gzt <- r centers; the LayerNorm backward forms zt rsum - that
  if ((rc = tc_gemm<TERMS, true, false>({cs, rs, P, M, Kp, bsc ? bsc + 1 : nullptr, 1, C, {0, Kp, 0, Kp}, CKp, Pp, M, CKp},
                                        TcSpaceGzEpi{gzt, (long long)M * P, P}, st))) return rc;
  // output rows K..Kp-1 of a channel are not computed (M = K): they would land in the next channel's gcenters
  return tc_gemm<TERMS, true, true>({rs, zs, K, P, M, bsc ? bsc + 2 : nullptr, 1, C, {Kp, 0, 0, (int)M}, M, CKp,
                                     (long long)C * M, Pp}, TcSpaceGcEpi{gcenters, centers, rcol, (long long)K * P, P, K}, st);
}
}  // namespace vadc

extern "C" int vadc_space_cluster_bwd(const float* x, const float* mu, const float* rstd,
                                      const void* zt_state, const float* ln_w, const float* ln_b,
                                      const float* centers,
                                      const float* Ds, const float* As, const float* gD,
                                      const float* gA, const float* g_loss_sq,
                                      int64_t M, int P, int C, int K, float alpha, float* gx,
                                      float* gcenters, float* g_ln_w, float* g_ln_b,
                                      void* workspace, size_t workspace_bytes, void* stream) {
  VADC_REQUIRE(M > 0 && P > 0 && C > 0 && K > 0 && (K % 4) == 0, VADC_ERR_BAD_SHAPE);
  VADC_REQUIRE(M * (int64_t)P < (1ll << 31) && M * (int64_t)C < (1ll << 31), VADC_ERR_UNSUPPORTED);
  VADC_REQUIRE(x && mu && rstd && zt_state && ln_w && ln_b && centers && Ds && As && gx && gcenters && g_ln_w &&
               g_ln_b && workspace, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(aligned16(zt_state), VADC_ERR_MISALIGNED);
  VADC_REQUIRE(workspace_bytes >= vadc_space_cluster_bwd_workspace_bytes(M, P, C, K), VADC_ERR_WORKSPACE);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Carver ws(workspace, workspace_bytes);
  const long long T = (long long)M * P;
  float* r = ws.take<float>((size_t)M * C * K);
  float* rsum = ws.take<float>((size_t)M * C);
  float* gzt = ws.take<float>((size_t)C * T);
  float* cpart = ws.take<float>((size_t)space_colsum_chunks(M, (long long)C * K) * C * K);
  float* rcol = ws.take<float>((size_t)C * K);
  const bool tc = space_tc_ok(M, P, C, K);
  const bool tiled = ln_bwd_tile_ok(C, P, tc);
  int nb = space_ln_bwd_blocks(T, C, tiled);
  float* lnpart = ws.take<float>((size_t)nb * 2 * C);
  unsigned* rbits = ws.take<unsigned>(64);       // max |r| (float bits) for the fp16 scale of r: comes out of the row pass
  int rc;
  cudaError_t e;
  if ((rc = launch_bwd_rows(Ds, As, nullptr, gD, gA, g_loss_sq, M * (long long)C, K, alpha, r, rsum, st,
                            (tc && space_nt(C) == 2) ? rbits : nullptr))) return rc;
  if (tc) {
    // r as [M, C Kp] (batch c = its Kp-column window), centers as [C Kp, Pp] and zt as [C M, Pp] (terms the forward kept):
    //   acc[c]^T = centers[c]^T r[:,c,:]^T   (gzt = zt rsum - acc is formed by the LayerNorm backward)   rows = positions p:
    //                                        A = centers MN-major, B = r K-major
    //   gcenters[c] = centers[c] rcol[c] - r[:,c,:]^T zt[c]    A MN-major (window offset along m), B MN-major
    void* rs = ws.take<uint8_t>(tc_terms_bytes(3, M, (long long)C * space_kp(K)));
    const int nt = space_nt(C);
    const void* zs = zt_state;
    const uint8_t* cs = static_cast<const uint8_t*>(zt_state) + space_zt_bytes(M, P, C);
    const float* fsc = reinterpret_cast<const float*>(cs + space_cen_bytes(P, C, K));
    e = launch_space_colsum(r, M, C * K, cpart, rcol, st);
    if (e != cudaSuccess) return record_cuda_error(e, "space colsum r");
    if ((rc = nt == 2 ? space_bwd_tc<2>(r, rs, rbits, fsc, zs, cs, centers, M, P, C, K, gzt, rcol, gcenters, ws, st)
                      : space_bwd_tc<3>(r, rs, rbits, fsc, zs, cs, centers, M, P, C, K, gzt, rcol, gcenters, ws, st))) return rc;
  } else {
    const float* zt = static_cast<const float*>(zt_state);
    // gzt[c] = zt[c] * rsum[:,c] - r[:,c,:] @ centers[c]
    {
      Operand Aop{r, (long long)C * K, 1}, Bop{centers, P, 1};
      SpaceGzEpilogue epi{gzt, zt, rsum, T, P, C};
      e = sgemm_auto((int)M, P, K, Aop, Bop, K, (long long)K * P, C, 1, epi, st);
      if (e != cudaSuccess) return record_cuda_error(e, "space bwd sgemm r.c");
    }
    // gcenters[c] = centers[c] * rcol[c] - r[:,c,:]^T @ zt[c]
    e = launch_space_colsum(r, M, C * K, cpart, rcol, st);
    if (e != cudaSuccess) return record_cuda_error(e, "space colsum r");
    Operand Aop{r, 1, (long long)C * K}, Bop{zt, P, 1};
    SpaceGcEpilogue epi{gcenters, centers, rcol, (long long)K * P, P, K};
    e = sgemm_auto(K, P, (int)M, Aop, Bop, K, T, C, 1, epi, st);
    if (e != cudaSuccess) return record_cuda_error(e, "space bwd sgemm rT.zt");
  }
  if (tiled) {
    if ((rc = launch_ln_bwd_tile(gzt, x, mu, rstd, ln_w, ln_b, tc ? rsum : nullptr, P, T, C, gx, lnpart, nb, st))) return rc;
  } else {
    size_t smem = ((size_t)32 * (C + 1) + (size_t)8 * 2 * C) * sizeof(float);
    if (smem > 48 * 1024)
      VADC_CUDA(cudaFuncSetAttribute(ln_bwd_transposed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ln_bwd_transposed_kernel<<<nb, 256, smem, st>>>(gzt, x, mu, rstd, ln_w, ln_b, tc ? rsum : nullptr, P, T, C, gx, lnpart);
    VADC_CHECK_LAUNCH("ln_bwd_transposed_kernel");
  }
  ln_bwd_finalize2_kernel<<<(2 * C + 31) / 32, 256, 0, st>>>(lnpart, nb, C, g_ln_w, g_ln_b);
  VADC_CHECK_LAUNCH("ln_bwd_finalize2_kernel");
  return VADC_OK;
}
