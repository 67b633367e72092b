// cluster_tc.cu — fused cluster forward (C1 + L1) on tcgen05 / TMEM / TMA.
//
//   model/cluster.py:81-99 + model/backbone.py:98 in ONE persistent kernel:
//   LayerNorm -> distance GEMM (tcgen05, TMEM accumulator) -> epilogue
//   {sqrt/clamp, row min + argmin, softmin, sum (D*A)^2} -> x_rec GEMM
//   (tcgen05) -> TMA tensor stores of D, A, x_rec.
//
// fp32-faithful tensor-core arithmetic: every fp32 operand v is split exactly
// into three bf16 terms v = v1 + v2 + v3 (8+8+8 mantissa bits) and the product
// is accumulated in fp32 TMEM from the six terms of order <= 2^-16
// (v1w1, v1w2, v2w1, v1w3, v2w2, v3w1); the dropped terms are <= 2^-24
// relative, i.e. below fp32 rounding.  kind::f16 is used rather than kind::tf32
// because bf16 K-major and MN-major SWIZZLE_128B tiles are byte-identical, so
// one shared-memory image of the centroids feeds both GEMMs (tf32 MN-major
// needs a different swizzle; tests/test_gpu_umma.py).
//
// One CTA (256 threads) per SM, persistent over 128-token tiles:
//   P1  8 warps: x rows (L2-prefetched one tile ahead by cp.async.bulk.prefetch)
//       -> LayerNorm in registers -> feature rows to HBM (coalesced float4) ->
//       3 bf16 terms into SWIZZLE_128B K-major operand tiles in shared memory
//   P2  1 thread: 6 x C/16 tcgen05.mma (M=128, N=K, K=16) -> TMEM cols [0,K)
//   P3  warps 0-3 (thread = token row): tcgen05.ld, distance / argmin / softmin /
//       loss, D and A rows into swizzled staging tiles (TMA tensor store), A's
//       3 bf16 terms as the (un-swizzled K-major) A operand of GEMM2
//   P4  1 thread: 6 x K/16 tcgen05.mma (M=128, N=C) against the SAME centroid
//       tiles read MN-major -> TMEM cols [K, K+C)
//   P5  8 warps: tcgen05.ld -> swizzled staging -> TMA tensor store of x_rec
// Shared memory (C=192, K=64): 144 KB token operand (re-used as staging after
// GEMM1), 72 KB centroid operand, loaded once per CTA by a bulk TMA copy.
#include <cuda.h>
#include <algorithm>
#include <stdio.h>
#include "common.cuh"
#include "tc_common.cuh"
#include "cluster.h"
#include "rows.cuh"

namespace vadc {
using namespace tc;

constexpr int kTileM = 128;
constexpr int kTcThreads = 256;

struct TcSmemPlan {
  uint32_t z_bytes, c_bytes, a_off, dst_off, ast_off, xst_off, alias_end;
  uint32_t cc_off, zz_off, misc_off, total;
};

__host__ __device__ inline TcSmemPlan tc_plan(int C, int K) {
  TcSmemPlan p;
  p.z_bytes = 3u * kTileM * C * 2u;                 // three bf16 terms of the 128 x C token tile
  p.c_bytes = 3u * K * C * 2u;                      // three bf16 terms of the K x C centroids
  p.a_off = 0;                                      // aliases the token operand after GEMM1
  p.dst_off = p.a_off + 2u * kTileM * K * 2u;       // (2 bf16 terms of A) then D staging [K/32][128 x 128 B]
  p.ast_off = p.dst_off + kTileM * K * 4u;          // A staging
  p.xst_off = p.ast_off + kTileM * K * 4u;          // x_rec staging, 2 slots of [128 x 128 B]
  p.alias_end = p.xst_off + 2u * kTileM * 128u;
  uint32_t off = p.z_bytes + p.c_bytes;
  p.cc_off = off; off += K * 4u;
  p.zz_off = off; off += kTileM * 4u;
  p.misc_off = off; off += 128u;
  p.total = off;
  return p;
}

// ---------------------------------------------------------------------------
// centroid prologue: 3-term bf16 split written as the shared-memory IMAGE
// (per term: C/64 blocks of [K rows x 128 B], SWIZZLE_128B), plus |c_k|^2.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
centroid_prep_kernel(const float* __restrict__ centers, int K, int C, uint8_t* __restrict__ image,
                     float* __restrict__ cc) {
  const int k = blockIdx.x;
  __shared__ float red[32];
  float s = 0.f;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float v = centers[(size_t)k * C + c];
    s += v * v;
    __nv_bfloat16 t[3];
    split_bf16x3(v, t);
    uint32_t off = (uint32_t)(c / 64) * (K * 128u) + sw128(k, (c % 64) * 2);
    const uint32_t term = (uint32_t)K * C * 2u;
    *reinterpret_cast<__nv_bfloat16*>(image + off) = t[0];
    *reinterpret_cast<__nv_bfloat16*>(image + term + off) = t[1];
    *reinterpret_cast<__nv_bfloat16*>(image + 2 * term + off) = t[2];
  }
  s = block_sum<float>(s, red);
  if (threadIdx.x == 0) cc[k] = s;
}

// packed 3-term split of two floats: one F2FP per term converts and packs both values
__device__ __forceinline__ uint32_t pack_rn(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);       // a -> low half, b -> high half
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ float bf_lo(uint32_t p) { return __uint_as_float(p << 16); }
__device__ __forceinline__ float bf_hi(uint32_t p) { return __uint_as_float(p & 0xFFFF0000u); }
__device__ __forceinline__ void split3_pair(float a, float b, uint32_t& p1, uint32_t& p2, uint32_t& p3) {
  p1 = pack_rn(a, b);
  float ra = a - bf_lo(p1), rb = b - bf_hi(p1);
  p2 = pack_rn(ra, rb);
  ra -= bf_lo(p2); rb -= bf_hi(p2);
  p3 = pack_rn(ra, rb);
}
__device__ __forceinline__ void split2_pair(float a, float b, uint32_t& p1, uint32_t& p2) {
  p1 = pack_rn(a, b);
  p2 = pack_rn(a - bf_lo(p1), b - bf_hi(p1));
}
__device__ __forceinline__ float fast_sqrt(float x) {
  float r;
  asm("sqrt.approx.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float fast_rcp(float x) {
  float r;
  asm("rcp.approx.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

__device__ __forceinline__ uint32_t pack2(__nv_bfloat16 a, __nv_bfloat16 b) {
  return (uint32_t)__bfloat16_as_ushort(a) | ((uint32_t)__bfloat16_as_ushort(b) << 16);
}

__device__ __forceinline__ void named_bar(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// 1D bulk copy global -> shared with mbarrier completion
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

struct TcParams {
  const float* x; const float* ln_w; const float* ln_b;
  const uint8_t* cimage; const float* cc;
  float* feature; long long* label; float* mu; float* rstd; double* partial;
  long long N; int C, K; float alpha, eps;
};

template <int F4, int KCH>
__global__ void __launch_bounds__(kTcThreads, 1)
cluster_fwd_tc_kernel(const __grid_constant__ CUtensorMap mapD, const __grid_constant__ CUtensorMap mapA,
                      const __grid_constant__ CUtensorMap mapR, const TcParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr int C = F4 * 32, K = KCH * 32;
  const TcSmemPlan pl = tc_plan(C, K);
  uint8_t* sZ = smem;                                   // [3][C/64][128 x 128 B]
  uint8_t* sC = smem + pl.z_bytes;                      // [3][C/64][K x 128 B]
  float* sCC = reinterpret_cast<float*>(smem + pl.cc_off);
  float* sZZ = reinterpret_cast<float*>(smem + pl.zz_off);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + pl.misc_off);     // [0] centroids, [1] gemm1, [2] gemm2
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + pl.misc_off + 32);
  double* loss_acc = reinterpret_cast<double*>(smem + pl.misc_off + 40);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const long long ntiles = (p.N + kTileM - 1) / kTileM;
  const uint32_t zterm = (uint32_t)kTileM * C * 2u;     // bytes per bf16 term of the token tile
  const uint32_t cterm = (uint32_t)K * C * 2u;
  uint32_t ncols = 32;
  while (ncols < (uint32_t)(K + C)) ncols <<= 1;

  if (tid == 0) {
    mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); mbar_init(&bars[2], 1);
    fence_mbar_init();
    *loss_acc = 0.0;
    prefetch_tmap(&mapD); prefetch_tmap(&mapA); prefetch_tmap(&mapR);
  }
  if (warp == 1) tmem_alloc(tmem_slot, ncols);
  for (int k = tid; k < K; k += kTcThreads) sCC[k] = p.cc[k];
  __syncthreads();
  if (tid == 0) {                                       // centroid operand image: bulk TMA copy, once per CTA
    mbar_expect_tx(&bars[0], pl.c_bytes);
    for (uint32_t off = 0; off < pl.c_bytes; off += 32768u) {
      uint32_t n = min(32768u, pl.c_bytes - off);
      bulk_g2s(sC + off, p.cimage + off, n, &bars[0]);
    }
    long long t0 = blockIdx.x;
    if (t0 < ntiles) {
      long long rows = min((long long)kTileM, p.N - t0 * kTileM);
      prefetch_l2_bulk(p.x + t0 * kTileM * C, (uint32_t)(rows * C * 4));
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t tmemD = tmem, tmemR = tmem + (uint32_t)K;

  // P1 mapping: 8 lanes per token row (lane j owns float4 chunks j, j+8, ...), 4 rows per warp
  // instruction; the two rows sharing a 16-lane store phase differ by 4 so that their swizzled
  // 64-byte pieces fall in disjoint banks.
  const int lj = lane & 7, lg = lane >> 3;
  const int rsel = (lg & 1) * 4 + (lg >> 1);            // rows +0, +4, +1, +5 within an 8-row block
  float4 gam[F4], bet[F4];
#pragma unroll
  for (int i = 0; i < F4; ++i) {
    gam[i] = __ldg(reinterpret_cast<const float4*>(p.ln_w) + lj + 8 * i);
    bet[i] = __ldg(reinterpret_cast<const float4*>(p.ln_b) + lj + 8 * i);
  }
  const uint32_t idesc1 = instr_desc(kFmtBF16, 128, K, 0, 0);
  const uint32_t idesc2 = instr_desc(kFmtBF16, 128, C, 0, 1);
  const float invC = 1.0f / (float)C;
  float loss_thread = 0.f;
  uint32_t phase = 0;

  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, phase ^= 1) {
    const long long row0 = tile * kTileM;
    if (tid == 0) {                                     // L2 prefetch of the next tile's tokens
      long long tn = tile + gridDim.x;
      if (tn < ntiles) {
        long long rows = min((long long)kTileM, p.N - tn * kTileM);
        prefetch_l2_bulk(p.x + tn * kTileM * C, (uint32_t)(rows * C * 4));
      }
    }
    // ------------------------------------------------------------------ P1
    for (int blk = warp; blk < kTileM / 8; blk += kTcThreads / 32) {
      float4 v[2][F4];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const long long row = row0 + blk * 8 + rsel + 2 * u;
        const float4* xr = reinterpret_cast<const float4*>(p.x + row * C) + lj;
#pragma unroll
        for (int i = 0; i < F4; ++i)
          v[u][i] = (row < p.N) ? ld_stream(xr + 8 * i) : make_float4(0, 0, 0, 0);
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int r = blk * 8 + rsel + 2 * u;
        const long long row = row0 + r;
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < F4; ++i) s += (v[u][i].x + v[u][i].y) + (v[u][i].z + v[u][i].w);
        s += __shfl_xor_sync(0xffffffffu, s, 1);
        s += __shfl_xor_sync(0xffffffffu, s, 2);
        s += __shfl_xor_sync(0xffffffffu, s, 4);
        const float mean = s * invC;
        float q = 0.f;
#pragma unroll
        for (int i = 0; i < F4; ++i) {
          v[u][i].x -= mean; v[u][i].y -= mean; v[u][i].z -= mean; v[u][i].w -= mean;
          q += (v[u][i].x * v[u][i].x + v[u][i].y * v[u][i].y) + (v[u][i].z * v[u][i].z + v[u][i].w * v[u][i].w);
        }
        q += __shfl_xor_sync(0xffffffffu, q, 1);
        q += __shfl_xor_sync(0xffffffffu, q, 2);
        q += __shfl_xor_sync(0xffffffffu, q, 4);
        const float rs = 1.0f / sqrtf(q * invC + p.eps);
        const bool live = row < p.N;
        float nz = 0.f;
        const uint32_t rowoff = (uint32_t)r * 128u;
        const uint32_t rx = (uint32_t)(r & 7);
        float4* frow = reinterpret_cast<float4*>(p.feature + row * C) + lj;
#pragma unroll
        for (int i = 0; i < F4; ++i) {
          float4 o;
          o.x = v[u][i].x * rs * gam[i].x + bet[i].x;
          o.y = v[u][i].y * rs * gam[i].y + bet[i].y;
          o.z = v[u][i].z * rs * gam[i].z + bet[i].z;
          o.w = v[u][i].w * rs * gam[i].w + bet[i].w;
          if (live) frow[8 * i] = o; else o = make_float4(0, 0, 0, 0);
          nz += (o.x * o.x + o.y * o.y) + (o.z * o.z + o.w * o.w);
          uint32_t a1, a2, a3, b1, b2, b3;
          split3_pair(o.x, o.y, a1, a2, a3);
          split3_pair(o.z, o.w, b1, b2, b3);
          const int f = lj + 8 * i;                          // float4 index in the row: channels 4f..4f+3
          const uint32_t byte = (uint32_t)(f & 15) * 8u;     // 8 bytes of bf16 in the 128-byte row of block f/16
          const uint32_t off = (uint32_t)(f >> 4) * (kTileM * 128u) + rowoff + ((((byte >> 4) ^ rx) << 4) | (byte & 15u));
          *reinterpret_cast<uint2*>(sZ + off) = make_uint2(a1, b1);
          *reinterpret_cast<uint2*>(sZ + zterm + off) = make_uint2(a2, b2);
          *reinterpret_cast<uint2*>(sZ + 2 * zterm + off) = make_uint2(a3, b3);
        }
        nz += __shfl_xor_sync(0xffffffffu, nz, 1);
        nz += __shfl_xor_sync(0xffffffffu, nz, 2);
        nz += __shfl_xor_sync(0xffffffffu, nz, 4);
        if (lj == 0) {
          sZZ[r] = nz;
          if (live) { p.mu[row] = mean; p.rstd[row] = rs; }
        }
      }
    }
    fence_async_smem();
    __syncthreads();
    // ------------------------------------------------------------------ P2
    if (tid == 0) {
      if (tile == (long long)blockIdx.x) mbar_wait(&bars[0], 0);        // centroid image landed
      tc_fence_after();
      const uint32_t zb = smem_u32(sZ), cb = smem_u32(sC);
      uint32_t acc = 0;
      const int pi[6] = {0, 0, 1, 0, 1, 2}, pj[6] = {0, 1, 0, 2, 1, 0};
#pragma unroll 1
      for (int t = 0; t < 6; ++t) {
        const uint32_t za = zb + pi[t] * zterm, ca = cb + pj[t] * cterm;
        for (int kk = 0; kk < C / 16; ++kk) {
          uint64_t ad = smem_desc_sw128(za + (kk >> 2) * (kTileM * 128u) + (kk & 3) * 32u, 0, 1024);
          uint64_t bd = smem_desc_sw128(ca + (kk >> 2) * (K * 128u) + (kk & 3) * 32u, 0, 1024);
          mma_f16(tmemD, ad, bd, idesc1, acc);
          acc = 1;
        }
      }
      mma_commit(&bars[1]);
    }
    // ------------------------------------------------------------------ P3
    if (warp < 4) {
      mbar_wait(&bars[1], phase);
      tc_fence_after();
      const int r = tid;                                 // token row of this thread (TMEM lane)
      const long long row = row0 + r;
      const uint32_t lane_addr = (uint32_t)(warp * 32) << 16;
      const float zz = sZZ[r];
      const bool live = row < p.N;
      const float nalpha = -p.alpha * 1.4426950408889634f;     // exp(-a t) = 2^(-a log2(e) t)
      float best = INFINITY; int bidx = 0;
      float dv[32];
      for (int c0 = 0; c0 < K; c0 += 32) {
        tmem_ld32(tmemD + lane_addr + c0, dv);
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          float d = fast_sqrt(fmaxf(zz + sCC[c0 + j] - 2.0f * dv[j], 0.f));
          if (d < best) { best = d; bidx = c0 + j; }
        }
      }
      float sum = 0.f;
      for (int c0 = 0; c0 < K; c0 += 32) {
        tmem_ld32(tmemD + lane_addr + c0, dv);
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          float d = fast_sqrt(fmaxf(zz + sCC[c0 + j] - 2.0f * dv[j], 0.f));
          sum += exp2f(nalpha * (d - best));
        }
      }
      for (int c0 = 0; c0 < K; c0 += 32) {
        float ev[32];
        tmem_ld32(tmemD + lane_addr + c0, dv);
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          dv[j] = fast_sqrt(fmaxf(zz + sCC[c0 + j] - 2.0f * dv[j], 0.f));
          ev[j] = exp2f(nalpha * (dv[j] - best));
        }
        const float inv = fast_rcp(sum);
        uint8_t* dblk = smem + pl.dst_off + (c0 >> 5) * (kTileM * 128u);
        uint8_t* ablk = smem + pl.ast_off + (c0 >> 5) * (kTileM * 128u);
        float lrow = 0.f;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            ev[4 * q + e] *= inv;
            float pr = dv[4 * q + e] * ev[4 * q + e];
            lrow = fmaf(pr, pr, lrow);
          }
          *reinterpret_cast<float4*>(dblk + sw128(r, q * 16)) = make_float4(dv[4 * q], dv[4 * q + 1], dv[4 * q + 2], dv[4 * q + 3]);
          *reinterpret_cast<float4*>(ablk + sw128(r, q * 16)) = make_float4(ev[4 * q], ev[4 * q + 1], ev[4 * q + 2], ev[4 * q + 3]);
        }
        if (live) loss_thread += lrow;
        // A operand of GEMM2: 2 bf16 terms, un-swizzled K-major core matrices (8 rows x 16 B)
#pragma unroll
        for (int kc = 0; kc < 4; ++kc) {
          uint32_t w1[4], w2[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) split2_pair(ev[8 * kc + 2 * e], ev[8 * kc + 2 * e + 1], w1[e], w2[e]);
          const uint32_t off = (uint32_t)((c0 >> 3) + kc) * 2048u + (r >> 3) * 128u + (r & 7) * 16u;
          const uint32_t aterm = (uint32_t)kTileM * K * 2u;
          *reinterpret_cast<uint4*>(smem + pl.a_off + off) = make_uint4(w1[0], w1[1], w1[2], w1[3]);
          *reinterpret_cast<uint4*>(smem + pl.a_off + aterm + off) = make_uint4(w2[0], w2[1], w2[2], w2[3]);
        }
      }
      if (row < p.N) p.label[row] = bidx;
      fence_async_smem();
      tc_fence_before();
      named_bar(1, 128);
      // ---------------------------------------------------------------- P4
      if (tid == 0) {
        tc_fence_after();
        for (int b = 0; b < K / 32; ++b) {
          tma_store_2d(&mapD, smem + pl.dst_off + b * (kTileM * 128u), b * 32, (int)row0);
          tma_store_2d(&mapA, smem + pl.ast_off + b * (kTileM * 128u), b * 32, (int)row0);
        }
        bulk_commit();
        const uint32_t ab = smem_u32(smem + pl.a_off), cb = smem_u32(sC);
        const uint32_t aterm = (uint32_t)kTileM * K * 2u;
        uint32_t acc = 0;
        const int pi[5] = {0, 0, 1, 0, 1}, pj[5] = {0, 1, 0, 2, 1};
#pragma unroll 1
        for (int t = 0; t < 5; ++t) {
          for (int ks = 0; ks < K / 16; ++ks) {
            uint64_t ad = smem_desc_noswz(ab + pi[t] * aterm + (uint32_t)(2 * ks) * 2048u, 2048, 128);
            uint64_t bd = smem_desc_sw128(cb + pj[t] * cterm + (uint32_t)(2 * ks) * 1024u, (uint32_t)K * 128u, 1024);
            mma_f16(tmemR, ad, bd, idesc2, acc);
            acc = 1;
          }
        }
        mma_commit(&bars[2]);
      }
    }
    // ------------------------------------------------------------------ P5
    {
      mbar_wait(&bars[2], phase);
      tc_fence_after();
      const int half = warp >> 2, q4 = warp & 3;
      const int r = q4 * 32 + lane;
      uint8_t* slot = smem + pl.xst_off + half * (kTileM * 128u);
      const bool issuer = (q4 == 0 && lane == 0);
      float xv[32];
      for (int ch = half; ch < C / 32; ch += 2) {
        tmem_ld32(tmemR + ((uint32_t)(q4 * 32) << 16) + ch * 32, xv);
        if (issuer) bulk_wait_read0();                   // previous store out of this slot has been read
        named_bar(2 + half, 128);
#pragma unroll
        for (int q = 0; q < 8; ++q)
          *reinterpret_cast<float4*>(slot + sw128(r, q * 16)) = make_float4(xv[4 * q], xv[4 * q + 1], xv[4 * q + 2], xv[4 * q + 3]);
        fence_async_smem();
        named_bar(2 + half, 128);
        if (issuer) { tma_store_2d(&mapR, slot, ch * 32, (int)row0); bulk_commit(); }
      }
      if (issuer || tid == 0) bulk_wait_read0();         // staging aliases the next tile's operand tiles
    }
    tc_fence_before();
    __syncthreads();
  }
  // ---- teardown
  loss_thread = warp_sum(loss_thread);
  if (lane == 0 && warp < 4) atomicAdd(loss_acc, (double)loss_thread);
  if (tid == 0 || tid == 128) bulk_wait0();
  __syncthreads();
  if (tid == 0) {
    if (ntiles <= (long long)blockIdx.x) mbar_wait(&bars[0], 0);     // never consumed: drain the bulk copy
    p.partial[blockIdx.x] = *loss_acc;
  }
  if (warp == 1) tmem_dealloc(tmem, ncols);
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* ptr = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess ||
      qres != cudaDriverEntryPointSuccess) {
    (void)cudaGetLastError();
    return nullptr;
  }
  fn = reinterpret_cast<EncodeTiledFn>(ptr);
  return fn;
}

// [rows, cols] fp32 row-major tensor, box = 32 columns x 128 rows, SWIZZLE_128B
static int make_map(CUtensorMap* m, float* base, long long rows, int cols) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return VADC_ERR_CUDA;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)cols * 4};
  cuuint32_t box[2] = {32, (cuuint32_t)kTileM};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    snprintf(g_last_cuda_error, sizeof(g_last_cuda_error), "cuTensorMapEncodeTiled failed: %d", (int)r);
    return VADC_ERR_CUDA;
  }
  return VADC_OK;
}

static bool tc_shape_ok(long long N, int C, int K) {
  if (N < 1 || N >= (1ll << 31)) return false;
  // the one instantiated shape: K = 32 runs cluster_fwd_ws, and at C = 64 / 128 the K = 64 staging does not fit
  if (C != 192 || K != 64) return false;
  TcSmemPlan pl = tc_plan(C, K);
  if (pl.alias_end > pl.z_bytes) return false;          // staging must fit in the dead operand tiles
  if (pl.total + 1024 > 227 * 1024) return false;
  return true;
}

}  // namespace vadc

using namespace vadc;

extern "C" size_t vadc_cluster_tc_extra_workspace_bytes(int64_t N, int C, int K) {
  if (!tc_shape_ok(N, C, K)) return 0;
  return align_up((size_t)3 * K * C * 2, 256) + align_up((size_t)(sm_count() + 1) * sizeof(double), 256) +
         align_up((size_t)K * sizeof(float), 256) + 256;
}

int vadc_cluster_fwd_tc(const float* x, const float* ln_w, const float* ln_b, const float* centers,
                        int64_t N, int C, int K, float alpha, float eps, float* D, float* A,
                        float* x_rec, float* feature, int64_t* label, float* mu, float* rstd,
                        float* loss_sq, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  if (!tc_shape_ok(N, C, K)) return VADC_ERR_UNSUPPORTED;
  if (!vadc_device_ok()) return VADC_ERR_NO_DEVICE;
  if (workspace_bytes < vadc_cluster_tc_extra_workspace_bytes(N, C, K)) return VADC_ERR_WORKSPACE;
  Carver ws(workspace, workspace_bytes);       // the SIMT carve is not live on this path
  uint8_t* image = ws.take<uint8_t>((size_t)3 * K * C * 2);
  const int grid = (int)std::min<long long>((N + kTileM - 1) / kTileM, sm_count());
  double* partial = ws.take<double>(sm_count() + 1);
  float* cc = ws.take<float>(K);

  CUtensorMap mD, mA, mR;
  int rc;
  if ((rc = make_map(&mD, D, N, K))) return rc;
  if ((rc = make_map(&mA, A, N, K))) return rc;
  if ((rc = make_map(&mR, x_rec, N, C))) return rc;

  centroid_prep_kernel<<<K, 256, 0, st>>>(centers, K, C, image, cc);
  VADC_CHECK_LAUNCH("centroid_prep_kernel");

  const TcSmemPlan pl = tc_plan(C, K);
  const size_t smem = pl.total + 1024;
  TcParams p{x, ln_w, ln_b, image, cc, feature, reinterpret_cast<long long*>(label), mu, rstd, partial,
             (long long)N, C, K, alpha, eps};
  VADC_CUDA(cudaFuncSetAttribute(cluster_fwd_tc_kernel<6, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  cluster_fwd_tc_kernel<6, 2><<<grid, kTcThreads, smem, st>>>(mD, mA, mR, p);
  VADC_CHECK_LAUNCH("cluster_fwd_tc_kernel");
  finalize_sum_kernel<<<1, 1024, 0, st>>>(partial, grid, loss_sq);
  VADC_CHECK_LAUNCH("finalize_sum_kernel");
  return VADC_OK;
}
