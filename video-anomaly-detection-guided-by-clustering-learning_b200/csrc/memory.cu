// memory.cu — Memory module (M1-M5), model/Memory.py:62-261 (MNAD memory):
// addressing scores with the two softmaxes, top-1/top-2 slots, read,
// gather / spread losses, weighted segmented update, separateness.
#include <algorithm>
#include "common.cuh"
#include "sgemm.cuh"
#include "tc_gemm.cuh"
#include "rows.cuh"
#include "cluster.h"

namespace vadc {

// ---- F.normalize(query, dim=1) + permute (Memory.py:148-149) --------------
// query [B, d, HW]: norms over d for every (b, hw); threads run along hw.
__global__ void __launch_bounds__(256)
query_norm_kernel(const float* __restrict__ query, int d, long long HW, float* __restrict__ inv) {
  // 32 positions per block (lanes), the eight warps split the channels: 128-byte reads, four independent chains per thread
  __shared__ float red[8][33];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const long long hw = (long long)blockIdx.x * 32 + lane;
  const int b = blockIdx.y;
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  if (hw < HW) {
    const float* p = query + (long long)b * d * HW + hw;
    int c = wid;
    for (; c + 24 < d; c += 32) {
      const float v0 = __ldg(p + (long long)c * HW), v1 = __ldg(p + (long long)(c + 8) * HW);
      const float v2 = __ldg(p + (long long)(c + 16) * HW), v3 = __ldg(p + (long long)(c + 24) * HW);
      s0 += v0 * v0; s1 += v1 * v1; s2 += v2 * v2; s3 += v3 * v3;
    }
    for (; c < d; c += 8) { const float v = __ldg(p + (long long)c * HW); s0 += v * v; }
  }
  red[wid][lane] = (s0 + s1) + (s2 + s3);
  __syncthreads();
  if (wid == 0 && hw < HW) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += red[w][lane];
    inv[(long long)b * HW + hw] = 1.0f / fmaxf(sqrtf(s), 1e-12f);
  }
}

// tiled transpose with the per-position scale: q[(b*HW+hw), c] = query[b,c,hw]*inv; a block moves 32 positions x 128
// channels (128-byte reads per channel row, 512 contiguous bytes per written token row)
__global__ void __launch_bounds__(256)
query_transpose_kernel(const float* __restrict__ query, const float* __restrict__ inv, int d,
                       long long HW, float* __restrict__ q) {
  __shared__ float tile[128][33];
  const int b = blockIdx.z;
  const long long hw0 = (long long)blockIdx.x * 32;
  const int c0 = blockIdx.y * 128;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
#pragma unroll 4
  for (int j = ty; j < 128; j += 8) {
    const int c = c0 + j;
    const long long hw = hw0 + tx;
    tile[j][tx] = (c < d && hw < HW) ? __ldg(query + ((long long)b * d + c) * HW + hw) : 0.f;
  }
  __syncthreads();
  for (int j = ty; j < 32; j += 8) {
    const long long hw = hw0 + j;
    if (hw >= HW) continue;
    const float sc = __ldg(inv + (long long)b * HW + hw);
    float* dst = q + ((long long)b * HW + hw) * d + c0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int c = tx + 32 * i;
      if (c0 + c < d) dst[c] = tile[c][j] * sc;
    }
  }
}


// ---- backward of Memory.forward with respect to `query` -------------------
// autograd of Memory.py:145-175.  What reaches `query` in the reference graph: the first half of
// updated_query (cat, :256 — the read softmax is .detach()ed, :255), MSELoss(q, keys[top1].detach())
// (:245) and TripletMarginLoss(margin=1, p=2, eps=1e-6)(q, pos.detach(), neg.detach()) (:229); then
// F.normalize(query, dim=1) (:148).  Everything is per token, so one kernel does it in the query's own
// [B, d, HW] layout: lanes run along hw (coalesced), the 8 warps of a block split the channels and meet
// in shared memory for the three per-token reductions (|x|^2; the two triplet distances; q . g).
//   g[c]  = gU[b,c,hw] + gQ[b,c,hw] + ag (q - k1) + cp (q - k1 + eps) - cn (q - k2 + eps)
//   gx[c] = (g[c] - q[c] (q . g)) / |x|            (g / 1e-12 where |x| < 1e-12: the clamp is constant)
// gQ (optional) is the gradient with respect to q-hat that the score matrices contribute (vadc_memory_scores_bwd).
// The per-token loss maths below is shared with the channel-last twin (memory_rows_bwd_kernel).
constexpr float kTripletEps = 1e-6f;            // pairwise_distance eps (TripletMarginLoss)

// the loss weights: ag = 2 g_gather / (N d) (MSELoss mean), gs = g_spread / N (TripletMarginLoss mean)
__device__ __forceinline__ void memory_loss_weights(const float* g_gather, const float* g_spread, bool spread,
                                                    long long N, int d, float& ag, float& gs) {
  ag = g_gather ? 2.0f * __ldg(g_gather) / ((float)N * (float)d) : 0.f;
  gs = (g_spread && spread) ? __ldg(g_spread) / (float)N : 0.f;
}

// triplet coefficients from the two squared distances |q - k1 + eps|^2, |q - k2 + eps|^2 (clamp_min(., 0) backward)
__device__ __forceinline__ void triplet_coefs(float dp2, float dn2, float gs, float& cp, float& cn) {
  const float dap = sqrtf(dp2), dan = sqrtf(dn2);
  const bool active = dap - dan + 1.0f >= 0.f;
  cp = (active && dap > 0.f) ? gs / dap : 0.f;
  cn = (active && dan > 0.f) ? gs / dan : 0.f;
}

// g + the gathering and spreading terms at one channel: ag (q - k1) + cp (q - k1 + eps) - cn (q - k2 + eps)
__device__ __forceinline__ float add_loss_grads(float g, float q, float k1, const float* k2, int c, float ag, float cp,
                                                float cn) {
  const float a = q - k1;
  g += ag * a + cp * (a + kTripletEps);
  if (k2) g -= cn * (q - __ldg(k2 + c) + kTripletEps);
  return g;
}

__global__ void __launch_bounds__(256)
memory_query_bwd_kernel(const float* __restrict__ query, const float* __restrict__ keys,
                        const long long* __restrict__ top1, const long long* __restrict__ top2,
                        const float* __restrict__ g_uq, const float* __restrict__ g_gather,
                        const float* __restrict__ g_spread, const float* __restrict__ g_qhat, int d, long long HW,
                        long long N, float* __restrict__ gquery) {
  __shared__ float red[2][8][32];
  __shared__ float tot[2][32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int b = blockIdx.y;
  const long long hw = (long long)blockIdx.x * 32 + lane;
  const bool live = hw < HW;
  const long long n = (long long)b * HW + hw;
  const float* xp = query + (long long)b * d * HW + hw;
  const float* gp = g_uq ? g_uq + (long long)b * 2 * d * HW + hw : nullptr;
  const float* hp = g_qhat ? g_qhat + (long long)b * d * HW + hw : nullptr;
  const float* k1 = live ? keys + top1[n] * d : keys;
  const float* k2 = (live && top2) ? keys + top2[n] * d : nullptr;
  float ag, gs;
  memory_loss_weights(g_gather, g_spread, top2 != nullptr, N, d, ag, gs);
  constexpr float kEps = kTripletEps;
  auto reduce2 = [&](float a, float c) {      // block-wide sums per lane (token) of two values
    red[0][wid][lane] = a; red[1][wid][lane] = c;
    __syncthreads();
    if (wid < 2) {
      float t = 0.f;
      for (int w = 0; w < 8; ++w) t += red[wid][w][lane];
      tot[wid][lane] = t;
    }
    __syncthreads();
  };
  // 1: |x|^2
  float s = 0.f;
  if (live) for (int c = wid; c < d; c += 8) { const float v = __ldg(xp + (long long)c * HW); s += v * v; }
  reduce2(s, 0.f);
  const float nrm = sqrtf(tot[0][lane]);
  const bool clamped = nrm < 1e-12f;
  const float inv = 1.0f / fmaxf(nrm, 1e-12f);
  __syncthreads();
  // 2: triplet distances
  float cp = 0.f, cn = 0.f;
  if (top2 != nullptr) {                       // block-uniform
    float dp = 0.f, dn = 0.f;
    if (live) for (int c = wid; c < d; c += 8) {
      const float q = __ldg(xp + (long long)c * HW) * inv;
      const float a = q - __ldg(k1 + c) + kEps, e = q - __ldg(k2 + c) + kEps;
      dp += a * a; dn += e * e;
    }
    reduce2(dp, dn);
    triplet_coefs(tot[0][lane], tot[1][lane], gs, cp, cn);
    __syncthreads();
  }
  auto grad_at = [&](int c, float q) {
    float g = gp ? __ldg(gp + (long long)c * HW) : 0.f;
    if (hp) g += __ldg(hp + (long long)c * HW);
    return add_loss_grads(g, q, __ldg(k1 + c), k2, c, ag, cp, cn);
  };
  // 3: q . g
  float dot = 0.f;
  if (live) for (int c = wid; c < d; c += 8) {
    const float q = __ldg(xp + (long long)c * HW) * inv;
    dot += q * grad_at(c, q);
  }
  reduce2(dot, 0.f);
  dot = clamped ? 0.f : tot[0][lane];
  // 4: through the normalisation
  if (live) for (int c = wid; c < d; c += 8) {
    const float q = __ldg(xp + (long long)c * HW) * inv;
    gquery[((long long)b * d + c) * HW + hw] = (grad_at(c, q) - q * dot) * inv;
  }
}

// ---- backward of the stand-alone methods, channel-last and without the normalisation -------------------------------
// read / gather_loss / spread_loss (Memory.py:214-261) take q [N, d] as passed, so the query gradient is per token:
//   g[n, c] = gU[b, c, hw] + gR[n, c] + ag (q - k1) + cp (q - k1 + eps) - cn (q - k2 + eps),   n = b HW + hw
// A block owns 32 tokens of one batch and each warp four of them.  The triplet distances are warp sums along the
// token's row (lanes along channels); gU ([B, 2d, HW], lanes along hw) is staged through shared memory 32 channels at
// a time, so that its reads and the [N, d] writes are both 128-byte lines.  g_rows may be the output (read, then
// written by the same thread).
__global__ void __launch_bounds__(256)
memory_rows_bwd_kernel(const float* __restrict__ q, const float* __restrict__ keys, const long long* __restrict__ top1,
                       const long long* __restrict__ top2, const float* __restrict__ g_uq,
                       const float* __restrict__ g_gather, const float* __restrict__ g_spread, const float* g_rows,
                       int d, long long HW, long long N, float* gquery) {
  __shared__ float tile[32][33];               // [channel][token]
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int b = blockIdx.y;
  const long long hw0 = (long long)blockIdx.x * 32;
  float ag, gs;
  memory_loss_weights(g_gather, g_spread, top2 != nullptr, N, d, ag, gs);
  const bool losses = g_gather || (g_spread && top2);
  const float* k1[4];
  const float* k2[4];
  float cp[4], cn[4];
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    const long long hw = hw0 + wid * 4 + t, n = (long long)b * HW + hw;
    const bool live = hw < HW && losses;
    k1[t] = live ? keys + top1[n] * d : keys;
    k2[t] = (live && top2) ? keys + top2[n] * d : nullptr;
    cp[t] = cn[t] = 0.f;
    if (k2[t]) {                               // warp-uniform
      const float* qr = q + n * d;
      float dp = 0.f, dn = 0.f;
      for (int c = lane; c < d; c += 32) {
        const float v = __ldg(qr + c);
        const float a = v - __ldg(k1[t] + c) + kTripletEps, e = v - __ldg(k2[t] + c) + kTripletEps;
        dp += a * a; dn += e * e;
      }
      triplet_coefs(warp_sum(dp), warp_sum(dn), gs, cp[t], cn[t]);
    }
  }
  for (int c0 = 0; c0 < d; c0 += 32) {
    if (g_uq) {                                // block-uniform
      const long long hw = hw0 + lane;
      for (int i = wid; i < 32; i += 8)
        tile[i][lane] = (hw < HW && c0 + i < d) ? __ldg(g_uq + ((long long)b * 2 * d + c0 + i) * HW + hw) : 0.f;
      __syncthreads();
    }
    const int c = c0 + lane;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int j = wid * 4 + t;
      const long long n = (long long)b * HW + hw0 + j;
      if (hw0 + j >= HW || c >= d) continue;
      float g = g_uq ? tile[lane][j] : 0.f;
      if (g_rows) g += g_rows[n * d + c];
      if (losses) g = add_loss_grads(g, __ldg(q + n * d + c), __ldg(k1[t] + c), k2[t], c, ag, cp[t], cn[t]);
      gquery[n * d + c] = g;
    }
    if (g_uq) __syncthreads();
  }
}

// prepare_query backward (F.normalize(query, dim=1) + permute, Memory.py:148-149): g arrives channel-last [B, HW, d],
// g_x [B, d, HW] = (g - q-hat (q-hat . g)) / max(|x|, 1e-12) per token (dot = 0 where the clamp holds: the clamp is a
// constant).  A block owns 32 positions (lanes along hw: query reads and g_x writes are 128-byte lines); g is staged
// through shared memory 32 channels at a time (read along its rows), once for |x|^2 and x . g, once for g_x.
__global__ void __launch_bounds__(256)
prepare_query_bwd_kernel(const float* __restrict__ g, const float* __restrict__ query, int d, long long HW,
                         float* __restrict__ gx) {
  __shared__ float tile[32][33];               // [channel][position]
  __shared__ float red[2][8][32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int b = blockIdx.y;
  const long long hw0 = (long long)blockIdx.x * 32, hw = hw0 + lane;
  const bool live = hw < HW;
  const float* xp = query + (long long)b * d * HW + hw;
  const float* gb = g + ((long long)b * HW + hw0) * d;
  auto stage = [&](int c0) {
    for (int j = wid; j < 32; j += 8)
      tile[lane][j] = (hw0 + j < HW && c0 + lane < d) ? __ldg(gb + (long long)j * d + c0 + lane) : 0.f;
    __syncthreads();
  };
  float s = 0.f, t = 0.f;
  for (int c0 = 0; c0 < d; c0 += 32) {
    stage(c0);
    for (int i = wid; i < 32; i += 8) {
      const int c = c0 + i;
      if (live && c < d) { const float x = __ldg(xp + (long long)c * HW); s += x * x; t += x * tile[i][lane]; }
    }
    __syncthreads();
  }
  red[0][wid][lane] = s; red[1][wid][lane] = t;
  __syncthreads();
  s = 0.f; t = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) { s += red[0][w][lane]; t += red[1][w][lane]; }
  const float nrm = sqrtf(s);
  const float inv = 1.0f / fmaxf(nrm, 1e-12f);
  const float dot = nrm < 1e-12f ? 0.f : t * inv;      // q-hat . g
  for (int c0 = 0; c0 < d; c0 += 32) {
    stage(c0);
    for (int i = wid; i < 32; i += 8) {
      const int c = c0 + i;
      if (live && c < d) {
        const float qh = __ldg(xp + (long long)c * HW) * inv;
        gx[((long long)b * d + c) * HW + hw] = (tile[i][lane] - qh * dot) * inv;
      }
    }
    __syncthreads();
  }
}

// (value desc, index asc) top-2 pairs of two lanes merged; used by both row-softmax kernels
__device__ __forceinline__ void top2_merge_warp(float& b1, int& i1, float& b2, int& i2) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    float ob1 = __shfl_xor_sync(0xffffffffu, b1, o), ob2 = __shfl_xor_sync(0xffffffffu, b2, o);
    int oi1 = __shfl_xor_sync(0xffffffffu, i1, o), oi2 = __shfl_xor_sync(0xffffffffu, i2, o);
    bool other_first = (ob1 > b1) || (ob1 == b1 && oi1 < i1);
    float n1, n2; int j1, j2;
    if (other_first) {
      n1 = ob1; j1 = oi1;
      bool s = (b1 > ob2) || (b1 == ob2 && i1 < oi2);
      n2 = s ? b1 : ob2; j2 = s ? i1 : oi2;
    } else {
      n1 = b1; j1 = i1;
      bool s = (ob1 > b2) || (ob1 == b2 && oi1 < i2);
      n2 = s ? ob1 : b2; j2 = s ? oi1 : i2;
    }
    b1 = n1; i1 = j1; b2 = n2; i2 = j2;
  }
}

// register-resident row: m % 4 == 0, m <= 128 V4, 16-byte aligned rows — the logits row is read ONCE (V4 float4 per lane,
// all in flight together), top-2, sum and output come from registers
// (writing score_query = exp(logit - colmax) / colsum from the same registers was tried: 190 registers, one block per SM,
// 823 us against 328 + 187 for this kernel and the separate column pass; capped at 128 registers it spills — not kept)
template <int V4>
__global__ void __launch_bounds__(256)
row_softmax_top2_reg_kernel(const float* __restrict__ logits, long long N, int m, float* __restrict__ out,
                            long long* __restrict__ top1, long long* __restrict__ top2, __half* __restrict__ terms) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= N) return;
  const float4* l4 = reinterpret_cast<const float4*>(logits + row * m);
  const int n4 = m >> 2;
  float4 v[V4];
#pragma unroll
  for (int k = 0; k < V4; ++k) {
    const int i = lane + 32 * k;
    v[k] = i < n4 ? ld_stream(l4 + i) : make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
  }
  float b1 = -INFINITY, b2 = -INFINITY;
  int i1 = 0x7fffffff, i2 = 0x7fffffff;
#pragma unroll
  for (int k = 0; k < V4; ++k) {
    const int base = 4 * (lane + 32 * k);
    const float e[4] = {v[k].x, v[k].y, v[k].z, v[k].w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (e[j] > b1) { b2 = b1; i2 = i1; b1 = e[j]; i1 = base + j; }
      else if (e[j] > b2) { b2 = e[j]; i2 = base + j; }
    }
  }
  top2_merge_warp(b1, i1, b2, i2);
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < V4; ++k) {
    v[k] = make_float4(expf(v[k].x - b1), expf(v[k].y - b1), expf(v[k].z - b1), expf(v[k].w - b1));
    s += (v[k].x + v[k].y) + (v[k].z + v[k].w);
  }
  s = warp_sum(s);
  float* orow = out + row * m;
#pragma unroll
  for (int k = 0; k < V4; ++k) {
    const int i = lane + 32 * k;
    if (i < n4) {
      const float4 p = make_float4(v[k].x / s, v[k].y / s, v[k].z / s, v[k].w / s);
      reinterpret_cast<float4*>(orow)[i] = p;
      if (terms) {                             // the operand split of the read GEMM, written in the same pass
        const float a[4] = {p.x * 8192.0f, p.y * 8192.0f, p.z * 8192.0f, p.w * 8192.0f};
        store_terms<2, 4>(terms, N * m, row * m + 4 * i, a);
      }
    }
  }
  if (lane == 0) {
    if (top1) top1[row] = i1;
    if (top2) top2[row] = (m > 1) ? i2 : 0;
  }
}

// ---- row softmax over m + top-1 / top-2 (Memory.py:141,185,223,241) -------
// one warp per token row of logits [N, m] (parking the row in shared memory for the second and third pass was measured
// slower — 519 vs 383 us at N = 65536, m = 2000: 64 KB per block leaves three blocks per SM)
__global__ void __launch_bounds__(256)
row_softmax_top2_kernel(const float* __restrict__ logits, long long N, int m,
                        float* __restrict__ out, long long* __restrict__ top1,
                        long long* __restrict__ top2,
                        __half* __restrict__ terms /* optional: two fp16 terms of out * 2^13, [2][N*m] */) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= N) return;
  const float* lr = logits + row * m;
  float b1 = -INFINITY, b2 = -INFINITY;
  int i1 = 0x7fffffff, i2 = 0x7fffffff;
  for (int i = lane; i < m; i += 32) {
    float v = lr[i];
    if (v > b1) { b2 = b1; i2 = i1; b1 = v; i1 = i; }
    else if (v > b2) { b2 = v; i2 = i; }
  }
  top2_merge_warp(b1, i1, b2, i2);
  float s = 0.f;
  float* orow = out + row * m;
  if ((m & 3) == 0 && ((reinterpret_cast<uintptr_t>(lr) | reinterpret_cast<uintptr_t>(orow)) & 15u) == 0) {
    // 16-byte accesses (the row is L1-resident after the top-2 pass); terms as 8-byte stores
    const float4* l4 = reinterpret_cast<const float4*>(lr);
    const int n4 = m >> 2;
    for (int i = lane; i < n4; i += 32) {
      const float4 v = l4[i];
      s += (expf(v.x - b1) + expf(v.y - b1)) + (expf(v.z - b1) + expf(v.w - b1));
    }
    s = warp_sum(s);
    for (int i = lane; i < n4; i += 32) {
      const float4 v = l4[i];
      const float4 p = make_float4(expf(v.x - b1) / s, expf(v.y - b1) / s, expf(v.z - b1) / s, expf(v.w - b1) / s);
      reinterpret_cast<float4*>(orow)[i] = p;
      if (terms) {                             // the operand split of the read GEMM, written in the same pass
        const float a[4] = {p.x * 8192.0f, p.y * 8192.0f, p.z * 8192.0f, p.w * 8192.0f};
        store_terms<2, 4>(terms, N * m, row * m + 4 * i, a);
      }
    }
    if (lane == 0) {
      if (top1) top1[row] = i1;
      if (top2) top2[row] = (m > 1) ? i2 : 0;
    }
    return;
  }
  for (int i = lane; i < m; i += 32) s += expf(lr[i] - b1);
  s = warp_sum(s);
  if (terms) {                                 // the operand split of the read GEMM, written in the same pass
    for (int i = lane; i < m; i += 32) {
      const float p = expf(lr[i] - b1) / s;
      orow[i] = p;
      store_terms<2>(terms, N * m, row * m + i, p * 8192.0f);
    }
  } else {
    for (int i = lane; i < m; i += 32) orow[i] = expf(lr[i] - b1) / s;
  }
  if (lane == 0) {
    if (top1) top1[row] = i1;
    if (top2) top2[row] = (m > 1) ? i2 : 0;
  }
}

// ---- column softmax over tokens (Memory.py:140): online max/sum per chunk --
__device__ __forceinline__ void online_add(float& mx, float& s, float v) {
  if (v > mx) { s = s * expf(mx - v) + 1.0f; mx = v; } else { s += expf(v - mx); }
}
__device__ __forceinline__ void online_merge(float& mx, float& s, float omx, float os) {
  if (omx == -INFINITY) return;
  if (omx > mx) { s = s * expf(mx - omx) + os; mx = omx; } else { s += os * expf(omx - mx); }
}

// a thread owns a column of a row chunk; four independent (max, sum) chains over interleaved rows, merged in a fixed order
__global__ void __launch_bounds__(256)
col_stats_stage1_kernel(const float* __restrict__ logits, long long N, int m, long long rpb,
                        float* __restrict__ pmax, float* __restrict__ psum) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= m) return;
  long long r0 = (long long)blockIdx.y * rpb, r1 = min(N, r0 + rpb);
  float mx[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY}, sm[4] = {0.f, 0.f, 0.f, 0.f};
  long long r = r0;
  for (; r + 3 < r1; r += 4) {
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = __ldg(logits + (r + j) * m + col);
#pragma unroll
    for (int j = 0; j < 4; ++j) online_add(mx[j], sm[j], v[j]);
  }
  for (; r < r1; ++r) online_add(mx[0], sm[0], __ldg(logits + r * m + col));
  online_merge(mx[0], sm[0], mx[1], sm[1]);
  online_merge(mx[2], sm[2], mx[3], sm[3]);
  online_merge(mx[0], sm[0], mx[2], sm[2]);
  pmax[(long long)blockIdx.y * m + col] = mx[0];
  psum[(long long)blockIdx.y * m + col] = sm[0];
}

// 32 columns per block, eight warps stride the chunks, merged through shared memory in warp order
__global__ void __launch_bounds__(256)
col_stats_stage2_kernel(const float* __restrict__ pmax, const float* __restrict__ psum, int chunks,
                        int m, float* __restrict__ colmax, float* __restrict__ colsum) {
  __shared__ float smx[8][32], ssm[8][32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int col = blockIdx.x * 32 + lane;
  float mx = -INFINITY, s = 0.f;
  if (col < m)
    for (int c = wid; c < chunks; c += 8) online_merge(mx, s, pmax[(long long)c * m + col], psum[(long long)c * m + col]);
  smx[wid][lane] = mx; ssm[wid][lane] = s;
  __syncthreads();
  if (wid == 0 && col < m) {
#pragma unroll
    for (int w = 1; w < 8; ++w) online_merge(mx, s, smx[w][lane], ssm[w][lane]);
    colmax[col] = mx;
    colsum[col] = s;
  }
}

// one level of the partial-statistics tree: [chunks_in, m] -> [gridDim.y, m], block y merges `per` consecutive chunks
__global__ void __launch_bounds__(256)
col_stats_merge_kernel(const float* __restrict__ pmax, const float* __restrict__ psum, int chunks_in, int per, int m,
                       float* __restrict__ omax, float* __restrict__ osum) {
  __shared__ float smx[8][32], ssm[8][32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int col = blockIdx.x * 32 + lane;
  const int c0 = blockIdx.y * per, c1 = min(chunks_in, c0 + per);
  float mx = -INFINITY, s = 0.f;
  if (col < m)
    for (int c = c0 + wid; c < c1; c += 8) online_merge(mx, s, pmax[(long long)c * m + col], psum[(long long)c * m + col]);
  smx[wid][lane] = mx; ssm[wid][lane] = s;
  __syncthreads();
  if (wid == 0 && col < m) {
#pragma unroll
    for (int w = 1; w < 8; ++w) online_merge(mx, s, smx[w][lane], ssm[w][lane]);
    omax[(long long)blockIdx.y * m + col] = mx;
    osum[(long long)blockIdx.y * m + col] = s;
  }
}

// out[r, c] = exp(logits[r, c] - colmax[c]) / colsum[c]: a thread keeps the statistics of its column(s) in registers and
// walks down a chunk of rows (VEC: four columns per thread, 16-byte accesses)
template <bool VEC>
__global__ void __launch_bounds__(256)
col_softmax_apply_kernel(const float* __restrict__ logits, const float* __restrict__ colmax,
                         const float* __restrict__ colsum, long long N, int m, long long rpb,
                         float* __restrict__ out) {
  const long long r0 = (long long)blockIdx.y * rpb, r1 = min(N, r0 + rpb);
  if constexpr (VEC) {
    const int c4 = blockIdx.x * blockDim.x + threadIdx.x;
    if (c4 >= m / 4) return;
    const float4 cm = __ldg(reinterpret_cast<const float4*>(colmax) + c4), cs = __ldg(reinterpret_cast<const float4*>(colsum) + c4);
    for (long long r = r0; r < r1; ++r) {
      const float4 v = ld_stream(reinterpret_cast<const float4*>(logits + r * m) + c4);
      float4 o;
      o.x = expf(v.x - cm.x) / cs.x; o.y = expf(v.y - cm.y) / cs.y; o.z = expf(v.z - cm.z) / cs.z; o.w = expf(v.w - cm.w) / cs.w;
      reinterpret_cast<float4*>(out + r * m)[c4] = o;
    }
  } else {
    const int col = blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= m) return;
    const float cm = __ldg(colmax + col), cs = __ldg(colsum + col);
    for (long long r = r0; r < r1; ++r) out[r * m + col] = expf(logits[r * m + col] - cm) / cs;
  }
}

struct StoreLogits {
  float* out; long long ld;
  __device__ __forceinline__ void operator()(int, int, int m, int n, float v) const {
    out[(long long)m * ld + n] = v;
  }
};

// ---- read (Memory.py:249-261): uq[n, 0:d] = q, uq[n, d:2d] = score_memory @ keys
struct ReadEpilogue {
  float* uq; const float* q; int d;
  __device__ __forceinline__ void operator()(int, int, int m, int n, float v) const {
    long long o = (long long)m * 2 * d;
    uq[o + n] = q[(long long)m * d + n];
    uq[o + d + n] = v;
  }
};

// ---- gather / spread losses (Memory.py:214-247), one warp per token --------
__global__ void __launch_bounds__(256)
memory_losses_kernel(const float* __restrict__ q, const float* __restrict__ keys,
                     const long long* __restrict__ top1, const long long* __restrict__ top2,
                     long long N, int d, double* __restrict__ partial /*[grid][2]*/) {
  __shared__ double red[32];
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  double g = 0.0, sp = 0.0;
  if (row < N) {
    const float* qr = q + row * d;
    const float* pos = keys + top1[row] * d;
    const float* neg = top2 ? keys + top2[row] * d : nullptr;
    float s1 = 0.f, sap = 0.f, san = 0.f;
    auto term = [&](float qv, float pv, float nv) {
      const float e = qv - pv;
      s1 += e * e;
      const float ep = e + 1e-6f;                 // pairwise_distance eps (TripletMarginLoss)
      sap += ep * ep;
      if (neg) { const float en = qv - nv + 1e-6f; san += en * en; }
    };
    if ((d & 3) == 0 && ((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(keys)) & 15u) == 0) {
      for (int c = lane; c < (d >> 2); c += 32) {            // 16-byte loads: a quarter of the load instructions in flight longer
        const float4 qv = ld_stream(reinterpret_cast<const float4*>(qr) + c);
        const float4 pv = __ldg(reinterpret_cast<const float4*>(pos) + c);
        const float4 nv = neg ? __ldg(reinterpret_cast<const float4*>(neg) + c) : make_float4(0.f, 0.f, 0.f, 0.f);
        term(qv.x, pv.x, nv.x); term(qv.y, pv.y, nv.y); term(qv.z, pv.z, nv.z); term(qv.w, pv.w, nv.w);
      }
    } else {
      for (int c = lane; c < d; c += 32) term(qr[c], __ldg(pos + c), neg ? __ldg(neg + c) : 0.f);
    }
    s1 = warp_sum(s1); sap = warp_sum(sap); san = warp_sum(san);
    if (lane == 0) {
      g = (double)s1;
      if (neg) sp = (double)fmaxf(sqrtf(sap) - sqrtf(san) + 1.0f, 0.f);
    }
  }
  double gt = block_sum<double>(g, red);
  double st = block_sum<double>(sp, red);
  if (threadIdx.x == 0) { partial[2 * blockIdx.x] = gt; partial[2 * blockIdx.x + 1] = st; }
}

__global__ void __launch_bounds__(1024)
memory_losses_finalize_kernel(const double* __restrict__ partial, int nb, double nd, double n,
                              float* __restrict__ out) {
  __shared__ double red[32];
  double g = 0.0, s = 0.0;
  for (int i = threadIdx.x; i < nb; i += blockDim.x) { g += partial[2 * i]; s += partial[2 * i + 1]; }
  g = block_sum<double>(g, red);
  s = block_sum<double>(s, red);
  if (threadIdx.x == 0) { out[0] = (float)(g / nd); out[1] = (float)(s / n); }
}

// ---- update (Memory.py:177-204, :94-131) ----------------------------------
// column max of score_query (the reference divides by torch.max(score[:, i]))
__global__ void __launch_bounds__(256)
colmax_stage1_kernel(const float* __restrict__ a, long long N, int m, long long rpb,
                     float* __restrict__ pmax) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= m) return;
  long long r0 = (long long)blockIdx.y * rpb, r1 = min(N, r0 + rpb);
  float mx = -INFINITY;
  for (long long r = r0; r < r1; ++r) mx = fmaxf(mx, __ldg(a + r * m + col));
  pmax[(long long)blockIdx.y * m + col] = mx;
}
__global__ void __launch_bounds__(256)
colmax_stage2_kernel(const float* __restrict__ pmax, int chunks, int m, float* __restrict__ out) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= m) return;
  float mx = -INFINITY;
  for (int c = 0; c < chunks; ++c) mx = fmaxf(mx, pmax[(long long)c * m + col]);
  out[col] = mx;
}

// stable counting sort of tokens by their top-1 slot: histogram per block of
// 1024 consecutive tokens, scan, then an in-order placement, so every slot's
// token list is in ascending token order and the weighted sum below is
// deterministic (the reference's python loop over slots with nonzero() visits
// tokens in the same ascending order).
constexpr int kSortChunk = 1024;

__global__ void __launch_bounds__(256)
slot_hist_kernel(const long long* __restrict__ top1, long long N, int m, int* __restrict__ hist /*[chunks][m]*/) {
  long long r0 = (long long)blockIdx.x * kSortChunk, r1 = min(N, r0 + kSortChunk);
  int* h = hist + (long long)blockIdx.x * m;
  for (long long r = r0 + threadIdx.x; r < r1; r += blockDim.x) atomicAdd(h + (int)top1[r], 1);
}

// offsets[chunk][slot] = start of that chunk's run inside slot's list; seg[slot] = list start
__global__ void __launch_bounds__(256)
slot_scan_kernel(int* __restrict__ hist, int chunks, int m, int* __restrict__ seg /*[m+1]*/) {
  // per-slot exclusive scan over chunks (threads over slots), then a serial scan over slots
  __shared__ int total_s[1];
  for (int s = blockIdx.x * blockDim.x + threadIdx.x; s < m; s += gridDim.x * blockDim.x) {
    int run = 0;
    for (int c = 0; c < chunks; ++c) { int v = hist[(long long)c * m + s]; hist[(long long)c * m + s] = run; run += v; }
    seg[s + 1] = run;     // count, turned into offsets by slot_scan2
  }
  (void)total_s;
}
__global__ void slot_scan2_kernel(int* __restrict__ seg, int m) {
  // single thread block, serial over m (m is a few thousand at most)
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    int run = 0;
    seg[0] = 0;
    for (int s = 0; s < m; ++s) { int c = seg[s + 1]; run += c; seg[s + 1] = run; }
  }
}

// one warp walks a chunk's tokens in order (32 at a time) and ranks equal slots
// with match_any so placement is stable
__global__ void __launch_bounds__(32)
slot_place_kernel(const long long* __restrict__ top1, long long N, int m,
                  const int* __restrict__ hist, const int* __restrict__ seg,
                  int* __restrict__ cursor /*[chunks][m] zeroed*/, int* __restrict__ order) {
  const int lane = threadIdx.x;
  long long r0 = (long long)blockIdx.x * kSortChunk, r1 = min(N, r0 + kSortChunk);
  const int* off = hist + (long long)blockIdx.x * m;
  int* cur = cursor + (long long)blockIdx.x * m;
  for (long long base = r0; base < r1; base += 32) {
    long long r = base + lane;
    bool valid = r < r1;
    int slot = valid ? (int)top1[r] : -1 - lane;
    unsigned peers = __match_any_sync(0xffffffffu, slot);
    int rank = __popc(peers & ((1u << lane) - 1u));
    int cnt = __popc(peers);
    int start = 0;
    if (valid) start = cur[slot];
    __syncwarp();
    if (valid) {
      order[seg[slot] + off[slot] + start + rank] = (int)r;
      if (rank == cnt - 1) cur[slot] = start + cnt;
    }
    __syncwarp();
  }
}

// one block per slot: u_i = sum_n (score_query[n,i]/colmax_sq[i]) q_n in token
// order (warps interleave tokens, partials combined in fixed warp order), then
// updated_memory[i] = normalize(u_i + keys[i])  (Memory.py:193)
__global__ void __launch_bounds__(256)
slot_update_kernel(const float* __restrict__ q, const float* __restrict__ keys,
                   const float* __restrict__ score_query, const float* __restrict__ colmax_sq,
                   const int* __restrict__ seg, const int* __restrict__ order, int m, int d,
                   float* __restrict__ query_update, float* __restrict__ updated) {
  extern __shared__ float sm[];        // [8][d] partials + [32] reduction
  const int slot = blockIdx.x;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int a = seg[slot], b = seg[slot + 1];
  const float inv = 1.0f / colmax_sq[slot];
  float* part = sm + (size_t)wid * d;
  for (int c = lane; c < d; c += 32) part[c] = 0.f;
  for (int j = a + wid; j < b; j += 8) {
    const long long n = order[j];
    const float wgt = score_query[n * m + slot] * inv;
    const float* qr = q + n * d;
    for (int c = lane; c < d; c += 32) part[c] += wgt * qr[c];
  }
  __syncthreads();
  float nrm = 0.f;
  for (int c = threadIdx.x; c < d; c += 256) {
    float u = 0.f;
    for (int w = 0; w < 8; ++w) u += sm[(size_t)w * d + c];
    query_update[(long long)slot * d + c] = u;
    float v = u + keys[(long long)slot * d + c];
    sm[c] = v;                        // safe: column c is only touched by this thread from here on
    nrm += v * v;
  }
  __shared__ float red[32];
  nrm = block_sum<float>(nrm, red);
  const float s = 1.0f / fmaxf(sqrtf(nrm), 1e-12f);
  for (int c = threadIdx.x; c < d; c += 256) updated[(long long)slot * d + c] = sm[c] * s;
}

// ---- global-batch memory under data parallelism (SURVEY 8e) ---------------------------------------
// softmax(score, dim=0) and max_n score_query[:, i] (Memory.py:140, :108) span ALL tokens of the batch.
// With the tokens sharded over ranks every rank has its own column maximum cm_l and exp-sum cs_l of the
// logits; with cm_g = max over ranks (all-reduce MAX) the global column sum is S = sum over ranks of
// cs_l exp(cm_l - cm_g) (all-reduce SUM of `contrib`), the global score_query is the local one times
// contrib / S, and the update weight exp(logit - cm_g) is the local weight times exp(cm_l - cm_g).
__global__ void __launch_bounds__(256)
memory_dp_contrib_kernel(const float* __restrict__ cm_l, const float* __restrict__ cs_l,
                         const float* __restrict__ cm_g, int m, float* __restrict__ contrib) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < m) contrib[i] = cs_l[i] * expf(cm_l[i] - cm_g[i]);
}

__global__ void __launch_bounds__(256)
scale_columns_kernel(float* __restrict__ x, const float* __restrict__ num, const float* __restrict__ den,
                     long long N, int m) {
  const long long total = N * m;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % m);
    x[i] *= num[c] / den[c];
  }
}

// u[i, :] *= exp(cm_l[i] - cm_g[i])   (local update sums -> this rank's share of the global ones)
__global__ void __launch_bounds__(256)
memory_dp_scale_update_kernel(float* __restrict__ u, const float* __restrict__ cm_l,
                              const float* __restrict__ cm_g, int d) {
  const int slot = blockIdx.x;
  const float f = expf(cm_l[slot] - cm_g[slot]);
  for (int c = threadIdx.x; c < d; c += blockDim.x) u[(long long)slot * d + c] *= f;
}

// updated_memory[i] = F.normalize(u_i + keys[i])  (Memory.py:193) from already reduced update sums
__global__ void __launch_bounds__(256)
memory_finish_update_kernel(const float* __restrict__ u, const float* __restrict__ keys, int d,
                            float* __restrict__ updated) {
  __shared__ float red[32];
  const int slot = blockIdx.x;
  float nrm = 0.f;
  for (int c = threadIdx.x; c < d; c += blockDim.x) {
    const float v = u[(long long)slot * d + c] + keys[(long long)slot * d + c];
    nrm += v * v;
  }
  nrm = block_sum<float>(nrm, red);
  const float s = 1.0f / fmaxf(sqrtf(nrm), 1e-12f);
  for (int c = threadIdx.x; c < d; c += blockDim.x)
    updated[(long long)slot * d + c] = (u[(long long)slot * d + c] + keys[(long long)slot * d + c]) * s;
}

__global__ void zero_int_kernel(int* p, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = 0;
}

// MemoryLoss (Memory.py:52-59)
struct SeparatenessEpilogue {
  float* out; int m;
  __device__ __forceinline__ void operator()(int, int, int r, int c, float v) const {
    out[(long long)r * m + c] = fabsf(v * 0.5f + 0.5f - (r == c ? 1.0f : 0.0f));
  }
};
__global__ void __launch_bounds__(256)
sum_all_kernel(const float* __restrict__ a, long long n, double scale, float* __restrict__ out) {
  __shared__ double red[32];
  double s = 0.0;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) s += (double)a[i];
  s = block_sum<double>(s, red);
  if (threadIdx.x == 0) out[0] = (float)(s * scale);
}

// ---- gradient with respect to the memory items ------------------------------------------------------------------
// read (Memory.py:255): updated_query[:, d:2d] = score_memory.detach() @ keys, so g_keys = score_memory^T G_r with
// G_r[n, c] = g_updated_query[b, d + c, hw], n = b HW + hw.  One GEMM, M = slots, N = channels, contraction over the
// tokens: score_memory is the A operand read MN-major ([tokens, slots] = [Kd, M]), G_r the K-major B operand
// ([channels, tokens]).  Both are split into their operand terms with row pitches padded to eight elements (TMA: 16-byte
// pitches) and zeros in the padding, so any m and any token count take the tensor-core path.
// score_memory [N, m] -> terms [TERMS][Np][m8] of score_memory * scale (fp16 x2: scale = 2^13, bf16 x3: 1)
template <int TERMS>
__global__ void __launch_bounds__(256)
keys_bwd_split_scores_kernel(const float* __restrict__ sm, long long N, int m, long long Np, int m8, float scale,
                             void* __restrict__ dst) {
  const long long plane = Np * m8;
  for (long long r = blockIdx.x; r < Np; r += gridDim.x) {
    const float* row = sm + r * m;
    for (int c = threadIdx.x; c < m8; c += blockDim.x) {
      const float v = (r < N && c < m) ? __ldg(row + c) * scale : 0.f;
      store_terms<TERMS>(dst, plane, r * m8 + c, v);
    }
  }
}

// channels c0..c0+d-1 of a [B, C, HW] tensor -> terms [TERMS][d][Np] of its transpose times scale[0] (NULL: 1) and,
// per token, tok[n] (NULL: 1); read and written along hw; the last batch's blocks also zero the padding columns N..Np-1.
// (G_r: g_updated_query with C = 2d, c0 = d; q-hat: query with C = d, c0 = 0, tok = 1 / |x|)
template <int TERMS>
__global__ void __launch_bounds__(256)
keys_bwd_split_grad_kernel(const float* __restrict__ src, int B, int C, int c0, int d, long long HW, long long Np,
                           const float* __restrict__ scale, const float* __restrict__ tok, void* __restrict__ dst) {
  const long long hw = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int c = blockIdx.y, b = blockIdx.z;
  const long long n = (long long)b * HW + hw;
  float v = 0.f;
  if (hw < HW) {
    v = __ldg(src + ((long long)b * C + c0 + c) * HW + hw) * (scale ? __ldg(scale) : 1.0f);
    if (tok) v *= __ldg(tok + n);
  } else if (b != B - 1 || n >= Np) {
    return;
  }
  store_terms<TERMS>(dst, (long long)d * Np, (long long)c * Np + n, v);
}

// g_keys[i, c] (+)= sum over split slots s (in slot order) of part[s][i][c]: repeated launches give identical bits
__global__ void __launch_bounds__(256)
keys_bwd_sum_partials_kernel(const float* __restrict__ part, int splits, long long split_stride, long long n,
                             bool accumulate, float* __restrict__ out) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int k = 0; k < splits; ++k) s += __ldg(part + k * split_stride + i);
    out[i] = accumulate ? out[i] + s : s;
  }
}

// ---- gradient through the returned score matrices -------------------------------------------------------------
// get_score (Memory.py:133-143): s = q-hat K^T, sq = softmax(s, dim=0), sm = softmax(s, dim=1).  With Gq, Gm the
// gradients of score_query, score_memory:
//   c_i = sum_n Gq[n,i] sq[n,i]  (over every token of the batch),  r_n = sum_i Gm[n,i] sm[n,i]
//   g_s = sq (Gq - 1 c^T) + sm (Gm - r 1^T);   g_qhat = g_s K,  g_keys += g_s^T q-hat

// column dots, first level: block y sums rows [y rpb, (y+1) rpb) of its column in four interleaved chains
__global__ void __launch_bounds__(256)
score_coldot_stage1_kernel(const float* __restrict__ sq, const float* __restrict__ gq, long long N, int m,
                           long long rpb, float* __restrict__ part) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= m) return;
  const long long r0 = (long long)blockIdx.y * rpb, r1 = min(N, r0 + rpb);
  float a[4] = {0.f, 0.f, 0.f, 0.f};
  long long r = r0;
  for (; r + 3 < r1; r += 4) {
#pragma unroll
    for (int j = 0; j < 4; ++j) a[j] += __ldg(sq + (r + j) * m + col) * __ldg(gq + (r + j) * m + col);
  }
  for (; r < r1; ++r) a[0] += __ldg(sq + r * m + col) * __ldg(gq + r * m + col);
  part[(long long)blockIdx.y * m + col] = (a[0] + a[1]) + (a[2] + a[3]);
}

// second level: 32 columns per block, eight warps stride the chunks, merged through shared memory in warp order
__global__ void __launch_bounds__(256)
score_coldot_stage2_kernel(const float* __restrict__ part, int chunks, int m, float* __restrict__ coldot) {
  __shared__ float red[8][32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int col = blockIdx.x * 32 + lane;
  float s = 0.f;
  if (col < m)
    for (int c = wid; c < chunks; c += 8) s += part[(long long)c * m + col];
  red[wid][lane] = s;
  __syncthreads();
  if (wid == 0 && col < m) {
#pragma unroll
    for (int w = 1; w < 8; ++w) s += red[w][lane];
    coldot[col] = s;
  }
}

// g_s in one pass, one warp per token row, written straight as operand terms [TERMS][Np][m8] of g_s * scale[0]
// (scale == NULL: 1; rows N..Np-1 and columns m..m8-1 zero).  Gq / Gm == NULL: that term is absent.
// V4 > 0 (m % 4 == 0, m <= 128 V4, 16-byte aligned rows): the row of sm and Gm stays in registers between the row dot
// and g_s, as in row_softmax_top2_reg_kernel; V4 == 0: two passes over the row, the second one served by L1.
template <int TERMS, int V4>
__global__ void __launch_bounds__(256)
scores_bwd_gs_kernel(const float* __restrict__ sq, const float* __restrict__ sm, const float* __restrict__ gq,
                     const float* __restrict__ gm, const float* __restrict__ coldot, long long N, int m, long long Np,
                     int m8, const float* __restrict__ scale, void* __restrict__ dst) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= Np) return;
  const long long plane = Np * m8;
  if (row >= N) {                                        // padding token: zeros for the contraction over the tokens
    for (int c = lane; c < m8; c += 32) store_terms<TERMS>(dst, plane, row * m8 + c, 0.f);
    return;
  }
  const float s = scale ? __ldg(scale) : 1.0f;
  const float* sqr = sq ? sq + row * m : nullptr;
  const float* gqr = gq ? gq + row * m : nullptr;
  const float* smr = gm ? sm + row * m : nullptr;
  const float* gmr = gm ? gm + row * m : nullptr;
  if constexpr (V4 > 0) {
    const int n4 = m >> 2;
    float4 vs[V4], vg[V4];
    float r = 0.f;
    if (gmr) {
#pragma unroll
      for (int k = 0; k < V4; ++k) {
        const int i = lane + 32 * k;
        vs[k] = i < n4 ? ld_stream(reinterpret_cast<const float4*>(smr) + i) : make_float4(0.f, 0.f, 0.f, 0.f);
        vg[k] = i < n4 ? ld_stream(reinterpret_cast<const float4*>(gmr) + i) : make_float4(0.f, 0.f, 0.f, 0.f);
        r += (vs[k].x * vg[k].x + vs[k].y * vg[k].y) + (vs[k].z * vg[k].z + vs[k].w * vg[k].w);
      }
      r = warp_sum(r);
    }
#pragma unroll
    for (int k = 0; k < V4; ++k) {
      const int i = lane + 32 * k;
      if (i >= n4) continue;
      float a[4] = {0.f, 0.f, 0.f, 0.f};
      if (gqr) {
        const float4 p = ld_stream(reinterpret_cast<const float4*>(sqr) + i);
        const float4 g = ld_stream(reinterpret_cast<const float4*>(gqr) + i);
        const float4 c = __ldg(reinterpret_cast<const float4*>(coldot) + i);
        a[0] = p.x * (g.x - c.x); a[1] = p.y * (g.y - c.y); a[2] = p.z * (g.z - c.z); a[3] = p.w * (g.w - c.w);
      }
      if (gmr) {
        a[0] += vs[k].x * (vg[k].x - r); a[1] += vs[k].y * (vg[k].y - r);
        a[2] += vs[k].z * (vg[k].z - r); a[3] += vs[k].w * (vg[k].w - r);
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) a[j] *= s;
      store_terms<TERMS, 4>(dst, plane, row * m8 + 4 * i, a);
    }
  } else {
    float r = 0.f;
    if (gmr) {
      for (int i = lane; i < m; i += 32) r += __ldg(smr + i) * __ldg(gmr + i);
      r = warp_sum(r);
    }
    for (int i = lane; i < m; i += 32) {
      float a = 0.f;
      if (gqr) a = __ldg(sqr + i) * (__ldg(gqr + i) - __ldg(coldot + i));
      if (gmr) a += __ldg(smr + i) * (__ldg(gmr + i) - r);
      store_terms<TERMS>(dst, plane, row * m8 + i, a * s);
    }
  }
  for (int c = m + lane; c < m8; c += 32) store_terms<TERMS>(dst, plane, row * m8 + c, 0.f);
}

// q [N, d] row-major -> terms [TERMS][d][Np] of its transpose times scale[0] (NULL: 1), tokens N..Np-1 zero: the
// K-major B operand of g_s^T q for the channel-last query.  A block moves 64 tokens x 32 channels through shared memory:
// a warp reads 128 bytes of a token row, and writes two tokens per lane along a channel row (128 bytes per term).
template <int TERMS>
__global__ void __launch_bounds__(256)
rows_transpose_terms_kernel(const float* __restrict__ q, long long N, int d, long long Np,
                            const float* __restrict__ scale, void* __restrict__ dst) {
  __shared__ float tile[32][65];               // [channel][token]
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const long long n0 = (long long)blockIdx.x * 64;
  const int c0 = blockIdx.y * 32;
  for (int j = wid; j < 64; j += 8) {
    const long long n = n0 + j;
    tile[lane][j] = (n < N && c0 + lane < d) ? __ldg(q + n * d + c0 + lane) : 0.f;
  }
  __syncthreads();
  const float s = scale ? __ldg(scale) : 1.0f;
  const long long plane = (long long)d * Np, n = n0 + 2 * lane;
  if (n >= Np) return;                         // Np is a multiple of eight: both tokens of a pair are in or out
  for (int i = wid; i < 32 && c0 + i < d; i += 8) {
    const float a[2] = {tile[i][2 * lane] * s, tile[i][2 * lane + 1] * s};
    store_terms<TERMS, 2>(dst, plane, (long long)(c0 + i) * Np + n, a);
  }
}

// keys [m, d] -> terms [TERMS][m8][d8] of keys * scale[0] (NULL: 1), zero padded: the MN-major B operand of g_s K
template <int TERMS>
__global__ void __launch_bounds__(256)
scores_bwd_split_keys_kernel(const float* __restrict__ keys, int m, int d, int m8, int d8,
                             const float* __restrict__ scale, void* __restrict__ dst) {
  const float s = scale ? __ldg(scale) : 1.0f;
  for (int r = blockIdx.x; r < m8; r += gridDim.x)
    for (int c = threadIdx.x; c < d8; c += blockDim.x)
      store_terms<TERMS>(dst, (long long)m8 * d8, (long long)r * d8 + c,
                         (r < m && c < d) ? __ldg(keys + (long long)r * d + c) * s : 0.f);
}

// power-of-two scales of the two contractions, from the measured bounds (float bits) of Gq, Gm, the column dots and K:
//   |g_s| <= max|Gq| + max|c| + 2 max|Gm|   (sq, sm in [0, 1]; |r_n| <= max|Gm|), put in [2^12, 2^13) like the softmax
//   weights of the read (small entries stay normal fp16 numbers); K in [4, 8) as in the forward; q-hat has unit rows: 2^13,
//   an unnormalised q (q_measured: its bound in bits[4]) is put in [2^12, 2^13) like g_s
//   out = {s_g, s_k, 1 / (s_g s_k), s_q, 1 / (s_g s_q)}
__global__ void scores_bwd_scales_kernel(const unsigned* __restrict__ bits, bool q_measured, float* __restrict__ out) {
  auto pow2 = [](float bound, int top) {                // 2^e with 2^e bound in [2^(top-1), 2^top); 1 for 0 / non-finite
    if (!(bound > 0.f) || !isfinite(bound)) return 1.0f;
    int e;
    (void)frexpf(bound, &e);
    return ldexpf(1.0f, max(-100, min(100, top - e)));
  };
  const float sg = pow2(__uint_as_float(bits[0]) + __uint_as_float(bits[2]) + 2.0f * __uint_as_float(bits[1]), 13);
  const float sk = pow2(__uint_as_float(bits[3]), 3), sq = q_measured ? pow2(__uint_as_float(bits[4]), 13) : 8192.0f;
  out[0] = sg; out[1] = sk; out[2] = 1.0f / (sg * sk); out[3] = sq; out[4] = 1.0f / (sg * sq);
}


// MemoryLoss (Memory.py:52-59) backward: G = sgn(S), S = K K^T / 2 + 1/2 - I from the same product and the same
// expression as SeparatenessEpilogue (sgn(0) = 0, the subgradient torch's abs backward takes)
struct SeparatenessSignEpilogue {
  float* out; int m;
  __device__ __forceinline__ void operator()(int, int, int r, int c, float v) const {
    const float s = v * 0.5f + 0.5f - (r == c ? 1.0f : 0.0f);
    out[(long long)r * m + c] = (s > 0.f) ? 1.0f : ((s < 0.f) ? -1.0f : 0.0f);
  }
};

// g_keys = g_out / (m (m - 1)) * (G K); G is symmetric by construction (the entries (r, c) and (c, r) come from the same
// operands in the same accumulation order), so G K = (G + G^T) / 2 K
struct ScaledStoreEpilogue {
  float* out; int ld; const float* g_out; float scale;
  __device__ __forceinline__ void operator()(int, int, int r, int c, float v) const {
    out[(long long)r * ld + c] = v * (__ldg(g_out) * scale);
  }
};

// split-K factor of the g_keys contraction ([m, d] output, contraction over the tokens): ~2 tiles per SM of a B200
// (148 SMs).  A function of the shape alone, so that the workspace query makes no CUDA call.
static int keys_bwd_splits(long long Np, int m8, int d) {
  const long long tiles = (long long)((m8 + 127) / 128) * ((d + 127) / 128);
  const long long nkb = (Np + 63) / 64;
  long long s = (2ll * 148 + tiles - 1) / tiles;
  if (s > nkb) s = nkb;
  if (s < 1) s = 1;
  return (int)s;
}

static int col_chunks(long long N) {
  long long c = (N + 255) / 256;
  if (c > 2048) c = 2048;
  if (c < 1) c = 1;
  return (int)c;
}

}  // namespace vadc

using namespace vadc;

extern "C" size_t vadc_memory_prepare_query_workspace_bytes(int B, int64_t HW) {
  return align_up((size_t)(B > 0 ? B : 1) * HW * sizeof(float), 256) + 256;
}

extern "C" int vadc_memory_prepare_query(const float* query, int B, int d, int64_t HW, float* q,
                                         void* workspace, size_t workspace_bytes, void* stream) {
  VADC_REQUIRE(B >= 0 && d > 0 && HW > 0, VADC_ERR_BAD_SHAPE);
  if (B == 0) return VADC_OK;
  VADC_REQUIRE(query && q && workspace, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(B <= 65535 && (d + 31) / 32 <= 65535, VADC_ERR_UNSUPPORTED);
  VADC_REQUIRE(workspace_bytes >= vadc_memory_prepare_query_workspace_bytes(B, HW), VADC_ERR_WORKSPACE);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* inv = static_cast<float*>(workspace);
  dim3 g1((unsigned)((HW + 31) / 32), B);
  query_norm_kernel<<<g1, 256, 0, st>>>(query, d, HW, inv);
  VADC_CHECK_LAUNCH("query_norm_kernel");
  dim3 g2((unsigned)((HW + 31) / 32), (d + 127) / 128, B);
  query_transpose_kernel<<<g2, 256, 0, st>>>(query, inv, d, HW, q);
  VADC_CHECK_LAUNCH("query_transpose_kernel");
  return VADC_OK;
}

extern "C" int vadc_memory_query_bwd(const float* query, const float* keys, const int64_t* top1,
                                     const int64_t* top2, const float* g_updated_query,
                                     const float* g_gather, const float* g_spread, int B, int d,
                                     int64_t HW, int m, float* g_query, void* stream) {
  return vadc_memory_query_bwd_ex(query, keys, top1, top2, g_updated_query, g_gather, g_spread, nullptr, B, d, HW, m,
                                  g_query, stream);
}

extern "C" int vadc_memory_query_bwd_ex(const float* query, const float* keys, const int64_t* top1,
                                        const int64_t* top2, const float* g_updated_query,
                                        const float* g_gather, const float* g_spread, const float* g_qhat, int B,
                                        int d, int64_t HW, int m, float* g_query, void* stream) {
  VADC_REQUIRE(B >= 0 && d > 0 && HW > 0 && m > 0, VADC_ERR_BAD_SHAPE);
  if (B == 0) return VADC_OK;
  VADC_REQUIRE(query && keys && top1 && g_query, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(B <= 65535, VADC_ERR_UNSUPPORTED);
  if (!vadc_device_ok()) return VADC_ERR_NO_DEVICE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  dim3 grid((unsigned)((HW + 31) / 32), B);
  memory_query_bwd_kernel<<<grid, 256, 0, st>>>(query, keys, reinterpret_cast<const long long*>(top1),
                                                reinterpret_cast<const long long*>(top2), g_updated_query,
                                                g_gather, g_spread, g_qhat, d, HW, (long long)B * HW, g_query);
  VADC_CHECK_LAUNCH("memory_query_bwd_kernel");
  return VADC_OK;
}

extern "C" size_t vadc_memory_score_workspace_bytes(int64_t N, int m, int d) {
  (void)d;
  size_t n = (size_t)(N > 0 ? N : 1);
  const size_t groups = std::max<size_t>((n + 31) / 32, (size_t)col_chunks(N));      // 32-token groups of the GEMM epilogue
  return align_up(n * m * sizeof(float), 256) + 2 * align_up(groups * m * sizeof(float), 256) +
         2 * align_up(((groups + 63) / 64) * m * sizeof(float), 256) +               // second level of the statistics tree
         tc_terms_bytes(3, (long long)n, d) + tc_terms_bytes(3, m, d) + 1024;     // operand terms of q and keys, scales
}

namespace vadc {
// q . keys^T on tcgen05 (m = 2000, d = 768 is tensor-bound: 244 flop/B).  TERMS = 3: fp32-faithful, six products.
// TERMS = 2: two fp16 terms of the operands scaled by a power of two from their measured bounds (unit-norm rows in the
// module: Memory.py:148, :222), three products, 22 significant bits: 2/3 of the operand bytes, half the MMAs.
// col_stats: score_query is wanted (fp16 x2 from m = 128 up: the epilogue leaves per-32-token column statistics in
// pmax / psum and sets have_groups)
template <int TERMS>
static int memory_score_tc(const float* q, const float* keys, long long N, int m, int d, bool col_stats, float* logits,
                           float* pmax, float* psum, bool& have_groups, Carver& ws, cudaStream_t st) {
  void* qs = ws.take<uint8_t>(tc_terms_bytes(3, N, d));
  void* ks = ws.take<uint8_t>(tc_terms_bytes(3, m, d));
  float* sc = nullptr;
  int rc;
  if constexpr (TERMS == 2) {
    unsigned* bits = ws.take<unsigned>(64);
    sc = ws.take<float>(64);
    if ((rc = tc_absmax_bits(q, (long long)N * d, bits, st))) return rc;
    if ((rc = tc_absmax_bits(keys, (long long)m * d, bits + 1, st))) return rc;
    if ((rc = tc_pair_scales(bits, 0.f, bits + 1, 0.f, sc, st))) return rc;
  }
  if ((rc = tc_split<TERMS>(q, N, d, sc, qs, st))) return rc;
  if ((rc = tc_split<TERMS>(keys, m, d, sc ? sc + 1 : nullptr, ks, st))) return rc;
  if constexpr (TERMS == 2) {
    // fp16 x2 only: operands swapped from m = 128 up (rows = memory slots): coalesced stores of the logits
    if (m >= 128) {
      have_groups = col_stats;
      if (col_stats) return tc_gemm<2, false, false>({ks, qs, m, N, d, sc + 2}, TcLogitsColStatsTEpi{logits, m, pmax, psum}, st);
      return tc_gemm<2, false, false>({ks, qs, m, N, d, sc + 2}, TcStoreTEpi{logits, m}, st);
    }
  }
  return tc_gemm<TERMS, false, false>({qs, ks, N, m, d, sc ? sc + 2 : nullptr}, TcStoreEpi{logits, m}, st);
}

// score_memory [N,m] . keys [m,d] (keys read MN-major) on tcgen05.  fp16 x2: the softmax weights (in [0, 1],
// Memory.py:139) scaled by 2^13 so that small weights stay normal numbers; their terms sm_terms may have been written by
// vadc_memory_score next to score_memory, else they are split here
template <int TERMS>
static int memory_read_tc(const float* q, const float* score_memory, const void* sm_terms, const float* keys, long long N,
                          int m, int d, float* updated_query, Carver& ws, cudaStream_t st) {
  void* ss = ws.take<uint8_t>(tc_terms_bytes(3, N, m));
  void* ks = ws.take<uint8_t>(tc_terms_bytes(3, m, d));
  float* sc = nullptr;
  int rc;
  if constexpr (TERMS == 2) {
    unsigned* bits = ws.take<unsigned>(64);
    sc = ws.take<float>(64);
    if ((rc = tc_absmax_bits(keys, (long long)m * d, bits, st))) return rc;
    if ((rc = tc_pair_scales(nullptr, 8192.0f, bits, 0.f, sc, st))) return rc;
  }
  if (!sm_terms) {
    if ((rc = tc_split<TERMS>(score_memory, N, m, sc, ss, st))) return rc;
    sm_terms = ss;
  }
  if ((rc = tc_split<TERMS>(keys, m, d, sc ? sc + 1 : nullptr, ks, st))) return rc;
  if constexpr (TERMS == 2) {
    if (d >= 128)   // fp16 x2 only: rows = channels (keys [m,d] as the MN-major A operand): coalesced output
      return tc_gemm<2, true, false>({ks, sm_terms, d, N, m, sc + 2}, TcReadTEpi{updated_query, q, d}, st);
  }
  return tc_gemm<TERMS, false, true>({sm_terms, ks, N, d, m, sc ? sc + 2 : nullptr}, TcReadEpi{updated_query, q, d}, st);
}
}  // namespace vadc

extern "C" int vadc_memory_score(const float* q, const float* keys, int64_t N, int m, int d,
                                 float* score_query, float* score_memory, float* colmax,
                                 float* colsum, int64_t* top1, int64_t* top2, void* score_memory_terms,
                                 void* workspace, size_t workspace_bytes, void* stream) {
  VADC_REQUIRE(N >= 0 && m > 0 && d > 0, VADC_ERR_BAD_SHAPE);
  if (N == 0) return VADC_OK;
  VADC_REQUIRE(q && keys && score_memory && workspace, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(!score_query || (colmax && colsum), VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(N < (1ll << 31), VADC_ERR_UNSUPPORTED);
  VADC_REQUIRE(workspace_bytes >= vadc_memory_score_workspace_bytes(N, m, d), VADC_ERR_WORKSPACE);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Carver ws(workspace, workspace_bytes);
  float* logits = ws.take<float>((size_t)N * m);
  int chunks = col_chunks(N);
  const size_t groups = std::max<size_t>(((size_t)N + 31) / 32, (size_t)chunks);
  float* pmax = ws.take<float>(groups * m);
  float* psum = ws.take<float>(groups * m);
  float* pmax2 = ws.take<float>(((groups + 63) / 64) * m);
  float* psum2 = ws.take<float>(((groups + 63) / 64) * m);
  bool have_groups = false;                    // the GEMM epilogue left per-32-token column statistics in pmax / psum
  if (tc_gemm_shape_ok(N, m, d, false) && !env_on("VADC_NO_TC_GEMM")) {
    // q . keys^T on tcgen05 (m = 2000, d = 768 is tensor-bound: 244 flop/B)
    int rc;
    if ((rc = env_int("VADC_MEMORY_TERMS", 2) == 3
                  ? memory_score_tc<3>(q, keys, N, m, d, score_query != nullptr, logits, pmax, psum, have_groups, ws, st)
                  : memory_score_tc<2>(q, keys, N, m, d, score_query != nullptr, logits, pmax, psum, have_groups, ws, st)))
      return rc;
  } else {
    Operand Aop{q, d, 1}, Bop{keys, 1, d};
    StoreLogits epi{logits, m};
    cudaError_t e = sgemm_auto((int)N, m, d, Aop, Bop, 0, 0, 1, 1, epi, st);
    if (e != cudaSuccess) return record_cuda_error(e, "memory score sgemm");
  }
  // column statistics first (score_query's softmax over the tokens): from the epilogue's 32-token groups through a
  // two-level tree, or from a pass over the logits
  if (score_query) {
    const float* lm = pmax;
    const float* ls = psum;
    int nch = chunks;
    if (have_groups) {
      const int ng = (int)(((size_t)N + 31) / 32);
      nch = (ng + 63) / 64;
      col_stats_merge_kernel<<<dim3((m + 31) / 32, nch), 256, 0, st>>>(pmax, psum, ng, 64, m, pmax2, psum2);
      VADC_CHECK_LAUNCH("col_stats_merge_kernel");
      lm = pmax2; ls = psum2;
    } else {
      long long rpb = (N + chunks - 1) / chunks;
      dim3 g1((m + 255) / 256, chunks);
      col_stats_stage1_kernel<<<g1, 256, 0, st>>>(logits, N, m, rpb, pmax, psum);
      VADC_CHECK_LAUNCH("col_stats_stage1_kernel");
    }
    col_stats_stage2_kernel<<<(m + 31) / 32, 256, 0, st>>>(lm, ls, nch, m, colmax, colsum);
    VADC_CHECK_LAUNCH("col_stats_stage2_kernel");
  }
  // with a terms buffer (fp16 x2 mode): the read GEMM's operand split of score_memory is written in the same pass
  __half* smt = (score_memory_terms && env_int("VADC_MEMORY_TERMS", 2) != 3) ? static_cast<__half*>(score_memory_terms) : nullptr;
  {
    const unsigned rg = (unsigned)((N + 7) / 8);
    long long* t1 = (long long*)top1;
    long long* t2 = (long long*)top2;
    const bool regs = (m % 4) == 0 && m <= 2048 && aligned16(logits) && aligned16(score_memory) && (!smt || aligned16(smt));
    if (regs && m <= 512) row_softmax_top2_reg_kernel<4><<<rg, 256, 0, st>>>(logits, N, m, score_memory, t1, t2, smt);
    else if (regs && m <= 1024) row_softmax_top2_reg_kernel<8><<<rg, 256, 0, st>>>(logits, N, m, score_memory, t1, t2, smt);
    else if (regs) row_softmax_top2_reg_kernel<16><<<rg, 256, 0, st>>>(logits, N, m, score_memory, t1, t2, smt);
    else row_softmax_top2_kernel<<<rg, 256, 0, st>>>(logits, N, m, score_memory, t1, t2, smt);
  }
  VADC_CHECK_LAUNCH("row_softmax_top2_kernel");
  if (score_query) {
    const bool vec = (m % 4) == 0 && aligned16(logits) && aligned16(score_query) && aligned16(colmax) && aligned16(colsum);
    const int cols = vec ? m / 4 : m;
    const unsigned gx = (unsigned)((cols + 255) / 256);
    long long ach = std::max<long long>(1, std::min<long long>((N + 15) / 16, (8ll * sm_count() + gx - 1) / gx));   // >= 16 rows each
    const long long arpb = (N + ach - 1) / ach;
    ach = (N + arpb - 1) / arpb;
    if (vec) col_softmax_apply_kernel<true><<<dim3(gx, (unsigned)ach), 256, 0, st>>>(logits, colmax, colsum, N, m, arpb, score_query);
    else col_softmax_apply_kernel<false><<<dim3(gx, (unsigned)ach), 256, 0, st>>>(logits, colmax, colsum, N, m, arpb, score_query);
    VADC_CHECK_LAUNCH("col_softmax_apply_kernel");
  }
  return VADC_OK;
}

extern "C" size_t vadc_memory_read_workspace_bytes(int64_t N, int m, int d) {
  size_t n = (size_t)(N > 0 ? N : 1);
  return tc_terms_bytes(3, (long long)n, m) + tc_terms_bytes(3, m, d) + 1024;     // operand terms of score_memory and keys, scales
}

extern "C" int vadc_memory_read(const float* q, const float* score_memory, const void* score_memory_terms,
                                const float* keys, int64_t N, int m, int d, float* updated_query,
                                void* workspace, size_t workspace_bytes, void* stream) {
  VADC_REQUIRE(N >= 0 && m > 0 && d > 0, VADC_ERR_BAD_SHAPE);
  if (N == 0) return VADC_OK;
  VADC_REQUIRE(q && score_memory && keys && updated_query, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(N < (1ll << 31), VADC_ERR_UNSUPPORTED);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (workspace && workspace_bytes >= vadc_memory_read_workspace_bytes(N, m, d) && tc_gemm_shape_ok(N, d, m, true) &&
      !env_on("VADC_NO_TC_GEMM")) {
    // score_memory [N,m] . keys [m,d] (keys read MN-major) on tcgen05
    Carver ws(workspace, workspace_bytes);
    return env_int("VADC_MEMORY_TERMS", 2) == 3
               ? memory_read_tc<3>(q, score_memory, nullptr, keys, N, m, d, updated_query, ws, st)
               : memory_read_tc<2>(q, score_memory, score_memory_terms, keys, N, m, d, updated_query, ws, st);
  }
  Operand Aop{score_memory, m, 1}, Bop{keys, d, 1};
  ReadEpilogue epi{updated_query, q, d};
  cudaError_t e = sgemm_auto((int)N, d, m, Aop, Bop, 0, 0, 1, 1, epi, st);
  if (e != cudaSuccess) return record_cuda_error(e, "memory read sgemm");
  return VADC_OK;
}

extern "C" size_t vadc_memory_losses_workspace_bytes(int64_t N, int d) {
  (void)d;
  return align_up((size_t)((N + 7) / 8 + 1) * 2 * sizeof(double), 256) + 256;
}

extern "C" int vadc_memory_losses(const float* q, const float* keys, const int64_t* top1,
                                  const int64_t* top2, int64_t N, int m, int d, float* out,
                                  void* workspace, size_t workspace_bytes, void* stream) {
  VADC_REQUIRE(N > 0 && m > 0 && d > 0, VADC_ERR_BAD_SHAPE);
  VADC_REQUIRE(q && keys && top1 && out && workspace, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(workspace_bytes >= vadc_memory_losses_workspace_bytes(N, d), VADC_ERR_WORKSPACE);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  double* partial = static_cast<double*>(workspace);
  int nb = (int)((N + 7) / 8);
  memory_losses_kernel<<<nb, 256, 0, st>>>(q, keys, (const long long*)top1, (const long long*)top2, N, d, partial);
  VADC_CHECK_LAUNCH("memory_losses_kernel");
  memory_losses_finalize_kernel<<<1, 1024, 0, st>>>(partial, nb, (double)N * d, (double)N, out);
  VADC_CHECK_LAUNCH("memory_losses_finalize_kernel");
  return VADC_OK;
}

static int sort_chunks(int64_t N) { return (int)((N + kSortChunk - 1) / kSortChunk); }

extern "C" size_t vadc_memory_update_workspace_bytes(int64_t N, int m, int d) {
  (void)d;
  size_t n = (size_t)(N > 0 ? N : 1);
  size_t b = 0;
  b += align_up((size_t)col_chunks(N) * m * sizeof(float), 256);     // column-max partials
  b += align_up((size_t)m * sizeof(float), 256);                     // column max of score_query
  b += 2 * align_up((size_t)sort_chunks(n) * m * sizeof(int), 256);  // hist/offsets + cursors
  b += align_up((size_t)(m + 1) * sizeof(int), 256);                 // segment starts
  b += align_up(n * sizeof(int), 256);                               // token order
  return b + 256;
}

extern "C" int vadc_memory_update(const float* q, const float* keys, const float* score_query,
                                  const int64_t* top1, int64_t N, int m, int d,
                                  float* query_update, float* updated_memory, void* workspace,
                                  size_t workspace_bytes, void* stream) {
  VADC_REQUIRE(N > 0 && m > 0 && d > 0, VADC_ERR_BAD_SHAPE);
  VADC_REQUIRE(q && keys && score_query && top1 && query_update && updated_memory && workspace, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(N < (1ll << 31), VADC_ERR_UNSUPPORTED);
  VADC_REQUIRE(workspace_bytes >= vadc_memory_update_workspace_bytes(N, m, d), VADC_ERR_WORKSPACE);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Carver ws(workspace, workspace_bytes);
  int cch = col_chunks(N), sch = sort_chunks(N);
  float* pmax = ws.take<float>((size_t)cch * m);
  float* cmax = ws.take<float>(m);
  int* hist = ws.take<int>((size_t)sch * m);
  int* cursor = ws.take<int>((size_t)sch * m);
  int* seg = ws.take<int>(m + 1);
  int* order = ws.take<int>(N);
  long long rpb = (N + cch - 1) / cch;
  dim3 g1((m + 255) / 256, cch);
  colmax_stage1_kernel<<<g1, 256, 0, st>>>(score_query, N, m, rpb, pmax);
  VADC_CHECK_LAUNCH("colmax_stage1_kernel");
  colmax_stage2_kernel<<<(m + 255) / 256, 256, 0, st>>>(pmax, cch, m, cmax);
  VADC_CHECK_LAUNCH("colmax_stage2_kernel");
  long long hz = (cursor + (long long)sch * m) - hist;   // hist and cursor are adjacent in the workspace
  zero_int_kernel<<<(unsigned)((hz + 255) / 256), 256, 0, st>>>(hist, hz);
  VADC_CHECK_LAUNCH("zero_int_kernel");
  slot_hist_kernel<<<sch, 256, 0, st>>>((const long long*)top1, N, m, hist);
  VADC_CHECK_LAUNCH("slot_hist_kernel");
  slot_scan_kernel<<<(m + 255) / 256, 256, 0, st>>>(hist, sch, m, seg);
  VADC_CHECK_LAUNCH("slot_scan_kernel");
  slot_scan2_kernel<<<1, 32, 0, st>>>(seg, m);
  VADC_CHECK_LAUNCH("slot_scan2_kernel");
  slot_place_kernel<<<sch, 32, 0, st>>>((const long long*)top1, N, m, hist, seg, cursor, order);
  VADC_CHECK_LAUNCH("slot_place_kernel");
  size_t smem = (size_t)8 * d * sizeof(float);
  if (smem > 48 * 1024)
    VADC_CUDA(cudaFuncSetAttribute(slot_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  slot_update_kernel<<<m, 256, smem, st>>>(q, keys, score_query, cmax, seg, order, m, d, query_update, updated_memory);
  VADC_CHECK_LAUNCH("slot_update_kernel");
  return VADC_OK;
}

extern "C" int vadc_memory_dp_contrib(const float* colmax_local, const float* colsum_local,
                                      const float* colmax_global, int m, float* contrib, void* stream) {
  VADC_REQUIRE(m > 0, VADC_ERR_BAD_SHAPE);
  VADC_REQUIRE(colmax_local && colsum_local && colmax_global && contrib, VADC_ERR_NULL_POINTER);
  memory_dp_contrib_kernel<<<(m + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(colmax_local, colsum_local,
                                                                                          colmax_global, m, contrib);
  VADC_CHECK_LAUNCH("memory_dp_contrib_kernel");
  return VADC_OK;
}

extern "C" int vadc_scale_columns(float* x, const float* num, const float* den, int64_t N, int m, void* stream) {
  VADC_REQUIRE(N >= 0 && m > 0, VADC_ERR_BAD_SHAPE);
  if (N == 0) return VADC_OK;
  VADC_REQUIRE(x && num && den, VADC_ERR_NULL_POINTER);
  const long long total = (long long)N * m;
  const int grid = (int)std::min<long long>((total + 255) / 256, (long long)sm_count() * 16);
  scale_columns_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(x, num, den, N, m);
  VADC_CHECK_LAUNCH("scale_columns_kernel");
  return VADC_OK;
}

extern "C" int vadc_memory_dp_scale_update(float* query_update, const float* colmax_local,
                                           const float* colmax_global, int m, int d, void* stream) {
  VADC_REQUIRE(m > 0 && d > 0, VADC_ERR_BAD_SHAPE);
  VADC_REQUIRE(query_update && colmax_local && colmax_global, VADC_ERR_NULL_POINTER);
  memory_dp_scale_update_kernel<<<m, 256, 0, static_cast<cudaStream_t>(stream)>>>(query_update, colmax_local, colmax_global, d);
  VADC_CHECK_LAUNCH("memory_dp_scale_update_kernel");
  return VADC_OK;
}

extern "C" int vadc_memory_finish_update(const float* query_update, const float* keys, int m, int d,
                                         float* updated_memory, void* stream) {
  VADC_REQUIRE(m > 0 && d > 0, VADC_ERR_BAD_SHAPE);
  VADC_REQUIRE(query_update && keys && updated_memory, VADC_ERR_NULL_POINTER);
  memory_finish_update_kernel<<<m, 256, 0, static_cast<cudaStream_t>(stream)>>>(query_update, keys, d, updated_memory);
  VADC_CHECK_LAUNCH("memory_finish_update_kernel");
  return VADC_OK;
}

extern "C" size_t vadc_memory_separateness_workspace_bytes(int m, int d) {
  (void)d;
  return align_up((size_t)m * m * sizeof(float), 256) + 256;
}

extern "C" int vadc_memory_separateness(const float* keys, int m, int d, float* out, void* workspace,
                                        size_t workspace_bytes, void* stream) {
  VADC_REQUIRE(m > 1 && d > 0, VADC_ERR_BAD_SHAPE);
  VADC_REQUIRE(keys && out && workspace, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(workspace_bytes >= vadc_memory_separateness_workspace_bytes(m, d), VADC_ERR_WORKSPACE);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* sim = static_cast<float*>(workspace);
  Operand Aop{keys, d, 1}, Bop{keys, 1, d};
  SeparatenessEpilogue epi{sim, m};
  cudaError_t e = sgemm_auto(m, m, d, Aop, Bop, 0, 0, 1, 1, epi, st);
  if (e != cudaSuccess) return record_cuda_error(e, "separateness sgemm");
  sum_all_kernel<<<1, 256, 0, st>>>(sim, (long long)m * m, 1.0 / ((double)m * (m - 1)), out);
  VADC_CHECK_LAUNCH("sum_all_kernel");
  return VADC_OK;
}

static long long pad8(long long v) { return (v + 7) / 8 * 8; }

extern "C" size_t vadc_memory_keys_bwd_workspace_bytes(int B, int d, int64_t HW, int m) {
  const long long Np = pad8((long long)(B > 0 ? B : 1) * (HW > 0 ? HW : 1)), m8 = pad8(m > 0 ? m : 1);
  const int dd = d > 0 ? d : 1;
  return tc_terms_bytes(3, Np, m8) + tc_terms_bytes(3, dd, Np) +       // operand terms (room for three)
         align_up((size_t)keys_bwd_splits(Np, (int)m8, dd) * m8 * dd * sizeof(float), 256) + 1024;   // partials, scales
}

// g_keys partials = score_memory^T G_r.  TERMS = 3: fp32-faithful, six products.  TERMS = 2: the softmax weights scaled
// by 2^13 as in vadc_memory_read, G_r by the power of two of its measured bound (over the channels d..2d-1 of every batch)
template <int TERMS>
static int keys_bwd_tc(const float* score_memory, const float* g_updated_query, int B, int d, int64_t HW, int m, void* sms,
                       void* gs, int sk, const TcPartialEpi& epi, Carver& ws, cudaStream_t st) {
  const long long N = (long long)B * HW, Np = pad8(N);
  const int m8 = (int)pad8(m);
  const unsigned srows = (unsigned)std::min<long long>(Np, 16ll * sm_count());
  const dim3 ggrid((unsigned)((HW + (Np - N) + 255) / 256), (unsigned)d, (unsigned)B);
  float* sc = nullptr;
  int rc;
  if constexpr (TERMS == 2) {
    unsigned* bits = ws.take<unsigned>(64);
    sc = ws.take<float>(64);
    if ((rc = tc_absmax_bits_seg(g_updated_query + (long long)d * HW, (long long)d * HW, B, 2ll * d * HW, bits, st))) return rc;
    if ((rc = tc_pair_scales(nullptr, 8192.0f, bits, 0.f, sc, st))) return rc;
  }
  keys_bwd_split_scores_kernel<TERMS><<<srows, 256, 0, st>>>(score_memory, N, m, Np, m8, TERMS == 2 ? 8192.0f : 1.0f, sms);
  VADC_CHECK_LAUNCH("keys_bwd_split_scores_kernel");
  keys_bwd_split_grad_kernel<TERMS><<<ggrid, 256, 0, st>>>(g_updated_query, B, 2 * d, d, d, HW, Np, sc ? sc + 1 : nullptr,
                                                           nullptr, gs);
  VADC_CHECK_LAUNCH("keys_bwd_split_grad_kernel");
  return tc_gemm<TERMS, true, false>({sms, gs, m8, d, Np, sc ? sc + 2 : nullptr, sk}, epi, st);
}

extern "C" int vadc_memory_keys_bwd(const float* score_memory, const float* g_updated_query, int B, int d, int64_t HW,
                                    int m, float* g_keys, void* workspace, size_t workspace_bytes, void* stream) {
  VADC_REQUIRE(B >= 0 && d > 0 && HW > 0 && m > 0, VADC_ERR_BAD_SHAPE);
  VADC_REQUIRE(g_keys && workspace, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(B == 0 || (score_memory && g_updated_query), VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(d >= 8 && d <= 65535 && B <= 65535 && (long long)B * HW < (1ll << 31) - 8, VADC_ERR_UNSUPPORTED);
  VADC_REQUIRE(workspace_bytes >= vadc_memory_keys_bwd_workspace_bytes(B, d, HW, m), VADC_ERR_WORKSPACE);
  if (!vadc_device_ok()) return VADC_ERR_NO_DEVICE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (B == 0) {                                          // no tokens: the read contributes nothing
    VADC_CUDA(cudaMemsetAsync(g_keys, 0, (size_t)m * d * sizeof(float), st));
    return VADC_OK;
  }
  const long long N = (long long)B * HW, Np = pad8(N);
  const int m8 = (int)pad8(m);
  const int sk = keys_bwd_splits(Np, m8, d);
  Carver ws(workspace, workspace_bytes);
  void* sms = ws.take<uint8_t>(tc_terms_bytes(3, Np, m8));
  void* gs = ws.take<uint8_t>(tc_terms_bytes(3, d, Np));
  float* part = ws.take<float>((size_t)sk * m8 * d);
  const TcPartialEpi epi{part, d, (long long)m8 * d};
  const int rc = env_int("VADC_MEMORY_TERMS", 2) == 3
                     ? keys_bwd_tc<3>(score_memory, g_updated_query, B, d, HW, m, sms, gs, sk, epi, ws, st)
                     : keys_bwd_tc<2>(score_memory, g_updated_query, B, d, HW, m, sms, gs, sk, epi, ws, st);
  if (rc) return rc;
  const long long md = (long long)m * d;
  keys_bwd_sum_partials_kernel<<<(unsigned)std::min<long long>((md + 255) / 256, 8ll * sm_count()), 256, 0, st>>>(
      part, sk, (long long)m8 * d, md, false, g_keys);
  VADC_CHECK_LAUNCH("keys_bwd_sum_partials_kernel");
  return VADC_OK;
}

extern "C" size_t vadc_memory_separateness_bwd_workspace_bytes(int m, int d) {
  (void)d;
  return align_up((size_t)(m > 0 ? m : 1) * (m > 0 ? m : 1) * sizeof(float), 256) + 256;
}

extern "C" int vadc_memory_separateness_bwd(const float* keys, const float* g_out, int m, int d, float* g_keys,
                                            void* workspace, size_t workspace_bytes, void* stream) {
  VADC_REQUIRE(m > 1 && d > 0, VADC_ERR_BAD_SHAPE);
  VADC_REQUIRE(keys && g_out && g_keys && workspace, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(workspace_bytes >= vadc_memory_separateness_bwd_workspace_bytes(m, d), VADC_ERR_WORKSPACE);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* sgn = static_cast<float*>(workspace);
  {
    Operand Aop{keys, d, 1}, Bop{keys, 1, d};                // K K^T exactly as vadc_memory_separateness forms it
    cudaError_t e = sgemm_auto(m, m, d, Aop, Bop, 0, 0, 1, 1, SeparatenessSignEpilogue{sgn, m}, st);
    if (e != cudaSuccess) return record_cuda_error(e, "separateness bwd sgemm K.K^T");
  }
  Operand Aop{sgn, m, 1}, Bop{keys, d, 1};
  cudaError_t e = sgemm_auto(m, d, m, Aop, Bop, 0, 0, 1, 1,
                             ScaledStoreEpilogue{g_keys, d, g_out, (float)(1.0 / ((double)m * (m - 1)))}, st);
  if (e != cudaSuccess) return record_cuda_error(e, "separateness bwd sgemm G.K");
  return VADC_OK;
}

extern "C" size_t vadc_memory_score_coldot_workspace_bytes(int64_t N, int m) {
  return align_up((size_t)col_chunks(N) * (m > 0 ? m : 1) * sizeof(float), 256) + 256;
}

extern "C" int vadc_memory_score_coldot(const float* score_query, const float* g_score_query, int64_t N, int m,
                                        float* coldot, void* workspace, size_t workspace_bytes, void* stream) {
  VADC_REQUIRE(N >= 0 && m > 0, VADC_ERR_BAD_SHAPE);
  VADC_REQUIRE(coldot && workspace, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(N == 0 || (score_query && g_score_query), VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(workspace_bytes >= vadc_memory_score_coldot_workspace_bytes(N, m), VADC_ERR_WORKSPACE);
  if (!vadc_device_ok()) return VADC_ERR_NO_DEVICE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (N == 0) {
    VADC_CUDA(cudaMemsetAsync(coldot, 0, (size_t)m * sizeof(float), st));
    return VADC_OK;
  }
  const int chunks = col_chunks(N);
  const long long rpb = (N + chunks - 1) / chunks;
  float* part = static_cast<float*>(workspace);
  score_coldot_stage1_kernel<<<dim3((m + 255) / 256, chunks), 256, 0, st>>>(score_query, g_score_query, N, m, rpb, part);
  VADC_CHECK_LAUNCH("score_coldot_stage1_kernel");
  score_coldot_stage2_kernel<<<(m + 31) / 32, 256, 0, st>>>(part, chunks, m, coldot);
  VADC_CHECK_LAUNCH("score_coldot_stage2_kernel");
  return VADC_OK;
}

extern "C" size_t vadc_memory_scores_bwd_workspace_bytes(int B, int d, int64_t HW, int m) {
  const long long Np = pad8((long long)(B > 0 ? B : 1) * (HW > 0 ? HW : 1)), m8 = pad8(m > 0 ? m : 1);
  const int dd = d > 0 ? d : 1;
  return tc_terms_bytes(3, Np, m8) + tc_terms_bytes(3, m8, pad8(dd)) + tc_terms_bytes(3, dd, Np) +  // terms
         align_up((size_t)Np * sizeof(float), 256) +                                                     // 1 / |x|
         align_up((size_t)keys_bwd_splits(Np, (int)m8, dd) * m8 * dd * sizeof(float), 256) + 1024;        // partials, scales
}

// the g_s pass and the two contractions of scores_bwd_impl.  TERMS = 3: fp32-faithful three-term bf16 split, six
// products.  TERMS = 2: g_s scaled from the bounds of the incoming gradients (no host sync), K from its measured max, and
// an unnormalised q (rows) from its measured max
template <int TERMS>
static int scores_bwd_tc(const float* query, bool rows, const float* keys, const float* score_query,
                         const float* score_memory, const float* g_score_query, const float* g_score_memory,
                         const float* coldot, int B, int d, int64_t HW, int m, float* g_q, float* g_keys, Carver& ws,
                         cudaStream_t st) {
  const long long N = (long long)B * HW, Np = pad8(N);
  const int m8 = (int)pad8(m), d8 = (int)pad8(d);
  const int sk = keys_bwd_splits(Np, m8, d);
  void* gst = ws.take<uint8_t>(tc_terms_bytes(3, Np, m8));
  void* kst = ws.take<uint8_t>(tc_terms_bytes(3, m8, d8));
  void* qst = ws.take<uint8_t>(tc_terms_bytes(3, d, Np));
  float* inv = ws.take<float>(Np);
  float* part = ws.take<float>((size_t)sk * m8 * d);
  unsigned* bits = ws.take<unsigned>(64);
  float* sc = ws.take<float>(64);
  auto at = [&](int i) -> const float* { return TERMS == 2 ? sc + i : nullptr; };
  int rc;
  if constexpr (TERMS == 2) {
    VADC_CUDA(cudaMemsetAsync(bits, 0, 4 * sizeof(unsigned), st));
    if (g_score_query) {
      if ((rc = tc_absmax_bits(g_score_query, N * m, bits, st))) return rc;
      if ((rc = tc_absmax_bits(coldot, m, bits + 2, st))) return rc;
    }
    if (g_score_memory && (rc = tc_absmax_bits(g_score_memory, N * m, bits + 1, st))) return rc;
    if (g_q && (rc = tc_absmax_bits(keys, (long long)m * d, bits + 3, st))) return rc;
    const bool q_measured = rows && g_keys;
    if (q_measured && (rc = tc_absmax_bits(query, N * d, bits + 4, st))) return rc;
    scores_bwd_scales_kernel<<<1, 1, 0, st>>>(bits, q_measured, sc);
    VADC_CHECK_LAUNCH("scores_bwd_scales_kernel");
  }
  {
    const unsigned rg = (unsigned)((Np + 7) / 8);
    const bool regs = (m % 4) == 0 && m <= 2048 && (!score_query || aligned16(score_query)) &&
                      (!score_memory || aligned16(score_memory)) && (!g_score_query || aligned16(g_score_query)) &&
                      (!g_score_memory || aligned16(g_score_memory)) && (!coldot || aligned16(coldot));
    const float* sq = g_score_query ? score_query : nullptr;
    const int V4 = !regs ? 0 : (m <= 512 ? 4 : (m <= 1024 ? 8 : 16));
#define VADC_GS_LAUNCH(V)                                                                                              \
  scores_bwd_gs_kernel<TERMS, V><<<rg, 256, 0, st>>>(sq, score_memory, g_score_query, g_score_memory, coldot, N, m, Np, \
                                                     m8, at(0), gst)
    if (V4 == 4) VADC_GS_LAUNCH(4); else if (V4 == 8) VADC_GS_LAUNCH(8);
    else if (V4 == 16) VADC_GS_LAUNCH(16); else VADC_GS_LAUNCH(0);
#undef VADC_GS_LAUNCH
    VADC_CHECK_LAUNCH("scores_bwd_gs_kernel");
  }
  if (g_q) {
    // g_q = g_s [Np, m8] . K [m8, d8].  Channel-first query: rows = tokens (g_s the K-major A operand, K the MN-major B),
    // stored into [B, d, HW].  Channel-last (rows): rows = channels (K the MN-major A operand, g_s the K-major B), stored
    // into [N, d] one 128-byte line of a token row per warp.
    const unsigned kr = (unsigned)std::min<long long>(m8, 16ll * sm_count());
    scores_bwd_split_keys_kernel<TERMS><<<kr, 256, 0, st>>>(keys, m, d, m8, d8, at(1), kst);
    VADC_CHECK_LAUNCH("scores_bwd_split_keys_kernel");
    rc = rows ? tc_gemm<TERMS, true, false>({kst, gst, d8, Np, m8, at(2)}, ScoresQRowsTEpi{g_q, N, d}, st)
              : tc_gemm<TERMS, false, true>({gst, kst, Np, d8, m8, at(2)}, ScoresQhatEpi{g_q, N, HW, d}, st);
    if (rc) return rc;
  }
  if (g_keys) {
    // g_keys [m8, d] += g_s^T q: g_s [Np, m8] the MN-major A operand, q^T [d, Np] (K-major B) written straight from the
    // query (channel-first: times 1 / |x|, i.e. q-hat; rows: one transposing pass); split-K over the tokens, the
    // partials then added to g_keys in slot order
    if (rows) {
      const dim3 tgrid((unsigned)((Np + 63) / 64), (unsigned)((d + 31) / 32));
      rows_transpose_terms_kernel<TERMS><<<tgrid, 256, 0, st>>>(query, N, d, Np, at(3), qst);
      VADC_CHECK_LAUNCH("rows_transpose_terms_kernel");
    } else {
      query_norm_kernel<<<dim3((unsigned)((HW + 31) / 32), B), 256, 0, st>>>(query, d, HW, inv);
      VADC_CHECK_LAUNCH("query_norm_kernel");
      const dim3 ggrid((unsigned)((HW + (Np - N) + 255) / 256), (unsigned)d, (unsigned)B);
      keys_bwd_split_grad_kernel<TERMS><<<ggrid, 256, 0, st>>>(query, B, d, 0, d, HW, Np, at(3), inv, qst);
      VADC_CHECK_LAUNCH("keys_bwd_split_grad_kernel");
    }
    if ((rc = tc_gemm<TERMS, true, false>({gst, qst, m8, d, Np, at(4), sk}, TcPartialEpi{part, d, (long long)m8 * d}, st)))
      return rc;
    const long long md = (long long)m * d;
    keys_bwd_sum_partials_kernel<<<(unsigned)std::min<long long>((md + 255) / 256, 8ll * sm_count()), 256, 0, st>>>(
        part, sk, (long long)m8 * d, md, true, g_keys);
    VADC_CHECK_LAUNCH("keys_bwd_sum_partials_kernel");
  }
  return VADC_OK;
}

// shared by vadc_memory_scores_bwd (query [B, d, HW], normalised where its operand terms are written) and
// vadc_memory_scores_bwd_rows (q [N, d] as passed: B = 1, HW = N): checks, scales, the g_s pass and the two contractions,
// whose query-side operand and epilogue follow the query's layout
static int scores_bwd_impl(const float* query, bool rows, const float* keys, const float* score_query,
                           const float* score_memory, const float* g_score_query, const float* g_score_memory,
                           const float* coldot, int B, int d, int64_t HW, int m, float* g_q, float* g_keys,
                           void* workspace, size_t workspace_bytes, void* stream) {
  VADC_REQUIRE(B >= 0 && d > 0 && HW > 0 && m > 0, VADC_ERR_BAD_SHAPE);
  VADC_REQUIRE(query && keys && workspace, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(g_score_query || g_score_memory, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(g_q || g_keys, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(!g_score_query || (score_query && coldot), VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(!g_score_memory || score_memory, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(d >= 8 && d <= 65535 && B <= 65535 && (long long)B * HW < (1ll << 31) - 8, VADC_ERR_UNSUPPORTED);
  VADC_REQUIRE(workspace_bytes >= vadc_memory_scores_bwd_workspace_bytes(B, d, HW, m), VADC_ERR_WORKSPACE);
  if (!vadc_device_ok()) return VADC_ERR_NO_DEVICE;
  if (B == 0) return VADC_OK;                            // no tokens: nothing to add to g_keys, g_q is empty
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Carver ws(workspace, workspace_bytes);
  return env_int("VADC_MEMORY_TERMS", 2) == 3
             ? scores_bwd_tc<3>(query, rows, keys, score_query, score_memory, g_score_query, g_score_memory, coldot, B, d, HW,
                                m, g_q, g_keys, ws, st)
             : scores_bwd_tc<2>(query, rows, keys, score_query, score_memory, g_score_query, g_score_memory, coldot, B, d, HW,
                                m, g_q, g_keys, ws, st);
}

extern "C" int vadc_memory_scores_bwd(const float* query, const float* keys, const float* score_query,
                                      const float* score_memory, const float* g_score_query,
                                      const float* g_score_memory, const float* coldot, int B, int d, int64_t HW,
                                      int m, float* g_qhat, float* g_keys, void* workspace, size_t workspace_bytes,
                                      void* stream) {
  return scores_bwd_impl(query, false, keys, score_query, score_memory, g_score_query, g_score_memory, coldot, B, d, HW,
                         m, g_qhat, g_keys, workspace, workspace_bytes, stream);
}

extern "C" size_t vadc_memory_scores_bwd_rows_workspace_bytes(int64_t N, int d, int m) {
  return vadc_memory_scores_bwd_workspace_bytes(1, d, N > 0 ? N : 1, m);
}

extern "C" int vadc_memory_scores_bwd_rows(const float* q, const float* keys, const float* score_query,
                                           const float* score_memory, const float* g_score_query,
                                           const float* g_score_memory, const float* coldot, int64_t N, int d, int m,
                                           float* g_q_rows, float* g_keys, void* workspace, size_t workspace_bytes,
                                           void* stream) {
  VADC_REQUIRE(N >= 0, VADC_ERR_BAD_SHAPE);
  return scores_bwd_impl(q, true, keys, score_query, score_memory, g_score_query, g_score_memory, coldot,
                         N > 0 ? 1 : 0, d, N > 0 ? N : 1, m, g_q_rows, g_keys, workspace, workspace_bytes, stream);
}

extern "C" int vadc_memory_rows_bwd(const float* q, const float* keys, const int64_t* top1, const int64_t* top2,
                                    const float* g_updated_query, const float* g_gather, const float* g_spread,
                                    const float* g_q_rows, int B, int d, int64_t HW, int m, float* g_query,
                                    void* stream) {
  VADC_REQUIRE(B >= 0 && d > 0 && HW > 0 && m > 0, VADC_ERR_BAD_SHAPE);
  if (B == 0) return VADC_OK;
  VADC_REQUIRE(q && keys && g_query, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(g_updated_query || g_gather || g_spread || g_q_rows, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(!(g_gather || g_spread) || top1, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(!g_spread || top2, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(B <= 65535 && (long long)B * HW < (1ll << 31), VADC_ERR_UNSUPPORTED);
  if (!vadc_device_ok()) return VADC_ERR_NO_DEVICE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  dim3 grid((unsigned)((HW + 31) / 32), B);
  memory_rows_bwd_kernel<<<grid, 256, 0, st>>>(q, keys, reinterpret_cast<const long long*>(top1),
                                               g_spread ? reinterpret_cast<const long long*>(top2) : nullptr,
                                               g_updated_query, g_gather, g_spread, g_q_rows, d, HW,
                                               (long long)B * HW, g_query);
  VADC_CHECK_LAUNCH("memory_rows_bwd_kernel");
  return VADC_OK;
}

extern "C" int vadc_memory_prepare_query_bwd(const float* g, const float* query, int B, int d, int64_t HW,
                                             float* g_x, void* stream) {
  VADC_REQUIRE(B >= 0 && d > 0 && HW > 0, VADC_ERR_BAD_SHAPE);
  if (B == 0) return VADC_OK;
  VADC_REQUIRE(g && query && g_x, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(B <= 65535, VADC_ERR_UNSUPPORTED);
  if (!vadc_device_ok()) return VADC_ERR_NO_DEVICE;
  prepare_query_bwd_kernel<<<dim3((unsigned)((HW + 31) / 32), B), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      g, query, d, HW, g_x);
  VADC_CHECK_LAUNCH("prepare_query_bwd_kernel");
  return VADC_OK;
}
