// tc_gemm.cuh — interface of the TMA-fed tcgen05 GEMM (tc_gemm.cu) and its epilogue functors.
// An epilogue receives 32 consecutive columns of one output row: epi(m, n, v[32], nvalid).
#pragma once
#include <cuda_bf16.h>
#include "common.cuh"

namespace vadc {

bool tc_gemm_shape_ok(long long M, long long N, long long Kd, bool b_mn);
size_t tc_gemm_split_bytes(long long rows, long long cols);     // workspace of one operand's three bf16 terms
int tc_split3(const float* src, long long rows, long long cols, void* dst, cudaStream_t st);

// C[m,n] = sum_k A[m,k] B(n,k); a_split / b_split from tc_split3 ([M,Kd]; [N,Kd] or, with B_MN, [Kd,N])
template <bool B_MN, class Epi>
int launch_tc_gemm(const void* a_split, const void* b_split, long long M, long long N, long long Kd, Epi epi,
                   cudaStream_t st);
// general form: A_MN = A given as [Kd, M] (e.g. a transposed token matrix), `splits` slots along the contraction,
// each handing its index to the epilogue (split-K partials for the centroid-gradient GEMMs, Kd = tokens)
template <bool A_MN, bool B_MN, class Epi>
int launch_tc_gemm_ex(const void* a_split, const void* b_split, long long M, long long N, long long Kd, int splits,
                      Epi epi, cudaStream_t st);

// two-term fp16 mode for bounded operands (tc_gemm.cu): operands pre-scaled by powers of two held in device memory,
// accumulators multiplied by *acc_scale before the epilogue
size_t tc_gemm_split2_bytes(long long rows, long long cols);
int tc_fwd_scales(const float* centers, const float* ln_w, const float* ln_b, long long KC, int C, float* out5,
                  cudaStream_t st);     // out (6 floats) = {s_z, s_c, 1/(s_z s_c), s_a, 1/(s_a s_c), 1/(s_c s_c)}
int tc_split2h(const float* src, long long rows, long long cols, const float* scale, void* dst, cudaStream_t st);
template <bool B_MN, class Epi>
int launch_tc_gemm_h2(const void* a_split, const void* b_split, long long M, long long N, long long Kd,
                      const float* acc_scale, Epi epi, cudaStream_t st);

// scales for operands whose bound has to be measured: max |src| as float bits (memset + atomicMax), then
// out3 = {s_a, s_b, 1 / (s_a s_b)} with s = the power of two that puts the bound in [4, 8), or the given constant
int tc_absmax_bits(const float* src, long long n, unsigned* out, cudaStream_t st);
// the same over nseg segments of n elements, `stride` elements apart (e.g. a channel slice of a [B, C, HW] tensor)
int tc_absmax_bits_seg(const float* src, long long n, int nseg, long long stride, unsigned* out, cudaStream_t st);
int tc_pair_scales(const unsigned* a_bits, float a_given, const unsigned* b_bits, float b_given, float* out3, cudaStream_t st);
int tc_fwd_scales_from_bits(const unsigned* cen_bits, const float* ln_w, const float* ln_b, int C, float* out6, cudaStream_t st);
int tc_cluster_bwd_scales(const unsigned* bits4, int stage, float* out9, cudaStream_t st);   // see tc_gemm.cu
int tc_space_bwd_scales(const unsigned* r_bits, const float* fwd_sc, float* out3, cudaStream_t st);   // {s_r, 1/(s_c s_r), 1/(s_r s_z)}

template <bool A_MN, bool B_MN, class Epi>
int launch_tc_gemm_ex_h2(const void* a_split, const void* b_split, long long M, long long N, long long Kd, int splits,
                         const float* acc_scale, Epi epi, cudaStream_t st);

// batched form (z = batch, handed to the epilogue): per-batch coordinate offsets along the operands' tensors — a_m / b_n along the
// output-row / output-column dimension, a_k / b_k along the contraction dimension
struct TcBatchOffsets { int a_m, a_k, b_n, b_k; };
template <bool A_MN, bool B_MN, class Epi>
int launch_tc_gemm_batched(const void* a_split, long long a_rows, long long a_cols, const void* b_split,
                           long long b_rows, long long b_cols, long long M, long long N, long long Kd, int nbatch,
                           TcBatchOffsets off, Epi epi, cudaStream_t st);

template <bool A_MN, bool B_MN, class Epi>
int launch_tc_gemm_batched_h2(const void* a_split, long long a_rows, long long a_cols, const void* b_split,
                              long long b_rows, long long b_cols, long long M, long long N, long long Kd, int nbatch,
                              TcBatchOffsets off, const float* acc_scale, Epi epi, cudaStream_t st);

__device__ __forceinline__ void tc_store_row32(float* o, const float (&v)[32], int nvalid) {
  if (nvalid == 32 && (reinterpret_cast<uintptr_t>(o) & 15u) == 0) {
#pragma unroll
    for (int j = 0; j < 8; ++j) reinterpret_cast<float4*>(o)[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j) if (j < nvalid) o[j] = v[j];
  }
}

// t[0..nvalid) = src[0..nvalid), the rest zero; never a predicated load followed by its use inside a branch
__device__ __forceinline__ void tc_load_row32(const float* src, float (&t)[32], int nvalid) {
  if (nvalid == 32 && (reinterpret_cast<uintptr_t>(src) & 15u) == 0) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(src) + j);
      t[4 * j] = a.x; t[4 * j + 1] = a.y; t[4 * j + 2] = a.z; t[4 * j + 3] = a.w;
    }
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j) t[j] = __ldg(src + min(j, nvalid - 1));
#pragma unroll
    for (int j = 0; j < 32; ++j) t[j] = j < nvalid ? t[j] : 0.f;
  }
}

struct TcStoreEpi {
  float* out; long long ldo;
  __device__ __forceinline__ void operator()(long long m, int n, float (&v)[32], int nvalid, int = 0) const {
    tc_store_row32(out + m * ldo + n, v, nvalid);
  }
};

// ---- transposed forms: the GEMM is launched with its operands swapped, so its rows (TMEM lanes = epilogue threads)
// run along the CONTIGUOUS dimension of the output and its 32 columns are 32 output rows: every store instruction of
// a warp writes 128 contiguous bytes of one output row (row-per-lane epilogues write 16 bytes to each of 32 rows).
// `c` = index along the output's contiguous dimension, `r0` = first of the 32 output rows.
// (full 32-row groups take a branch-free path: one pointer bump and one store per row)
__device__ __forceinline__ void tc_store_col32(float* o, long long ld, const float (&v)[32], int nvalid) {
  if (nvalid == 32) {
#pragma unroll
    for (int j = 0; j < 32; ++j) { *o = v[j]; o += ld; }
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j) { if (j < nvalid) *o = v[j]; o += ld; }
  }
}

struct TcStoreTEpi {
  float* out; long long ldo;
  __device__ __forceinline__ void operator()(long long c, int r0, float (&v)[32], int nvalid, int = 0) const {
    tc_store_col32(out + (long long)r0 * ldo + c, ldo, v, nvalid);
  }
};

// memory logits (Memory.py:133-143), transposed (c = memory slot, rows = tokens): stores the logits and, from the same
// registers, the slot's online (max, sum exp) over this group of 32 tokens — the column-softmax statistics of
// `score_query` without another pass over [N, m]; pmax / psum [ceil(N / 32), m]
struct TcLogitsColStatsTEpi {
  float* out; long long ldo; float* pmax; float* psum;
  __device__ __forceinline__ void operator()(long long c, int r0, float (&v)[32], int nvalid, int = 0) const {
    tc_store_col32(out + (long long)r0 * ldo + c, ldo, v, nvalid);
    float mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < 32; ++j) mx = fmaxf(mx, j < nvalid ? v[j] : -INFINITY);
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < 32; ++j) s += j < nvalid ? expf(v[j] - mx) : 0.f;
    const long long g = (long long)(r0 >> 5) * ldo + c;
    pmax[g] = mx; psum[g] = s;
  }
};

// sqrt for the two-term fp16 paths (22 significant bits already): MUFU.SQRT, <= 1 ulp, no slow-path branch per element
__device__ __forceinline__ float sqrt_approx(float x) {
  float y;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// torch.cdist (mm form), transposed: out[r, c] = sqrt(max(0, |row r|^2 + |col c|^2 - 2 dot)); cn = norms along c, rn along r
struct TcDistTEpi {
  float* out; const float* cn; const float* rn; long long ldo;
  __device__ __forceinline__ void operator()(long long c, int r0, float (&v)[32], int nvalid, int = 0) const {
    const float cc = cn[c];
    float rr[32];
    if (nvalid == 32 && ((r0 & 3) == 0)) {               // rn + r0 is 16-byte aligned (rn comes from the workspace carver)
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(rn + r0) + j);
        rr[4 * j] = t.x; rr[4 * j + 1] = t.y; rr[4 * j + 2] = t.z; rr[4 * j + 3] = t.w;
      }
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j) rr[j] = __ldg(rn + r0 + min(j, nvalid - 1));
    }
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = sqrt_approx(fmaxf(fmaf(-2.0f, v[j], rr[j] + cc), 0.f));
    tc_store_col32(out + (long long)r0 * ldo + c, ldo, v, nvalid);
  }
};

// encoder downsample stage (model/swin_transformer.py:575-585): bias + exact GELU, transposed (c = output channel, rows =
// tokens, channel-last output); `pre` (optional) keeps the pre-activation for the backward
struct TcBiasGeluTEpi {
  float* out; float* pre; const float* bias; long long ld;
  __device__ __forceinline__ void operator()(long long c, int r0, float (&v)[32], int nvalid, int = 0) const {
    const float b = bias[c];
    float* o = out + (long long)r0 * ld + c;
    float* p = pre ? pre + (long long)r0 * ld + c : nullptr;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float a = v[j] + b;
      const float g = 0.5f * a * (1.0f + erff(a * 0.70710678118654752f));
      if (j < nvalid) {
        o[(long long)j * ld] = g;
        if (p) p[(long long)j * ld] = a;
      }
    }
  }
};

// out[m, n] = acc + bias[n] (row per lane; for outputs with fewer than 8 rows the transposed form cannot take)
struct TcBiasEpi {
  float* out; const float* bias; long long ld;
  __device__ __forceinline__ void operator()(long long m, int n, float (&v)[32], int nvalid, int = 0) const {
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] += bias[n + min(j, nvalid - 1)];
    tc_store_row32(out + m * ld + n, v, nvalid);
  }
};

// out[r, c] = acc + bias[c], transposed (c = output channel, rows = tokens): the predict-mode decoder entry
struct TcBiasTEpi {
  float* out; const float* bias; long long ld;
  __device__ __forceinline__ void operator()(long long c, int r0, float (&v)[32], int nvalid, int = 0) const {
    const float b = bias[c];
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] += b;
    tc_store_col32(out + (long long)r0 * ld + c, ld, v, nvalid);
  }
};

// Memory.read (Memory.py:249-261), transposed: c = channel, rows = tokens
struct TcReadTEpi {
  float* uq; const float* q; int d;
  __device__ __forceinline__ void operator()(long long c, int r0, float (&v)[32], int nvalid, int = 0) const {
    float t[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) t[j] = __ldg(q + (long long)(r0 + min(j, nvalid - 1)) * d + c);
    tc_store_col32(uq + (long long)r0 * 2 * d + c, 2ll * d, t, nvalid);
    tc_store_col32(uq + (long long)r0 * 2 * d + d + c, 2ll * d, v, nvalid);
  }
};

// gz = feature * rsum - r @ centers + gF (cluster backward, generic path), transposed: c = channel, rows = tokens
struct TcGzTEpi {
  float* out; const float* feature; const float* rsum; const float* gF; long long ld;
  __device__ __forceinline__ void operator()(long long c, int r0, float (&v)[32], int nvalid, int = 0) const {
    float f[32], rs[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const long long r = r0 + min(j, nvalid - 1);
      f[j] = __ldg(feature + r * ld + c); rs[j] = __ldg(rsum + r);
    }
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = f[j] * rs[j] - v[j];
    if (gF) {
#pragma unroll
      for (int j = 0; j < 32; ++j) f[j] = __ldg(gF + (long long)(r0 + min(j, nvalid - 1)) * ld + c);
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] += f[j];
    }
    tc_store_col32(out + (long long)r0 * ld + c, ld, v, nvalid);
  }
};

// torch.cdist, mm form: sqrt(max(0, |a|^2 + |b|^2 - 2 a.b))
struct TcDistEpi {
  float* out; const float* aa; const float* bb; long long ldo;
  __device__ __forceinline__ void operator()(long long m, int n, float (&v)[32], int nvalid, int = 0) const {
    const float am = aa[m];
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float b = (j < nvalid) ? bb[n + j] : 0.f;
      v[j] = sqrtf(fmaxf(am + b - 2.0f * v[j], 0.f));
    }
    tc_store_row32(out + m * ldo + n, v, nvalid);
  }
};

// batched torch.cdist (mm form): out[z out_z + m ldo + n] from |a|^2 [z aa_z + m], |b|^2 [z bb_z + n]
struct TcBatchDistEpi {
  float* out; const float* aa; const float* bb; long long ldo, out_z, aa_z, bb_z;
  __device__ __forceinline__ void operator()(long long m, int n, float (&v)[32], int nvalid, int z) const {
    const float am = aa[z * aa_z + m];
    const float* b = bb + z * bb_z + n;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float bj = (j < nvalid) ? b[j] : 0.f;
      v[j] = sqrtf(fmaxf(am + bj - 2.0f * v[j], 0.f));
    }
    tc_store_row32(out + z * out_z + m * ldo + n, v, nvalid);
  }
};

// space head backward (model/cluster.py:127-149 under autograd): gzt[c,m,p] = zt[c,m,p] rsum[m,c] - (r centers)[m,p].
// The GEMM writes only the contraction, acc[c,m,p] = (r[:,c,:] centers[c])[m,p]; the LayerNorm backward that consumes
// it forms zt rsum - acc itself from the x-hat it has in registers (zt = x-hat gamma + beta), so nothing is re-read
// here.  Computed TRANSPOSED — the GEMM's rows (TMEM lanes = epilogue threads) are the positions p, its columns the
// frames m — so that for every frame a warp stores 32 consecutive p (128 contiguous bytes).
struct TcSpaceGzEpi {
  float* out; long long MP; int P;
  __device__ __forceinline__ void operator()(long long p, int n, float (&v)[32], int nvalid, int z) const {
    tc_store_col32(out + (long long)z * MP + (long long)n * P + p, P, v, nvalid);
  }
};

// gcenters[c,k,p] = centers[c,k,p] rcol[c,k] - (r^T zt)[k,p]
struct TcSpaceGcEpi {
  float* out; const float* centers; const float* rcol; long long KP; int P, K;
  __device__ __forceinline__ void operator()(long long m, int n, float (&v)[32], int nvalid, int z) const {
    const long long i = (long long)z * KP + m * P + n;
    const float rc = rcol[(long long)z * K + m];
    if (nvalid == 32 && (reinterpret_cast<uintptr_t>(centers + i) & 15u) == 0) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(centers + i) + j);
        v[4 * j] = t.x * rc - v[4 * j]; v[4 * j + 1] = t.y * rc - v[4 * j + 1];
        v[4 * j + 2] = t.z * rc - v[4 * j + 2]; v[4 * j + 3] = t.w * rc - v[4 * j + 3];
      }
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j) if (j < nvalid) v[j] = centers[i + j] * rc - v[j];
    }
    tc_store_row32(out + i, v, nvalid);
  }
};

// Memory.read (Memory.py:249-261): uq[m, 0:d] = q[m], uq[m, d:2d] = score_memory @ keys
// (the row loads of these two are unconditional — 128-bit where the row is aligned, clamped indices otherwise: a
// predicated load + use per column compiles to one branch region per column, every load waited for alone)
struct TcReadEpi {
  float* uq; const float* q; int d;
  __device__ __forceinline__ void operator()(long long m, int n, float (&v)[32], int nvalid, int = 0) const {
    float* o = uq + m * 2 * d;
    tc_store_row32(o + d + n, v, nvalid);
    const float* qs = q + m * d + n;
    float t[32];
    tc_load_row32(qs, t, nvalid);
    tc_store_row32(o + n, t, nvalid);
  }
};

// gz = feature * rsum - r @ centers + gF   (cluster backward, generic path)
struct TcGzEpi {
  float* out; const float* feature; const float* rsum; const float* gF; long long ld;
  __device__ __forceinline__ void operator()(long long m, int n, float (&v)[32], int nvalid, int = 0) const {
    const float rs = rsum[m];
    float t[32];
    tc_load_row32(feature + m * ld + n, t, nvalid);
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = t[j] * rs - v[j];
    if (gF) {
      tc_load_row32(gF + m * ld + n, t, nvalid);
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] += t[j];
    }
    tc_store_row32(out + m * ld + n, v, nvalid);
  }
};

// decoder entry (model/swin_decoder_predict.py:590-602; bias may be null: the predict-mode entry's backward reuses the
// scatter): ConvTranspose3d(C -> C, kernel (2,1,1), stride (2,1,1)) of the
// channel-last tokens as ONE GEMM [N, C] x [C, 2C]: column j*C + co of token n = (frame f, pixel hw) is channel co of
// output frame 2f + j, written channel-last: out[((f * 2 + j) * HW + hw) * C + co] + bias[co]
struct TcTimeDebedEpi {
  float* out; const float* bias; long long HW; int C;
  __device__ __forceinline__ void operator()(long long m, int n, float (&v)[32], int nvalid, int = 0) const {
    const int j = n / C, co = n - j * C;
    const long long f = m / HW, hw = m - f * HW;
    if (bias) {
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] += bias[co + min(i, nvalid - 1)];
    }
    tc_store_row32(out + ((f * 2 + j) * HW + hw) * C + co, v, nvalid);
  }
};

// Memory: gradient with respect to q-hat through the score matrices, g_qhat = g_s K (vadc_memory_scores_bwd).  The
// GEMM's rows (TMEM lanes = epilogue threads) are the tokens, its columns the channels: for each channel a warp stores
// 32 consecutive tokens, one 128-byte line of the query's [B, d, HW] layout (two where the 32 tokens straddle a batch
// boundary, n = b HW + hw).  Rows N..Np-1 and channels d..d8-1 are padding.
struct ScoresQhatEpi {
  float* out; long long N, HW; int d;
  __device__ __forceinline__ void operator()(long long n, int c, float (&v)[32], int nvalid, int = 0) const {
    if (n >= N) return;
    const long long b = n / HW, hw = n - b * HW;
    tc_store_col32(out + (b * d + c) * HW + hw, HW, v, min(nvalid, d - c));
  }
};

// Memory: g_q = g_s K for the stand-alone methods' channel-last query [N, d] (vadc_memory_scores_bwd_rows), transposed:
// the GEMM's rows are the channels (K's terms [m8, d8] the MN-major A operand), its columns the tokens, so for each token
// a warp stores 32 consecutive channels, one 128-byte line of its row.  Channels d..d8-1 and tokens N..Np-1 are padding.
struct ScoresQRowsTEpi {
  float* out; long long N; int d;
  __device__ __forceinline__ void operator()(long long c, int r0, float (&v)[32], int nvalid, int = 0) const {
    if (c >= d) return;
    tc_store_col32(out + (long long)r0 * d + c, d, v, (int)min((long long)nvalid, N - r0));
  }
};

// split-K partial: out[split][m][n]
struct TcPartialEpi {
  float* out; long long ld, split_stride;
  __device__ __forceinline__ void operator()(long long m, int n, float (&v)[32], int nvalid, int split) const {
    tc_store_row32(out + (long long)split * split_stride + m * ld + n, v, nvalid);
  }
};

}  // namespace vadc
