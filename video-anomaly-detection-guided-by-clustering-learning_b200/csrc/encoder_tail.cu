// encoder_tail.cu — SURVEY.md 8f-3: the encoder's downsample stage (model/swin_transformer.py:575-585:
// Conv3d(Cin -> Cout, kernel (1,2,2), stride (1,2,2)) + GELU) as a producer of CHANNEL-LAST tokens, so that the
// 'n c d h w -> n d h w c' rearranges that follow it (swin_transformer.py:745, model/backbone.py:82) are views and the
// cluster head reads its input without a transposing copy.
//
// A stride == kernel convolution is a GEMM over non-overlapping patches:
//   out[(b,d,h,w), co] = gelu( sum_{ci,dy,dx} x[b,ci,d,2h+dy,2w+dx] W[co,ci,0,dy,dx] + bias[co] )
// forward : patchify x into the bf16 x3 operand terms of A [tokens, Cin*4] (k = ci*4 + dy*2 + dx, the order of
//           W.reshape(Cout, Cin*4)), then W . A^T on tcgen05 with the operands swapped (rows = output channels) so
//           that every store of the channel-last result is one 128-byte line per warp; bias + exact (erf) GELU in the
//           epilogue, which also keeps the pre-activation for the backward.
// backward: g_pre = g_out * gelu'(pre) (with its operand terms), g_bias = column sums, g_A = g_pre . W scattered back
//           to the channel-first input by the inverse patch permutation, g_W = g_pre^T . A split over the tokens.
#include <cuda_bf16.h>
#include <algorithm>
#include "common.cuh"
#include "tc_gemm.cuh"
#include "cluster.h"

namespace vadc {

constexpr int kPatchTok = 32;       // tokens (consecutive w) per block of the patch permutation kernels

__device__ __forceinline__ void split3_pair(float a, float b, __nv_bfloat162& h0, __nv_bfloat162& h1, __nv_bfloat162& h2) {
  h0 = __floats2bfloat162_rn(a, b);
  const float r0 = a - __low2float(h0), r1 = b - __high2float(h0);
  h1 = __floats2bfloat162_rn(r0, r1);
  h2 = __floats2bfloat162_rn(r0 - __low2float(h1), r1 - __high2float(h1));
}

// x [B, Cin, D, 2H, 2W] -> the three bf16 terms of A [B*D*H*W, Cin*4]; a block owns 32 consecutive w of one (b, d, h):
// coalesced float2 reads per (ci, dy) into a [32][K4+1] tile, then a token's K4 values written contiguously
__global__ void __launch_bounds__(256)
patchify_split3_kernel(const float* __restrict__ x, int Cin, int D, int H, int W, long long NT,
                       __nv_bfloat16* __restrict__ terms) {
  extern __shared__ float tile[];
  const int K4 = Cin * 4, ld = K4 + 1;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const long long bdh = blockIdx.x;
  const int h = (int)(bdh % H), d = (int)((bdh / H) % D);
  const long long b = bdh / ((long long)H * D);
  const int w0 = blockIdx.y * kPatchTok, nw = min(kPatchTok, W - w0);
  for (int i = wid; i < 2 * Cin; i += 8) {
    const int ci = i >> 1, dy = i & 1;
    if (lane < nw) {
      const float* src = x + ((((b * Cin + ci) * D + d) * (2ll * H) + 2 * h + dy) * (2ll * W)) + 2 * (w0 + lane);
      const float2 v = __ldg(reinterpret_cast<const float2*>(src));
      tile[lane * ld + ci * 4 + dy * 2] = v.x;
      tile[lane * ld + ci * 4 + dy * 2 + 1] = v.y;
    }
  }
  __syncthreads();
  const long long row0 = bdh * W + w0, n = NT * K4;
  for (int tok = wid; tok < nw; tok += 8) {
    __nv_bfloat16* dst = terms + (row0 + tok) * K4;
    for (int k = 2 * lane; k < K4; k += 64) {
      __nv_bfloat162 h0, h1, h2;
      split3_pair(tile[tok * ld + k], tile[tok * ld + k + 1], h0, h1, h2);
      *reinterpret_cast<__nv_bfloat162*>(dst + k) = h0;
      *reinterpret_cast<__nv_bfloat162*>(dst + n + k) = h1;
      *reinterpret_cast<__nv_bfloat162*>(dst + 2 * n + k) = h2;
    }
  }
}

// the inverse permutation: gA [B*D*H*W, Cin*4] fp32 -> gx [B, Cin, D, 2H, 2W]
__global__ void __launch_bounds__(256)
unpatchify_kernel(const float* __restrict__ ga, int Cin, int D, int H, int W, float* __restrict__ gx) {
  extern __shared__ float tile[];
  const int K4 = Cin * 4, ld = K4 + 1;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const long long bdh = blockIdx.x;
  const int h = (int)(bdh % H), d = (int)((bdh / H) % D);
  const long long b = bdh / ((long long)H * D);
  const int w0 = blockIdx.y * kPatchTok, nw = min(kPatchTok, W - w0);
  const long long row0 = bdh * W + w0;
  for (int tok = wid; tok < nw; tok += 8) {
    const float* src = ga + (row0 + tok) * K4;
    for (int k = 2 * lane; k < K4; k += 64) {
      const float2 v = __ldg(reinterpret_cast<const float2*>(src + k));
      tile[tok * ld + k] = v.x; tile[tok * ld + k + 1] = v.y;
    }
  }
  __syncthreads();
  for (int i = wid; i < 2 * Cin; i += 8) {
    const int ci = i >> 1, dy = i & 1;
    if (lane < nw) {
      float* dst = gx + ((((b * Cin + ci) * D + d) * (2ll * H) + 2 * h + dy) * (2ll * W)) + 2 * (w0 + lane);
      *reinterpret_cast<float2*>(dst) = make_float2(tile[lane * ld + ci * 4 + dy * 2], tile[lane * ld + ci * 4 + dy * 2 + 1]);
    }
  }
}

// g_pre = g_out * d gelu(pre) / d pre (exact GELU: Phi(p) + p phi(p)), fp32 and as bf16 x3 operand terms
__global__ void __launch_bounds__(256)
gelu_bwd_split3_kernel(const float* __restrict__ pre, const float* __restrict__ gout, long long n4, float* __restrict__ gpre,
                       __nv_bfloat16* __restrict__ t0, __nv_bfloat16* __restrict__ t1, __nv_bfloat16* __restrict__ t2) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 p = __ldg(reinterpret_cast<const float4*>(pre) + i), g = __ldg(reinterpret_cast<const float4*>(gout) + i);
    const float pv[4] = {p.x, p.y, p.z, p.w}, gv[4] = {g.x, g.y, g.z, g.w};
    float o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float cdf = 0.5f * (1.0f + erff(pv[j] * 0.70710678118654752f));
      const float pdf = 0.39894228040143268f * expf(-0.5f * pv[j] * pv[j]);
      o[j] = gv[j] * (cdf + pv[j] * pdf);
    }
    reinterpret_cast<float4*>(gpre)[i] = make_float4(o[0], o[1], o[2], o[3]);
    __nv_bfloat162 h[3][2];
    split3_pair(o[0], o[1], h[0][0], h[1][0], h[2][0]);
    split3_pair(o[2], o[3], h[0][1], h[1][1], h[2][1]);
    reinterpret_cast<uint2*>(t0)[i] = *reinterpret_cast<uint2*>(h[0]);
    reinterpret_cast<uint2*>(t1)[i] = *reinterpret_cast<uint2*>(h[1]);
    reinterpret_cast<uint2*>(t2)[i] = *reinterpret_cast<uint2*>(h[2]);
  }
}

__global__ void __launch_bounds__(256)
tail_sum_partials_kernel(const float* __restrict__ q, int splits, long long n, float* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float s = 0.f;
  for (int sp = 0; sp < splits; ++sp) s += q[sp * n + i];       // fixed order: deterministic
  out[i] = s;
}

// column sums of a [R, C] matrix in two deterministic stages (R is large here: tokens)
__global__ void __launch_bounds__(256)
tail_colsum_stage1_kernel(const float* __restrict__ a, long long R, int C, long long rpb, float* __restrict__ part) {
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c >= C) return;
  const long long r0 = (long long)blockIdx.y * rpb, r1 = min(R, r0 + rpb);
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  long long r = r0;
  for (; r + 3 < r1; r += 4) {
    s0 += __ldg(a + r * C + c); s1 += __ldg(a + (r + 1) * C + c); s2 += __ldg(a + (r + 2) * C + c); s3 += __ldg(a + (r + 3) * C + c);
  }
  for (; r < r1; ++r) s0 += __ldg(a + r * C + c);
  part[(long long)blockIdx.y * C + c] = (s0 + s1) + (s2 + s3);
}

// partial [chunks, C] -> out [C]: a block owns 32 columns, eight warps stride the chunks (fixed order: deterministic)
__global__ void __launch_bounds__(256)
tail_colsum_stage2_kernel(const float* __restrict__ part, int chunks, int C, float* __restrict__ out) {
  __shared__ float red[8][33];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + lane;
  float s = 0.f;
  if (c < C)
    for (int b = wid; b < chunks; b += 8) s += part[(size_t)b * C + c];
  red[wid][lane] = s;
  __syncthreads();
  if (wid == 0 && c < C) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += red[w][lane];
    out[c] = t;
  }
}

static int tail_splits(long long NT, int Cout, int K4) {
  const long long tiles = (long long)((Cout + 127) / 128) * ((K4 + 127) / 128);
  const long long nkb = (NT + 63) / 64;
  long long s = (2ll * sm_count() + tiles - 1) / tiles;
  return (int)std::max<long long>(1, std::min(s, nkb));
}
static int tail_colsum_chunks(long long NT) { return (int)std::max<long long>(1, std::min<long long>(1024, (NT + 255) / 256)); }

static bool tail_shape_ok(int B, int Cin, int D, int H, int W, int Cout) {
  const long long NT = (long long)B * D * H * W;
  return B > 0 && Cin > 0 && D > 0 && H > 0 && W > 0 && Cout >= 8 && (Cout % 8) == 0 && (Cin % 2) == 0 && NT >= 8 && NT < (1ll << 31) &&
         (W + kPatchTok - 1) / kPatchTok <= 65535 && (size_t)kPatchTok * (Cin * 4 + 1) * sizeof(float) <= 200 * 1024 && tc_gemm_shape_ok(Cout, NT, Cin * 4, false) &&
         tc_gemm_shape_ok(Cin * 4, NT, Cout, false);
}

static int launch_patchify(const float* x, int B, int Cin, int D, int H, int W, void* terms, cudaStream_t st) {
  const size_t smem = (size_t)kPatchTok * (Cin * 4 + 1) * sizeof(float);
  if (smem > 48 * 1024) VADC_CUDA(cudaFuncSetAttribute(patchify_split3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const long long bdh = (long long)B * D * H;
  dim3 grid((unsigned)bdh, (unsigned)((W + kPatchTok - 1) / kPatchTok));
  patchify_split3_kernel<<<grid, 256, smem, st>>>(x, Cin, D, H, W, bdh * W, static_cast<__nv_bfloat16*>(terms));
  VADC_CHECK_LAUNCH("patchify_split3_kernel");
  return VADC_OK;
}

}  // namespace vadc

using namespace vadc;

extern "C" int vadc_downsample_gelu_supported(int B, int Cin, int D, int H, int W, int Cout) {
  return tail_shape_ok(B, Cin, D, H, W, Cout) ? 1 : 0;
}

extern "C" size_t vadc_downsample_gelu_workspace_bytes(int B, int Cin, int D, int H, int W, int Cout) {
  const long long NT = (long long)std::max(B, 1) * std::max(D, 1) * std::max(H, 1) * std::max(W, 1);
  const int K4 = Cin * 4;
  size_t b = 0;
  b += tc_terms_bytes(3, NT, K4);                                   // A terms
  b += tc_terms_bytes(3, Cout, K4);                                 // W terms
  b += align_up((size_t)NT * Cout * sizeof(float), 256);              // g_pre
  b += tc_terms_bytes(3, NT, Cout);                                 // g_pre terms
  b += align_up((size_t)NT * K4 * sizeof(float), 256);                // g_A
  b += align_up((size_t)tail_splits(NT, Cout, K4) * Cout * K4 * sizeof(float), 256);
  b += align_up((size_t)tail_colsum_chunks(NT) * Cout * sizeof(float), 256);
  return b + 256;
}

// x [B, Cin, D, 2H, 2W] contiguous (channel-first, as the Swin stage leaves it); weight [Cout, Cin*4] =
// Conv3d.weight.reshape(Cout, -1); out / pre [B, D, H, W, Cout] channel-last (pre may be NULL: inference)
extern "C" int vadc_downsample_gelu_fwd(const float* x, const float* weight, const float* bias, int B, int Cin, int D, int H,
                                        int W, int Cout, float* out, float* pre, void* workspace, size_t workspace_bytes,
                                        void* stream) {
  VADC_REQUIRE(x && weight && bias && out && workspace, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(tail_shape_ok(B, Cin, D, H, W, Cout), VADC_ERR_UNSUPPORTED);
  VADC_REQUIRE(aligned16(x) && aligned16(weight) && aligned16(out) && (!pre || aligned16(pre)), VADC_ERR_MISALIGNED);
  VADC_REQUIRE(workspace_bytes >= vadc_downsample_gelu_workspace_bytes(B, Cin, D, H, W, Cout), VADC_ERR_WORKSPACE);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long NT = (long long)B * D * H * W;
  const int K4 = Cin * 4;
  Carver ws(workspace, workspace_bytes);
  void* as = ws.take<uint8_t>(tc_terms_bytes(3, NT, K4));
  void* wsp = ws.take<uint8_t>(tc_terms_bytes(3, Cout, K4));
  int rc;
  if ((rc = launch_patchify(x, B, Cin, D, H, W, as, st))) return rc;
  if ((rc = tc_split<3>(weight, Cout, K4, nullptr, wsp, st))) return rc;
  // rows = output channels, columns = tokens: out[token, co] stored 128 contiguous bytes per warp
  return tc_gemm<3, false, false>({wsp, as, Cout, NT, K4}, TcBiasGeluTEpi{out, pre, bias, Cout}, st);
}

extern "C" int vadc_downsample_gelu_bwd(const float* x, const float* weight, const float* pre, const float* gout, int B,
                                        int Cin, int D, int H, int W, int Cout, float* gx, float* gweight, float* gbias,
                                        void* workspace, size_t workspace_bytes, void* stream) {
  VADC_REQUIRE(x && weight && pre && gout && gx && gweight && gbias && workspace, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(tail_shape_ok(B, Cin, D, H, W, Cout), VADC_ERR_UNSUPPORTED);
  VADC_REQUIRE(aligned16(x) && aligned16(weight) && aligned16(pre) && aligned16(gout) && aligned16(gx), VADC_ERR_MISALIGNED);
  VADC_REQUIRE(workspace_bytes >= vadc_downsample_gelu_workspace_bytes(B, Cin, D, H, W, Cout), VADC_ERR_WORKSPACE);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long NT = (long long)B * D * H * W;
  const int K4 = Cin * 4;
  const int sk = tail_splits(NT, Cout, K4), cch = tail_colsum_chunks(NT);
  Carver ws(workspace, workspace_bytes);
  void* as = ws.take<uint8_t>(tc_terms_bytes(3, NT, K4));
  void* wsp = ws.take<uint8_t>(tc_terms_bytes(3, Cout, K4));
  float* gpre = ws.take<float>((size_t)NT * Cout);
  __nv_bfloat16* gps = reinterpret_cast<__nv_bfloat16*>(ws.take<uint8_t>(tc_terms_bytes(3, NT, Cout)));
  float* ga = ws.take<float>((size_t)NT * K4);
  float* part = ws.take<float>((size_t)sk * Cout * K4);
  float* cpart = ws.take<float>((size_t)cch * Cout);
  int rc;
  {
    const long long n = NT * Cout, n4 = n / 4;                         // Cout % 8 == 0
    const int grid = (int)std::min<long long>((n4 + 255) / 256, (long long)sm_count() * 8);
    gelu_bwd_split3_kernel<<<grid, 256, 0, st>>>(pre, gout, n4, gpre, gps, gps + n, gps + 2 * n);
    VADC_CHECK_LAUNCH("gelu_bwd_split3_kernel");
  }
  {
    const long long rpb = (NT + cch - 1) / cch;
    tail_colsum_stage1_kernel<<<dim3((Cout + 255) / 256, cch), 256, 0, st>>>(gpre, NT, Cout, rpb, cpart);
    VADC_CHECK_LAUNCH("tail_colsum_stage1_kernel");
    tail_colsum_stage2_kernel<<<(Cout + 31) / 32, 256, 0, st>>>(cpart, cch, Cout, gbias);
    VADC_CHECK_LAUNCH("tail_colsum_stage2_kernel");
  }
  // g_A[token, k] = sum_co g_pre[token, co] W[co, k]: rows = k (W [Cout, K4] is the MN-major A operand), columns = tokens
  if ((rc = tc_split<3>(weight, Cout, K4, nullptr, wsp, st))) return rc;
  if ((rc = tc_gemm<3, true, false>({wsp, gps, K4, NT, Cout}, TcStoreTEpi{ga, K4}, st))) return rc;
  {
    const size_t smem = (size_t)kPatchTok * (K4 + 1) * sizeof(float);
    if (smem > 48 * 1024) VADC_CUDA(cudaFuncSetAttribute(unpatchify_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid((unsigned)((long long)B * D * H), (unsigned)((W + kPatchTok - 1) / kPatchTok));
    unpatchify_kernel<<<grid, 256, smem, st>>>(ga, Cin, D, H, W, gx);
    VADC_CHECK_LAUNCH("unpatchify_kernel");
  }
  // g_W [Cout, K4] = g_pre^T A: both operands given as [tokens, .] (MN-major), split over the tokens
  if ((rc = launch_patchify(x, B, Cin, D, H, W, as, st))) return rc;
  if ((rc = tc_gemm<3, true, true>({gps, as, Cout, K4, NT, nullptr, sk}, TcPartialEpi{part, K4, (long long)Cout * K4}, st))) return rc;
  {
    const long long n = (long long)Cout * K4;
    tail_sum_partials_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(part, sk, n, gweight);
    VADC_CHECK_LAUNCH("tail_sum_partials_kernel");
  }
  return VADC_OK;
}
