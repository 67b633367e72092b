// tc_terms.cuh — the operand-term format of tc_gemm (tc_gemm.cuh): an fp32 operand becomes TERMS 16-bit matrices of its
// shape, stored one after another ("planes", `plane` elements apart), whose sum is the operand.
//   TERMS = 3 (bf16 x3): t0 = rn(a), t1 = rn(a - t0), t2 = rn(a - t0 - t1); exact for any fp32 a (3 x 8 mantissa bits)
//   TERMS = 2 (fp16 x2): h0 = rn(a), h1 = rn(a - h0) of an operand pre-scaled by a power of two into fp16's range
//                        (22 significant bits); the caller multiplies by the scale before the split
// Every kernel that writes operand terms, stand-alone or fused into a row pass, splits through these helpers.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

namespace vadc {

template <int TERMS> struct TcTerm;
template <> struct TcTerm<2> { using T = __half; };
template <> struct TcTerm<3> { using T = __nv_bfloat16; };

__device__ __forceinline__ void split_f16x2(float a, __half (&h)[2]) {
  h[0] = __float2half_rn(a);
  h[1] = __float2half_rn(a - __half2float(h[0]));
}

__device__ __forceinline__ void split_bf16x3(float a, __nv_bfloat16 (&b)[3]) {
  b[0] = __float2bfloat16_rn(a);
  const float r1 = a - __bfloat162float(b[0]);
  b[1] = __float2bfloat16_rn(r1);
  b[2] = __float2bfloat16_rn(r1 - __bfloat162float(b[1]));
}

template <int TERMS>
__device__ __forceinline__ void split_terms(float a, typename TcTerm<TERMS>::T (&t)[TERMS]) {
  if constexpr (TERMS == 2) split_f16x2(a, t);
  else split_bf16x3(a, t);
}

// the terms of W consecutive elements as one W-wide store per plane (W = 4: the 8-byte stores of the row kernels)
template <int W> struct TcPack;
template <> struct TcPack<1> { using T = uint16_t; };
template <> struct TcPack<2> { using T = uint32_t; };
template <> struct TcPack<4> { using T = uint2; };

template <int TERMS, int W>
__device__ __forceinline__ void split_terms(const float (&a)[W], typename TcTerm<TERMS>::T (&t)[TERMS][W]) {
#pragma unroll
  for (int j = 0; j < W; ++j) {
    typename TcTerm<TERMS>::T e[TERMS];
    split_terms<TERMS>(a[j], e);
#pragma unroll
    for (int k = 0; k < TERMS; ++k) t[k][j] = e[k];
  }
}

// terms of a[0..W) to elements i..i+W-1 of every plane of dst (i a multiple of W)
template <int TERMS, int W>
__device__ __forceinline__ void store_terms(void* dst, long long plane, long long i, const float (&a)[W]) {
  using E = typename TcTerm<TERMS>::T;
  using P = typename TcPack<W>::T;
  E t[TERMS][W];
  split_terms<TERMS, W>(a, t);
  E* o = static_cast<E*>(dst) + i;
#pragma unroll
  for (int k = 0; k < TERMS; ++k) {
    if constexpr (W == 1) o[k * plane] = t[k][0];
    else *reinterpret_cast<P*>(o + k * plane) = *reinterpret_cast<const P*>(t[k]);
  }
}

template <int TERMS>
__device__ __forceinline__ void store_terms(void* dst, long long plane, long long i, float a) {
  const float v[1] = {a};
  store_terms<TERMS, 1>(dst, plane, i, v);
}

}  // namespace vadc
