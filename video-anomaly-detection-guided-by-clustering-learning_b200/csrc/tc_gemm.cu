// tc_gemm.cu — fp32-faithful GEMM on tcgen05 / TMEM fed by TMA, for the contractions of the path
// that are NOT covered by the fused K == 32 kernels and are tensor-bound (SURVEY 8(d)): the
// distance / x_rec GEMMs of the cluster head at C = 768 or K >= 64 (BASELINE configs[2], the
// reference-native K = 1024 head) and the memory score / read GEMMs (m = 2000, d = 768: 244 flop/B).
//
//   C[m,n] = sum_k A[m,k] B(n,k)      A [M,Kd] row-major;  B [N,Kd] row-major (K-major) or [Kd,N] row-major (MN-major)
//
// fp32 inputs are first split into THREE bf16 terms v = t0 + t1 + t2 (exact: 3 x 8 mantissa bits; tc_terms.cuh),
// written once as bf16 matrices of the same layout (6 bytes per element of workspace);
// the GEMM keeps the six products t0t0, t0t1, t1t0, t0t2, t1t1, t2t0 in the fp32 TMEM accumulator
// (dropped terms <= 2^-24 relative), which is what keeps argmin bit-exact against the fp32 reference.
//
// One kernel for every launch, plain, batched and split-K: tc_gemm_persist_kernel on min(work items, SMs) CTAs, one per
// SM, each walking 128 x BN output tiles.  Warp 0 = TMA producer (3-D tensor maps {cols, rows, term}, SWIZZLE_128B boxes
// land directly as UMMA operand tiles), warp 1 = MMA issuer, warps 2-9 = epilogue (thread = output row = TMEM lane,
// functor per 32 columns).
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <algorithm>
#include <stdio.h>
#include "common.cuh"
#include "tc_common.cuh"
#include "tc_gemm.cuh"

namespace vadc {
using namespace tc;

namespace tg {

constexpr int BM = 128, BK = 64;
constexpr int kThreads = 320;            // warp 0 TMA, warp 1 MMA, warps 2-9 epilogue

// fp32 [n4 * 4] -> its TERMS term planes (tc_terms.cuh); fp16 x2: of src * scale[0].  ld > cols: src is [rows, cols]
// (any cols, any alignment), the terms [rows, ld] (n4 = rows ld / 4) with zeros in columns cols..ld-1
template <int TERMS>
__global__ void __launch_bounds__(256)
split_kernel(const float* __restrict__ src, long long n4, const float* __restrict__ scale, void* __restrict__ dst,
             long long cols, long long ld) {
  const float s = TERMS == 2 ? __ldg(scale) : 1.0f;
  if (ld == cols) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
      const float4 v = reinterpret_cast<const float4*>(src)[i];
      const float a[4] = {v.x * s, v.y * s, v.z * s, v.w * s};
      store_terms<TERMS, 4>(dst, 4 * n4, 4 * i, a);
    }
    return;
  }
  const long long q = ld / 4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / q, c = 4 * (i - r * q);
    const float* p = src + r * cols + c;
    float a[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) a[j] = c + j < cols ? __ldg(p + j) * s : 0.f;
    store_terms<TERMS, 4>(dst, 4 * n4, 4 * i, a);
  }
}

// split_kernel for row groups (tc_split's group < gpitch): term row g gpitch + k [.., ld] holds source row g group + k
// [.., cols] for k < group; the other rows and columns cols..ld-1 are zeros (a kernel of its own, so that the ungrouped
// splits keep their instruction stream)
template <int TERMS>
__global__ void __launch_bounds__(256)
split_groups_kernel(const float* __restrict__ src, long long n4, const float* __restrict__ scale, void* __restrict__ dst,
                    long long cols, long long ld, long long group, long long gpitch) {
  const float s = TERMS == 2 ? __ldg(scale) : 1.0f;
  const long long q = ld / 4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / q, c = 4 * (i - r * q), g = r / gpitch, k = r - g * gpitch;
    const float* p = src + (g * group + k) * cols + c;
    float a[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) a[j] = k < group && c + j < cols ? __ldg(p + j) * s : 0.f;
    store_terms<TERMS, 4>(dst, 4 * n4, 4 * i, a);
  }
}

__device__ __forceinline__ void tma_load_3d(const void* tmap, uint32_t smem_dst, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
               ::"r"(smem_dst), "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}

// One CTA per SM walks the work items (output tiles, the nz slices along z slowest).  Within a slice the dimension with
// FEWER tiles varies fastest (m_fast = the m-tiles): the CTAs in flight then share the small operand and stream the big
// one from DRAM once (with 16 m-tiles x 512 n-tiles the other order re-read the n-side operand 16 times).  The operand
// ring (STAGES stages) runs across tile boundaries, the accumulator is double-buffered in TMEM (2 x BN columns), and EIGHT
// epilogue warps (two per TMEM lane quarter, splitting the columns) drain tile i while the MMA warp is already in tile
// i+1: load, MMA and epilogue are three concurrent streams.  A CTA with a single tile still overlaps its loads with the
// MMAs of the k-loop.
//
// TERMS = 3: three bf16 terms per operand, six products (fp32-faithful for any fp32 data).
// TERMS = 2: two fp16 terms of operands pre-scaled by a power of two into fp16's range (bounded data: LayerNorm
// output, centroids, softmax weights), three products hh + hl + lh (22 significant bits) — two thirds of the operand
// bytes, half the MMAs, and a 64 KB stage; the accumulators are multiplied by *acc_scale (= 1 / (s_a s_b)) before the
// epilogue sees them.
__device__ __forceinline__ void mbar_arrive1(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

template <int BN, int TERMS, int STAGES, bool A_MN, bool B_MN, class Epi>
__global__ void __launch_bounds__(kThreads, 1)
tc_gemm_persist_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                       int M, int N, int Kd, int mt, int nt, int nz, int m_fast, int kb_per_split, const TcBatchOffsets zo,
                       const float* __restrict__ acc_scale, Epi epi) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr uint32_t kATerm = BM * 128u, kBTerm = BN * 128u;
  constexpr uint32_t kStage = (uint32_t)TERMS * (kATerm + kBTerm);
  __shared__ uint64_t full[STAGES], empty[STAGES], accfull[2], accempty[2];
  __shared__ uint32_t tmem_slot;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nkb = (Kd + BK - 1) / BK;
  // nz (z slowest) = independent problems of a batched launch, or — kb_per_split > 0 — split-K slots of one problem: slot z
  // contracts k-blocks [z kb_per_split, ...) and hands z to the epilogue (partial outputs; an empty slot writes zeros)
  const long long per_z = (long long)mt * nt, ntiles = per_z * nz;
  auto k_range = [&](int z, int& kb0, int& kcnt) {
    kb0 = kb_per_split > 0 ? z * kb_per_split : 0;
    kcnt = kb_per_split > 0 ? max(0, min(nkb - kb0, kb_per_split)) : nkb;
  };
  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&accfull[b], 1); mbar_init(&accempty[b], 8); }
    fence_mbar_init();
    prefetch_tmap(&mapA); prefetch_tmap(&mapB);
  }
  if (warp == 1) tmem_alloc(&tmem_slot, 2 * BN);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_slot;
  const uint32_t s0 = smem_u32(smem);
  auto tile_mn = [&](long long t, int& m0, int& n0, int& z) {
    z = (int)(t / per_z);
    const long long r = t - (long long)z * per_z;
    const int a = (int)(r % (m_fast ? mt : nt)), b = (int)(r / (m_fast ? mt : nt));
    m0 = (m_fast ? a : b) * BM; n0 = (m_fast ? b : a) * BN;
  };

  if (warp == 0 && lane == 0) {
    // ---------------------------------------------------------------- TMA producer
    uint32_t it = 0;
    for (long long t = blockIdx.x; t < ntiles; t += gridDim.x) {
      int m0, n0, z;
      tile_mn(t, m0, n0, z);
      const int am = m0 + z * zo.a_m, ak = z * zo.a_k, bn = n0 + z * zo.b_n, bk = z * zo.b_k;
      int kb0, kcnt;
      k_range(z, kb0, kcnt);
      for (int kb = 0; kb < kcnt; ++kb, ++it) {
        const uint32_t s = it % STAGES;
        mbar_wait(&empty[s], ((it / STAGES) & 1) ^ 1);
        mbar_expect_tx(&full[s], kStage);
        const uint32_t a = s0 + s * kStage, b = a + (uint32_t)TERMS * kATerm;
        const int k0 = (kb0 + kb) * BK;
#pragma unroll
        for (int tt = 0; tt < TERMS; ++tt) {
          if constexpr (!A_MN) {
            tma_load_3d(&mapA, a + tt * kATerm, &full[s], k0 + ak, am, tt);
          } else {
#pragma unroll
            for (int mb = 0; mb < BM / 64; ++mb) tma_load_3d(&mapA, a + tt * kATerm + mb * 8192u, &full[s], am + mb * 64, k0 + ak, tt);
          }
          if constexpr (!B_MN) {
            tma_load_3d(&mapB, b + tt * kBTerm, &full[s], k0 + bk, bn, tt);
          } else {
#pragma unroll
            for (int nb = 0; nb < BN / 64; ++nb) tma_load_3d(&mapB, b + tt * kBTerm + nb * 8192u, &full[s], bn + nb * 64, k0 + bk, tt);
          }
        }
      }
    }
  } else if (warp == 1 && lane == 0) {
    // ---------------------------------------------------------------- MMA issuer
    const uint32_t idesc = instr_desc(TERMS == 2 ? 0u /* fp16 */ : kFmtBF16, BM, BN, A_MN ? 1 : 0, B_MN ? 1 : 0);
    constexpr int kProducts = TERMS == 2 ? 3 : 6;
    constexpr int ta[6] = {TERMS == 2 ? 1 : 2, TERMS == 2 ? 0 : 1, 0, 1, 0, 0};   // small products first
    constexpr int tb[6] = {0, 1, TERMS == 2 ? 0 : 2, 0, 1, 0};
    uint32_t it = 0, lt = 0;
    for (long long t = blockIdx.x; t < ntiles; t += gridDim.x, ++lt) {
      const uint32_t buf = lt & 1;
      mbar_wait(&accempty[buf], ((lt >> 1) & 1) ^ 1);           // the epilogue has drained this accumulator
      tc_fence_after();
      const uint32_t acc = tmem + buf * BN;
      int kb0, kcnt;
      k_range((int)(t / per_z), kb0, kcnt);
      if (kcnt == 0) { mbar_arrive1(&accfull[buf]); continue; }  // empty split-K slot: nothing to contract
      for (int kb = 0; kb < kcnt; ++kb, ++it) {
        const uint32_t s = it % STAGES;
        mbar_wait(&full[s], (it / STAGES) & 1);
        tc_fence_after();
        const uint32_t a = s0 + s * kStage, b = a + (uint32_t)TERMS * kATerm;
#pragma unroll
        for (int pr = 0; pr < kProducts; ++pr) {
#pragma unroll
          for (int kk = 0; kk < BK / 16; ++kk) {
            const uint64_t ad = A_MN ? smem_desc_sw128(a + ta[pr] * kATerm + kk * 2048u, 8192, 1024)
                                     : smem_desc_sw128(a + ta[pr] * kATerm + kk * 32u, 0, 1024);
            const uint64_t bd = B_MN ? smem_desc_sw128(b + tb[pr] * kBTerm + kk * 2048u, 8192, 1024)
                                     : smem_desc_sw128(b + tb[pr] * kBTerm + kk * 32u, 0, 1024);
            mma_f16(acc, ad, bd, idesc, (kb > 0 || pr > 0 || kk > 0) ? 1u : 0u);
          }
        }
        mma_commit(&empty[s]);
      }
      mma_commit(&accfull[buf]);
    }
  } else if (warp >= 2) {
    // ---------------------------------------------------------------- epilogue: thread = row = TMEM lane, two warps per quarter
    const int q = warp & 3, hh = (warp - 2) >> 2;
    const float sc = acc_scale ? __ldg(acc_scale) : 1.0f;
    uint32_t lt = 0;
    for (long long t = blockIdx.x; t < ntiles; t += gridDim.x, ++lt) {
      int m0, n0, z;
      tile_mn(t, m0, n0, z);
      const uint32_t buf = lt & 1;
      mbar_wait(&accfull[buf], (lt >> 1) & 1);
      tc_fence_after();
      const long long m = (long long)m0 + q * 32 + lane;
      int kb0, kcnt;
      k_range(z, kb0, kcnt);
#pragma unroll 1
      for (int c = 0; c < BN / 64; ++c) {
        float v[32];
        const int col = hh * (BN / 2) + c * 32;
        if (kcnt > 0) {
          tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + buf * BN + (uint32_t)col, v);
          if (TERMS == 2) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] *= sc;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = 0.f;
        }
        const int n = n0 + col;
        if (m < M && n < N) epi(m, n, v, min(32, N - n), z);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive1(&accempty[buf]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) { tc_fence_after(); tmem_dealloc(tmem, 2 * BN); }
}

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

// three bf16 term matrices [rows, cols] stored back to back -> 3-D map {cols, rows, 3}, box {64, box_rows, 1}
static int make_map3(CUtensorMap* m, const void* base, long long rows, long long cols, int box_rows, int terms = 3) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return VADC_ERR_CUDA;
  cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)terms};
  cuuint64_t strides[2] = {(cuuint64_t)cols * 2, (cuuint64_t)rows * (cuuint64_t)cols * 2};
  cuuint32_t box[3] = {64, (cuuint32_t)box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(m, terms == 2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    snprintf(g_last_cuda_error, sizeof(g_last_cuda_error), "cuTensorMapEncodeTiled(3d) failed: %d", (int)r);
    return VADC_ERR_CUDA;
  }
  return VADC_OK;
}

}  // namespace tg

bool tc_gemm_shape_ok(long long M, long long N, long long Kd, bool b_mn) {
  if (M < 1 || N < 8 || Kd < 8 || M >= (1ll << 31) || N >= (1ll << 31) || Kd >= (1ll << 31)) return false;
  if (Kd % 8) return false;                 // TMA row pitch (bf16) must be a multiple of 16 bytes
  if (b_mn && (N % 8)) return false;
  return vadc_device_ok() != 0;
}

size_t tc_terms_bytes(int terms, long long rows, long long cols) {
  return align_up((size_t)terms * rows * cols * sizeof(uint16_t), 256);
}

template <int TERMS>
int tc_split(const float* src, long long rows, long long cols, const float* scale, void* dst, cudaStream_t st,
             long long ld, long long group, long long gpitch) {
  static_assert(TERMS == 2 || TERMS == 3, "operand terms: fp16 x2 or bf16 x3");
  if (ld == 0) ld = cols;
  if (ld < cols || (ld != cols && ld % 8)) return VADC_ERR_BAD_SHAPE;
  if (group == 0 && gpitch == 0) group = gpitch = 1;
  if (group < 1 || gpitch < group || rows % group) return VADC_ERR_BAD_SHAPE;
  if (gpitch != group && ld % 4) return VADC_ERR_BAD_SHAPE;
  const long long n = rows / group * gpitch * ld;
  if (n % 4) return VADC_ERR_BAD_SHAPE;
  if (TERMS == 2 && !scale) return VADC_ERR_NULL_POINTER;
  const long long n4 = n / 4;
  const int grid = (int)std::min<long long>((n4 + 255) / 256, (long long)sm_count() * 8);
  if (gpitch == group) {
    tg::split_kernel<TERMS><<<grid, 256, 0, st>>>(src, n4, scale, dst, cols, ld);
    VADC_CHECK_LAUNCH("split_kernel");
  } else {
    tg::split_groups_kernel<TERMS><<<grid, 256, 0, st>>>(src, n4, scale, dst, cols, ld, group, gpitch);
    VADC_CHECK_LAUNCH("split_groups_kernel");
  }
  return VADC_OK;
}
template int tc_split<2>(const float*, long long, long long, const float*, void*, cudaStream_t, long long, long long, long long);
template int tc_split<3>(const float*, long long, long long, const float*, void*, cudaStream_t, long long, long long, long long);

// nz work slices along z of an [M, N] output on min(work items, SMs) persistent CTAs with three 64 KB (fp16 x2) or two
// 96 KB (bf16 x3) operand stages.  Split matrices MN-major: [Kd rows, M / N cols], boxes of 64 k-rows x 64 cols; K-major:
// [M / N rows, Kd cols], boxes of 128 rows x 64 k-cols.  Split-K: kb_per_split k-blocks per slot; batched: 0.
template <int TERMS, bool A_MN, bool B_MN, class Epi>
int tc_gemm(const TcGemm& g, Epi epi, cudaStream_t st) {
  constexpr int BN = 128, kStages = TERMS == 2 ? 3 : 2;
  if (TERMS == 2 && !g.acc_scale) return VADC_ERR_NULL_POINTER;
  if (g.nbatch < 1 || g.nbatch > 65535) return VADC_ERR_UNSUPPORTED;
  const int splits = g.splits < 1 ? 1 : g.splits;
  if (splits > 1 && g.nbatch > 1) return VADC_ERR_UNSUPPORTED;
  const long long M = g.M, N = g.N, Kd = g.Kd;
  const int nkb = (int)((Kd + tg::BK - 1) / tg::BK);
  const int kb_per_split = splits > 1 ? (nkb + splits - 1) / splits : 0;
  const int nz = splits > 1 ? splits : g.nbatch;
  const long long a_rows = g.a_rows ? g.a_rows : (A_MN ? Kd : M), a_cols = g.a_cols ? g.a_cols : (A_MN ? M : Kd);
  const long long b_rows = g.b_rows ? g.b_rows : (B_MN ? Kd : N), b_cols = g.b_cols ? g.b_cols : (B_MN ? N : Kd);
  CUtensorMap mA, mB;
  int rc;
  if ((rc = tg::make_map3(&mA, g.a, a_rows, a_cols, A_MN ? 64 : tg::BM, TERMS))) return rc;
  if ((rc = tg::make_map3(&mB, g.b, b_rows, b_cols, B_MN ? 64 : BN, TERMS))) return rc;
  const int mt = (int)((M + tg::BM - 1) / tg::BM), nt = (int)((N + BN - 1) / BN);
  const int grid = (int)std::min<long long>((long long)mt * nt * nz, sm_count());
  const size_t smem = (size_t)kStages * TERMS * (tg::BM * 128 + BN * 128) + 1024;
  auto kern = tg::tc_gemm_persist_kernel<BN, TERMS, kStages, A_MN, B_MN, Epi>;
  VADC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<grid, tg::kThreads, smem, st>>>(mA, mB, (int)M, (int)N, (int)Kd, mt, nt, nz, mt < nt ? 1 : 0, kb_per_split, g.off,
                                         g.acc_scale, epi);
  VADC_CHECK_LAUNCH("tc_gemm_persist_kernel");
  return VADC_OK;
}

// one line per (terms, operand layouts, epilogue) the library launches
#define VADC_TC_GEMM(TERMS, A_MN, B_MN, EPI) template int tc_gemm<TERMS, A_MN, B_MN, EPI>(const TcGemm&, EPI, cudaStream_t);
VADC_TC_GEMM(2, false, false, TcDistEpi)
VADC_TC_GEMM(2, false, true, TcStoreEpi)
VADC_TC_GEMM(2, false, false, TcStoreEpi)
VADC_TC_GEMM(2, false, true, TcReadEpi)
VADC_TC_GEMM(2, false, false, TcLogitsColStatsTEpi)
VADC_TC_GEMM(2, false, false, TcStoreTEpi)
VADC_TC_GEMM(2, false, false, TcDistTEpi)
VADC_TC_GEMM(2, false, true, TcGzEpi)
VADC_TC_GEMM(2, true, false, TcStoreTEpi)
VADC_TC_GEMM(2, true, false, TcReadTEpi)
VADC_TC_GEMM(2, true, false, TcGzTEpi)
VADC_TC_GEMM(2, true, false, TcPartialEpi)
VADC_TC_GEMM(2, true, true, TcPartialEpi)
VADC_TC_GEMM(2, false, true, ScoresQhatEpi)
VADC_TC_GEMM(2, true, false, ScoresQRowsTEpi)
VADC_TC_GEMM(2, false, false, TcBatchDistEpi)
VADC_TC_GEMM(2, true, false, TcSpaceGzEpi)
VADC_TC_GEMM(2, true, true, TcSpaceGcEpi)
VADC_TC_GEMM(2, true, false, TcCdistGaTEpi)
VADC_TC_GEMM(3, false, false, TcStoreEpi)
VADC_TC_GEMM(3, false, true, TcStoreEpi)
VADC_TC_GEMM(3, false, false, TcDistEpi)
VADC_TC_GEMM(3, false, true, TcReadEpi)
VADC_TC_GEMM(3, false, true, TcGzEpi)
VADC_TC_GEMM(3, false, false, TcTimeDebedEpi)
VADC_TC_GEMM(3, false, true, TcTimeDebedEpi)
VADC_TC_GEMM(3, true, false, TcPartialEpi)
VADC_TC_GEMM(3, true, true, TcPartialEpi)
VADC_TC_GEMM(3, false, true, ScoresQhatEpi)
VADC_TC_GEMM(3, true, false, ScoresQRowsTEpi)
VADC_TC_GEMM(3, true, false, TcStoreTEpi)
VADC_TC_GEMM(3, false, false, TcBiasEpi)
VADC_TC_GEMM(3, false, false, TcBiasTEpi)
VADC_TC_GEMM(3, false, false, TcBiasGeluTEpi)
VADC_TC_GEMM(3, false, false, TcBatchDistEpi)
VADC_TC_GEMM(3, true, false, TcSpaceGzEpi)
VADC_TC_GEMM(3, true, true, TcSpaceGcEpi)
VADC_TC_GEMM(3, true, false, TcCdistGaTEpi)
#undef VADC_TC_GEMM

// ---- two-term fp16 mode -------------------------------------------------------------------------
namespace tg {
__device__ __forceinline__ float pow2_scale(float bound) {   // power of two s with s * bound in [4, 8); 1 for 0 / non-finite
  if (!(bound > 0.f) || !isfinite(bound)) return 1.0f;
  int e;
  (void)frexpf(bound, &e);
  e = max(-96, min(96, e));
  return ldexpf(1.0f, 3 - e);
}

// scales of the cluster forward (one block): s_z from the LayerNorm bound sqrt(C) max|gamma| + max|beta|, s_c from
// max|centers|, s_a = 2^13 for the softmin weights in [0, 1]
//   out[0] = s_z, [1] = s_c, [2] = 1 / (s_z s_c), [3] = s_a, [4] = 1 / (s_a s_c), [5] = 1 / (s_c s_c)
__global__ void __launch_bounds__(1024)
fwd_scales_kernel(const float* __restrict__ centers, const float* __restrict__ ln_w, const float* __restrict__ ln_b,
                  long long KC, int C, float* __restrict__ out) {
  __shared__ float red[3][32];
  float mc = 0.f, mg = 0.f, mb = 0.f;
  if ((KC & 3) == 0 && (reinterpret_cast<uintptr_t>(centers) & 15u) == 0) {
    float m4[4] = {0.f, 0.f, 0.f, 0.f};                      // four independent chains, 16-byte loads
    for (long long i = threadIdx.x; i < KC / 4; i += blockDim.x) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(centers) + i);
      m4[0] = fmaxf(m4[0], fabsf(v.x)); m4[1] = fmaxf(m4[1], fabsf(v.y));
      m4[2] = fmaxf(m4[2], fabsf(v.z)); m4[3] = fmaxf(m4[3], fabsf(v.w));
    }
    mc = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
  } else {
    for (long long i = threadIdx.x; i < KC; i += blockDim.x) mc = fmaxf(mc, fabsf(centers[i]));
  }
  for (int i = threadIdx.x; i < C; i += blockDim.x) { mg = fmaxf(mg, fabsf(ln_w[i])); mb = fmaxf(mb, fabsf(ln_b[i])); }
  mc = warp_max(mc); mg = warp_max(mg); mb = warp_max(mb);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) { red[0][w] = mc; red[1][w] = mg; red[2][w] = mb; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < 32; ++i) { mc = fmaxf(mc, red[0][i]); mg = fmaxf(mg, red[1][i]); mb = fmaxf(mb, red[2][i]); }
    mc = fmaxf(mc, red[0][0]); mg = fmaxf(mg, red[1][0]); mb = fmaxf(mb, red[2][0]);
    const float s_z = pow2_scale(sqrtf((float)C) * mg + mb), s_c = pow2_scale(mc), s_a = 8192.0f;
    out[0] = s_z; out[1] = s_c; out[2] = 1.0f / (s_z * s_c); out[3] = s_a; out[4] = 1.0f / (s_a * s_c);
    out[5] = 1.0f / (s_c * s_c);                             // centroid self-distance
  }
}

}  // namespace tg

int tc_fwd_scales(const float* centers, const float* ln_w, const float* ln_b, long long KC, int C, float* out,
                  cudaStream_t st) {
  tg::fwd_scales_kernel<<<1, 1024, 0, st>>>(centers, ln_w, ln_b, KC, C, out);
  VADC_CHECK_LAUNCH("fwd_scales_kernel");
  return VADC_OK;
}

namespace tg {
// max |src| as the bit pattern of a non-negative float (ordered like unsigned integers): deterministic atomicMax;
// blockIdx.y walks segments of n elements `stride` apart
__global__ void __launch_bounds__(256)
absmax_bits_kernel(const float* __restrict__ src, long long n, long long stride, unsigned* __restrict__ out) {
  src += (long long)blockIdx.y * stride;
  float m = 0.f;
  const long long n4 = ((reinterpret_cast<uintptr_t>(src) & 15u) == 0) ? n / 4 : 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(src) + i);
    m = fmaxf(fmaxf(m, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
  }
  for (long long i = 4 * n4 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    m = fmaxf(m, fabsf(src[i]));
  m = warp_max(m);
  if ((threadIdx.x & 31) == 0 && m > 0.f && isfinite(m)) atomicMax(out, __float_as_uint(m));
}

// out[0] = s_a, out[1] = s_b, out[2] = 1 / (s_a s_b); a scale comes from a measured bound (bits) or is given
__global__ void pair_scales_kernel(const unsigned* a_bits, float a_given, const unsigned* b_bits, float b_given, float* out) {
  const float sa = a_bits ? pow2_scale(__uint_as_float(*a_bits)) : a_given;
  const float sb = b_bits ? pow2_scale(__uint_as_float(*b_bits)) : b_given;
  out[0] = sa; out[1] = sb; out[2] = 1.0f / (sa * sb);
}
}  // namespace tg

// space head backward: r scaled from its measured bound, against the forward's s_z, s_c (fwd_sc = tc_fwd_scales output)
//   out[0] = s_r, [1] = 1 / (s_c s_r), [2] = 1 / (s_r s_z)
namespace tg {
__global__ void space_bwd_scales_kernel(const unsigned* r_bits, const float* fwd_sc, float* out) {
  const float sr = pow2_scale(__uint_as_float(*r_bits));
  out[0] = sr; out[1] = 1.0f / (fwd_sc[1] * sr); out[2] = 1.0f / (sr * fwd_sc[0]);
}
}  // namespace tg
int tc_space_bwd_scales(const unsigned* r_bits, const float* fwd_sc, float* out3, cudaStream_t st) {
  tg::space_bwd_scales_kernel<<<1, 1, 0, st>>>(r_bits, fwd_sc, out3);
  VADC_CHECK_LAUNCH("space_bwd_scales_kernel");
  return VADC_OK;
}

// the forward scales (layout of fwd_scales_kernel) from an already measured max |centers| (tc_absmax_bits: every SM
// takes part — the one-block scan of fwd_scales_kernel is for the cluster head's small [K, C] centroid matrix)
namespace tg {
__global__ void __launch_bounds__(256)
fwd_scales_from_bits_kernel(const unsigned* cen_bits, const float* __restrict__ ln_w, const float* __restrict__ ln_b, int C,
                            float* __restrict__ out) {
  __shared__ float red[2][8];
  float mg = 0.f, mb = 0.f;
  for (int i = threadIdx.x; i < C; i += blockDim.x) { mg = fmaxf(mg, fabsf(ln_w[i])); mb = fmaxf(mb, fabsf(ln_b[i])); }
  mg = warp_max(mg); mb = warp_max(mb);
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = mg; red[1][threadIdx.x >> 5] = mb; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 0; i < 8; ++i) { mg = fmaxf(mg, red[0][i]); mb = fmaxf(mb, red[1][i]); }
    const float s_z = pow2_scale(sqrtf((float)C) * mg + mb), s_c = pow2_scale(__uint_as_float(*cen_bits)), s_a = 8192.0f;
    out[0] = s_z; out[1] = s_c; out[2] = 1.0f / (s_z * s_c); out[3] = s_a; out[4] = 1.0f / (s_a * s_c);
    out[5] = 1.0f / (s_c * s_c);
  }
}
}  // namespace tg
int tc_fwd_scales_from_bits(const unsigned* cen_bits, const float* ln_w, const float* ln_b, int C, float* out, cudaStream_t st) {
  tg::fwd_scales_from_bits_kernel<<<1, 256, 0, st>>>(cen_bits, ln_w, ln_b, C, out);
  VADC_CHECK_LAUNCH("fwd_scales_from_bits_kernel");
  return VADC_OK;
}

// generic cluster backward in fp16 x2: scales of gR, centers, feature (measured), A (2^13) and — once bwd_rows has run — r
//   out[0] = s_g, [1] = s_c, [2] = s_f, [3] = s_a, [4] = s_r, [5] = 1/(s_g s_c), [6] = 1/(s_a s_g), [7] = 1/(s_r s_c), [8] = 1/(s_r s_f)
// bits[0..3] = max |gR|, |centers|, |feature|, |r|; stage 0 fills everything that does not need r, stage 1 the rest
namespace tg {
__global__ void cluster_bwd_scales_kernel(const unsigned* bits, int stage, float* out) {
  if (stage == 0) {
    const float sg = pow2_scale(__uint_as_float(bits[0])), sc = pow2_scale(__uint_as_float(bits[1]));
    const float sf = pow2_scale(__uint_as_float(bits[2])), sa = 8192.0f;
    out[0] = sg; out[1] = sc; out[2] = sf; out[3] = sa; out[5] = 1.0f / (sg * sc); out[6] = 1.0f / (sa * sg);
  } else {
    const float sr = pow2_scale(__uint_as_float(bits[3]));
    out[4] = sr; out[7] = 1.0f / (sr * out[1]); out[8] = 1.0f / (sr * out[2]);
  }
}
}  // namespace tg
int tc_cluster_bwd_scales(const unsigned* bits, int stage, float* out, cudaStream_t st) {
  tg::cluster_bwd_scales_kernel<<<1, 1, 0, st>>>(bits, stage, out);
  VADC_CHECK_LAUNCH("cluster_bwd_scales_kernel");
  return VADC_OK;
}

int tc_absmax_bits_seg(const float* src, long long n, int nseg, long long stride, unsigned* out, cudaStream_t st) {
  if (nseg < 1 || nseg > 65535) return VADC_ERR_UNSUPPORTED;
  VADC_CUDA(cudaMemsetAsync(out, 0, sizeof(unsigned), st));
  const long long per = std::max<long long>(1, (long long)sm_count() * 8 / nseg);
  const int grid = (int)std::max<long long>(1, std::min<long long>((n / 4 + 255) / 256, per));
  tg::absmax_bits_kernel<<<dim3(grid, nseg), 256, 0, st>>>(src, n, stride, out);
  VADC_CHECK_LAUNCH("absmax_bits_kernel");
  return VADC_OK;
}

int tc_absmax_bits(const float* src, long long n, unsigned* out, cudaStream_t st) {
  return tc_absmax_bits_seg(src, n, 1, 0, out, st);
}

int tc_pair_scales(const unsigned* a_bits, float a_given, const unsigned* b_bits, float b_given, float* out3, cudaStream_t st) {
  tg::pair_scales_kernel<<<1, 1, 0, st>>>(a_bits, a_given, b_bits, b_given, out3);
  VADC_CHECK_LAUNCH("pair_scales_kernel");
  return VADC_OK;
}

}  // namespace vadc

// ---------------------------------------------------------------------------
// self-test entry: out[M,N] = A[M,Kd] . B^T  (b_mn = 0: B is [N,Kd]; b_mn = 1: B is [Kd,N])
// ---------------------------------------------------------------------------
extern "C" size_t vadc_debug_tc_gemm_workspace_bytes(int64_t M, int64_t N, int64_t Kd) {
  return vadc::tc_terms_bytes(3, M, Kd) + vadc::tc_terms_bytes(3, N, Kd) + 256;
}

extern "C" int vadc_debug_tc_gemm(const float* A, const float* B, int64_t M, int64_t N, int64_t Kd, int b_mn,
                                  float* out, void* workspace, size_t workspace_bytes, void* stream) {
  using namespace vadc;
  VADC_REQUIRE(A && B && out && workspace, VADC_ERR_NULL_POINTER);
  VADC_REQUIRE(tc_gemm_shape_ok(M, N, Kd, b_mn != 0), VADC_ERR_UNSUPPORTED);
  VADC_REQUIRE(workspace_bytes >= vadc_debug_tc_gemm_workspace_bytes(M, N, Kd), VADC_ERR_WORKSPACE);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Carver ws(workspace, workspace_bytes);
  void* as = ws.take<uint8_t>(tc_terms_bytes(3, M, Kd));
  void* bs = ws.take<uint8_t>(tc_terms_bytes(3, N, Kd));
  int rc;
  if ((rc = tc_split<3>(A, M, Kd, nullptr, as, st))) return rc;
  if ((rc = b_mn ? tc_split<3>(B, Kd, N, nullptr, bs, st) : tc_split<3>(B, N, Kd, nullptr, bs, st))) return rc;
  const TcGemm g{as, bs, M, N, Kd};
  TcStoreEpi epi{out, N};
  return b_mn ? tc_gemm<3, false, true>(g, epi, st) : tc_gemm<3, false, false>(g, epi, st);
}
