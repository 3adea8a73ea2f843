// K2 / K4 on the 5th-generation tensor cores: TMA-fed tcgen05.mma (kind::tf32) with TMEM accumulators,
// 3xTF32 split for fp32-class accuracy.
//
//   cov       : Ct (n x k)   = Xt (n x d) . W (d x k)          [dictionary @ X.T, sklearn/_dict_learning.py:426]
//   surrogate : P (k x (k+d)) = [ Ht^T Ht | Ht^T Xt ]           [np.dot(H1.T,H1), np.dot(H1.T,X.T), src/ontf.py:147-148]
//
// Precision: plain TF32 inputs cost 1.5e-3 per-atom dictionary error (SURVEY.md §0.9), so every fp32 operand is
// split once into hi = rna_tf32(x) and lo = x - hi (both exactly representable where the tensor core reads
// them) and each product is three MMAs, hi*hi + hi*lo + lo*hi, accumulated in fp32 in TMEM.
//
// Kernel shape: one CTA per (128 x BN output tile, K split).  Warp 0 = TMA producer (one elected lane),
// warp 1 = MMA issuer (one elected lane), warp 2 = TMEM allocator, warps 4-7 = epilogue (TMEM -> registers ->
// padded smem -> coalesced global stores).  A stage holds the hi and lo tiles of A (128 x 32) and B (BN x 32)
// in the 128-byte-swizzled canonical layouts; operands that are K-contiguous in global memory (Xt for cov) use
// the K-major form, operands that are MN-contiguous (W, Ht, Xt as right-hand sides of the transposed products)
// use the MN-major form directly -- no transposed copies are ever made.  The surrogate products reduce over
// the sample axis and are split-K across the grid with a fixed-order second-pass reduction (deterministic).
#include <cuda.h>

#include <algorithm>

#include "common.cuh"

namespace onmf {
namespace tc {

constexpr int BM = 128;
constexpr int BK = 32;                 // fp32 elements per K block = 128 bytes = one swizzle row
constexpr uint32_t CHUNK_BYTES = BK * 128;   // one 32-wide MN chunk of an MN-major tile: 32 k-rows x 128 B

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
  } while (!done);
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      :
      : "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor: start>>4 [0,14), LBO>>4 [16,30), SBO>>4 [32,46),
// version=1 [46,48), layout type [61,64))
//   K-major : SWIZZLE_128B (2): rows of 128 B (32 tf32 along K), 8-row atoms 1024 B apart (SBO); LBO unused (1)
//   MN-major: 32-bit operands only exist in the SWIZZLE_128B_BASE32B (1) form: 32 MN elements contiguous (128 B)
//             per k-row, 32-byte chunks XOR-swizzled with (k-row mod 4), 4-k-row atoms 512 B apart (SBO), next
//             32-wide MN chunk CHUNK_BYTES further (LBO).  TMA writes it with CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B.
template <bool MN>
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {
  const uint64_t lbo = MN ? (CHUNK_BYTES >> 4) : 1;
  const uint64_t sbo = MN ? (512 >> 4) : (1024 >> 4);
  const uint64_t lay = MN ? 1 : 2;
  return (uint64_t)((saddr >> 4) & 0x3FFF) | (lbo << 16) | (sbo << 32) | (1ull << 46) | (lay << 61);
}

template <int BN>
struct Cfg {
  static constexpr int STAGES = BN == 256 ? 2 : (BN == 128 ? 3 : 4);
  static constexpr uint32_t A_BYTES = BM * BK * 4;
  static constexpr uint32_t B_BYTES = BN * BK * 4;
  static constexpr uint32_t STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;
  static constexpr uint32_t SMEM_BYTES = STAGES * STAGE_BYTES + 1024;
  static constexpr int STG_LD = BN + 4;                      // padded row of the epilogue staging tile (floats)
  static_assert((size_t)BM * STG_LD * 4 <= (size_t)STAGES * STAGE_BYTES, "staging tile must fit in the pipeline buffers");
};

template <int BN, bool A_MN, bool B_MN>
__global__ void __launch_bounds__(256, 1)
gemm3_kernel(const __grid_constant__ CUtensorMap tmA_hi, const __grid_constant__ CUtensorMap tmA_lo,
             const __grid_constant__ CUtensorMap tmB_hi, const __grid_constant__ CUtensorMap tmB_lo,
             float* __restrict__ D, long long ldd, int M, int N, int kblocks, int kb_per_split, long long split_stride) {
  using C = Cfg<BN>;
  constexpr int STAGES = C::STAGES;
  extern __shared__ uint8_t smem_dyn[];
  __shared__ __align__(8) uint64_t full_bar[4];
  __shared__ __align__(8) uint64_t empty_bar[4];
  __shared__ __align__(8) uint64_t tmem_full_bar;
  __shared__ uint32_t tmem_slot;

  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~uintptr_t(1023));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
  const int kb0 = blockIdx.z * kb_per_split;
  int kb1 = kb0 + kb_per_split;
  if (kb1 > kblocks) kb1 = kblocks;
  const int nkb = kb1 - kb0;

  auto stage_ptr = [&](int s) -> uint8_t* { return smem + (size_t)s * C::STAGE_BYTES; };

  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
    mbar_init(smem_u32(&tmem_full_bar), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  } else if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"((uint32_t)BN)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      for (int i = 0; i < nkb; ++i) {
        const int s = i % STAGES;
        const uint32_t ph = (i / STAGES) & 1;
        mbar_wait(smem_u32(&empty_bar[s]), ph ^ 1);
        const uint32_t fb = smem_u32(&full_bar[s]);
        mbar_expect_tx(fb, C::STAGE_BYTES);
        const int kc = (kb0 + i) * BK;
        const uint32_t a_hi = smem_u32(stage_ptr(s));
        const uint32_t a_lo = a_hi + C::A_BYTES;
        const uint32_t b_hi = a_lo + C::A_BYTES;
        const uint32_t b_lo = b_hi + C::B_BYTES;
        if (A_MN) {
#pragma unroll
          for (int c = 0; c < BM / 32; ++c) {
            tma_load_2d(a_hi + c * CHUNK_BYTES, &tmA_hi, fb, m0 + 32 * c, kc);
            tma_load_2d(a_lo + c * CHUNK_BYTES, &tmA_lo, fb, m0 + 32 * c, kc);
          }
        } else {
          tma_load_2d(a_hi, &tmA_hi, fb, kc, m0);
          tma_load_2d(a_lo, &tmA_lo, fb, kc, m0);
        }
        if (B_MN) {
#pragma unroll
          for (int c = 0; c < BN / 32; ++c) {
            tma_load_2d(b_hi + c * CHUNK_BYTES, &tmB_hi, fb, n0 + 32 * c, kc);
            tma_load_2d(b_lo + c * CHUNK_BYTES, &tmB_lo, fb, n0 + 32 * c, kc);
          }
        } else {
          tma_load_2d(b_hi, &tmB_hi, fb, kc, n0);
          tma_load_2d(b_lo, &tmB_lo, fb, kc, n0);
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    if (lane == 0) {
      // instruction descriptor (cute::UMMA::InstrDescriptor): D=F32 [4,6), A=TF32 [7,10), B=TF32 [10,13),
      // A major [15], B major [16], N>>3 [17,23), M>>4 [24,29)
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((A_MN ? 1u : 0u) << 15) | ((B_MN ? 1u : 0u) << 16) |
                             ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
      for (int i = 0; i < nkb; ++i) {
        const int s = i % STAGES;
        const uint32_t ph = (i / STAGES) & 1;
        mbar_wait(smem_u32(&full_bar[s]), ph);
        tc_fence_after();
        const uint32_t a_hi = smem_u32(stage_ptr(s));
        const uint32_t a_lo = a_hi + C::A_BYTES;
        const uint32_t b_hi = a_lo + C::A_BYTES;
        const uint32_t b_lo = b_hi + C::B_BYTES;
#pragma unroll
        for (int ks = 0; ks < BK / 8; ++ks) {
          const uint32_t adv_a = A_MN ? ks * 1024 : ks * 32;
          const uint32_t adv_b = B_MN ? ks * 1024 : ks * 32;
          const uint64_t dah = make_desc<A_MN>(a_hi + adv_a), dal = make_desc<A_MN>(a_lo + adv_a);
          const uint64_t dbh = make_desc<B_MN>(b_hi + adv_b), dbl = make_desc<B_MN>(b_lo + adv_b);
          umma_tf32(tmem_base, dah, dbh, idesc, (i > 0 || ks > 0) ? 1u : 0u);
          umma_tf32(tmem_base, dah, dbl, idesc, 1u);
          umma_tf32(tmem_base, dal, dbh, idesc, 1u);
        }
        umma_commit(smem_u32(&empty_bar[s]));     // frees the stage when the MMAs above have read it
      }
      umma_commit(smem_u32(&tmem_full_bar));       // accumulator complete
    }
  } else if (warp >= 4) {
    // ===== epilogue: TMEM -> registers -> padded smem -> coalesced global =====
    const int ew = warp - 4;                        // == warp % 4: the TMEM lane quarter this warp may read
    float* stg = reinterpret_cast<float*>(smem);    // pipeline buffers are free once tmem_full has fired
    const int row = ew * 32 + lane;
    if (nkb > 0) {
      mbar_wait(smem_u32(&tmem_full_bar), 0);
      tc_fence_after();
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 32) {
        uint32_t v[32];
        const uint32_t taddr = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)c0;
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
            "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
            : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
              "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
              "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
              "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
            : "r"(taddr)
            : "memory");
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        float4* dst = reinterpret_cast<float4*>(stg + (size_t)row * C::STG_LD + c0);
#pragma unroll
        for (int j = 0; j < 8; ++j)
          dst[j] = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]),
                               __uint_as_float(v[4 * j + 3]));
      }
    } else {
      for (int c0 = 0; c0 < BN; c0 += 4)
        *reinterpret_cast<float4*>(stg + (size_t)row * C::STG_LD + c0) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    __syncwarp();
    // each warp stores the 32 rows it staged: one row per iteration, 128 floats per pass
    float* Dz = D + (size_t)blockIdx.z * split_stride;
    for (int r = 0; r < 32; ++r) {
      const int gr = m0 + ew * 32 + r;
      if (gr >= M) break;
      const float* src = stg + (size_t)(ew * 32 + r) * C::STG_LD;
#pragma unroll
      for (int c = lane * 4; c < BN; c += 128) {
        const int gc = n0 + c;
        if (gc + 3 < N) {
          *reinterpret_cast<float4*>(Dz + (size_t)gr * ldd + gc) = *reinterpret_cast<const float4*>(src + c);
        } else {
          for (int e = 0; e < 4; ++e)
            if (gc + e < N) Dz[(size_t)gr * ldd + gc + e] = src[c + e];
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)BN) : "memory");
  }
}

// hi = rna_tf32(x), lo = x - hi
__global__ void split_tf32_kernel(const float* __restrict__ src, float* __restrict__ hi, float* __restrict__ lo, long long count4) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < count4; i += stride) {
    float4 x = reinterpret_cast<const float4*>(src)[i];
    float4 h, l;
    uint32_t t;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(t) : "f"(x.x)); h.x = __uint_as_float(t); l.x = x.x - h.x;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(t) : "f"(x.y)); h.y = __uint_as_float(t); l.y = x.y - h.y;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(t) : "f"(x.z)); h.z = __uint_as_float(t); l.z = x.z - h.z;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(t) : "f"(x.w)); h.w = __uint_as_float(t); l.w = x.w - h.w;
    reinterpret_cast<float4*>(hi)[i] = h;
    reinterpret_cast<float4*>(lo)[i] = l;
  }
}

// out[r, c] (leading dim ldo) = sum_z part[z][r][c] in fixed order
__global__ void split_reduce2d_kernel(const float* __restrict__ part, int splits, int rows, int cols, float* __restrict__ out,
                                      long long ldo) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)rows * cols) return;
  const int r = (int)(i / cols), c = (int)(i - (long long)r * cols);
  float s = 0.f;
  const size_t stride = (size_t)rows * cols;
  for (int z = 0; z < splits; ++z) s += part[z * stride + i];
  out[(size_t)r * ldo + c] = s;
}

// ------------------------------------------------------------------------------------------------ host
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// row-major fp32 matrix [outer x inner] (leading dim ld elements); box = [box_outer x box_inner], 128B swizzle
static int make_map(CUtensorMap* m, const float* ptr, long long inner, long long outer, long long ld, int box_inner, int box_outer,
                    bool mn_major = false) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(ONMF_E_CUDA, "cuTensorMapEncodeTiled unavailable");
  cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
  cuuint32_t box[2] = {(cuuint32_t)box_inner, (cuuint32_t)box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, mn_major ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    snprintf(g_err, sizeof(g_err), "cuTensorMapEncodeTiled failed (%d): inner=%lld outer=%lld ld=%lld box=%dx%d", (int)r, inner,
             outer, ld, box_inner, box_outer);
    return ONMF_E_CUDA;
  }
  return ONMF_OK;
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

struct Operand {
  const float* hi;
  const float* lo;
  long long mn;     // extent along M (A) or N (B)
  long long ld;     // leading dimension (elements)
  bool mn_major;    // true: stored [K x MN] row-major (MN contiguous); false: stored [MN x K] row-major (K contiguous)
};

template <int BN, bool A_MN, bool B_MN>
static int launch_gemm3(const Operand& A, const Operand& B, long long K, float* D, long long ldd, int splits, long long split_stride,
                        cudaStream_t st) {
  CUtensorMap ma_hi, ma_lo, mb_hi, mb_lo;
  int rc;
  if (A_MN) {
    if ((rc = make_map(&ma_hi, A.hi, A.mn, K, A.ld, 32, BK, true))) return rc;
    if ((rc = make_map(&ma_lo, A.lo, A.mn, K, A.ld, 32, BK, true))) return rc;
  } else {
    if ((rc = make_map(&ma_hi, A.hi, K, A.mn, A.ld, BK, BM))) return rc;
    if ((rc = make_map(&ma_lo, A.lo, K, A.mn, A.ld, BK, BM))) return rc;
  }
  if (B_MN) {
    if ((rc = make_map(&mb_hi, B.hi, B.mn, K, B.ld, 32, BK, true))) return rc;
    if ((rc = make_map(&mb_lo, B.lo, B.mn, K, B.ld, 32, BK, true))) return rc;
  } else {
    if ((rc = make_map(&mb_hi, B.hi, K, B.mn, B.ld, BK, BN))) return rc;
    if ((rc = make_map(&mb_lo, B.lo, K, B.mn, B.ld, BK, BN))) return rc;
  }
  const int kblocks = (int)cdiv<long long>(K, BK);
  if (splits > kblocks) splits = kblocks;
  if (splits < 1) splits = 1;
  int kbps = cdiv(kblocks, splits);
  splits = cdiv(kblocks, kbps);                       // every split owns at least one K block
  auto kern = gemm3_kernel<BN, A_MN, B_MN>;
  ONMF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg<BN>::SMEM_BYTES));
  dim3 grid((unsigned)cdiv<long long>(A.mn, BM), (unsigned)cdiv<long long>(B.mn, BN), (unsigned)splits);
  kern<<<grid, 256, Cfg<BN>::SMEM_BYTES, st>>>(ma_hi, ma_lo, mb_hi, mb_lo, D, ldd, (int)A.mn, (int)B.mn, kblocks, kbps, split_stride);
  ONMF_LAUNCH_CHECK("gemm3_kernel");
  return splits;   // >= 1: number of partial tiles written
}

template <bool A_MN, bool B_MN>
static int dispatch_bn(const Operand& A, const Operand& B, long long K, float* D, long long ldd, int splits, long long split_stride,
                       cudaStream_t st) {
  if (B.mn <= 64) return launch_gemm3<64, A_MN, B_MN>(A, B, K, D, ldd, splits, split_stride, st);
  if (B.mn <= 128) return launch_gemm3<128, A_MN, B_MN>(A, B, K, D, ldd, splits, split_stride, st);
  return launch_gemm3<256, A_MN, B_MN>(A, B, K, D, ldd, splits, split_stride, st);
}

// The tensor core adds each MMA into the fp32 accumulator with round-toward-zero, a bias of ~1.6e-8 relative per
// accumulation (measured: 1.0e-5 at 384 MMAs + ...).  Chains are therefore capped at MAX_CHAIN_KB K-blocks
// (12 MMAs each) per split -- the partial tiles are then summed in fp32 round-to-nearest by the second pass --
// and every surrogate product uses the same chain length so that A and B carry the same (cancelling) scale bias.
constexpr int MAX_CHAIN_KB = 32;
static int pick_splits(long long tiles, long long kblocks) {
  long long fill = cdiv<long long>(num_sms(), tiles);
  long long chain = cdiv<long long>(kblocks, MAX_CHAIN_KB);
  long long s = fill > chain ? fill : chain;
  if (s > kblocks) s = kblocks;
  if (s < 1) s = 1;
  return (int)s;
}

static long long tiles_of(long long m, long long n) {
  int bn = n <= 64 ? 64 : n <= 128 ? 128 : 256;
  return cdiv<long long>(m, BM) * cdiv<long long>(n, bn);
}

}  // namespace tc
}  // namespace onmf

using namespace onmf;

extern "C" int onmf_tc_supported(int k, int d) {
  // TMA needs 16-byte global strides; the 3xTF32 path is fp32 only
  return (k % 4 == 0 && d % 4 == 0 && k >= 32 && d >= 32) ? 1 : 0;
}

extern "C" int onmf_split_tf32(const void* src, void* hi, void* lo, int64_t count, void* stream) {
  if (!src || !hi || !lo || count < 0 || count % 4) return fail(ONMF_E_ARG, "split_tf32: bad argument (count must be a multiple of 4)");
  if (!tc::aligned16(src) || !tc::aligned16(hi) || !tc::aligned16(lo)) return fail(ONMF_E_ARG, "split_tf32: pointers must be 16-byte aligned");
  if (count == 0) return ONMF_OK;
  long long c4 = count / 4;
  int grid = (int)std::min<long long>(cdiv<long long>(c4, 256), 16LL * num_sms());
  tc::split_tf32_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const float*)src, (float*)hi, (float*)lo, c4);
  ONMF_LAUNCH_CHECK("split_tf32_kernel");
  return ONMF_OK;
}

extern "C" int onmf_cov_tc(const void* Xt_hi, const void* Xt_lo, int64_t n, int d, const void* W_hi, const void* W_lo, int k, void* Ct,
                           void* stream) {
  if (!Xt_hi || !Xt_lo || !W_hi || !W_lo || !Ct || n < 0 || !onmf_tc_supported(k, d)) return fail(ONMF_E_ARG, "cov_tc: bad argument / unsupported shape");
  if (n == 0) return ONMF_OK;
  tc::Operand A{(const float*)Xt_hi, (const float*)Xt_lo, n, d, false};       // K-major (K = d contiguous)
  tc::Operand B{(const float*)W_hi, (const float*)W_lo, k, k, true};          // W is (d x k): N contiguous
  int rc = tc::dispatch_bn<false, true>(A, B, d, (float*)Ct, k, 1, 0, (cudaStream_t)stream);
  return rc < 0 ? rc : ONMF_OK;
}

extern "C" size_t onmf_surrogate_tc_workspace(int64_t n, int k, int d) {
  if (n < 0 || k <= 0 || d <= 0) return 0;
  long long kblocks = cdiv<long long>(n > 0 ? n : 1, tc::BK);
  size_t s1 = tc::pick_splits(tc::tiles_of(k, d), kblocks), s2 = s1;
  return (s1 * (size_t)k * k + s2 * (size_t)k * d) * 4 + 512;
}

extern "C" int onmf_surrogate_partial_tc(const void* Ht_hi, const void* Ht_lo, const void* Xt_hi, const void* Xt_lo, int64_t n, int k,
                                         int d, void* P, void* workspace, size_t workspace_bytes, void* stream) {
  if (!Ht_hi || !Ht_lo || !Xt_hi || !Xt_lo || !P || n < 0 || !onmf_tc_supported(k, d)) return fail(ONMF_E_ARG, "surrogate_partial_tc: bad argument / unsupported shape");
  if (!workspace || workspace_bytes < onmf_surrogate_tc_workspace(n, k, d)) return fail(ONMF_E_WORKSPACE, "surrogate_partial_tc: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  float* Pf = (float*)P;
  const long long ldp = k + d;
  if (n == 0) {
    ONMF_CUDA(cudaMemsetAsync(P, 0, (size_t)k * ldp * 4, st));
    return ONMF_OK;
  }
  const long long kblocks = cdiv<long long>(n, tc::BK);
  const int s1 = tc::pick_splits(tc::tiles_of(k, d), kblocks), s2 = s1;   // equal chain lengths for HtH and HtX
  float* part1 = (float*)workspace;
  float* part2 = part1 + (size_t)s1 * k * k;
  tc::Operand A{(const float*)Ht_hi, (const float*)Ht_lo, k, k, true};        // Ht (n x k): M = k contiguous
  tc::Operand B1{(const float*)Ht_hi, (const float*)Ht_lo, k, k, true};
  tc::Operand B2{(const float*)Xt_hi, (const float*)Xt_lo, d, d, true};       // Xt (n x d): N = d contiguous
  int w1 = tc::dispatch_bn<true, true>(A, B1, n, part1, k, s1, (long long)k * k, st);
  if (w1 < 0) return w1;
  int w2 = tc::dispatch_bn<true, true>(A, B2, n, part2, d, s2, (long long)k * d, st);
  if (w2 < 0) return w2;
  tc::split_reduce2d_kernel<<<(unsigned)cdiv<long long>((long long)k * k, 256), 256, 0, st>>>(part1, w1, k, k, Pf, ldp);
  ONMF_LAUNCH_CHECK("split_reduce2d_kernel");
  tc::split_reduce2d_kernel<<<(unsigned)cdiv<long long>((long long)k * d, 256), 256, 0, st>>>(part2, w2, k, d, Pf + k, ldp);
  ONMF_LAUNCH_CHECK("split_reduce2d_kernel");
  return ONMF_OK;
}
