// K1 + K2 and K4 fused on the tensor cores: the minibatch is read ONCE per product, as stored.
//
//   cov_fused : Ct (n x k)      = X[idx] (n x d) . W (d x k)                  [sklearn/_dict_learning.py:426 + src/ontf.py:231]
//   sur_fused : P (k x (k+d))   = [ Ht^T Ht | Ht^T X[idx] ]   (+ blend)       [src/ontf.py:147-148]
//
// gemm_tc.cu feeds tcgen05 from TF32 hi/lo copies that a gather/split kernel first materialises in HBM (3x the minibatch
// in traffic).  Here "loader" warps read the minibatch rows straight from the resident pool (fp32, or the narrow storage
// formats uint8 / fp16) through the minibatch indices, split every value into hi = rna_tf32(x) and lo = x - hi in
// registers and store both tiles into shared memory in exactly the swizzled canonical layouts the UMMA descriptors
// expect (K-major SWIZZLE_128B for cov's A operand, MN-major SWIZZLE_128B_BASE32B for both surrogate operands), then
// fence the generic->async proxy and arrive on the stage's mbarrier.  The small dictionary operand of cov (W hi/lo, L2
// resident) still arrives by TMA.  Both kernels are persistent (one CTA per SM looping over work items), warp
// specialised (TMA / MMA issuer / TMEM allocator / 4 epilogue warps / 2 x 8 loader warps), and keep FP32 accumulators in
// TMEM; cov double-buffers the accumulator so the epilogue of tile i overlaps the MMAs of tile i+1.
//
// sur_fused: one CTA owns both 128-row halves of the k <= 256 atoms (two TMEM accumulators sharing every B tile), a
// 256-column slab of [H | X] and a contiguous range of samples; the tensor core accumulates with round-toward-zero
// (~1.6e-8 relative per MMA), so a chain is capped at 1024 samples, after which the epilogue warps add the accumulator
// into the CTA's partial tile in global memory (L2 resident) in fp32 round-to-nearest.  A second small kernel sums the
// per-range partial tiles in fixed order (deterministic) and -- on one GPU -- applies the blend
// A <- (1-w) A + w P_A, B <- (1-w) B + w P_B in the same pass (SURVEY.md §2 K4).
#include <cuda.h>
#include <cuda_fp16.h>

#include <algorithm>

#include "common.cuh"

namespace onmf {
namespace tcf {

constexpr int BM = 128;
constexpr int NLW = 8;                     // loader warps per group
constexpr int NLG = 2;                     // loader groups (alternate over k-blocks)
constexpr int THREADS = (8 + NLG * NLW) * 32;   // 768

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
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
// generic-proxy writes (st.shared) -> visible to the async proxy (tcgen05.mma operand reads)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
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
}

// shared-memory matrix descriptor (see gemm_tc.cu make_desc): K-major SWIZZLE_128B, or MN-major SWIZZLE_128B_BASE32B with
// the byte distance `lbo` between consecutive 32-element MN chunks
__device__ __forceinline__ uint64_t desc_kmajor(uint32_t saddr) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ uint64_t desc_mnmajor(uint32_t saddr, uint32_t lbo) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(512 >> 4) << 32) | (1ull << 46) | (1ull << 61);
}

// ---- source element access: 4 consecutive values of a stored row -> fp32 ------------------------------------------
template <typename S> struct Src;
template <> struct Src<float> {
  static __device__ __forceinline__ float4 ld4(const void* row, long long e, float) {
    return *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(row) + e);
  }
};
template <> struct Src<unsigned char> {
  static __device__ __forceinline__ float4 ld4(const void* row, long long e, float sc) {
    const uchar4 v = *reinterpret_cast<const uchar4*>(reinterpret_cast<const unsigned char*>(row) + e);
    return make_float4((float)v.x * sc, (float)v.y * sc, (float)v.z * sc, (float)v.w * sc);
  }
};
template <> struct Src<__half> {
  static __device__ __forceinline__ float4 ld4(const void* row, long long e, float sc) {
    const uint2 raw = *reinterpret_cast<const uint2*>(reinterpret_cast<const __half*>(row) + e);
    const __half2 a = *reinterpret_cast<const __half2*>(&raw.x), b = *reinterpret_cast<const __half2*>(&raw.y);
    const float2 fa = __half22float2(a), fb = __half22float2(b);
    return make_float4(fa.x * sc, fa.y * sc, fb.x * sc, fb.y * sc);
  }
};

__device__ __forceinline__ void split4(const float4& x, float4& h, float4& l) {
  uint32_t t;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(t) : "f"(x.x)); h.x = __uint_as_float(t); l.x = x.x - h.x;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(t) : "f"(x.y)); h.y = __uint_as_float(t); l.y = x.y - h.y;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(t) : "f"(x.z)); h.z = __uint_as_float(t); l.z = x.z - h.z;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(t) : "f"(x.w)); h.w = __uint_as_float(t); l.w = x.w - h.w;
}

// The loaders read the minibatch through a SOURCE VIEW:
//   row<S>(src, rp)  -> false for a sample that must become a NaN row (never dereferenced), else rp = its base address
//   off(e)           -> where features e .. e+3 sit relative to a row's base (a function of e alone: computed once per
//                       k-block / item and shared by every row the thread loads)
//   ld4<S>(rp, o)    -> the 4 values widened to fp32 (value = (float)stored * scale for the narrow formats)
struct PoolView {
  const void* base;       // stored minibatch pool, one sample per row
  long long ld;           // row pitch in ELEMENTS of the storage type
  const long long* idx;   // minibatch row indices into the pool, or nullptr (rows 0..n-1)
  long long n_pool;       // rows in the pool (indices outside [0, n_pool) contribute NaN rows, like the K1 gather)
  float scale;            // narrow formats: value = (float)stored * scale

  struct Off { long long e; };
  __device__ __forceinline__ Off off(int e) const { return Off{e}; }
  template <typename S>
  __device__ __forceinline__ bool row(long long src, const void*& rp) const {
    rp = base;
    if (src < 0 || src >= n_pool) return false;
    rp = reinterpret_cast<const unsigned char*>(base) + (size_t)src * (size_t)ld * sizeof(S);
    return true;
  }
  template <typename S>
  __device__ __forceinline__ float4 ld4(const void* rp, const Off& o) const { return Src<S>::ld4(rp, o.e, scale); }
};

// A minibatch of image patches by reference: sample j is the p x p (x C) patch of the HWC image whose top-left corner is
// coords[idx[j]], feature e = (r*p + c)*C + ch  ->  image element (y + r, x + c, ch).  A row's base is its corner; the
// offset of feature e inside a patch is r*W*C + (c*C + ch), the same for every patch.  When p*C % 4 != 0 a 4-feature
// chunk can straddle two patch rows, so the four offsets are kept separately and the values loaded as scalars (the
// chunk is contiguous but in general unaligned in the image when p*C % 4 == 0: scalar loads as well).  Corner bases
// are 64-bit; intra-patch offsets are 32-bit (the host checks (p+32)*W*C < 2^31).
struct PatchView {
  const void* img;        // (H x W x C) row-major
  int H, W, C, p;
  const int* coords;      // (n_coords x 2) int32 top-left corners (y, x)
  long long n_coords;
  const long long* idx;   // minibatch indices into coords, or nullptr (0..n-1)
  float scale;

  struct Off { int o[4]; };
  __device__ __forceinline__ Off off(int e) const {
    const int run = p * C, pitch = W * C;
    int r = e / run, c = e - r * run;
    Off f;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      f.o[t] = r * pitch + c;
      if (++c == run) { c = 0; ++r; }
    }
    return f;
  }
  template <typename S>
  __device__ __forceinline__ bool row(long long src, const void*& rp) const {
    rp = img;
    if (src < 0 || src >= n_coords) return false;
    const int y = __ldg(coords + 2 * src), x = __ldg(coords + 2 * src + 1);
    if (y < 0 || x < 0 || y > H - p || x > W - p) return false;          // the patch leaves the image
    rp = reinterpret_cast<const S*>(img) + ((size_t)y * (size_t)W + (size_t)x) * (size_t)C;
    return true;
  }
  template <typename S>
  __device__ __forceinline__ float4 ld4(const void* rp, const Off& f) const {
    const S* q = reinterpret_cast<const S*>(rp);
    return make_float4(wide(__ldg(q + f.o[0])), wide(__ldg(q + f.o[1])), wide(__ldg(q + f.o[2])), wide(__ldg(q + f.o[3])));
  }
  __device__ __forceinline__ float wide(float v) const { return v; }
  __device__ __forceinline__ float wide(unsigned char v) const { return (float)v * scale; }   // as Src<unsigned char>::ld4
};

// =====================================================================================================================
// cov_fused
// =====================================================================================================================
template <int BN>
struct CovCfg {
  static constexpr int BK = 32;
  static constexpr int STAGES = BN == 256 ? 2 : 3;
  static constexpr uint32_t A_BYTES = BM * BK * 4;                 // one of hi / lo
  static constexpr uint32_t B_BYTES = BN * BK * 4;
  static constexpr uint32_t STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;
  static constexpr uint32_t SMEM_BYTES = STAGES * STAGE_BYTES + 1024;
  static constexpr uint32_t CHUNK_BYTES = BK * 128;                // MN-major B: 32-wide N chunk = 32 k-rows x 128 B
};

template <int BN, typename S, typename V>
__global__ void __launch_bounds__(THREADS, 1)
cov_fused_kernel(const __grid_constant__ CUtensorMap tmW_hi, const __grid_constant__ CUtensorMap tmW_lo, V X, long long n,
                 int d, int k, float* __restrict__ Ct) {
  using C = CovCfg<BN>;
  constexpr int STAGES = C::STAGES;
  extern __shared__ uint8_t smem_dyn[];
  __shared__ __align__(8) uint64_t full_bar[STAGES];
  __shared__ __align__(8) uint64_t empty_bar[STAGES];
  __shared__ __align__(8) uint64_t tmem_full_bar[2];
  __shared__ __align__(8) uint64_t tmem_empty_bar[2];
  __shared__ uint32_t tmem_slot;

  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~uintptr_t(1023));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nkb = (d + C::BK - 1) / C::BK;
  const long long ntiles = (n + BM - 1) / BM;

  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(smem_u32(&full_bar[s]), NLW + 1);       // 8 loader warps + the TMA thread's expect_tx arrive
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(smem_u32(&tmem_full_bar[a]), 1);
      mbar_init(smem_u32(&tmem_empty_bar[a]), 4);        // one arrive per epilogue warp
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  } else if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"((uint32_t)(2 * BN))
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;

  auto stage_ptr = [&](int s) -> uint8_t* { return smem + (size_t)s * C::STAGE_BYTES; };

  if (warp == 0) {
    // ===== TMA producer: the dictionary operand (W hi / lo, MN-major chunks of 32 atoms) =====
    if (lane == 0) {
      long long c = 0;
      for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        for (int kb = 0; kb < nkb; ++kb, ++c) {
          const int s = (int)(c % STAGES);
          const uint32_t ph = (uint32_t)((c / STAGES) & 1);
          mbar_wait(smem_u32(&empty_bar[s]), ph ^ 1);
          const uint32_t fb = smem_u32(&full_bar[s]);
          mbar_expect_tx(fb, 2 * C::B_BYTES);
          const uint32_t b_hi = smem_u32(stage_ptr(s)) + 2 * C::A_BYTES;
          const uint32_t b_lo = b_hi + C::B_BYTES;
#pragma unroll
          for (int ch = 0; ch < BN / 32; ++ch) {
            tma_load_2d(b_hi + ch * C::CHUNK_BYTES, &tmW_hi, fb, 32 * ch, kb * C::BK);
            tma_load_2d(b_lo + ch * C::CHUNK_BYTES, &tmW_lo, fb, 32 * ch, kb * C::BK);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    if (lane == 0) {
      // instruction descriptor: D=F32 [4,6), A=TF32 [7,10), B=TF32 [10,13), A K-major [15]=0, B MN-major [16]=1, N>>3 [17,23), M>>4 [24,29)
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 16) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
      long long c = 0;
      int it = 0;
      for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
        const int acc = it & 1;
        mbar_wait(smem_u32(&tmem_empty_bar[acc]), (uint32_t)(((it >> 1) & 1) ^ 1));      // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t tacc = tmem_base + (uint32_t)(acc * BN);
        for (int kb = 0; kb < nkb; ++kb, ++c) {
          const int s = (int)(c % STAGES);
          const uint32_t ph = (uint32_t)((c / STAGES) & 1);
          mbar_wait(smem_u32(&full_bar[s]), ph);
          tc_fence_after();
          const uint32_t a_hi = smem_u32(stage_ptr(s));
          const uint32_t a_lo = a_hi + C::A_BYTES;
          const uint32_t b_hi = a_lo + C::A_BYTES;
          const uint32_t b_lo = b_hi + C::B_BYTES;
#pragma unroll
          for (int ks = 0; ks < C::BK / 8; ++ks) {
            const uint64_t dah = desc_kmajor(a_hi + ks * 32), dal = desc_kmajor(a_lo + ks * 32);
            const uint64_t dbh = desc_mnmajor(b_hi + ks * 1024, C::CHUNK_BYTES), dbl = desc_mnmajor(b_lo + ks * 1024, C::CHUNK_BYTES);
            umma_tf32(tacc, dah, dbh, idesc, (kb > 0 || ks > 0) ? 1u : 0u);
            umma_tf32(tacc, dah, dbl, idesc, 1u);
            umma_tf32(tacc, dal, dbh, idesc, 1u);
          }
          umma_commit(smem_u32(&empty_bar[s]));
        }
        umma_commit(smem_u32(&tmem_full_bar[acc]));
      }
    }
  } else if (warp >= 4 && warp < 8) {
    // ===== epilogue: TMEM -> registers -> global (each thread owns one row: 128 contiguous bytes per 32 columns) =====
    const int q = warp - 4;
    int it = 0;
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
      const int acc = it & 1;
      mbar_wait(smem_u32(&tmem_full_bar[acc]), (uint32_t)((it >> 1) & 1));
      tc_fence_after();
      const long long row = tile * BM + q * 32 + lane;
      float* dst = Ct + (size_t)row * k;
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 32) {
        if (c0 >= k) break;
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BN + c0), v);
        if (row < n) {
#pragma unroll
          for (int j = 0; j < 8; ++j)
            if (c0 + 4 * j < k)      // k % 4 == 0
              *reinterpret_cast<float4*>(dst + c0 + 4 * j) = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                                                         __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&tmem_empty_bar[acc]));
    }
  } else if (warp >= 8) {
    // ===== loaders: gather + widen + TF32 split of the minibatch rows, straight into the K-major swizzled A tiles =====
    const int g = (warp - 8) / NLW;                    // loader group: handles the k-blocks with (global counter % NLG) == g
    const int u = threadIdx.x - (8 + g * NLW) * 32;    // 0..255 inside the group
    const int r0 = u >> 3, ch = u & 7;                 // rows r0 + 32 i (i < 4), 16-byte chunk ch of the 128-byte K slice
    long long c_tile0 = 0;                             // global k-block counter at the start of the current tile
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, c_tile0 += nkb) {
      const void* rowp[4];
      bool rok[4], rnan[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const long long j = tile * BM + r0 + 32 * i;
        rok[i] = j < n;
        long long src = 0;
        if (rok[i]) src = X.idx ? X.idx[j] : j;
        rnan[i] = !X.template row<S>(src, rowp[i]) && rok[i];
      }
      // first k-block of this group within the tile
      int kb = (int)((NLG - (c_tile0 % NLG) + g) % NLG);
      for (; kb < nkb; kb += NLG) {
        const long long c = c_tile0 + kb;
        const int s = (int)(c % STAGES);
        const uint32_t ph = (uint32_t)((c / STAGES) & 1);
        const int e = kb * C::BK + ch * 4;             // first feature of this thread's chunk (d % 4 == 0)
        const typename V::Off eo = X.off(e);           // shared by the thread's 4 rows
        float4 x[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          x[i] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (rnan[i]) { const float qn = __int_as_float(0x7fc00000); x[i] = make_float4(qn, qn, qn, qn); }
          else if (rok[i] && e < d) x[i] = X.template ld4<S>(rowp[i], eo);
        }
        mbar_wait(smem_u32(&empty_bar[s]), ph ^ 1);    // the MMAs that read this stage last time have completed
        uint8_t* a_hi = stage_ptr(s);
        uint8_t* a_lo = a_hi + C::A_BYTES;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int r = r0 + 32 * i;
          const uint32_t off = (uint32_t)((r >> 3) * 1024 + (r & 7) * 128 + ((ch ^ (r & 7)) << 4));
          float4 h, l;
          split4(x[i], h, l);
          *reinterpret_cast<float4*>(a_hi + off) = h;
          *reinterpret_cast<float4*>(a_lo + off) = l;
        }
        fence_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&full_bar[s]));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)(2 * BN)) : "memory");
  }
}

// =====================================================================================================================
// sur_fused
// =====================================================================================================================
struct SurCfg {
  static constexpr int BK = 16;                                    // samples per k-block
  static constexpr int BN = 256;
  static constexpr int STAGES = 3;
  static constexpr uint32_t CHUNK = BK * 128;                      // a 32-wide MN chunk: 16 k-rows x 128 B
  static constexpr uint32_t A_BYTES = 8 * CHUNK;                   // 256 atoms (both halves), one of hi / lo
  static constexpr uint32_t B_BYTES = (BN / 32) * CHUNK;
  static constexpr uint32_t STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;   // 64 KB
  static constexpr uint32_t SMEM_BYTES = STAGES * STAGE_BYTES + 1024;
  static constexpr int CHAIN = 64;                                 // k-blocks per accumulation chain (1024 samples)
};

// byte offset of the 16-byte piece holding MN elements [mn, mn+4) of k-row kr inside an MN-major SWIZZLE_128B_BASE32B tile
__device__ __forceinline__ uint32_t mn_off(int kr, int mn) {
  return (uint32_t)((mn >> 5) * SurCfg::CHUNK + (kr >> 2) * 512 + (kr & 3) * 128 + ((((mn & 31) >> 3) ^ (kr & 3)) << 5) + ((mn & 7) >> 2) * 16);
}

template <typename S, typename V>
__global__ void __launch_bounds__(THREADS, 1)
sur_fused_kernel(const float* __restrict__ Ht, V X, long long n, int k, int d, int n_tiles, int splits, long long kb_per_split,
                 float* __restrict__ part) {
  using C = SurCfg;
  extern __shared__ uint8_t smem_dyn[];
  __shared__ __align__(8) uint64_t full_bar[C::STAGES];
  __shared__ __align__(8) uint64_t empty_bar[C::STAGES];
  __shared__ __align__(8) uint64_t tmem_full_bar;
  __shared__ __align__(8) uint64_t tmem_empty_bar;
  __shared__ uint32_t tmem_slot;

  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~uintptr_t(1023));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int MH = (k + 127) / 128;                      // 128-row halves of the atom axis (1 or 2)
  const long long kb_total = (n + C::BK - 1) / C::BK;
  const long long items = (long long)n_tiles * splits;
  const int ncat = k + d;

  if (warp == 1 && lane == 0) {
    for (int s = 0; s < C::STAGES; ++s) {
      mbar_init(smem_u32(&full_bar[s]), NLW);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
    mbar_init(smem_u32(&tmem_full_bar), 1);
    mbar_init(smem_u32(&tmem_empty_bar), 4);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  } else if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;
  auto stage_ptr = [&](int s) -> uint8_t* { return smem + (size_t)s * C::STAGE_BYTES; };
  // k-block range of an item
  auto item_range = [&](long long item, long long& kb0, long long& kb1, int& nt) {
    nt = (int)(item % n_tiles);
    const long long sp = item / n_tiles;
    kb0 = sp * kb_per_split;
    kb1 = kb0 + kb_per_split;
    if (kb1 > kb_total) kb1 = kb_total;
    if (kb0 > kb1) kb0 = kb1;
  };

  if (warp == 1) {
    // ===== MMA issuer =====
    if (lane == 0) {
      // A MN-major [15]=1, B MN-major [16]=1
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(C::BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
      long long c = 0, chains = 0;
      for (long long item = blockIdx.x; item < items; item += gridDim.x) {
        long long kb0, kb1; int nt;
        item_range(item, kb0, kb1, nt);
        for (long long kc = kb0; kc < kb1; kc += C::CHAIN, ++chains) {
          const long long kce = kc + C::CHAIN < kb1 ? kc + C::CHAIN : kb1;
          mbar_wait(smem_u32(&tmem_empty_bar), (uint32_t)((chains & 1) ^ 1));          // the epilogue has drained the accumulators
          tc_fence_after();
          for (long long kb = kc; kb < kce; ++kb, ++c) {
            const int s = (int)(c % C::STAGES);
            const uint32_t ph = (uint32_t)((c / C::STAGES) & 1);
            mbar_wait(smem_u32(&full_bar[s]), ph);
            tc_fence_after();
            const uint32_t a_hi = smem_u32(stage_ptr(s));
            const uint32_t a_lo = a_hi + C::A_BYTES;
            const uint32_t b_hi = a_lo + C::A_BYTES;
            const uint32_t b_lo = b_hi + C::B_BYTES;
            for (int h = 0; h < MH; ++h) {
              const uint32_t tacc = tmem_base + (uint32_t)(h * C::BN);
              const uint32_t ah = a_hi + h * 4 * C::CHUNK, al = a_lo + h * 4 * C::CHUNK;
#pragma unroll
              for (int ks = 0; ks < C::BK / 8; ++ks) {
                const uint64_t dah = desc_mnmajor(ah + ks * 1024, C::CHUNK), dal = desc_mnmajor(al + ks * 1024, C::CHUNK);
                const uint64_t dbh = desc_mnmajor(b_hi + ks * 1024, C::CHUNK), dbl = desc_mnmajor(b_lo + ks * 1024, C::CHUNK);
                umma_tf32(tacc, dah, dbh, idesc, (kb > kc || ks > 0) ? 1u : 0u);
                umma_tf32(tacc, dah, dbl, idesc, 1u);
                umma_tf32(tacc, dal, dbh, idesc, 1u);
              }
            }
            umma_commit(smem_u32(&empty_bar[s]));
          }
          umma_commit(smem_u32(&tmem_full_bar));
        }
      }
    }
  } else if (warp >= 4 && warp < 8) {
    // ===== epilogue: after every chain, partial tile (+)= accumulator (fp32 round-to-nearest; the tile stays in L2) =====
    const int q = warp - 4;
    long long chains = 0;
    for (long long item = blockIdx.x; item < items; item += gridDim.x) {
      long long kb0, kb1; int nt;
      item_range(item, kb0, kb1, nt);
      float* tile = part + (size_t)item * (size_t)(MH * 128) * C::BN;
      if (kb0 >= kb1) {                                   // empty sample range: the partial tile is zero
        for (int h = 0; h < MH; ++h) {
          float* dst = tile + (size_t)(h * 128 + q * 32 + lane) * C::BN;
          for (int c0 = 0; c0 < C::BN; c0 += 4) *reinterpret_cast<float4*>(dst + c0) = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        continue;
      }
      for (long long kc = kb0; kc < kb1; kc += C::CHAIN, ++chains) {
        mbar_wait(smem_u32(&tmem_full_bar), (uint32_t)(chains & 1));
        tc_fence_after();
        const bool first = (kc == kb0);
        for (int h = 0; h < MH; ++h) {
          float* dst = tile + (size_t)(h * 128 + q * 32 + lane) * C::BN;
#pragma unroll 1
          for (int c0 = 0; c0 < C::BN; c0 += 32) {
            uint32_t v[32];
            float4 old[8];
            if (!first) {
#pragma unroll
              for (int j = 0; j < 8; ++j) old[j] = *reinterpret_cast<const float4*>(dst + c0 + 4 * j);
            }
            tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(h * C::BN + c0), v);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              float4 o = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]),
                                     __uint_as_float(v[4 * j + 3]));
              if (!first) { o.x += old[j].x; o.y += old[j].y; o.z += old[j].z; o.w += old[j].w; }
              *reinterpret_cast<float4*>(dst + c0 + 4 * j) = o;
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&tmem_empty_bar));
      }
    }
  } else if (warp >= 8) {
    // ===== loaders: both operands, MN-major.  A = rows of Ht (all atoms), B = 256 columns of [Ht | X[idx]] =====
    const int g = (warp - 8) / NLW;
    const int u = threadIdx.x - (8 + g * NLW) * 32;    // 0..255
    const int kr = u >> 4;                             // k-row (sample inside the k-block) 0..15
    const int f0 = u & 15;                             // float4 column f0 + 16 p, p < 4  (64 float4 = 256 columns per row)
    long long c0 = 0;                                  // global k-block counter at the start of the current item
    for (long long item = blockIdx.x; item < items; item += gridDim.x) {
      long long kb0, kb1; int nt;
      item_range(item, kb0, kb1, nt);
      const int n0 = nt * C::BN;                       // first column of [Ht | X] of this item
      typename V::Off xo[4];                           // feature offsets of the thread's X columns: fixed for the item
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        const int col = n0 + (f0 + 16 * p) * 4;
        xo[p] = X.off(col >= k && col < ncat ? col - k : 0);
      }
      long long kb = kb0 + (long long)((NLG - (c0 % NLG) + g) % NLG);
      long long src_next = -1;                         // pool row of sample (kb, kr), fetched one k-block ahead
      {
        const long long j = kb * C::BK + kr;
        if (kb < kb1 && j < n) src_next = X.idx ? X.idx[j] : j;
      }
      for (; kb < kb1; kb += NLG) {
        const long long c = c0 + (kb - kb0);
        const int s = (int)(c % C::STAGES);
        const uint32_t ph = (uint32_t)((c / C::STAGES) & 1);
        const long long j = kb * C::BK + kr;
        const bool jok = j < n;
        const long long src = src_next;
        {
          const long long jn = (kb + NLG) * C::BK + kr;
          src_next = -1;
          if (kb + NLG < kb1 && jn < n) src_next = X.idx ? X.idx[jn] : jn;
        }
        const void* xrow;
        const bool bad = !X.template row<S>(jok ? src : 0, xrow) && jok;
        const float* hrow = Ht + (size_t)(jok ? j : 0) * k;
        float4 a[4], b[4];
#pragma unroll
        for (int p = 0; p < 4; ++p) {
          const int m = (f0 + 16 * p) * 4;             // atom (A operand)
          a[p] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (jok && m < k) a[p] = *reinterpret_cast<const float4*>(hrow + m);
          const int col = n0 + m;                      // column of [Ht | X] (B operand); k % 4 == 0 so a float4 never straddles
          b[p] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (jok && col < ncat) {
            if (col < k) b[p] = *reinterpret_cast<const float4*>(hrow + col);
            else if (bad) { const float qn = __int_as_float(0x7fc00000); b[p] = make_float4(qn, qn, qn, qn); }
            else b[p] = X.template ld4<S>(xrow, xo[p]);
          }
        }
        mbar_wait(smem_u32(&empty_bar[s]), ph ^ 1);
        uint8_t* a_hi = stage_ptr(s);
        uint8_t* a_lo = a_hi + C::A_BYTES;
        uint8_t* b_hi = a_lo + C::A_BYTES;
        uint8_t* b_lo = b_hi + C::B_BYTES;
#pragma unroll
        for (int p = 0; p < 4; ++p) {
          const uint32_t off = mn_off(kr, (f0 + 16 * p) * 4);
          float4 h, l;
          split4(a[p], h, l);
          *reinterpret_cast<float4*>(a_hi + off) = h;
          *reinterpret_cast<float4*>(a_lo + off) = l;
          split4(b[p], h, l);
          *reinterpret_cast<float4*>(b_hi + off) = h;
          *reinterpret_cast<float4*>(b_lo + off) = l;
        }
        fence_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&full_bar[s]));
      }
      c0 += kb1 - kb0;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

// P[r, c] = sum over sample ranges (fixed order) of the partial tiles; BLEND: A, B <- (1-w) A, B + w P in the same pass
template <bool BLEND>
__global__ void sur_reduce_kernel(const float* __restrict__ part, int n_tiles, int splits, int mrows, int k, int d,
                                  float* __restrict__ P, const double* __restrict__ w_dev, double w_host, float* __restrict__ A,
                                  float* __restrict__ B) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int ncat = k + d;
  if (i >= (long long)k * ncat) return;
  const int r = (int)(i / ncat), c = (int)(i - (long long)r * ncat);
  const int nt = c / SurCfg::BN, cc = c - nt * SurCfg::BN;
  const size_t tile_elems = (size_t)mrows * SurCfg::BN;
  float s = 0.f;
  for (int sp = 0; sp < splits; ++sp) s += part[((size_t)sp * n_tiles + nt) * tile_elems + (size_t)r * SurCfg::BN + cc];
  if (P) P[i] = s;
  if (BLEND) {
    const float w = (float)(w_dev ? *w_dev : w_host);
    const float om = 1.f - w;
    if (c < k) {
      const size_t o = (size_t)r * k + c;
      A[o] = om * A[o] + w * s;
    } else {
      const size_t o = (size_t)r * d + (c - k);
      B[o] = om * B[o] + w * s;
    }
  }
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
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}
// MN-major map of a row-major [K x MN] fp32 matrix: boxes of 32 (MN) x box_k, SWIZZLE_128B_ATOM_32B
static int make_map_mn(CUtensorMap* m, const float* ptr, long long mn, long long K, long long ld, int box_k) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(ONMF_E_CUDA, "cuTensorMapEncodeTiled unavailable");
  cuuint64_t dims[2] = {(cuuint64_t)mn, (cuuint64_t)K};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
  cuuint32_t box[2] = {32u, (cuuint32_t)box_k};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    snprintf(g_err, sizeof(g_err), "cuTensorMapEncodeTiled failed (%d): mn=%lld K=%lld ld=%lld", (int)r, mn, K, ld);
    return ONMF_E_CUDA;
  }
  return ONMF_OK;
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

static int check_pool(int src_kind, const void* pool, int64_t ld, int d, const char* who) {
  if (!pool || ld < d) return fail(ONMF_E_ARG, who);
  const size_t esz = src_kind == ONMF_F32 ? 4 : src_kind == ONMF_STORE_F16 ? 2 : src_kind == ONMF_STORE_U8 ? 1 : 0;
  if (!esz) return fail(ONMF_E_ARG, "fused tensor-core products: minibatch storage must be ONMF_F32, ONMF_STORE_U8 or ONMF_STORE_F16");
  // every 4-element group must be naturally aligned: 16 B (fp32), 8 B (fp16), 4 B (u8)
  if ((reinterpret_cast<uintptr_t>(pool) % (4 * esz)) || (ld % 4) || (d % 4)) return fail(ONMF_E_ARG, "fused tensor-core products: pool base / pitch / d must be multiples of 4 elements");
  return ONMF_OK;
}

template <int BN, typename S, typename V>
static int launch_cov(const CUtensorMap& mh, const CUtensorMap& ml, const V& X, long long n, int d, int k, float* Ct, cudaStream_t st) {
  auto kern = cov_fused_kernel<BN, S, V>;
  ONMF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CovCfg<BN>::SMEM_BYTES));
  const long long ntiles = cdiv<long long>(n, BM);
  const int grid = (int)std::min<long long>(ntiles, num_sms());
  kern<<<grid, THREADS, CovCfg<BN>::SMEM_BYTES, st>>>(mh, ml, X, n, d, k, Ct);
  ONMF_LAUNCH_CHECK("cov_fused_kernel");
  return ONMF_OK;
}

template <typename S, typename V>
static int dispatch_cov(const CUtensorMap& mh, const CUtensorMap& ml, const V& X, long long n, int d, int k, float* Ct, cudaStream_t st) {
  if (k <= 64) return launch_cov<64, S>(mh, ml, X, n, d, k, Ct, st);
  if (k <= 128) return launch_cov<128, S>(mh, ml, X, n, d, k, Ct, st);
  return launch_cov<256, S>(mh, ml, X, n, d, k, Ct, st);
}

// split-K plan of the surrogate products: sample ranges x 256-column slabs of [Ht | X]
static void sur_plan(long long n, int k, int d, int* n_tiles, int* splits, long long* kb_per_split) {
  const int nt = cdiv(k + d, SurCfg::BN);
  const long long kb_total = cdiv<long long>(n > 0 ? n : 1, SurCfg::BK);
  long long s = num_sms() / nt;                         // one item per CTA when the column slabs allow it
  if (s < 1) s = 1;
  const long long s_work = cdiv<long long>(kb_total, 4);  // at least 64 samples per item
  if (s > s_work) s = s_work;
  long long per = cdiv<long long>(kb_total, s);
  s = cdiv<long long>(kb_total, per);
  *n_tiles = nt; *splits = (int)s; *kb_per_split = per;
}

template <typename S, typename V>
static int launch_sur(const float* Ht, const V& X, long long n, int k, int d, int nt, int sp, long long per, float* part, cudaStream_t st) {
  auto kern = sur_fused_kernel<S, V>;
  ONMF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SurCfg::SMEM_BYTES));
  const int grid = (int)std::min<long long>((long long)nt * sp, num_sms());
  kern<<<grid, THREADS, SurCfg::SMEM_BYTES, st>>>(Ht, X, n, k, d, nt, sp, per, part);
  ONMF_LAUNCH_CHECK("sur_fused_kernel");
  return ONMF_OK;
}

// fixed-order sum of the per-range partial tiles into P (and, blend != 0, the A / B recursion in the same pass)
static int sur_reduce(const float* part, int nt, int sp, int mrows, int k, int d, void* P, int blend, double w, const double* w_dev,
                      void* A, void* B, cudaStream_t st) {
  const long long tot = (long long)k * (k + d);
  const unsigned grid2 = (unsigned)cdiv<long long>(tot, 256);
  if (blend) sur_reduce_kernel<true><<<grid2, 256, 0, st>>>(part, nt, sp, mrows, k, d, (float*)P, w_dev, w, (float*)A, (float*)B);
  else sur_reduce_kernel<false><<<grid2, 256, 0, st>>>(part, nt, sp, mrows, k, d, (float*)P, nullptr, 0.0, nullptr, nullptr);
  ONMF_LAUNCH_CHECK("sur_reduce_kernel");
  return ONMF_OK;
}

// a patch minibatch the fused kernels can read: fp32 / u8 image, sane geometry, 32-bit intra-patch offsets
static int check_patches(const onmf_patch_minibatch* pm, const char* who) {
  if (!pm || !pm->img || pm->H <= 0 || pm->W <= 0 || pm->C <= 0 || pm->p <= 0 || pm->p > pm->H || pm->p > pm->W || pm->n < 0 ||
      pm->n_coords < 0 || (pm->n_coords > 0 && !pm->coords))
    return fail(ONMF_E_ARG, who);
  if (pm->kind != ONMF_F32 && pm->kind != ONMF_STORE_U8)
    return fail(ONMF_E_ARG, "fused tensor-core products: a patch minibatch's image must be ONMF_F32 or ONMF_STORE_U8");
  if ((long long)(pm->p + 32) * pm->W * pm->C >= (1LL << 31))
    return fail(ONMF_E_UNSUPPORTED, "fused tensor-core products: image rows too wide for 32-bit offsets inside a patch ((p+32)*W*C >= 2^31)");
  return ONMF_OK;
}

static PatchView patch_view(const onmf_patch_minibatch* pm) {
  return PatchView{pm->img, pm->H, pm->W, pm->C, pm->p, pm->coords, pm->n_coords, (const long long*)pm->idx, (float)pm->scale};
}

}  // namespace tcf
}  // namespace onmf

using namespace onmf;

extern "C" int onmf_fused_tc_supported(int k, int d) {
  // k <= 256: both 128-row halves of the atom axis live in one CTA's tensor memory (two 256-column accumulators)
  return (onmf_tc_supported(k, d) && k <= 256) ? 1 : 0;
}

extern "C" int onmf_cov_fused_tc(int src_kind, const void* pool, int64_t n_pool, int64_t ld_pool, const int64_t* idx, int64_t n, int d,
                                 double scale, const void* W_hi, const void* W_lo, int k, void* Ct, void* stream) {
  if (!W_hi || !W_lo || !Ct || n < 0 || n_pool <= 0 || !onmf_fused_tc_supported(k, d)) return fail(ONMF_E_ARG, "cov_fused_tc: bad argument / unsupported shape");
  int rc = tcf::check_pool(src_kind, pool, ld_pool, d, "cov_fused_tc: bad pool");
  if (rc) return rc;
  if (!tcf::aligned16(W_hi) || !tcf::aligned16(W_lo) || !tcf::aligned16(Ct)) return fail(ONMF_E_ARG, "cov_fused_tc: W_hi / W_lo / Ct must be 16-byte aligned");
  if (n == 0) return ONMF_OK;
  CUtensorMap mh, ml;
  if ((rc = tcf::make_map_mn(&mh, (const float*)W_hi, k, d, k, 32))) return rc;
  if ((rc = tcf::make_map_mn(&ml, (const float*)W_lo, k, d, k, 32))) return rc;
  tcf::PoolView X{pool, ld_pool, (const long long*)idx, n_pool, (float)scale};
  cudaStream_t st = (cudaStream_t)stream;
  if (src_kind == ONMF_F32) return tcf::dispatch_cov<float>(mh, ml, X, n, d, k, (float*)Ct, st);
  if (src_kind == ONMF_STORE_U8) return tcf::dispatch_cov<unsigned char>(mh, ml, X, n, d, k, (float*)Ct, st);
  return tcf::dispatch_cov<__half>(mh, ml, X, n, d, k, (float*)Ct, st);
}

extern "C" size_t onmf_surrogate_fused_tc_workspace(int64_t n, int k, int d) {
  if (n < 0 || k <= 0 || d <= 0) return 0;
  int nt, sp; long long per;
  tcf::sur_plan(n, k, d, &nt, &sp, &per);
  const size_t mrows = (size_t)cdiv(k, 128) * 128;
  return (size_t)nt * sp * mrows * tcf::SurCfg::BN * sizeof(float) + 256;
}

extern "C" int onmf_surrogate_fused_tc(const void* Ht, int src_kind, const void* pool, int64_t n_pool, int64_t ld_pool, const int64_t* idx,
                                       int64_t n, int k, int d, double scale, void* P, int blend, double w, const double* w_dev, void* A,
                                       void* B, void* workspace, size_t workspace_bytes, void* stream) {
  if (!Ht || n < 0 || n_pool <= 0 || !onmf_fused_tc_supported(k, d)) return fail(ONMF_E_ARG, "surrogate_fused_tc: bad argument / unsupported shape");
  if (!P && !blend) return fail(ONMF_E_ARG, "surrogate_fused_tc: nothing to write (P == NULL and blend == 0)");
  if (blend && (!A || !B)) return fail(ONMF_E_ARG, "surrogate_fused_tc: blend needs A and B");
  int rc = tcf::check_pool(src_kind, pool, ld_pool, d, "surrogate_fused_tc: bad pool");
  if (rc) return rc;
  if (!tcf::aligned16(Ht)) return fail(ONMF_E_ARG, "surrogate_fused_tc: Ht must be 16-byte aligned");
  if (!workspace || workspace_bytes < onmf_surrogate_fused_tc_workspace(n, k, d)) return fail(ONMF_E_WORKSPACE, "surrogate_fused_tc: workspace too small");
  if ((uintptr_t)workspace % 16) return fail(ONMF_E_ARG, "surrogate_fused_tc: workspace must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  int nt, sp; long long per;
  tcf::sur_plan(n, k, d, &nt, &sp, &per);
  const int mrows = cdiv(k, 128) * 128;
  float* part = (float*)workspace;
  const long long items = (long long)nt * sp;
  if (n == 0) {
    ONMF_CUDA(cudaMemsetAsync(part, 0, (size_t)items * mrows * tcf::SurCfg::BN * sizeof(float), st));
  } else {
    tcf::PoolView X{pool, ld_pool, (const long long*)idx, n_pool, (float)scale};
    if (src_kind == ONMF_F32) rc = tcf::launch_sur<float>((const float*)Ht, X, n, k, d, nt, sp, per, part, st);
    else if (src_kind == ONMF_STORE_U8) rc = tcf::launch_sur<unsigned char>((const float*)Ht, X, n, k, d, nt, sp, per, part, st);
    else rc = tcf::launch_sur<__half>((const float*)Ht, X, n, k, d, nt, sp, per, part, st);
    if (rc) return rc;
  }
  return tcf::sur_reduce(part, nt, sp, mrows, k, d, P, blend, w, w_dev, A, B, st);
}

// ---- the same two products on a patch minibatch (PatchView loaders) ----
extern "C" int onmf_cov_fused_tc_patches(const onmf_patch_minibatch* pm, const void* W_hi, const void* W_lo, int k, void* Ct, void* stream) {
  int rc = tcf::check_patches(pm, "cov_fused_tc_patches: bad patch minibatch");
  if (rc) return rc;
  const int d = pm->p * pm->p * pm->C;
  if (!W_hi || !W_lo || !Ct || !onmf_fused_tc_supported(k, d)) return fail(ONMF_E_ARG, "cov_fused_tc_patches: bad argument / unsupported shape");
  if (!tcf::aligned16(W_hi) || !tcf::aligned16(W_lo) || !tcf::aligned16(Ct)) return fail(ONMF_E_ARG, "cov_fused_tc_patches: W_hi / W_lo / Ct must be 16-byte aligned");
  if (pm->n == 0) return ONMF_OK;
  CUtensorMap mh, ml;
  if ((rc = tcf::make_map_mn(&mh, (const float*)W_hi, k, d, k, 32))) return rc;
  if ((rc = tcf::make_map_mn(&ml, (const float*)W_lo, k, d, k, 32))) return rc;
  const tcf::PatchView X = tcf::patch_view(pm);
  cudaStream_t st = (cudaStream_t)stream;
  if (pm->kind == ONMF_F32) return tcf::dispatch_cov<float>(mh, ml, X, pm->n, d, k, (float*)Ct, st);
  return tcf::dispatch_cov<unsigned char>(mh, ml, X, pm->n, d, k, (float*)Ct, st);
}

extern "C" int onmf_surrogate_fused_tc_patches(const void* Ht, const onmf_patch_minibatch* pm, int k, void* P, int blend, double w,
                                               const double* w_dev, void* A, void* B, void* workspace, size_t workspace_bytes,
                                               void* stream) {
  int rc = tcf::check_patches(pm, "surrogate_fused_tc_patches: bad patch minibatch");
  if (rc) return rc;
  const int d = pm->p * pm->p * pm->C;
  const long long n = pm->n;
  if (!Ht || !onmf_fused_tc_supported(k, d)) return fail(ONMF_E_ARG, "surrogate_fused_tc_patches: bad argument / unsupported shape");
  if (!P && !blend) return fail(ONMF_E_ARG, "surrogate_fused_tc_patches: nothing to write (P == NULL and blend == 0)");
  if (blend && (!A || !B)) return fail(ONMF_E_ARG, "surrogate_fused_tc_patches: blend needs A and B");
  if (!tcf::aligned16(Ht)) return fail(ONMF_E_ARG, "surrogate_fused_tc_patches: Ht must be 16-byte aligned");
  if (!workspace || workspace_bytes < onmf_surrogate_fused_tc_workspace(n, k, d)) return fail(ONMF_E_WORKSPACE, "surrogate_fused_tc_patches: workspace too small");
  if ((uintptr_t)workspace % 16) return fail(ONMF_E_ARG, "surrogate_fused_tc_patches: workspace must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  int nt, sp; long long per;
  tcf::sur_plan(n, k, d, &nt, &sp, &per);
  const int mrows = cdiv(k, 128) * 128;
  float* part = (float*)workspace;
  if (n == 0) {
    ONMF_CUDA(cudaMemsetAsync(part, 0, (size_t)nt * sp * mrows * tcf::SurCfg::BN * sizeof(float), st));
  } else {
    const tcf::PatchView X = tcf::patch_view(pm);
    if (pm->kind == ONMF_F32) rc = tcf::launch_sur<float>((const float*)Ht, X, n, k, d, nt, sp, per, part, st);
    else rc = tcf::launch_sur<unsigned char>((const float*)Ht, X, n, k, d, nt, sp, per, part, st);
    if (rc) return rc;
  }
  return tcf::sur_reduce(part, nt, sp, mrows, k, d, P, blend, w, w_dev, A, B, st);
}
