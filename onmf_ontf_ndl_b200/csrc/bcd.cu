// K5 -- dictionary update: one Gauss-Seidel block-coordinate sweep over the k atoms.
//
// Replaces update_dict (reference src/ontf.py:91-115 == src/onmf.py:92-116):
//   for j in 0..k-1:  W[:,j] -= (1/(A[j,j]+1)) * (W A[:,j] - B[j,:]);  W[:,j] = max(W[:,j], 0);
//                     W[:,j] *= 1 / max(1, ||W[:,j]||_2)
//
// The sweep is sequential in j but separable over the d rows of W except for the column norm.  ONE
// thread-block cluster owns the whole dictionary: CTA r keeps a row slab of W resident in shared memory
// (global W is read once and written once per sweep), TPR lanes cooperate on one row's dot product with
// the current column of A, and the k column norms are cluster-wide reductions through distributed
// shared memory (every CTA pushes its partial sum of squares into every peer's slot, one
// barrier.cluster per atom, partials summed in rank order so all CTAs -- and all GPUs of a
// data-parallel run -- get bit-identical dictionaries).
#include <cooperative_groups.h>
#include <stdlib.h>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace onmf {

constexpr int BCD_MAX_CLUSTER = 16;

// ---- point-to-point cluster signalling (PTX): a remote store into a peer CTA's shared memory followed by a release-arrive
// on that peer's mbarrier; the peer's threads acquire-wait on their own mbarrier.  Lighter than barrier.cluster, which makes
// every thread of every CTA of the cluster rendezvous once per atom.
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void st_cluster(uint32_t raddr, float v) { asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(raddr), "f"(v) : "memory"); }
__device__ __forceinline__ void st_cluster(uint32_t raddr, double v) { asm volatile("st.shared::cluster.f64 [%0], %1;" ::"r"(raddr), "d"(v) : "memory"); }
__device__ __forceinline__ void mbar_init(uint32_t mbar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t rmbar) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(rmbar) : "memory");
}
// st.async: the value and the completion signal travel together (complete_tx on the destination CTA's mbarrier) -- no
// release fence on the sender (ncu of the release-arrive form: `membar` among the top stall reasons of the atom chain)
__device__ __forceinline__ void st_async_cluster(uint32_t raddr, float v, uint32_t rmbar) {
  asm volatile("st.async.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];" ::"r"(raddr), "r"(__float_as_uint(v)), "r"(rmbar) : "memory");
}
__device__ __forceinline__ void st_async_cluster(uint32_t raddr, double v, uint32_t rmbar) {
  asm volatile("st.async.shared::cluster.mbarrier::complete_tx::bytes.b64 [%0], %1, [%2];" ::"r"(raddr), "l"(__double_as_longlong(v)), "r"(rmbar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t mbar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t mbar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(mbar), "r"(parity)
        : "memory");
  } while (!ok);
}

// REGW (fp32, k % 4 == 0, 4 <= tpr, k <= 32 * tpr, <= 512 threads, pitch ks a multiple of 4: e.g. 1024 x 128, not cfg5 --
// see bcd_plan_of): every lane keeps its share of its row of W
// -- up to eight 4-element chunks, chunk c = tl + tpr * i -- in REGISTERS next to the shared-memory slab (which stays the
// master copy for W[row, j] reads and the final store).  The per-atom dot product then reads only the column of A from
// shared memory, 16 bytes per load and the same address for every row of a warp (broadcast): 8 LDS.128 + 32 FFMA per lane
// instead of 64 scalar LDS + 32 FFMA (ncu of the shared-memory form: issue-active 45 % on the 16 SMs, ~600 warp-instructions
// per atom).  The one entry that changes per atom is written into the owner lane's register through a uniform switch.
template <typename T, bool REGW>
__global__ void __launch_bounds__(REGW ? 512 : 1024, 1) bcd_kernel(const T* __restrict__ Win, const T* __restrict__ A, const T* __restrict__ B,
                           T* __restrict__ Wout, int d, int k, int rpc, int ks, int tpr, int use_mbar) {
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const int csize = (int)cluster.num_blocks();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* Ws = reinterpret_cast<T*>(smem_raw);                  // rpc x ks slab
  T* aj = Ws + (size_t)rpc * ks;                           // 2 x k   (double-buffered column of A)
  T* warp_part = aj + 2 * k;                               // 32
  T* slots = warp_part + 32;                               // 2 x BCD_MAX_CLUSTER (written by peers)
  // (Ws, aj, warp_part, slots hold rpc*ks + 2k + 64 elements; the mbarrier sits at the next 8-byte boundary)
  const uint32_t mbar = (smem_u32(slots + 2 * BCD_MAX_CLUSTER) + 7u) & ~7u;
  // step table 1 / (A_jj + 1), one FP64 division per atom per CTA instead of one per thread per atom
  double* cs = reinterpret_cast<double*>((reinterpret_cast<uintptr_t>(slots + 2 * BCD_MAX_CLUSTER) + 7u) & ~(uintptr_t)7u) + 2;
  const int tid = threadIdx.x, nthr = blockDim.x;
  if (use_mbar && tid == 0) {                              // two mbarriers, one per atom parity (see the push below)
    // mode 1: csize release-arrives per phase; mode 2: one local arrive.expect_tx + csize st.async completions per phase
    mbar_init(mbar, use_mbar == 2 ? 1u : (uint32_t)csize);
    mbar_init(mbar + 8, use_mbar == 2 ? 1u : (uint32_t)csize);
    if (use_mbar == 2) {                                   // armed for atoms 0 and 1; re-armed for atom j+2 right after the wait of atom j,
      mbar_expect_tx(mbar, (uint32_t)(csize * sizeof(T)));        // so an expect_tx always precedes the completions it counts
      mbar_expect_tx(mbar + 8, (uint32_t)(csize * sizeof(T)));
    }
  }
  const int row0 = rank * rpc;
  const int nrows = max(0, min(rpc, d - row0));

  // slab load (coalesced along k)
  for (int idx = tid; idx < rpc * k; idx += nthr) {
    int r = idx / k, q = idx - r * k;
    Ws[(size_t)r * ks + q] = (r < nrows) ? Win[(size_t)(row0 + r) * k + q] : T(0);
  }
  for (int q = tid; q < k; q += nthr) aj[q] = A[(size_t)q * k + 0];
  for (int q = tid; q < k; q += nthr) cs[q] = 1.0 / ((double)A[(size_t)q * k + q] + 1.0);
  if (tid < 2 * BCD_MAX_CLUSTER) slots[tid] = T(0);
  cluster.sync();

  const int rl = tid / tpr;          // local row handled by this lane team
  const int tl = tid % tpr;          // lane inside the team
  const bool has_row = rl < nrows;
  const T* wrow = Ws + (size_t)rl * ks;

  // software pipeline over atoms: column j+1 of A (strided, L2 resident) and B[j+1, row] are requested one full atom
  // step before they are consumed, so their latency never sits on the k-step dependency chain
  constexpr int PF = 4;              // per-thread slice of a column of A (k <= PF * blockDim.x, else the tail is loaded directly)
  T pend[PF];
  T bnext = T(0);
  auto issue_col = [&](int col) {
    int i = 0;
    for (int q = tid; q < k && i < PF; q += nthr) pend[i++] = A[(size_t)q * k + col];
  };
  auto store_col = [&](int col, T* dst) {
    int i = 0;
    for (int q = tid; q < k && i < PF; q += nthr) dst[q] = pend[i++];
    for (int q = tid + PF * nthr; q < k; q += nthr) dst[q] = A[(size_t)q * k + col];
  };
  if (k > 1) issue_col(1);
  T bcur = has_row ? B[(size_t)0 * d + row0 + rl] : T(0);

  // W A[:,j] and B[j,:] are O(A_jj) while their difference is the O(1e-2 .. 1e-4) update.  Every lane sums its k/tpr
  // products in the working precision (two independent chains); the partial sums are combined across the team, and the
  // difference with B is formed, in FP64.  (Accumulating every product in FP64 costs two f32->f64 conversions per product
  // on the quarter-rate conversion pipe: measured 0.81 -> 1.32 ms at d=1024, k=256 -- ncu: XU pipe 46 % -- for no
  // measurable change of the dictionary; profiles/r2_other_kernels_ncu.md.)
  // team dot product of this row with column `a` of A (whatever the shared-memory slab holds at the moment)
  struct __align__(4 * sizeof(T)) V4 { T x, y, z, w; };
  constexpr int NCH = REGW ? 8 : 1;
  V4 wr[NCH];
  int ltpr = 0;                                              // log2(tpr)
  while ((1 << ltpr) < tpr) ++ltpr;
  if (REGW) {
#pragma unroll
    for (int i = 0; i < NCH; ++i) {
      const int c = tl + tpr * i;
      wr[i] = (has_row && 4 * c < k) ? *reinterpret_cast<const V4*>(wrow + 4 * c) : V4{T(0), T(0), T(0), T(0)};
    }
  }
  auto team_dot = [&](const T* a) -> double {
    if (REGW) {
      T a0 = T(0), a1 = T(0), a2 = T(0), a3 = T(0);
#pragma unroll
      for (int i = 0; i < NCH; ++i) {
        const int c = tl + tpr * i;
        if (4 * c < k) {
          const V4 av = *reinterpret_cast<const V4*>(a + 4 * c);
          a0 += wr[i].x * av.x; a1 += wr[i].y * av.y; a2 += wr[i].z * av.z; a3 += wr[i].w * av.w;
        }
      }
      double dsum = ((double)a0 + (double)a1) + ((double)a2 + (double)a3);
      for (int off = tpr >> 1; off > 0; off >>= 1) dsum += __shfl_xor_sync(0xffffffffu, dsum, off);
      return dsum;
    }
    T acc0 = T(0), acc1 = T(0);
    if (has_row) {
      int q = tl;
      for (; q + tpr < k; q += 2 * tpr) {
        acc0 += wrow[q] * a[q];
        acc1 += wrow[q + tpr] * a[q + tpr];
      }
      if (q < k) acc0 += wrow[q] * a[q];
    }
    double dsum = (double)acc0 + (double)acc1;
    for (int off = tpr >> 1; off > 0; off >>= 1) dsum += __shfl_xor_sync(0xffffffffu, dsum, off);
    return dsum;
  };
  double dot = team_dot(aj);                     // atom 0: nothing pending
  double cj = cs[0];                             // step of atom j

  // Software pipeline over atoms.  Column j of W is final only after the cluster-wide norm of its new entries; column
  // j+1's dot product needs it in ONE term (W[row, j] A[j, j+1]).  So the norm reduction of atom j (DSMEM pushes + one
  // split-phase barrier.cluster) is in flight while every team already forms atom j+1's dot product with the OLD entry
  // W[row, j] still in the slab; after the barrier that one term is exchanged: dot += (w_final - w_old) A[j, j+1].  Column j+1 of A (strided, L2 resident) and B[j+1, row] are requested one
  // full atom step before they are consumed.
  for (int j = 0; j < k; ++j) {
    const int par = j & 1;
    const T* a = aj + par * k;
    const T* an = aj + (par ^ 1) * k;
    if (j + 1 < k) {
      store_col(j + 1, aj + (par ^ 1) * k);       // requested during the previous step; nobody reads this buffer now
      if (has_row) bnext = B[(size_t)(j + 1) * d + row0 + rl];
    }
    if (j + 2 < k) issue_col(j + 2);
    T wnew = T(0), wold = T(0);
    if (has_row) {
      wold = wrow[j];
      const double v = (double)wold - cj * (dot - (double)bcur);
      wnew = v > 0.0 ? (T)v : T(0);
    }
    bcur = bnext;
    T sq = (has_row && tl == 0) ? wnew * wnew : T(0);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, off);
    if ((tid & 31) == 0) warp_part[tid >> 5] = sq;
    __syncthreads();                               // (also: column j+1 of A is now visible to every team)
    if (tid < 32) {
      T v = (tid < (nthr + 31) / 32) ? warp_part[tid] : T(0);
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
      if (use_mbar == 2) {
        if (tid < csize)
          st_async_cluster(mapa_u32(smem_u32(slots + par * BCD_MAX_CLUSTER + rank), (uint32_t)tid), v,
                           mapa_u32(mbar + 8u * (uint32_t)par, (uint32_t)tid));
      } else if (tid < csize) {
        if (use_mbar) {
          // slot (par, rank) of peer `tid`, then a release-arrive on that peer's mbarrier of this parity (csize arrivals per
          // atom).  Slot and mbarrier are reused at atom j+2: this CTA gets there only after it has seen the peer's arrival
          // for atom j+1, which the peer issues after its own phase j has completed (every arrival of atom j delivered)
          // and after all its threads have read the slots of atom j.  With ONE mbarrier an early arrival for atom j+1
          // could be counted into a peer's still incomplete phase j.
          st_cluster(mapa_u32(smem_u32(slots + par * BCD_MAX_CLUSTER + rank), (uint32_t)tid), v);
          mbar_arrive_remote(mapa_u32(mbar + 8u * (uint32_t)par, (uint32_t)tid));
        } else {
          T* peer = cluster.map_shared_rank(slots, tid);
          peer[par * BCD_MAX_CLUSTER + rank] = v;
        }
      }
    }
    if (!use_mbar) cluster.barrier_arrive();       // release: the pushes above are visible to whoever passes the wait
    // ---- in the shadow of the reduction: atom j+1's dot product without its j-th term, and its step ----
    double pdot = 0.0;
    if (j + 1 < k) {
      pdot = team_dot(an);                         // (the team's lanes share a warp: these reads precede the write below)
      cj = cs[j + 1];
    }
    if (use_mbar) {
      mbar_wait(mbar + 8u * (uint32_t)par, (uint32_t)((j >> 1) & 1));
      if (use_mbar == 2 && tid == 0 && j + 2 < k) mbar_expect_tx(mbar + 8u * (uint32_t)par, (uint32_t)(csize * sizeof(T)));
    } else {
      cluster.barrier_wait();
    }
    T tot = T(0);
    for (int r = 0; r < csize; ++r) tot += slots[par * BCD_MAX_CLUSTER + r];
    const T nrm = sqrt(tot);
    const T sc = T(1) / (nrm > T(1) ? nrm : T(1));
    const T wfin = sc * wnew;
    if (has_row && tl == 0) Ws[(size_t)rl * ks + j] = wfin;
    if (REGW) {
      const int cj4 = j >> 2;                                // chunk of entry j; owner lane cj4 % tpr, its chunk slot cj4 / tpr
      if (has_row && tl == (cj4 & (tpr - 1))) {
        switch (((cj4 >> ltpr) << 2) | (j & 3)) {           // (uniform)
#define ONMF_BCD_SET(I) \
          case 4 * I: wr[I < NCH ? I : 0].x = wfin; break;     \
          case 4 * I + 1: wr[I < NCH ? I : 0].y = wfin; break; \
          case 4 * I + 2: wr[I < NCH ? I : 0].z = wfin; break; \
          case 4 * I + 3: wr[I < NCH ? I : 0].w = wfin; break;
          ONMF_BCD_SET(0) ONMF_BCD_SET(1) ONMF_BCD_SET(2) ONMF_BCD_SET(3)
          ONMF_BCD_SET(4) ONMF_BCD_SET(5) ONMF_BCD_SET(6) ONMF_BCD_SET(7)
#undef ONMF_BCD_SET
          default: break;
        }
      }
    }
    if (j + 1 < k) dot = pdot + (has_row ? ((double)wfin - (double)wold) * (double)an[j] : 0.0);
    __syncwarp();
  }
  __syncthreads();
  for (int idx = tid; idx < nrows * k; idx += nthr) {
    int r = idx / k, q = idx - r * k;
    Wout[(size_t)(row0 + r) * k + q] = Ws[(size_t)r * ks + q];
  }
  cluster.sync();                                  // no CTA leaves while a peer could still address its shared memory
}

// Small dictionaries (d <= 1024 rows, W and A together within one CTA's shared memory: BASELINE configs 1-4, every per-patch
// driver call): ONE CTA, one thread per row, no cluster and no global memory inside the atom loop.  The cluster kernel above
// pays ~2.3 us per atom even as a cluster of one (barrier.cluster + the L2 latency of the prefetched column of A on the
// k-step chain; bench.py --workload next: 57 us at d=100, k=25 -- the longest kernel of a cfg1 step); here W (row-padded to
// an odd pitch: conflict-free), A and the warp partials live in shared memory, B[j, row] rides a four-deep register ring,
// and an atom costs k multiply-adds per thread (four fp32 chains, combined and differenced with B in FP64 like above), one
// warp reduction and ONE __syncthreads (the partial-sum buffer alternates with the atom's parity).  Partials are summed in
// warp order by every thread: deterministic, bit-identical on every GPU of a data-parallel run.
template <typename T>
struct BcdVec;
template <>
struct BcdVec<float> {
  static constexpr int N = 4;
  typedef float4 type;
  static __device__ __forceinline__ void fma4(const float4& w, const float4& a, float (&acc)[4], int) {
    acc[0] += w.x * a.x; acc[1] += w.y * a.y; acc[2] += w.z * a.z; acc[3] += w.w * a.w;
  }
};
template <>
struct BcdVec<double> {
  static constexpr int N = 2;
  typedef double2 type;
  static __device__ __forceinline__ void fma4(const double2& w, const double2& a, double (&acc)[4], int c) {
    if (c & 1) { acc[2] += w.x * a.x; acc[3] += w.y * a.y; }
    else { acc[0] += w.x * a.x; acc[1] += w.y * a.y; }
  }
};

// shared-memory pitches of bcd_small_kernel: 16-byte chunks; an ODD number of chunks per row of W makes the 16-byte row
// reads of eight consecutive threads (one shared-memory wavefront) hit eight different bank groups
template <typename T>
static inline int bcd_small_ks(int k) {
  const int V = 16 / (int)sizeof(T);
  int ks = round_up(k, V);
  if (((ks / V) & 1) == 0) ks += V;
  return ks;
}
template <typename T>
static inline int bcd_small_ka(int k) { return round_up(k, 16 / (int)sizeof(T)); }

template <typename T>
__global__ void __launch_bounds__(1024, 1) bcd_small_kernel(const T* __restrict__ Win, const T* __restrict__ A, const T* __restrict__ B,
                                                            T* __restrict__ Wout, int d, int k, int ks, int ka) {
  typedef typename BcdVec<T>::type V;
  constexpr int VN = BcdVec<T>::N;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* Ws = reinterpret_cast<T*>(smem_raw);                  // d x ks, zero beyond column k
  T* At = Ws + (size_t)d * ks;                             // k x ka: At[j][q] = A[q][j] (column j of A, contiguous), zero padded
  T* part = At + (size_t)k * ka;                           // 2 x 32
  double* cjs = reinterpret_cast<double*>(part + 64);      // k: 1 / (A_jj + 1), off the atom chain (an FP64 division each)
  const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarp = nthr >> 5;
  for (int j = tid; j < k; j += nthr) cjs[j] = 1.0 / ((double)A[(size_t)j * k + j] + 1.0);
  for (int idx = tid; idx < d * ks; idx += nthr) {
    const int r = idx / ks, q = idx - r * ks;
    Ws[idx] = q < k ? Win[(size_t)r * k + q] : T(0);
  }
  for (int idx = tid; idx < k * ka; idx += nthr) {
    const int j = idx / ka, q = idx - j * ka;
    At[idx] = q < k ? A[(size_t)q * k + j] : T(0);
  }
  const bool has_row = tid < d;
  T bq[4];
#pragma unroll
  for (int s = 0; s < 4; ++s) bq[s] = (has_row && s < k) ? B[(size_t)s * d + tid] : T(0);
  __syncthreads();
  T* wrow = Ws + (size_t)(has_row ? tid : 0) * ks;
  const int nch = ka / VN;
  for (int j0 = 0; j0 < k; j0 += 4) {
#pragma unroll
    for (int s = 0; s < 4; ++s) {
      const int j = j0 + s;
      if (j < k) {                                         // (uniform)
        const int par = j & 1;
        T wnew = T(0);
        if (has_row) {
          T acc[4] = {T(0), T(0), T(0), T(0)};
          const V* wv = reinterpret_cast<const V*>(wrow);
          const V* av = reinterpret_cast<const V*>(At + (size_t)j * ka);
#pragma unroll 4
          for (int c = 0; c < nch; ++c) BcdVec<T>::fma4(wv[c], av[c], acc, c);
          const double dot = ((double)acc[0] + (double)acc[1]) + ((double)acc[2] + (double)acc[3]);
          const double cj = cjs[j];
          const double v = (double)wrow[j] - cj * (dot - (double)bq[s]);
          wnew = v > 0.0 ? (T)v : T(0);
          bq[s] = (j + 4 < k) ? B[(size_t)(j + 4) * d + tid] : T(0);
        }
        T sq = wnew * wnew;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, off);
        if (lane == 0) part[par * 32 + warp] = sq;
        __syncthreads();
        T tot = T(0);
        for (int w = 0; w < nwarp; ++w) tot += part[par * 32 + w];
        const T nrm = sqrt(tot);
        const T sc = T(1) / (nrm > T(1) ? nrm : T(1));
        if (has_row) wrow[j] = sc * wnew;
      }
    }
  }
  __syncthreads();
  for (int idx = tid; idx < d * k; idx += nthr) {
    const int r = idx / k, q = idx - r * k;
    Wout[idx] = Ws[(size_t)r * ks + q];
  }
}

template <typename T>
static size_t bcd_small_smem(int d, int k) {
  return ((size_t)d * bcd_small_ks<T>(k) + (size_t)k * bcd_small_ka<T>(k) + 64) * sizeof(T) + (size_t)k * sizeof(double) + 8;
}

template <typename T>
static bool bcd_small_fits(int d, int k) {
  static const int off = [] { const char* e = getenv("ONMF_BCD_SMALL"); return (e && atoi(e) == 0) ? 1 : 0; }();   // (A/B runs)
  return !off && d <= 1024 && bcd_small_smem<T>(d, k) <= (size_t)max_smem_optin() - 1024;
}

// Fallback for dictionaries that do not fit one cluster's shared memory (d*k beyond ~0.9 M fp32 / 0.45 M fp64 entries, e.g.
// joint unfoldings of large tensors): a cooperative grid keeps W in global memory (L2 resident), every CTA owns a row
// slab -- rows are only ever read and written by their owner, the sweep is row-separable -- and the column norm is a
// fixed-order sum of per-CTA partials exchanged through global memory with ONE grid.sync() per atom.
template <typename T>
__global__ void __launch_bounds__(256) bcd_global_kernel(const T* __restrict__ Win, const T* __restrict__ A, const T* __restrict__ B,
                                                         T* __restrict__ Wout, int d, int k, int rpb, T* __restrict__ partials) {
  cg::grid_group grid = cg::this_grid();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* aj = reinterpret_cast<T*>(smem_raw);              // k     column j of A
  T* wn = aj + k;                                      // rpb   the slab's new (unnormalised) column j
  T* warp_part = wn + rpb;                             // 8
  __shared__ T tot_s;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = blockDim.x >> 5;
  const int nb = gridDim.x;
  const int row0 = blockIdx.x * rpb;
  const int nrows = max(0, min(rpb, d - row0));
  if (Win != Wout)
    for (long long idx = tid; idx < (long long)nrows * k; idx += blockDim.x) Wout[(size_t)row0 * k + idx] = Win[(size_t)row0 * k + idx];
  __syncthreads();
  for (int j = 0; j < k; ++j) {
    const int par = j & 1;
    for (int q = tid; q < k; q += blockDim.x) aj[q] = A[(size_t)q * k + j];
    __syncthreads();
    const double c = 1.0 / ((double)aj[j] + 1.0);
    T sq = T(0);
    for (int r = warp; r < nrows; r += nwarp) {        // one warp per row, rows of a warp in increasing order
      const T* wrow = Wout + (size_t)(row0 + r) * k;
      double dot = 0.0;                                  // FP64 accumulation: see bcd_kernel
      for (int q = lane; q < k; q += 32) dot += (double)wrow[q] * (double)aj[q];
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, off);
      const double vd = (double)wrow[j] - (double)c * (dot - (double)B[(size_t)j * d + row0 + r]);
      const T v = vd > 0.0 ? (T)vd : T(0);
      if (lane == 0) { wn[r] = v; sq += v * v; }
    }
    if (lane == 0) warp_part[warp] = sq;
    __syncthreads();
    if (tid == 0) {
      T v = T(0);
      for (int w = 0; w < nwarp; ++w) v += warp_part[w];
      partials[(size_t)par * nb + blockIdx.x] = v;
    }
    grid.sync();
    if (warp == 0) {                                   // fixed-order total: lane-strided partial sums, then a shuffle tree
      T v = T(0);
      for (int b = lane; b < nb; b += 32) v += partials[(size_t)par * nb + b];
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
      if (lane == 0) tot_s = v;
    }
    __syncthreads();
    const T nrm = sqrt(tot_s);
    const T sc = T(1) / (nrm > T(1) ? nrm : T(1));
    for (int r = tid; r < nrows; r += blockDim.x) Wout[(size_t)(row0 + r) * k + j] = sc * wn[r];
    __syncthreads();
  }
}

template <typename T>
static bool cluster_fits(int d, int k) {
  const size_t smem_cap = (size_t)max_smem_optin() - 1024;
  const int rpc = cdiv(d, BCD_MAX_CLUSTER);
  if (rpc > 1024) return false;
  int tpr = 32;
  while (tpr > 1 && rpc * tpr > 1024) tpr >>= 1;
  while (tpr > 1 && tpr * 2 > k) tpr >>= 1;
  const int ks = round_up(k, 32) + (tpr < 32 ? tpr : 1);
  return ((size_t)rpc * ks + 2 * (size_t)k + 32 + 2 * BCD_MAX_CLUSTER) * sizeof(T) + 32 + (size_t)k * 8 <= smem_cap;
}

// Every decision of the launcher in one host function (onmf_update_dict_plan exposes it): which kernel, cluster / grid
// size, rows per CTA, lanes per row, slab pitch, register form, signalling form and dynamic shared memory.  Reads the
// A/B switches ONMF_BCD_SMALL / _TPR / _REGW / _MBAR (once per process) and the device limits (the B200's 227 KB and 148
// SMs when no device is visible).  Returns ONMF_E_UNSUPPORTED when no kernel takes the shape.
template <typename T>
static int bcd_plan_of(int d, int k, onmf_bcd_plan* p) {
  *p = onmf_bcd_plan{};
  if (bcd_small_fits<T>(d, k)) {
    p->kind = ONMF_BCD_KIND_SMALL;
    p->ctas = 1;
    p->rows_per_cta = d;
    p->tpr = 1;
    p->ks = bcd_small_ks<T>(k);
    p->threads = round_up(d, 32);
    p->smem = bcd_small_smem<T>(d, k);
    return ONMF_OK;
  }
  const size_t smem_cap = (size_t)max_smem_optin() - 1024;
  if (cluster_fits<T>(d, k)) {
    // smallest power-of-two cluster whose slabs fit; prefer <= 128 rows per CTA so several lanes share a row
    for (int cs = 1; cs <= BCD_MAX_CLUSTER; cs *= 2) {
      const int rpc = cdiv(d, cs);
      int tpr = 32;
      while (tpr > 1 && rpc * tpr > 512) tpr >>= 1;    // 512 threads per CTA: 16 warps to synchronise per atom (measured 9 % faster than 1024)
      while (tpr > 1 && tpr * 2 > k) tpr >>= 1;
      static const int tpr_cap = [] { const char* e = getenv("ONMF_BCD_TPR"); return e ? atoi(e) : 0; }();   // (experiments)
      while (tpr_cap > 0 && tpr > tpr_cap) tpr >>= 1;
      const int ks = round_up(k, 32) + (tpr < 32 ? tpr : 1);
      const size_t smem = ((size_t)rpc * ks + 2 * (size_t)k + 32 + 2 * BCD_MAX_CLUSTER) * sizeof(T) + 32 + (size_t)k * 8;
      const bool fits = smem <= smem_cap && rpc <= 1024;
      if (!fits || (rpc > 128 && cs < 8)) continue;
      p->kind = ONMF_BCD_KIND_CLUSTER;
      p->ctas = cs;
      p->rows_per_cta = rpc;
      p->tpr = tpr;
      p->ks = ks;
      p->threads = min(round_up(rpc * tpr, 32), 1024);
      static const int regw_on = [] { const char* e = getenv("ONMF_BCD_REGW"); return (e && atoi(e) == 0) ? 0 : 1; }();   // (A/B runs)
      // the register form reads rows of the slab and the column of A (at rpc * ks) as 16-byte vectors: the pitch must be a
      // multiple of 4 floats, which rules out tpr = 32 (odd pitch, chosen for conflict-free scalar reads)
      p->regw = regw_on && sizeof(T) == 4 && k % 4 == 0 && tpr >= 4 && k <= 32 * tpr && p->threads <= 512 && ks % 4 == 0;
      static const int use_mbar = [] { const char* e = getenv("ONMF_BCD_MBAR"); return e ? atoi(e) : 2; }();   // (A/B runs: 0 barrier.cluster, 1 release-arrive, 2 st.async [default])
      p->mbar = use_mbar;
      p->smem = smem;
      return ONMF_OK;
    }
    // (a shape at the edge of one cluster's shared memory whose lane count at 512 threads needs a wider pitch than
    // cluster_fits assumed: the cooperative grid below takes it)
  }
  int nb = num_sms();
  if (nb > d) nb = d;
  const int rpb = cdiv(d, nb);
  p->kind = ONMF_BCD_KIND_GRID;
  p->ctas = cdiv(d, rpb);
  p->rows_per_cta = rpb;
  p->tpr = 32;
  p->ks = k;
  p->threads = 256;
  p->smem = ((size_t)k + rpb + 8) * sizeof(T);
  if (p->smem > (size_t)max_smem_optin()) return fail(ONMF_E_UNSUPPORTED, "update_dict: dictionary too large (row slab exceeds shared memory)");
  return ONMF_OK;
}

template <typename T>
static int update_dict_t(const T* Win, const T* A, const T* B, int d, int k, T* Wout, void* ws, size_t ws_bytes, cudaStream_t st) {
  onmf_bcd_plan p;
  int rc = bcd_plan_of<T>(d, k, &p);
  if (rc) return rc;
  if (p.kind == ONMF_BCD_KIND_SMALL) {
    auto kern = bcd_small_kernel<T>;
    ONMF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
    kern<<<1, p.threads, p.smem, st>>>(Win, A, B, Wout, d, k, p.ks, bcd_small_ka<T>(k));
    ONMF_LAUNCH_CHECK("bcd_small_kernel");
    return ONMF_OK;
  }
  if (p.kind == ONMF_BCD_KIND_GRID) {
    int dev = 0, coop = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
    if (!coop) return fail(ONMF_E_UNSUPPORTED, "update_dict: dictionary too large for one cluster and no cooperative launch");
    if (!ws || ws_bytes < 2 * (size_t)num_sms() * sizeof(double))
      return fail(ONMF_E_WORKSPACE, "update_dict: this dictionary needs onmf_update_dict_ws with a workspace of onmf_update_dict_workspace bytes");
    auto kern = bcd_global_kernel<T>;
    ONMF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
    T* partials = (T*)ws;
    int rpb = p.rows_per_cta;
    void* args[] = {(void*)&Win, (void*)&A, (void*)&B, (void*)&Wout, (void*)&d, (void*)&k, (void*)&rpb, (void*)&partials};
    ONMF_CUDA(cudaLaunchCooperativeKernel((void*)kern, dim3(p.ctas), dim3(p.threads), args, p.smem, st));
    ++g_launches;
    return ONMF_OK;
  }
  const int cs = p.ctas;
  auto kern = p.regw ? bcd_kernel<T, sizeof(T) == 4> : bcd_kernel<T, false>;
  ONMF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
  if (cs > 8) ONMF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(cs);
  cfg.blockDim = dim3(p.threads);
  cfg.dynamicSmemBytes = p.smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cs;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  ONMF_CUDA(cudaLaunchKernelEx(&cfg, kern, Win, A, B, Wout, d, k, p.rows_per_cta, p.ks, p.tpr, p.mbar));
  ++g_launches;
  return ONMF_OK;
}

}  // namespace onmf

extern "C" size_t onmf_update_dict_workspace(int dtype, int d, int k) {
  using namespace onmf;
  if (d <= 0 || k <= 0) return 0;
  onmf_bcd_plan p;
  const int rc = dtype == ONMF_F64 ? bcd_plan_of<double>(d, k, &p) : bcd_plan_of<float>(d, k, &p);
  return (rc == ONMF_OK && p.kind == ONMF_BCD_KIND_GRID) ? 2 * (size_t)num_sms() * sizeof(double) : 0;
}

extern "C" int onmf_update_dict_plan(int dtype, int d, int k, onmf_bcd_plan* out) {
  using namespace onmf;
  if (!out || d <= 0 || k <= 0 || (dtype != ONMF_F32 && dtype != ONMF_F64)) return fail(ONMF_E_ARG, "update_dict_plan: bad argument");
  return dtype == ONMF_F64 ? bcd_plan_of<double>(d, k, out) : bcd_plan_of<float>(d, k, out);
}

extern "C" int onmf_update_dict_ws(int dtype, const void* W_in, const void* A, const void* B, int d, int k, void* W_out,
                                   void* workspace, size_t workspace_bytes, void* stream) {
  using namespace onmf;
  if (!W_in || !A || !B || !W_out || d <= 0 || k <= 0) return fail(ONMF_E_ARG, "update_dict: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == ONMF_F32)
    return update_dict_t<float>((const float*)W_in, (const float*)A, (const float*)B, d, k, (float*)W_out, workspace, workspace_bytes, st);
  if (dtype == ONMF_F64)
    return update_dict_t<double>((const double*)W_in, (const double*)A, (const double*)B, d, k, (double*)W_out, workspace, workspace_bytes, st);
  return fail(ONMF_E_ARG, "update_dict: bad dtype");
}

extern "C" int onmf_update_dict(int dtype, const void* W_in, const void* A, const void* B, int d, int k, void* W_out,
                                void* stream) {
  return onmf_update_dict_ws(dtype, W_in, A, B, d, k, W_out, nullptr, 0, stream);
}
