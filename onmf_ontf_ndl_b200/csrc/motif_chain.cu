// ------------------------------------------------------------------------------------------------
// NDL motif embeddings on the device (DESIGN.md §0 f.5): batched Glauber chains of homomorphisms of the path
// 0 - 1 - ... - kk-1 into a symmetric CSR graph -- the MCMC of network_reconstruction_nx.py (tree_sample,
// get_single_patch_glauber) run as thousands of independent chains instead of one host walk.  The chain's law depends
// only on the graph, so every chain samples the same distribution; one warp advances one chain (lane q holds x[q]).
//
// Randomness is counter-based (Philox4x32-10, common.cuh; no cuRAND), keyed by the seed and addressed by (global step,
// global chain index), so a chain's trajectory does not depend on the launch shape, on n_chains, or on how a run is split
// into calls.  oracle/motif_chain.py restates both kernels in numpy bit for bit.
// ------------------------------------------------------------------------------------------------
#include <mutex>

#include "common.cuh"

namespace onmf {

// tree_sample of a path, one thread per chain: root uniform over the nodes with a neighbour (redrawn from counter
// (0, a, c, 1), a = 1, 2, ... while it has none), then x[q] uniform in N(x[q-1]) from counter (q, 0, c, 1).
__global__ void motif_chain_init_kernel(const long long* __restrict__ rowptr, const int* __restrict__ colidx, unsigned n_nodes,
                                        int kk, long long n_chains, unsigned chain0, uint2 key, int* __restrict__ state) {
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_chains) return;
  const unsigned cg = chain0 + (unsigned)c;
  int u = (int)__umulhi(philox4x32_10(make_uint4(0u, 0u, cg, 1u), key).x, n_nodes);
  for (unsigned a = 1; __ldg(rowptr + u + 1) == __ldg(rowptr + u); ++a)     // the caller checked the graph has an edge
    u = (int)__umulhi(philox4x32_10(make_uint4(0u, a, cg, 1u), key).x, n_nodes);
  int* x = state + c * kk;
  x[0] = u;
  for (int q = 1; q < kk; ++q) {
    const long long base = __ldg(rowptr + u);
    const unsigned deg = (unsigned)(__ldg(rowptr + u + 1) - base);
    if (deg) u = __ldg(colidx + base + __umulhi(philox4x32_10(make_uint4((unsigned)q, 0u, cg, 1u), key).x, deg));
    x[q] = u;
  }
}

// *bad = 1 when a state names a node outside [0, n_nodes) or a consecutive pair that is not an edge; one thread per (c, q).
__global__ void motif_chain_check_kernel(const long long* __restrict__ rowptr, const int* __restrict__ colidx, int n_nodes, int kk,
                                         long long n_chains, const int* __restrict__ state, unsigned* __restrict__ bad) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_chains * kk) return;
  const int q = (int)(idx % kk);
  const int u = state[idx];
  if ((unsigned)u >= (unsigned)n_nodes) { *bad = 1u; return; }
  if (q == kk - 1) return;
  const int v = state[idx + 1];
  if ((unsigned)v >= (unsigned)n_nodes) return;                 // reported by its own thread
  const long long base = __ldg(rowptr + u);
  const int len = (int)(__ldg(rowptr + u + 1) - base);
  int lo = 0, hi = len;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(colidx + base + mid) < v) lo = mid + 1;
    else hi = mid;
  }
  if (lo >= len || __ldg(colidx + base + lo) != v) *bad = 1u;
}

// lower bound of v in row[0, len)
__device__ __forceinline__ bool row_contains(const int* __restrict__ row, int len, int v) {
  int lo = 0, hi = len;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(row + mid) < v) lo = mid + 1;
    else hi = mid;
  }
  return lo < len && __ldg(row + lo) == v;
}

// One warp per chain, lane q holds x[q].  Step t: site i = mulhi(word0, kk); S = N(x[i-1]) & N(x[i+1]) (one row at the ends),
// x[i] <- S[mulhi(word1, |S|)].  An interior S is found by the lanes striding over the shorter row and binary-searching the
// longer one; ballot + popcount give |S| and the rank of every hit, so the chosen element does not depend on timing.
__global__ void __launch_bounds__(256) motif_chain_kernel(const long long* __restrict__ rowptr, const int* __restrict__ colidx, int kk,
                                                          long long n_chains, unsigned chain0, uint2 key, unsigned long long step0,
                                                          long long n_samples, long long sps, int* __restrict__ state,
                                                          int* __restrict__ out) {
  const long long c = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (c >= n_chains) return;                                    // warp-uniform
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const unsigned cg = chain0 + (unsigned)c;
  int x = lane < kk ? state[c * kk + lane] : 0;
  unsigned long long t = step0;
  for (long long s = 0; s < n_samples; ++s) {
    for (long long k = 0; k < sps; ++k) {
      ++t;
      const uint4 w = philox4x32_10(make_uint4((unsigned)t, (unsigned)(t >> 32), cg, 0u), key);
      const int i = (int)__umulhi(w.x, (unsigned)kk);
      const int xi = __shfl_sync(FULL, x, i);
      const int a = __shfl_sync(FULL, x, i == 0 ? 1 : i - 1);
      const int b = __shfl_sync(FULL, x, i == kk - 1 ? kk - 2 : i + 1);
      int v = xi;
      if (i == 0 || i == kk - 1) {
        const long long base = __ldg(rowptr + a);
        const unsigned deg = (unsigned)(__ldg(rowptr + a + 1) - base);
        if (deg) v = __ldg(colidx + base + __umulhi(w.y, deg));
      } else {
        const long long ba = __ldg(rowptr + a), bb = __ldg(rowptr + b);
        const int la = (int)(__ldg(rowptr + a + 1) - ba), lb = (int)(__ldg(rowptr + b + 1) - bb);
        const bool a_short = la <= lb;
        const int* srow = colidx + (a_short ? ba : bb);
        const int* lrow = colidx + (a_short ? bb : ba);
        const int ls = a_short ? la : lb, ll = a_short ? lb : la;
        unsigned m = 0, mask = 0;
        int e = 0;
        for (int j0 = 0; j0 < ls; j0 += 32) {                   // |S|
          const int j = j0 + lane;
          e = j < ls ? __ldg(srow + j) : 0;
          mask = __ballot_sync(FULL, j < ls && row_contains(lrow, ll, e));
          m += __popc(mask);
        }
        if (m) {
          unsigned r = __umulhi(w.y, m);
          if (ls > 32) {                                        // find the stride holding hit r
            for (int j0 = 0;; j0 += 32) {
              const int j = j0 + lane;
              e = j < ls ? __ldg(srow + j) : 0;
              mask = __ballot_sync(FULL, j < ls && row_contains(lrow, ll, e));
              const unsigned h = __popc(mask);
              if (r < h) break;
              r -= h;
            }
          }
          v = __shfl_sync(FULL, e, __fns(mask, 0, (int)r + 1));
        }
      }
      if (lane == i) x = v;
    }
    if (lane < kk) out[(s * n_chains + c) * kk + lane] = x;
  }
  if (lane < kk) state[c * kk + lane] = x;
}

__device__ unsigned g_motif_bad;     // validation flag of onmf_motif_chain (one per device; calls are serialised by a host lock)
static std::mutex g_motif_lock;

static int chain_args(const int64_t* rowptr, const int32_t* colidx, int64_t n_nodes, int kk, int64_t n_chains, int64_t chain0,
               const int32_t* state, const char* what) {
  if (!rowptr || !colidx || !state || n_nodes <= 0 || n_nodes > INT32_MAX || kk < 2 || n_chains <= 0 || chain0 < 0 ||
      chain0 + n_chains > (int64_t(1) << 32))
    return fail(ONMF_E_ARG, what);
  if (kk > 32) return fail(ONMF_E_UNSUPPORTED, "motif_chain: kk > 32 (one warp holds a state)");
  return ONMF_OK;
}

}  // namespace onmf

using namespace onmf;

extern "C" int onmf_motif_chain_init(const int64_t* rowptr, const int32_t* colidx, int64_t n_nodes, int kk, int64_t n_chains,
                                     int64_t chain0, uint64_t seed, int32_t* state, void* stream) {
  int rc = chain_args(rowptr, colidx, n_nodes, kk, n_chains, chain0, state, "motif_chain_init: bad argument");
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  long long nnz = 0;                                           // a graph without an edge has no homomorphism of a path
  ONMF_CUDA(cudaMemcpyAsync(&nnz, rowptr + n_nodes, sizeof(nnz), cudaMemcpyDeviceToHost, st));
  ONMF_CUDA(cudaStreamSynchronize(st));
  if (nnz <= 0) return fail(ONMF_E_ARG, "motif_chain_init: the graph has no edge");
  const unsigned grid = (unsigned)cdiv<long long>(n_chains, 256);
  motif_chain_init_kernel<<<grid, 256, 0, st>>>((const long long*)rowptr, colidx, (unsigned)n_nodes, kk, n_chains,
                                                (unsigned)chain0, seed_key(seed), state);
  ONMF_LAUNCH_CHECK("motif_chain_init_kernel");
  return ONMF_OK;
}

extern "C" int onmf_motif_chain(const int64_t* rowptr, const int32_t* colidx, int64_t n_nodes, int kk, int64_t n_chains,
                                int64_t chain0, uint64_t seed, uint64_t step0, int64_t n_samples, int64_t steps_per_sample,
                                int32_t* state, int32_t* out, void* stream) {
  int rc = chain_args(rowptr, colidx, n_nodes, kk, n_chains, chain0, state, "motif_chain: bad argument");
  if (rc) return rc;
  if (!out || n_samples <= 0 || steps_per_sample <= 0) return fail(ONMF_E_ARG, "motif_chain: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  {
    // every state must be a homomorphism before a step reads the CSR through it
    std::lock_guard<std::mutex> lock(g_motif_lock);
    unsigned* bad = nullptr;
    unsigned host_bad = 0;
    ONMF_CUDA(cudaGetSymbolAddress((void**)&bad, g_motif_bad));
    ONMF_CUDA(cudaMemsetAsync(bad, 0, sizeof(unsigned), st));
    const long long tot = n_chains * (long long)kk;
    motif_chain_check_kernel<<<(unsigned)cdiv<long long>(tot, 256), 256, 0, st>>>((const long long*)rowptr, colidx, (int)n_nodes, kk,
                                                                                   n_chains, state, bad);
    ONMF_LAUNCH_CHECK("motif_chain_check_kernel");
    ONMF_CUDA(cudaMemcpyAsync(&host_bad, bad, sizeof(unsigned), cudaMemcpyDeviceToHost, st));
    ONMF_CUDA(cudaStreamSynchronize(st));
    if (host_bad) return fail(ONMF_E_ARG, "motif_chain: a state is not a homomorphism of the path into the graph");
  }
  const unsigned grid = (unsigned)cdiv<long long>(n_chains * 32, 256);
  motif_chain_kernel<<<grid, 256, 0, st>>>((const long long*)rowptr, colidx, kk, n_chains, (unsigned)chain0, seed_key(seed),
                                           (unsigned long long)step0, n_samples, steps_per_sample, state, out);
  ONMF_LAUNCH_CHECK("motif_chain_kernel");
  return ONMF_OK;
}
