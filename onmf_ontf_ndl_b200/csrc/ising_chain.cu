// ------------------------------------------------------------------------------------------------
// Ising lattices on the device (DESIGN.md §0 f.6): n_chains independent checkerboard heat-bath chains of the Ising model
// (J = 1, no field) on an H x W torus -- the trajectory source of the Ising driver (ising_simulator.ising_update), run as many
// chains instead of one host loop over sites.  Heat bath, not the reference's Metropolis: a checkerboard sweep with the
// Metropolis acceptance forces every site with sigma * s <= 0 to flip and does not sample the Gibbs law (DESIGN.md §7),
// while the heat bath sets each site from its conditional law, so one colour's sites are conditionally independent and a
// checkerboard sweep is exact.
//
// Randomness is Philox4x32-10 (common.cuh) addressed by (global sweep, global chain, Philox group of a colour), so the
// result depends on the counters only: the shared-memory and global forms, the launch shape, n_chains and the split of a
// run into calls give the same bits.  oracle/ising_chain.py restates both entry points in numpy.
// ------------------------------------------------------------------------------------------------
#include <math.h>

#include <algorithm>

#include "common.cuh"

namespace onmf {

struct IsingThr { unsigned v[5]; };     // thr[(s + 4) / 2], s the neighbour sum

// thr[(s + 4) / 2] by selects, so no address depends on a spin value (a state that is not +-1 gives +-1 spins, never a fault)
__device__ __forceinline__ unsigned thr_of(const IsingThr& thr, int s) {
  return s <= -4 ? thr.v[0] : s <= -2 ? thr.v[1] : s <= 0 ? thr.v[2] : s <= 2 ? thr.v[3] : thr.v[4];
}

// One Philox group (sites 4g .. 4g+3 of `colour`, in row-major order of that colour) of one lattice at sweep t: each site
// becomes +1 iff its word < thr[(s + 4) / 2].  The sites of a group never neighbour each other (same colour), so groups run
// concurrently; lat may be shared or global memory.
__device__ __forceinline__ void update_group(int8_t* lat, int H, int W, int half, int g, int colour, unsigned long long t,
                                             unsigned chain, uint2 key, const IsingThr& thr) {
  const uint4 w4 = philox4x32_10(make_uint4((unsigned)t, (unsigned)(t >> 32), chain, 2u * (unsigned)g + (unsigned)colour), key);
  const unsigned w[4] = {w4.x, w4.y, w4.z, w4.w};
  const int hw = W >> 1;
  const int m0 = 4 * g;
  int y = m0 / hw, j = m0 - y * hw;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    if (m0 + q < half) {
      const int x = 2 * j + ((y + colour) & 1);
      const int up = (y == 0 ? H - 1 : y - 1) * W, dn = (y == H - 1 ? 0 : y + 1) * W, row = y * W;
      const int s = lat[up + x] + lat[dn + x] + lat[row + (x == 0 ? W - 1 : x - 1)] + lat[row + (x == W - 1 ? 0 : x + 1)];
      lat[row + x] = w[q] < thr_of(thr, s) ? 1 : -1;
    }
    if (++j == hw) { j = 0; ++y; }
  }
}

// Shared-memory form: one CTA per chain (grid-striding over chains), the lattice resident in shared memory for every sweep
// of the call; HBM sees the initial state, the frames and the final state only.
template <typename T>
__global__ void __launch_bounds__(1024) ising_chain_smem_kernel(int H, int W, long long n_chains, unsigned chain0, uint2 key,
                                                                IsingThr thr, unsigned long long sweep0, long long n_samples,
                                                                long long sps, int8_t* __restrict__ state, T* __restrict__ out) {
  extern __shared__ int8_t lat[];
  const int HW = H * W, half = HW >> 1, groups = (half + 3) >> 2;
  for (long long c = blockIdx.x; c < n_chains; c += gridDim.x) {
    int8_t* st = state + c * (long long)HW;
    for (int i = threadIdx.x; i < HW; i += blockDim.x) lat[i] = st[i];
    __syncthreads();
    const unsigned cg = chain0 + (unsigned)c;
    unsigned long long t = sweep0;
    for (long long s = 0; s < n_samples; ++s) {
      for (long long k = 0; k < sps; ++k) {
        ++t;
        for (int colour = 0; colour < 2; ++colour) {
          for (int g = threadIdx.x; g < groups; g += blockDim.x) update_group(lat, H, W, half, g, colour, t, cg, key, thr);
          __syncthreads();
        }
      }
      T* o = out + (s * n_chains + c) * (long long)HW;
      for (int i = threadIdx.x; i < HW; i += blockDim.x) o[i] = (T)lat[i];
      __syncthreads();                                          // the frame is read before the next sweep writes
    }
    for (int i = threadIdx.x; i < HW; i += blockDim.x) st[i] = lat[i];
    __syncthreads();                                            // before the next chain's lattice overwrites lat
  }
}

// Global form, one half-sweep of every chain: one thread per (chain, Philox group), the lattices in place in `state`.
__global__ void __launch_bounds__(256) ising_half_sweep_kernel(int H, int W, long long n_chains, unsigned chain0, uint2 key,
                                                               IsingThr thr, unsigned long long t, int colour,
                                                               int8_t* __restrict__ state) {
  const int HW = H * W, half = HW >> 1, groups = (half + 3) >> 2;
  const long long total = n_chains * groups;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long c = i / groups;
    update_group(state + c * (long long)HW, H, W, half, (int)(i - c * groups), colour, t, chain0 + (unsigned)c, key, thr);
  }
}

// out[i] = state[i] for n entries (the frames of the global form)
template <typename T>
__global__ void __launch_bounds__(256) ising_frame_kernel(const int8_t* __restrict__ state, long long n, T* __restrict__ out) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = (T)state[i];
}

// Initial state: sweep 0 with every threshold 2^31, one thread per (chain, colour, Philox group).  No neighbour is read.
__global__ void __launch_bounds__(256) ising_init_kernel(int H, int W, long long n_chains, unsigned chain0, uint2 key,
                                                         int8_t* __restrict__ state) {
  const int HW = H * W, half = HW >> 1, groups = (half + 3) >> 2, hw = W >> 1;
  const long long total = n_chains * 2 * groups;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long c = i / (2 * groups);
    const int r = (int)(i - c * 2 * groups), colour = r / groups, g = r - colour * groups;
    const uint4 w4 = philox4x32_10(make_uint4(0u, 0u, chain0 + (unsigned)c, 2u * (unsigned)g + (unsigned)colour), key);
    const unsigned w[4] = {w4.x, w4.y, w4.z, w4.w};
    int8_t* lat = state + c * (long long)HW;
    const int m0 = 4 * g;
    int y = m0 / hw, j = m0 - y * hw;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      if (m0 + q < half) lat[y * W + 2 * j + ((y + colour) & 1)] = w[q] < 0x80000000u ? 1 : -1;
      if (++j == hw) { j = 0; ++y; }
    }
  }
}

static int ising_shape_ok(int H, int W) {
  return H >= 4 && W >= 4 && !(H & 1) && !(W & 1) && (int64_t)H * W < (int64_t(1) << 31);
}

static int ising_plan_of(int H, int W, onmf_ising_plan* p) {
  if (!ising_shape_ok(H, W)) return fail(ONMF_E_ARG, "ising_chain: H and W must be even, >= 4, with H*W < 2^31");
  const int64_t HW = (int64_t)H * W;
  const int groups = (int)((HW / 2 + 3) / 4);
  p->form = HW <= max_smem_optin() ? ONMF_ISING_FORM_SMEM : ONMF_ISING_FORM_GLOBAL;
  p->threads = p->form == ONMF_ISING_FORM_SMEM ? (int)std::min<int64_t>(1024, round_up<int64_t>(groups, 32)) : 256;
  p->smem = p->form == ONMF_ISING_FORM_SMEM ? (size_t)HW : 0;
  return ONMF_OK;
}

static int ising_args(int H, int W, int64_t n_chains, int64_t chain0, const int8_t* state, const char* what) {
  if (!state || !ising_shape_ok(H, W) || n_chains <= 0 || chain0 < 0 || chain0 + n_chains > (int64_t(1) << 32))
    return fail(ONMF_E_ARG, what);
  return ONMF_OK;
}

static unsigned grid_for(long long work, int threads) {
  return (unsigned)std::min<long long>(cdiv<long long>(work, threads), (long long)num_sms() * 32);
}

template <typename T>
static int ising_run(const onmf_ising_plan& p, int H, int W, int64_t n_chains, unsigned chain0, uint2 key, const IsingThr& thr,
                     uint64_t sweep0, int64_t n_samples, int64_t sps, int8_t* state, T* out, cudaStream_t st) {
  const long long HW = (long long)H * W;
  if (p.form == ONMF_ISING_FORM_SMEM) {
    auto kern = ising_chain_smem_kernel<T>;
    ONMF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
    int per_sm = 0;
    ONMF_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, p.threads, p.smem));
    const unsigned grid = (unsigned)std::min<long long>(n_chains, (long long)num_sms() * std::max(per_sm, 1));
    kern<<<grid, p.threads, p.smem, st>>>(H, W, n_chains, chain0, key, thr, sweep0, n_samples, sps, state, out);
    ONMF_LAUNCH_CHECK("ising_chain_smem_kernel");
    return ONMF_OK;
  }
  const int groups = (int)((HW / 2 + 3) / 4);
  unsigned long long t = sweep0;
  for (long long s = 0; s < n_samples; ++s) {
    for (long long k = 0; k < sps; ++k) {
      ++t;
      for (int colour = 0; colour < 2; ++colour) {
        ising_half_sweep_kernel<<<grid_for(n_chains * groups, p.threads), p.threads, 0, st>>>(H, W, n_chains, chain0, key, thr, t,
                                                                                            colour, state);
        ONMF_LAUNCH_CHECK("ising_half_sweep_kernel");
      }
    }
    ising_frame_kernel<T><<<grid_for(n_chains * HW, 256), 256, 0, st>>>(state, n_chains * HW, out + s * n_chains * HW);
    ONMF_LAUNCH_CHECK("ising_frame_kernel");
  }
  return ONMF_OK;
}

}  // namespace onmf

using namespace onmf;

extern "C" int onmf_ising_thresholds(double beta, uint32_t thr[5]) {
  if (!thr || !isfinite(beta)) return fail(ONMF_E_ARG, "ising_thresholds: beta must be finite");
  for (int j = 0; j < 5; ++j) {
    const double v = floor(4294967296.0 / (1.0 + exp(-2.0 * beta * (2 * j - 4))));
    thr[j] = v >= 4294967295.0 ? 0xFFFFFFFFu : (uint32_t)v;
  }
  return ONMF_OK;
}

extern "C" int onmf_ising_chain_plan(int H, int W, onmf_ising_plan* out) {
  if (!out) return fail(ONMF_E_ARG, "ising_chain_plan: null output");
  return ising_plan_of(H, W, out);
}

extern "C" int onmf_ising_chain_init(int H, int W, int64_t n_chains, int64_t chain0, uint64_t seed, int8_t* state, void* stream) {
  int rc = ising_args(H, W, n_chains, chain0, state, "ising_chain_init: bad argument");
  if (rc) return rc;
  const int groups = (int)(((int64_t)H * W / 2 + 3) / 4);
  ising_init_kernel<<<grid_for(n_chains * 2 * groups, 256), 256, 0, (cudaStream_t)stream>>>(H, W, n_chains, (unsigned)chain0,
                                                                                          seed_key(seed), state);
  ONMF_LAUNCH_CHECK("ising_init_kernel");
  return ONMF_OK;
}

extern "C" int onmf_ising_chain(int H, int W, int64_t n_chains, int64_t chain0, uint64_t seed, double beta, uint64_t sweep0,
                                int64_t n_samples, int64_t sweeps_per_sample, int8_t* state, void* out, int out_dtype,
                                void* stream) {
  int rc = ising_args(H, W, n_chains, chain0, state, "ising_chain: bad argument");
  if (rc) return rc;
  if (!out || n_samples <= 0 || sweeps_per_sample <= 0 || (out_dtype != ONMF_F32 && out_dtype != ONMF_F64) ||
      n_samples > INT64_MAX / sweeps_per_sample || (uint64_t)(n_samples * sweeps_per_sample) > UINT64_MAX - sweep0)
    return fail(ONMF_E_ARG, "ising_chain: bad argument");
  IsingThr thr;
  if ((rc = onmf_ising_thresholds(beta, thr.v))) return rc;
  onmf_ising_plan p;
  if ((rc = ising_plan_of(H, W, &p))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const uint2 key = seed_key(seed);
  if (out_dtype == ONMF_F32)
    return ising_run<float>(p, H, W, n_chains, (unsigned)chain0, key, thr, sweep0, n_samples, sweeps_per_sample, state,
                            (float*)out, st);
  return ising_run<double>(p, H, W, n_chains, (unsigned)chain0, key, thr, sweep0, n_samples, sweeps_per_sample, state,
                           (double*)out, st);
}
