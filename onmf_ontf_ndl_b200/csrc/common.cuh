// Shared helpers for the sm_100a kernels of libonmf_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/onmf_b200.h"

namespace onmf {

extern thread_local char g_err[512];
extern thread_local int g_lars_reserved_sms;     // SMs the persistent coder leaves free for concurrently running kernels
extern thread_local int g_lars_fast;             // 1: the warp-uniform fast first tier of the fp32 coder (k > 128) is used
extern thread_local long long g_launches;        // kernels launched by this host thread (every launch site counts itself)

inline int fail(int code, const char* msg) {
  snprintf(g_err, sizeof(g_err), "%s", msg);
  return code;
}

inline int cuda_fail(cudaError_t e, const char* where) {
  snprintf(g_err, sizeof(g_err), "%s: %s", where, cudaGetErrorString(e));
  return ONMF_E_CUDA;
}

#define ONMF_CUDA(call)                                            \
  do {                                                             \
    cudaError_t e__ = (call);                                      \
    if (e__ != cudaSuccess) return onmf::cuda_fail(e__, #call);    \
  } while (0)

#define ONMF_LAUNCH_CHECK(where)                                   \
  do {                                                             \
    cudaError_t e__ = cudaGetLastError();                          \
    if (e__ != cudaSuccess) return onmf::cuda_fail(e__, where);    \
    ++onmf::g_launches;                                            \
  } while (0)

inline int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

inline int max_smem_optin() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (n <= 0) n = 227 * 1024;
  }
  return n;
}

// Philox4x32-10 (Salmon et al., SC'11; the Random123 constants), the counter-based generator of the device chains
// (motif_chain.cu, ising_chain.cu); oracle/motif_chain.py restates it.
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r) { k.x += 0x9E3779B9u; k.y += 0xBB67AE85u; }
    const unsigned lo0 = 0xD2511F53u * c.x, hi0 = __umulhi(0xD2511F53u, c.x);
    const unsigned lo1 = 0xCD9E8D57u * c.z, hi1 = __umulhi(0xCD9E8D57u, c.z);
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
  }
  return c;
}

// the Philox key of a 64-bit seed
inline uint2 seed_key(uint64_t seed) { return make_uint2((unsigned)seed, (unsigned)(seed >> 32)); }

template <typename T>
__host__ __device__ inline T cdiv(T a, T b) { return (a + b - 1) / b; }

template <typename T>
__host__ __device__ inline T round_up(T a, T b) { return cdiv(a, b) * b; }

}  // namespace onmf
