// K2 / K4 -- dense products of the ONMF step, FP32/FP64 CUDA-core version.
//
//   cov   : Ct (n x k)       = Xt (n x d) . W (d x k)            [replaces dictionary @ X.T,
//                                                                  sklearn/_dict_learning.py:426]
//   gram  : G  (k x k)       = W^T W                              [_dict_learning.py:422]
//   surrogate partial sums:  P (k x (k+d)) = [ Ht^T Ht | Ht^T Xt ] [np.dot(H1.T,H1), np.dot(H1.T,X.T),
//                                                                  src/ontf.py:147-148]
//   blend : A = (1-w) A + w P[:, :k],  B = (1-w) B + w P[:, k:]
//
// This file is the exact-FP32 (and FP64 parity-mode) path: register-tiled 128 x BN x 16 CTA tiles,
// 8 x TN micro-tiles, split-K over the sample axis for the surrogate sums with a fixed-order
// (deterministic) second-pass reduction.  The tensor-core (tcgen05, 3xTF32) versions of the two large
// products live in gemm_tc.cu and are checked against this file.
#include "common.cuh"

namespace onmf {

constexpr int BM = 128, BK = 16, NT = 256;      // BM: the large row tile (64 and 32 for few rows / few CTAs, see launch_gemm)

// C[M x N] (+ split z) = op(A) . B ; A is (M x K) row-major (AKM=false) or (K x M) row-major (AKM=true);
// B is (K x N) row-major with leading dim ldb; C row-major with leading dim ldc.
template <typename T, int BN, bool AKM, int BM = 128>
__global__ void __launch_bounds__(NT) gemm_kernel(const T* __restrict__ A, int lda, const T* __restrict__ B, int ldb,
                                                  T* __restrict__ C, int ldc, long long M, int N, long long K,
                                                  long long kchunk, long long split_stride) {
  constexpr int TN = BN / 16, TM = BM / 16;
  __shared__ T As[BK][BM + 4];
  __shared__ T Bs[BK][BN + 4];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const long long m0 = (long long)blockIdx.x * BM;
  const int n0 = blockIdx.y * BN;
  const long long kbeg = (long long)blockIdx.z * kchunk;
  long long kend = kbeg + kchunk;
  if (kend > K) kend = K;
  T acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = T(0);

  for (long long k0 = kbeg; k0 < kend; k0 += BK) {
    if (AKM) {
      // A tile BK x BM from rows k0.., contiguous along M
      const int kk = tid >> 4, mm = (tid & 15) * TM;
      const long long kr = k0 + kk;
#pragma unroll
      for (int e = 0; e < TM; ++e) {
        long long m = m0 + mm + e;
        As[kk][mm + e] = (kr < kend && m < M) ? A[kr * lda + m] : T(0);
      }
    } else {
      // A tile BM x BK from row-major (M x K): thread -> (row, EK consecutive k)
      constexpr int TPR = NT / BM, EK = BK / TPR;
      const int row = tid / TPR, kq = (tid % TPR) * EK;
      const long long m = m0 + row;
#pragma unroll
      for (int e = 0; e < EK; ++e) {
        long long kr = k0 + kq + e;
        As[kq + e][row] = (m < M && kr < kend) ? A[m * lda + kr] : T(0);
      }
    }
    {
      const int kk = tid >> 4, nn = (tid & 15) * TN;
      const long long kr = k0 + kk;
#pragma unroll
      for (int e = 0; e < TN; ++e) {
        int nc = n0 + nn + e;
        Bs[kk][nn + e] = (kr < kend && nc < N) ? B[kr * ldb + nc] : T(0);
      }
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      T a[TM], b[TN];
#pragma unroll
      for (int i = 0; i < TM; ++i) a[i] = As[kk][ty * TM + i];
#pragma unroll
      for (int j = 0; j < TN; ++j) b[j] = Bs[kk][tx * TN + j];
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] += a[i] * b[j];
    }
    __syncthreads();
  }
  T* Cz = C + (size_t)blockIdx.z * split_stride;
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    long long m = m0 + ty * TM + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      int nc = n0 + tx * TN + j;
      if (nc < N) Cz[m * ldc + nc] = acc[i][j];
    }
  }
}

// out[i] = sum_z part[z][i] in fixed order z = 0..splits-1
template <typename T>
__global__ void split_reduce_kernel(const T* __restrict__ part, int splits, long long count, long long stride,
                                    T* __restrict__ out) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  T s = T(0);
  for (int z = 0; z < splits; ++z) s += part[(size_t)z * stride + i];
  out[i] = s;
}

template <typename T>
__global__ void blend_kernel(const T* __restrict__ P, int k, int d, T w, T* __restrict__ A, T* __restrict__ B) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long tot = (long long)k * (k + d);
  if (i >= tot) return;
  int r = (int)(i / (k + d)), c = (int)(i - (long long)r * (k + d));
  T p = P[i];
  T om = T(1) - w;
  if (c < k) {
    size_t o = (size_t)r * k + c;
    A[o] = om * A[o] + w * p;
  } else {
    size_t o = (size_t)r * d + (c - k);
    B[o] = om * B[o] + w * p;
  }
}

// same, blend weight read from device memory (the CUDA-graph form of the step: w = t^-beta changes every replay)
template <typename T>
__global__ void blend_dev_kernel(const T* __restrict__ P, int k, int d, const double* __restrict__ w_dev, T* __restrict__ A,
                                 T* __restrict__ B) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long tot = (long long)k * (k + d);
  if (i >= tot) return;
  const T w = (T)(*w_dev);
  int r = (int)(i / (k + d)), c = (int)(i - (long long)r * (k + d));
  T p = P[i];
  T om = T(1) - w;
  if (c < k) {
    size_t o = (size_t)r * k + c;
    A[o] = om * A[o] + w * p;
  } else {
    size_t o = (size_t)r * d + (c - k);
    B[o] = om * B[o] + w * p;
  }
}

template <typename T>
__global__ void axpby_kernel(long long count, T a, const T* __restrict__ x, T b, T* __restrict__ y) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) y[i] = a * x[i] + b * y[i];
}

template <typename T, bool AKM>
static int launch_gemm(const T* A, int lda, const T* B, int ldb, T* C, int ldc, long long M, int N, long long K,
                       int splits, long long split_stride, cudaStream_t st) {
  if (M <= 0 || N <= 0) return ONMF_OK;
  long long kchunk = round_up<long long>(cdiv<long long>(K, splits), BK);
  if (kchunk < BK) kchunk = BK;
  dim3 block(NT);
  const int bn = N <= 32 ? 32 : N <= 64 ? 64 : 128;
  // row tile: 32 / 64 rows when the product has no more (the surrogate sums of the small dictionaries: M = k <= 64 -- a
  // 128-row tile would compute 2-5 x the needed entries), 64 rows when 128-row tiles would leave SMs without a CTA.  The
  // order of the k-loop inside a CTA does not depend on the tile, so the results do not either.
  const long long ctas128 = cdiv<long long>(M, 128) * cdiv(N, bn) * splits;
  const int bm = M <= 32 ? 32 : (M <= 64 || ctas128 < num_sms()) ? 64 : 128;
  dim3 grid((unsigned)cdiv<long long>(M, bm), (unsigned)cdiv(N, bn), splits);
#define ONMF_GEMM_CASE(BN_, BM_)                                                                                       \
  if (bn == BN_ && bm == BM_) gemm_kernel<T, BN_, AKM, BM_><<<grid, block, 0, st>>>(A, lda, B, ldb, C, ldc, M, N, K, kchunk, split_stride);
  ONMF_GEMM_CASE(32, 32) ONMF_GEMM_CASE(32, 64) ONMF_GEMM_CASE(32, 128)
  ONMF_GEMM_CASE(64, 32) ONMF_GEMM_CASE(64, 64) ONMF_GEMM_CASE(64, 128)
  ONMF_GEMM_CASE(128, 32) ONMF_GEMM_CASE(128, 64) ONMF_GEMM_CASE(128, 128)
#undef ONMF_GEMM_CASE
  ONMF_LAUNCH_CHECK("gemm_kernel");
  return ONMF_OK;
}

static int pick_splits(long long n, int k, int d) {
  // enough CTAs to fill the GPU: tiles(M=k, N=k+d) * splits >= 2 * SMs, each split >= 64 samples (the small configurations
  // -- 1,000 to 16,384 samples, k <= 100 -- have one or two output tiles: with 256 samples per split they ran on 4-8 CTAs and
  // the two products took longer than the coder)
  long long tiles = cdiv(k, BM) * (cdiv(k, 128) + cdiv(d, 128));
  long long want = cdiv<long long>(2LL * num_sms(), tiles);
  long long cap = cdiv<long long>(n, 64);
  long long s = want < cap ? want : cap;
  if (s < 1) s = 1;
  if (s > 256) s = 256;
  return (int)s;
}

template <typename T>
static int surrogate_partial_t(const T* Ht, const T* Xt, long long n, int k, int d, T* P, T* ws, cudaStream_t st) {
  const int splits = pick_splits(n, k, d);
  const long long ldp = k + d;
  const long long stride = (long long)k * ldp;
  T* dst = splits == 1 ? P : ws;
  // [Ht^T Ht] -> columns 0..k-1 ; [Ht^T Xt] -> columns k..k+d-1 of the packed (k x (k+d)) buffer
  int rc = launch_gemm<T, true>(Ht, k, Ht, k, dst, (int)ldp, k, k, n, splits, stride, st);
  if (rc) return rc;
  rc = launch_gemm<T, true>(Ht, k, Xt, d, dst + k, (int)ldp, k, d, n, splits, stride, st);
  if (rc) return rc;
  if (splits > 1) {
    int threads = 256;
    split_reduce_kernel<T><<<(unsigned)cdiv<long long>(stride, threads), threads, 0, st>>>(ws, splits, stride, stride, P);
    ONMF_LAUNCH_CHECK("split_reduce_kernel");
  }
  return ONMF_OK;
}

// ------------------------------------------------------------------------------------------------
// FP64-accumulated Gram matrix of an fp32 (or fp64) dictionary.  The sparse coder inverts active blocks of G; an fp32
// G carries independent rounding errors of ~6e-8 per entry which the inverse amplifies by cond(G) (~4e5 on the early
// online dictionaries), whereas the exact Gram of the stored (fp32) W only sees cond(W) = sqrt(cond(G)).  So the Gram
// is accumulated and kept in FP64 (k x k doubles: 0.5 MB at k = 256), upper-triangle tiles only, mirrored on reduce.
// ------------------------------------------------------------------------------------------------
constexpr int G64_T = 64, G64_BK = 16;

template <typename Tin>
__global__ void __launch_bounds__(256) gram64_kernel(const Tin* __restrict__ W, int d, int k, int dchunk, int ntile,
                                                     double* __restrict__ part) {
  __shared__ double As[G64_BK][G64_T + 2];
  __shared__ double Bs[G64_BK][G64_T + 2];
  // linear tile id -> (bi <= bj)
  int t = blockIdx.x, bi = 0;
  while (t >= ntile - bi) { t -= ntile - bi; ++bi; }
  const int bj = bi + t;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int r0 = blockIdx.y * dchunk;
  int r1 = r0 + dchunk;
  if (r1 > d) r1 = d;
  double acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0;
  for (int rr = r0; rr < r1; rr += G64_BK) {
    {
      const int kk = tid >> 4, c4 = (tid & 15) * 4;
      const int r = rr + kk;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int ci = bi * G64_T + c4 + e, cj = bj * G64_T + c4 + e;
        As[kk][c4 + e] = (r < r1 && ci < k) ? (double)W[(size_t)r * k + ci] : 0.0;
        Bs[kk][c4 + e] = (r < r1 && cj < k) ? (double)W[(size_t)r * k + cj] : 0.0;
      }
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < G64_BK; ++kk) {
      double a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = As[kk][ty * 4 + i]; b[i] = Bs[kk][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] += a[i] * b[j];
    }
    __syncthreads();
  }
  double* out = part + (size_t)blockIdx.y * k * k;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int gi = bi * G64_T + ty * 4 + i;
    if (gi >= k) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int gj = bj * G64_T + tx * 4 + j;
      if (gj < k) out[(size_t)gi * k + gj] = acc[i][j];
    }
  }
}

// G64[i][j] = sum_z part[z][min-tile-ordered (i, j)] in fixed order; optional fp32 copy
__global__ void gram64_reduce_kernel(const double* __restrict__ part, int splits, int k, double* __restrict__ G64,
                                     float* __restrict__ G32) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= k * k) return;
  int i = idx / k, j = idx - i * k;
  // only tiles with bi <= bj were computed; inside a diagonal tile both orders exist and are bitwise equal
  const bool swap = (i / G64_T) > (j / G64_T);
  const size_t src = swap ? (size_t)j * k + i : (size_t)i * k + j;
  double s = 0.0;
  for (int z = 0; z < splits; ++z) s += part[(size_t)z * k * k + src];
  G64[idx] = s;
  if (G32) G32[idx] = (float)s;
}

static int gram64_splits(int d) {
  int s = d / 64;
  return s < 1 ? 1 : s > 16 ? 16 : s;
}

// surrogate loss read-out  tr(W A W^T) - 2 tr(W B) + tr(C)  (reference ising_reconstruction.py:133,164):
//   out[0] = <W^T W, A> = tr(W A W^T)   (the FP64 Gram of W is already maintained for the coder)
//   out[1] = tr(W B) = sum_{r,j} W[r,j] B[j,r]        out[2] = tr(C)
// One CTA, FP64 accumulation, fixed summation order (deterministic); the three sums are ~3e5 terms at cfg5.
template <typename T>
__global__ void __launch_bounds__(1024) surrogate_error_kernel(const T* __restrict__ W, const double* __restrict__ G64,
                                                               const T* __restrict__ A, const T* __restrict__ B,
                                                               const T* __restrict__ C, int d, int k, double* __restrict__ out) {
  __shared__ double red[3][32];
  double s0 = 0.0, s1 = 0.0, s2 = 0.0;
  for (int i = threadIdx.x; i < k * k; i += blockDim.x) s0 += G64[i] * (double)A[i];
  for (long long i = threadIdx.x; i < (long long)d * k; i += blockDim.x) {
    const int j = (int)(i / d), r = (int)(i - (long long)j * d);          // B is (k x d): coalesced along r
    s1 += (double)B[i] * (double)W[(size_t)r * k + j];
  }
  if (C != nullptr)
    for (int i = threadIdx.x; i < d; i += blockDim.x) s2 += (double)C[(size_t)i * d + i];
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    s0 += __shfl_xor_sync(0xffffffffu, s0, off);
    s1 += __shfl_xor_sync(0xffffffffu, s1, off);
    s2 += __shfl_xor_sync(0xffffffffu, s2, off);
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { red[0][warp] = s0; red[1][warp] = s1; red[2][warp] = s2; }
  __syncthreads();
  if (warp == 0) {
    const int nw = (blockDim.x + 31) / 32;
    s0 = lane < nw ? red[0][lane] : 0.0;
    s1 = lane < nw ? red[1][lane] : 0.0;
    s2 = lane < nw ? red[2][lane] : 0.0;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      s0 += __shfl_xor_sync(0xffffffffu, s0, off);
      s1 += __shfl_xor_sync(0xffffffffu, s1, off);
      s2 += __shfl_xor_sync(0xffffffffu, s2, off);
    }
    if (lane == 0) { out[0] = s0; out[1] = s1; out[2] = s2; }
  }
}

}  // namespace onmf

using namespace onmf;

extern "C" int onmf_gram(int dtype, const void* W, int d, int k, void* G, void* stream) {
  if (!W || !G || d <= 0 || k <= 0) return fail(ONMF_E_ARG, "gram: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == ONMF_F32) return launch_gemm<float, true>((const float*)W, k, (const float*)W, k, (float*)G, k, k, k, d, 1, 0, st);
  if (dtype == ONMF_F64) return launch_gemm<double, true>((const double*)W, k, (const double*)W, k, (double*)G, k, k, k, d, 1, 0, st);
  return fail(ONMF_E_ARG, "gram: bad dtype");
}

extern "C" size_t onmf_gram_f64_workspace(int d, int k) {
  if (d <= 0 || k <= 0) return 0;
  return (size_t)onmf::gram64_splits(d) * k * k * sizeof(double) + 256;
}

extern "C" int onmf_gram_f64(int dtype_in, const void* W, int d, int k, double* G64, float* G32, void* workspace,
                             size_t workspace_bytes, void* stream) {
  using namespace onmf;
  if (!W || !G64 || !workspace || d <= 0 || k <= 0) return fail(ONMF_E_ARG, "gram_f64: bad argument");
  if (workspace_bytes < onmf_gram_f64_workspace(d, k)) return fail(ONMF_E_WORKSPACE, "gram_f64: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  const int splits = gram64_splits(d);
  int dchunk = round_up(cdiv(d, splits), G64_BK);
  const int ntile = cdiv(k, G64_T);
  dim3 grid(ntile * (ntile + 1) / 2, splits);
  double* part = (double*)workspace;
  if (dtype_in == ONMF_F32) gram64_kernel<float><<<grid, 256, 0, st>>>((const float*)W, d, k, dchunk, ntile, part);
  else if (dtype_in == ONMF_F64) gram64_kernel<double><<<grid, 256, 0, st>>>((const double*)W, d, k, dchunk, ntile, part);
  else return fail(ONMF_E_ARG, "gram_f64: bad dtype");
  ONMF_LAUNCH_CHECK("gram64_kernel");
  gram64_reduce_kernel<<<cdiv(k * k, 256), 256, 0, st>>>(part, splits, k, G64, G32);
  ONMF_LAUNCH_CHECK("gram64_reduce_kernel");
  return ONMF_OK;
}

// ------------------------------------------------------------------------------------------------
// Spectral norm of a tall matrix M (n x k, sample-major): sqrt(lambda_max(M^T M)).  The stopping test of the reference's
// projected-gradient coder takes two of them per outer iteration (np.linalg.norm(., 2), src/onmf.py:265).
// M^T M comes from the FP64 Gram kernels above; lambda_max of the k x k matrix by repeated squaring in one CTA:
// B_0 = G / tr G, B_{m+1} = B_m^2 / tr(B_m^2) -- the dominant eigenspace takes over quadratically -- then the Rayleigh
// quotient of G at the column of B with the largest diagonal entry.  With SQ squarings, x = 1 - lambda_2/lambda_1,
// eps = (1 - x)^(2^SQ) and m eigenvalues at lambda_2 (m up to k - 1), the relative error of sqrt(lambda) is about
// (x / 2) m eps^2 / (1 + m eps^2) when the top eigenvector is flat: largest, ~ln k / 2^(SQ+3), at x ~ ln k / 2^(SQ+1).
// At SQ = 16 that reaches 1.3e-5 for k = 256 and 1.5e-5 for k = 512; SQ = 17 keeps every spectrum below 1e-5 for k <= 512
// (tests/test_pgd_coder_variants.py restates this kernel in numpy and runs those spectra on both).  The 17th squaring
// costs one more k^3 product: onmf_spectral_norm of a 4096 x k matrix 2.42 -> 2.57 ms at k = 64, 148 -> 157 ms at
// k = 256, 1184 -> 1258 ms at k = 512 (+6 %; B200, 1000 W power limit, CUDA events over 20-50 calls).
namespace onmf {
constexpr int LMAX_SQUARINGS = 17;
__global__ void __launch_bounds__(1024) lambda_max_kernel(const double* __restrict__ G, int k, double* __restrict__ b0,
                                                          double* __restrict__ b1, int squarings, double* __restrict__ out) {
  __shared__ double red[32];
  __shared__ double bc;
  __shared__ int best_col;
  const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31, warp = tid >> 5;
  auto block_sum = [&](double v) -> double {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    __syncthreads();                     // (red is free again)
    if (lane == 0) red[warp] = v;
    __syncthreads();
    if (warp == 0) {
      double t = lane < (nthr + 31) / 32 ? red[lane] : 0.0;
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) t += __shfl_xor_sync(0xffffffffu, t, off);
      if (lane == 0) bc = t;
    }
    __syncthreads();
    return bc;
  };
  double tr = 0.0;
  for (int i = tid; i < k; i += nthr) tr += G[(size_t)i * k + i];
  tr = block_sum(tr);
  if (!(tr > 0.0)) {                     // the zero matrix (or NaN input: propagate)
    if (tid == 0) *out = (tr == 0.0) ? 0.0 : tr;
    return;
  }
  double* cur = b0;
  double* nxt = b1;
  const double itr = 1.0 / tr;
  for (int idx = tid; idx < k * k; idx += nthr) cur[idx] = G[idx] * itr;
  __syncthreads();
  for (int m = 0; m < squarings; ++m) {
    double dsum = 0.0;
    for (int idx = tid; idx < k * k; idx += nthr) {
      const int i = idx / k, j = idx - i * k;
      const double* ri = cur + (size_t)i * k;
      const double* rj = cur + (size_t)j * k;      // (symmetric: column j is row j)
      double a0 = 0.0, a1 = 0.0;
      int q = 0;
      for (; q + 1 < k; q += 2) { a0 += ri[q] * rj[q]; a1 += ri[q + 1] * rj[q + 1]; }
      if (q < k) a0 += ri[q] * rj[q];
      const double v = a0 + a1;
      nxt[idx] = v;
      if (i == j) dsum += v;
    }
    const double t2 = block_sum(dsum);             // (its barriers also order the writes of nxt before the rescale)
    const double it2 = 1.0 / t2;
    for (int idx = tid; idx < k * k; idx += nthr) nxt[idx] *= it2;
    __syncthreads();
    double* sw = cur; cur = nxt; nxt = sw;
  }
  // x = the column with the largest diagonal entry (a vector of the dominant eigenspace); lambda = x^T G x / x^T x
  if (tid == 0) {
    int bcol = 0;
    double bd = -1.0;
    for (int i = 0; i < k; ++i) { const double dv = cur[(size_t)i * k + i]; if (dv > bd) { bd = dv; bcol = i; } }
    best_col = bcol;
  }
  __syncthreads();
  const double* x = cur + (size_t)best_col * k;
  double num = 0.0, den = 0.0;
  for (int i = tid; i < k; i += nthr) {
    const double* gi = G + (size_t)i * k;
    double gx = 0.0;
    for (int q = 0; q < k; ++q) gx += gi[q] * x[q];
    num += x[i] * gx;
    den += x[i] * x[i];
  }
  num = block_sum(num);
  den = block_sum(den);
  if (tid == 0) *out = sqrt(num / den);
}
}  // namespace onmf

extern "C" size_t onmf_spectral_norm_workspace(int64_t n, int k) {
  if (n <= 0 || k <= 0 || n > 0x7fffffffLL) return 0;
  return onmf_gram_f64_workspace((int)n, k) + 3 * (size_t)k * k * sizeof(double) + 256;
}

extern "C" int onmf_spectral_norm(int dtype, const void* M, int64_t n, int k, double* out, void* workspace, size_t workspace_bytes,
                                  void* stream) {
  using namespace onmf;
  if (!M || !out || !workspace || n <= 0 || k <= 0 || n > 0x7fffffffLL) return fail(ONMF_E_ARG, "spectral_norm: bad argument");
  if (workspace_bytes < onmf_spectral_norm_workspace(n, k)) return fail(ONMF_E_WORKSPACE, "spectral_norm: workspace too small");
  if ((uintptr_t)workspace % 256) return fail(ONMF_E_ARG, "spectral_norm: workspace must be 256-byte aligned");
  const size_t gws = round_up<size_t>(onmf_gram_f64_workspace((int)n, k), 256);
  double* G64 = reinterpret_cast<double*>((unsigned char*)workspace + gws);
  int rc = onmf_gram_f64(dtype, M, (int)n, k, G64, nullptr, workspace, gws, stream);
  if (rc) return rc;
  lambda_max_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(G64, k, G64 + (size_t)k * k, G64 + 2 * (size_t)k * k, LMAX_SQUARINGS, out);
  ONMF_LAUNCH_CHECK("lambda_max_kernel");
  return ONMF_OK;
}

extern "C" int onmf_cov(int dtype, const void* Xt, int64_t n, int d, const void* W, int k, void* Ct, void* stream) {
  if (!Xt || !W || !Ct || n < 0 || d <= 0 || k <= 0) return fail(ONMF_E_ARG, "cov: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == ONMF_F32) return launch_gemm<float, false>((const float*)Xt, d, (const float*)W, k, (float*)Ct, k, n, k, d, 1, 0, st);
  if (dtype == ONMF_F64) return launch_gemm<double, false>((const double*)Xt, d, (const double*)W, k, (double*)Ct, k, n, k, d, 1, 0, st);
  return fail(ONMF_E_ARG, "cov: bad dtype");
}

extern "C" size_t onmf_surrogate_workspace(int dtype, int64_t n, int k, int d) {
  if (n < 0 || k <= 0 || d <= 0) return 0;
  size_t tsz = dtype == ONMF_F64 ? 8 : 4;
  return (size_t)pick_splits(n, k, d) * (size_t)k * (size_t)(k + d) * tsz + 256;
}

extern "C" int onmf_surrogate_partial(int dtype, const void* Ht, const void* Xt, int64_t n, int k, int d, void* P,
                                      void* workspace, size_t workspace_bytes, void* stream) {
  if (!Ht || !Xt || !P || n < 0 || k <= 0 || d <= 0) return fail(ONMF_E_ARG, "surrogate_partial: bad argument");
  if (!workspace || workspace_bytes < onmf_surrogate_workspace(dtype, n, k, d))
    return fail(ONMF_E_WORKSPACE, "surrogate_partial: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  if (n == 0) {
    ONMF_CUDA(cudaMemsetAsync(P, 0, (size_t)k * (k + d) * (dtype == ONMF_F64 ? 8 : 4), st));
    return ONMF_OK;
  }
  if (dtype == ONMF_F32) return surrogate_partial_t<float>((const float*)Ht, (const float*)Xt, n, k, d, (float*)P, (float*)workspace, st);
  if (dtype == ONMF_F64) return surrogate_partial_t<double>((const double*)Ht, (const double*)Xt, n, k, d, (double*)P, (double*)workspace, st);
  return fail(ONMF_E_ARG, "surrogate_partial: bad dtype");
}

extern "C" int onmf_xxt_partial(int dtype, const void* Xt, int64_t n, int d, void* P2, void* workspace,
                                size_t workspace_bytes, void* stream) {
  if (!Xt || !P2 || n < 0 || d <= 0) return fail(ONMF_E_ARG, "xxt_partial: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  size_t tsz = dtype == ONMF_F64 ? 8 : 4;
  if (n == 0) {
    ONMF_CUDA(cudaMemsetAsync(P2, 0, (size_t)d * d * tsz, st));
    return ONMF_OK;
  }
  long long tiles = cdiv(d, BM) * cdiv(d, 128);
  long long want = cdiv<long long>(2LL * num_sms(), tiles);
  long long cap = cdiv<long long>(n, 256);
  int splits = (int)(want < cap ? want : cap);
  if (splits < 1) splits = 1;
  long long stride = (long long)d * d;
  // as many splits as the workspace holds: one split is one CTA per tile summing every sample in sequence
  const long long fit = workspace ? (long long)(workspace_bytes / ((size_t)stride * tsz)) : 0;
  if (splits > fit) splits = fit > 1 ? (int)fit : 1;
  int rc;
  if (dtype == ONMF_F32) {
    float* dst = splits == 1 ? (float*)P2 : (float*)workspace;
    rc = launch_gemm<float, true>((const float*)Xt, d, (const float*)Xt, d, dst, d, d, d, n, splits, stride, st);
    if (!rc && splits > 1) split_reduce_kernel<float><<<(unsigned)cdiv<long long>(stride, 256), 256, 0, st>>>((float*)workspace, splits, stride, stride, (float*)P2);
  } else if (dtype == ONMF_F64) {
    double* dst = splits == 1 ? (double*)P2 : (double*)workspace;
    rc = launch_gemm<double, true>((const double*)Xt, d, (const double*)Xt, d, dst, d, d, d, n, splits, stride, st);
    if (!rc && splits > 1) split_reduce_kernel<double><<<(unsigned)cdiv<long long>(stride, 256), 256, 0, st>>>((double*)workspace, splits, stride, stride, (double*)P2);
  } else {
    return fail(ONMF_E_ARG, "xxt_partial: bad dtype");
  }
  if (rc) return rc;
  ONMF_LAUNCH_CHECK("xxt_partial");
  return ONMF_OK;
}

extern "C" int onmf_surrogate_blend(int dtype, const void* P, int k, int d, double w, void* A, void* B, void* stream) {
  if (!P || !A || !B || k <= 0 || d <= 0) return fail(ONMF_E_ARG, "surrogate_blend: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  long long tot = (long long)k * (k + d);
  unsigned grid = (unsigned)cdiv<long long>(tot, 256);
  if (dtype == ONMF_F32) blend_kernel<float><<<grid, 256, 0, st>>>((const float*)P, k, d, (float)w, (float*)A, (float*)B);
  else if (dtype == ONMF_F64) blend_kernel<double><<<grid, 256, 0, st>>>((const double*)P, k, d, w, (double*)A, (double*)B);
  else return fail(ONMF_E_ARG, "surrogate_blend: bad dtype");
  ONMF_LAUNCH_CHECK("blend_kernel");
  return ONMF_OK;
}

template <typename TI, typename TO>
__global__ void convert_kernel(const TI* __restrict__ src, long long count, TO* __restrict__ dst) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < count; i += stride) dst[i] = (TO)src[i];
}

extern "C" int onmf_convert(int dtype_in, int dtype_out, const void* src, int64_t count, void* dst, void* stream) {
  if (!src || !dst || count < 0) return fail(ONMF_E_ARG, "convert: bad argument");
  if (count == 0) return ONMF_OK;
  cudaStream_t st = (cudaStream_t)stream;
  int grid = (int)cdiv<long long>(count, 256);
  if (grid > 16 * num_sms()) grid = 16 * num_sms();
  if (dtype_in == ONMF_F32 && dtype_out == ONMF_F64) convert_kernel<float, double><<<grid, 256, 0, st>>>((const float*)src, count, (double*)dst);
  else if (dtype_in == ONMF_F64 && dtype_out == ONMF_F32) convert_kernel<double, float><<<grid, 256, 0, st>>>((const double*)src, count, (float*)dst);
  else return fail(ONMF_E_ARG, "convert: f32 <-> f64 only");
  ONMF_LAUNCH_CHECK("convert_kernel");
  return ONMF_OK;
}

extern "C" int onmf_surrogate_blend_dev(int dtype, const void* P, int k, int d, const double* w_dev, void* A, void* B,
                                        void* stream) {
  if (!P || !A || !B || !w_dev || k <= 0 || d <= 0) return fail(ONMF_E_ARG, "surrogate_blend_dev: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  long long tot = (long long)k * (k + d);
  unsigned grid = (unsigned)cdiv<long long>(tot, 256);
  if (dtype == ONMF_F32) blend_dev_kernel<float><<<grid, 256, 0, st>>>((const float*)P, k, d, w_dev, (float*)A, (float*)B);
  else if (dtype == ONMF_F64) blend_dev_kernel<double><<<grid, 256, 0, st>>>((const double*)P, k, d, w_dev, (double*)A, (double*)B);
  else return fail(ONMF_E_ARG, "surrogate_blend_dev: bad dtype");
  ONMF_LAUNCH_CHECK("blend_dev_kernel");
  return ONMF_OK;
}

extern "C" int onmf_axpby(int dtype, int64_t count, double a, const void* x, double b, void* y, void* stream) {
  if (!x || !y || count < 0) return fail(ONMF_E_ARG, "axpby: bad argument");
  if (count == 0) return ONMF_OK;
  cudaStream_t st = (cudaStream_t)stream;
  unsigned grid = (unsigned)cdiv<long long>(count, 256);
  if (dtype == ONMF_F32) axpby_kernel<float><<<grid, 256, 0, st>>>(count, (float)a, (const float*)x, (float)b, (float*)y);
  else if (dtype == ONMF_F64) axpby_kernel<double><<<grid, 256, 0, st>>>(count, a, (const double*)x, b, (double*)y);
  else return fail(ONMF_E_ARG, "axpby: bad dtype");
  ONMF_LAUNCH_CHECK("axpby_kernel");
  return ONMF_OK;
}

extern "C" int onmf_surrogate_error(int dtype, const void* W, const double* G64, const void* A, const void* B, const void* C,
                                    int d, int k, double* out3, void* stream) {
  if (!W || !G64 || !A || !B || !out3 || d <= 0 || k <= 0) return fail(ONMF_E_ARG, "surrogate_error: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == ONMF_F32)
    surrogate_error_kernel<float><<<1, 1024, 0, st>>>((const float*)W, G64, (const float*)A, (const float*)B, (const float*)C, d, k, out3);
  else if (dtype == ONMF_F64)
    surrogate_error_kernel<double><<<1, 1024, 0, st>>>((const double*)W, G64, (const double*)A, (const double*)B, (const double*)C, d, k, out3);
  else
    return fail(ONMF_E_ARG, "surrogate_error: bad dtype");
  ONMF_LAUNCH_CHECK("surrogate_error_kernel");
  return ONMF_OK;
}
