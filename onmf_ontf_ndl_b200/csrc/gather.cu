// K1 -- patch gather, minibatch row gather, layout/precision conversion; plus the secondary
// projected-gradient coder sweep.
//
// Replaces the drivers' O(N^2) np.append patch loops (reference image_reconstruction.py:184-205,
// image_reconstruction_tensor.py:102-123, ising_reconstruction.py:56-65), the matricization
// tl_unfold(...)[.T] (src/ontf.py:203-208) and the minibatch slice X_unfold[:, idx] (src/ontf.py:231).
// All three are pure data movement: one coalesced read and one coalesced write per element, output in
// the sample-major layout (one sample per row) every other kernel consumes.
#include "common.cuh"

namespace onmf {

template <typename T> __device__ __forceinline__ T nan_of();
template <> __device__ __forceinline__ float nan_of<float>() { return __int_as_float(0x7fc00000); }
template <> __device__ __forceinline__ double nan_of<double>() { return __longlong_as_double(0x7ff8000000000000LL); }

// stored image element -> output element: a copy, or the u8 widening (float)v * scale of onmf_widen
template <typename T> __device__ __forceinline__ T widen_to(float v, float) { return (T)v; }
template <typename T> __device__ __forceinline__ T widen_to(double v, float) { return (T)v; }
template <typename T> __device__ __forceinline__ T widen_to(unsigned char v, float sc) { return (T)((float)v * sc); }

// corner of minibatch sample j: coords[idx[j]] (idx == nullptr: coords[j]); false -> NaN row (index outside [0, n_coords)
// or a patch that leaves the image), never read
__device__ __forceinline__ bool patch_corner(const int32_t* __restrict__ coords, long long n_coords, const long long* __restrict__ idx,
                                             long long j, int H, int Wd, int p, int& a, int& b) {
  long long s = j;
  if (idx) {
    s = idx[j];
    if (s < 0 || s >= n_coords) return false;
  }
  a = coords[2 * s]; b = coords[2 * s + 1];
  return !(a < 0 || b < 0 || a > H - p || b > Wd - p);
}

// S: stored image type, T: output type.  idx == nullptr: sample j is coords[j] (n_coords == n); else coords[idx[j]].
template <typename S, typename T>
__global__ void gather_patches_kernel(const S* __restrict__ img, int H, int Wd, int C, const int32_t* __restrict__ coords,
                                      long long n_coords, const long long* __restrict__ idx, long long n, int p, float scale,
                                      T* __restrict__ Xt, long long ld) {
  // one warp per (patch, patch-row): the p*C values of a patch row are contiguous in the image and in Xt
  const int lane = threadIdx.x & 31;
  const long long wid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
  const int run = p * C;
  for (long long t = wid; t < n * p; t += nw) {
    const long long j = t / p;
    const int r = (int)(t - j * p);
    int a, b;
    T* dst = Xt + (size_t)j * ld + (size_t)r * run;
    if (!patch_corner(coords, n_coords, idx, j, H, Wd, p, a, b)) {   // never read out of bounds,
      for (int e = lane; e < run; e += 32) dst[e] = nan_of<T>();     // poison the patch so the error is loud downstream
      continue;
    }
    const S* src = img + ((size_t)(a + r) * Wd + b) * C;
    for (int e = lane; e < run; e += 32) dst[e] = widen_to<T>(src[e], scale);
  }
}

// Vector form (the default whenever a patch's feature count and the output pitch are multiples of 16 bytes): one thread per
// 16 bytes of OUTPUT.  The output (n x d, every byte written once) is the only HBM stream of this kernel -- the image is read
// n*d/(H*W) times over and stays in L1/L2 -- so the store side is what has to be coalesced: consecutive threads write
// consecutive 16-byte pieces of consecutive patches, while the source elements (arbitrary alignment: b*C is any integer)
// are fetched as scalars through L1.  IdxT = 32-bit when n*d/V fits (a 64-bit division per thread costs more than the copy).
template <typename T, int V, typename IdxT>
__global__ void __launch_bounds__(256) gather_patches_vec_kernel(const T* __restrict__ img, int H, int Wd, int C,
                                                                 const int32_t* __restrict__ coords, long long n, int p,
                                                                 T* __restrict__ Xt, long long ld, int dv) {
  struct __align__(16) Vec { T v[V]; };
  const int run = p * C;
  const IdxT total = (IdxT)n * (IdxT)dv;
  const IdxT stride = (IdxT)gridDim.x * blockDim.x;
  auto fetch = [&](IdxT g, Vec& out) -> T* {
    const IdxT j = g / (IdxT)dv;
    const int e0 = (int)(g - j * (IdxT)dv) * V;
    const int2 ab = reinterpret_cast<const int2*>(coords)[j];
    const int a = ab.x, b = ab.y;
    if (a < 0 || b < 0 || a > H - p || b > Wd - p) {          // corner outside the image: poison, never read out of bounds
#pragma unroll
      for (int t = 0; t < V; ++t) out.v[t] = nan_of<T>();
    } else {
      int r = e0 / run, c = e0 - r * run;
      const T* src = img + ((size_t)(a + r) * Wd + b) * C + c;
#pragma unroll
      for (int t = 0; t < V; ++t) {
        out.v[t] = __ldg(src);
        ++src;
        if (++c == run) {                                    // next patch row (the pointer past the last row is never read)
          c = 0;
          ++r;
          src = img + ((size_t)(a + r) * Wd + b) * C;
        }
      }
    }
    return Xt + (size_t)j * ld + e0;
  };
  for (IdxT g = (IdxT)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += stride) {
    Vec o;
    T* dst = fetch(g, o);
    *reinterpret_cast<Vec*>(dst) = o;
  }
}

// Tiled form of the same copy (the default: d / V <= 1024 vectors per patch, image below 2^31 elements): blockDim.x = the
// vectors of ONE patch, blockDim.y = patches per CTA.  A thread keeps its position inside the patch for the whole grid-stride
// loop, so the two integer divisions and the row-crossing logic of the flat kernel (which made it issue-bound at 0.45 of the
// HBM rate) are paid once per thread: the V source offsets relative to the patch corner are loop invariants, and a patch costs
// one broadcast corner load, V scalar loads and one 16-byte store.  Linear thread order == output order, stores stay coalesced.
template <typename S, typename T, int V>
__global__ void __launch_bounds__(1024) gather_patches_tile_kernel(const S* __restrict__ img, int H, int Wd, int C,
                                                                   const int32_t* __restrict__ coords, long long n_coords,
                                                                   const long long* __restrict__ idx, long long n, int p,
                                                                   float scale, T* __restrict__ Xt, long long ld) {
  struct __align__(16) Vec { T v[V]; };
  const int run = p * C;
  const int e0 = threadIdx.x * V;
  int off[V];
  {
    int r = e0 / run, c = e0 - r * run;
#pragma unroll
    for (int t = 0; t < V; ++t) {
      off[t] = r * Wd * C + c;
      if (++c == run) { c = 0; ++r; }
    }
  }
  const long long step = (long long)gridDim.x * blockDim.y;
  for (long long j = (long long)blockIdx.x * blockDim.y + threadIdx.y; j < n; j += step) {
    long long s = j;
    bool ok = true;
    if (idx) {                                          // minibatch through an index (onmf_gather_patches_mb)
      s = idx[j];
      ok = s >= 0 && s < n_coords;
    }
    const int2 ab = ok ? __ldg(reinterpret_cast<const int2*>(coords) + s) : make_int2(-1, -1);
    Vec out;
    if (ab.x < 0 || ab.y < 0 || ab.x > H - p || ab.y > Wd - p) {
#pragma unroll
      for (int t = 0; t < V; ++t) out.v[t] = nan_of<T>();
    } else {
      const S* src = img + ((size_t)ab.x * Wd + ab.y) * C;
#pragma unroll
      for (int t = 0; t < V; ++t) out.v[t] = widen_to<T>(__ldg(src + off[t]), scale);
    }
    *reinterpret_cast<Vec*>(Xt + (size_t)j * ld + e0) = out;
  }
}

template <typename T>
__global__ void gather_rows_kernel(const T* __restrict__ pool, long long n_pool, int d, const long long* __restrict__ idx,
                                   long long n, T* __restrict__ Xt) {
  const int lane = threadIdx.x & 31;
  const long long wid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long j = wid; j < n; j += nw) {
    const long long i = idx[j];
    T* dst = Xt + (size_t)j * d;
    if (i < 0 || i >= n_pool) {                               // bad index: NaN row instead of an out-of-bounds read
      for (int e = lane; e < d; e += 32) dst[e] = nan_of<T>();
      continue;
    }
    const T* src = pool + (size_t)i * d;
    for (int e = lane; e < d; e += 32) dst[e] = src[e];
  }
}

// dst (cols x rows) = src (rows x cols)^T with conversion; 32 x 32 tiles through shared memory
template <typename TI, typename TO>
__global__ void transpose_kernel(const TI* __restrict__ src, long long rows, long long cols, TO* __restrict__ dst) {
  __shared__ TO tile[32][33];
  const long long c0 = (long long)blockIdx.x * 32, r0 = (long long)blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    long long r = r0 + i, c = c0 + threadIdx.x;
    if (r < rows && c < cols) tile[i][threadIdx.x] = (TO)src[(size_t)r * cols + c];
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    long long c = c0 + i, r = r0 + threadIdx.x;
    if (r < rows && c < cols) dst[(size_t)c * rows + r] = tile[threadIdx.x][i];
  }
}

// Vector form: 64 x 64 tiles, 256 threads, four elements per access on both sides (16 bytes of fp32, 32 of fp64) -- used when
// rows and cols are multiples of 4 and both pointers are 32-byte aligned.  The 32 x 32 scalar kernel above reached 0.44-0.55
// of the HBM copy rate at the matricization shapes (profiles/r2_next_rows.md); this one moves 4x the bytes per instruction.
template <typename TI, typename TO>
__global__ void __launch_bounds__(256) transpose64_kernel(const TI* __restrict__ src, long long rows, long long cols,
                                                          TO* __restrict__ dst) {
  struct __align__(sizeof(TI) * 4) VI { TI v[4]; };
  struct __align__(sizeof(TO) * 4) VO { TO v[4]; };
  __shared__ TO tile[64][65];
  const long long c0 = (long long)blockIdx.x * 64, r0 = (long long)blockIdx.y * 64;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;          // 16 four-element vectors across, 16 lines down
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int rr = ty + 16 * i;
    const long long r = r0 + rr, c = c0 + 4 * tx;
    if (r < rows && c < cols) {                                    // cols % 4 == 0: a vector is inside or outside as a whole
      const VI v = *reinterpret_cast<const VI*>(src + (size_t)r * cols + c);
#pragma unroll
      for (int e = 0; e < 4; ++e) tile[rr][4 * tx + e] = (TO)v.v[e];
    }
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int cc = ty + 16 * i;
    const long long c = c0 + cc, r = r0 + 4 * tx;
    if (c < cols && r < rows) {
      VO v;
#pragma unroll
      for (int e = 0; e < 4; ++e) v.v[e] = tile[4 * tx + e][cc];
      *reinterpret_cast<VO*>(dst + (size_t)c * rows + r) = v;
    }
  }
}

// one outer iteration of the shipped projected-gradient coder (reference src/onmf.py:252-263, r=None):
// for q in 0..k-1:  h_q <- max(h_q - (G[q,:] h - c_q + alpha) / (sqrt(it+10) (G_qq+1)), 0), Gauss-Seidel in q,
// independently per sample.  One warp per sample; h lives in registers (atom i on lane i%32).
template <typename T, int NA>
__global__ void pgd_sweep_kernel(const T* __restrict__ G, const T* __restrict__ Ct, long long n, int k, T alpha, T scale,
                                 T* __restrict__ Ht, int q_begin, int q_end, int gsm) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const T* Gs = G;                 // Gram matrices beyond the shared-memory capacity are read through L1/L2
  if (gsm) {
    T* Gw = reinterpret_cast<T*>(smem_raw);
    for (int i = threadIdx.x; i < k * k; i += blockDim.x) Gw[i] = G[i];
    __syncthreads();
    Gs = Gw;
  }
  const int lane = threadIdx.x & 31;
  const long long wid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long j = wid; j < n; j += nw) {
    T h[NA];
#pragma unroll
    for (int m = 0; m < NA; ++m) {
      int i = lane + 32 * m;
      h[m] = i < k ? Ht[(size_t)j * k + i] : T(0);
    }
    for (int q = q_begin; q < q_end; ++q) {
      T part = T(0);
#pragma unroll
      for (int m = 0; m < NA; ++m) {
        int i = lane + 32 * m;
        if (i < k) part += Gs[q * k + i] * h[m];
      }
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) part += __shfl_xor_sync(0xffffffffu, part, off);
      const T grad = part - Ct[(size_t)j * k + q] + alpha;
      const T step = T(1) / (scale * (Gs[q * k + q] + T(1)));
#pragma unroll
      for (int m = 0; m < NA; ++m)
        if (lane + 32 * m == q) {
          T v = h[m] - step * grad;
          h[m] = v > T(0) ? v : T(0);
        }
    }
#pragma unroll
    for (int m = 0; m < NA; ++m) {
      int i = lane + 32 * m;
      if (i < k) Ht[(size_t)j * k + i] = h[m];
    }
  }
}

// The whole projected-gradient coder per sample, in-kernel: what the reference does when it codes ONE patch per call
// (image_reconstruction.py:384: update_code_within_radius(patch, W, H0=None, r=None, alpha, sub_iter, stopping_diff)):
// outer iterations i < sub_iter while dist > stopping_diff, dist = ||h - h_old||_2 / ||h_old||_2 (for a single column
// the spectral norm of src/onmf.py:265 is the vector 2-norm).  One warp per sample; Ht holds H0 on entry.
template <typename T, int NA>
__global__ void pgd_columns_kernel(const T* __restrict__ G, const T* __restrict__ Ct, long long n, int k, T alpha, int sub_iter,
                                   T stopping_diff, T* __restrict__ Ht, int gsm) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const T* Gs = G;                 // Gram matrices beyond the shared-memory capacity are read through L1/L2
  if (gsm) {
    T* Gw = reinterpret_cast<T*>(smem_raw);
    for (int i = threadIdx.x; i < k * k; i += blockDim.x) Gw[i] = G[i];
    __syncthreads();
    Gs = Gw;
  }
  const int lane = threadIdx.x & 31;
  const long long wid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long j = wid; j < n; j += nw) {
    T h[NA], c[NA];
#pragma unroll
    for (int m = 0; m < NA; ++m) {
      int i = lane + 32 * m;
      h[m] = i < k ? Ht[(size_t)j * k + i] : T(0);
      c[m] = i < k ? Ct[(size_t)j * k + i] : T(0);
    }
    T dist = T(1);
    for (int it = 0; it < sub_iter && dist > stopping_diff; ++it) {
      const T scale = (T)sqrt((double)it + 10.0);
      T hold[NA];
#pragma unroll
      for (int m = 0; m < NA; ++m) hold[m] = h[m];
      for (int q = 0; q < k; ++q) {
        T part = T(0);
#pragma unroll
        for (int m = 0; m < NA; ++m) {
          int i = lane + 32 * m;
          if (i < k) part += Gs[q * k + i] * h[m];
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) part += __shfl_xor_sync(0xffffffffu, part, off);
        T cq = T(0);
#pragma unroll
        for (int m = 0; m < NA; ++m)
          if (lane + 32 * m == q) cq = c[m];
        cq = __shfl_sync(0xffffffffu, cq, q & 31);
        const T grad = part - cq + alpha;
        const T step = T(1) / (scale * (Gs[q * k + q] + T(1)));
#pragma unroll
        for (int m = 0; m < NA; ++m)
          if (lane + 32 * m == q) {
            T v = h[m] - step * grad;
            h[m] = v > T(0) ? v : T(0);
          }
      }
      T num = T(0), den = T(0);
#pragma unroll
      for (int m = 0; m < NA; ++m) {
        T dv = h[m] - hold[m];
        num += dv * dv;
        den += hold[m] * hold[m];
      }
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) {
        num += __shfl_xor_sync(0xffffffffu, num, off);
        den += __shfl_xor_sync(0xffffffffu, den, off);
      }
      dist = sqrt(num) / sqrt(den);
    }
#pragma unroll
    for (int m = 0; m < NA; ++m) {
      int i = lane + 32 * m;
      if (i < k) Ht[(size_t)j * k + i] = h[m];
    }
  }
}

// The same per-sample coder for small dictionaries (k <= 32) on LARGE batches -- image reconstruction codes every grid patch
// of an image in one call (reconstruct.py: 252,004 patches of a 512 x 512 image at k = 25): ONE THREAD per sample.  The
// warp-per-sample kernel above spends ~100 warp-instructions (five shuffles, the lane select, a division) on a Gauss-Seidel
// coordinate whose arithmetic is k multiply-adds; here the code vector lives in the thread's registers (KP = k rounded up to
// a multiple of 4, fully unrolled), the zero-padded Gram is read from shared memory at warp-uniform addresses (broadcast,
// 16 bytes per load) and the per-coordinate step 1 / (G_qq + 1) is tabulated once per CTA.  Same iteration, same stopping
// test; the dot products are summed in index order instead of the butterfly order, so results agree with the kernel above to
// rounding (fp64: ~1e-16), not bit for bit.  Rows of Ct / Ht are read and written directly: the 32 rows of a warp are one
// contiguous block, every line is used completely through L1.
template <typename T, int KP>
__global__ void __launch_bounds__(128) pgd_columns_tps_kernel(const T* __restrict__ G, const T* __restrict__ Ct, long long n, int k,
                                                             T alpha, int sub_iter, T stopping_diff, T* __restrict__ Ht) {
  __shared__ __align__(16) T Gs[KP * KP];
  __shared__ T inv[KP];
  for (int i = threadIdx.x; i < KP * KP; i += blockDim.x) {
    const int q = i / KP, c = i - q * KP;
    Gs[i] = (q < k && c < k) ? G[q * k + c] : T(0);
  }
  for (int q = threadIdx.x; q < KP; q += blockDim.x) inv[q] = q < k ? T(1) / (G[q * k + q] + T(1)) : T(0);
  __syncthreads();
  const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  T h[KP], c[KP];
#pragma unroll
  for (int i = 0; i < KP; ++i) {
    h[i] = i < k ? Ht[(size_t)j * k + i] : T(0);
    c[i] = i < k ? Ct[(size_t)j * k + i] - alpha : T(0);       // grad = G[q,:] h - (c_q - alpha)
  }
  T dist = T(1);
  for (int it = 0; it < sub_iter && dist > stopping_diff; ++it) {
    const T rscale = T(1) / (T)sqrt((double)it + 10.0);
    T num = T(0), den = T(0);
    int off = 0;
    asm volatile("" : "+r"(off));              // the Gram is re-read every sweep (hoisting k^2 loads out of the loop spills)
    const T* Gp = Gs + off;
    const T* ip = inv + off;
#pragma unroll
    for (int q = 0; q < KP; ++q) {
      T p0 = T(0), p1 = T(0), p2 = T(0), p3 = T(0);
#pragma unroll
      for (int i = 0; i < KP; i += 4) {
        p0 += Gp[q * KP + i] * h[i];
        p1 += Gp[q * KP + i + 1] * h[i + 1];
        p2 += Gp[q * KP + i + 2] * h[i + 2];
        p3 += Gp[q * KP + i + 3] * h[i + 3];
      }
      const T grad = ((p0 + p1) + (p2 + p3)) - c[q];
      T v = h[q] - (rscale * ip[q]) * grad;
      v = (q < k && v > T(0)) ? v : T(0);
      const T dv = v - h[q];
      num += dv * dv;
      den += h[q] * h[q];
      h[q] = v;
    }
    dist = sqrt(num) / sqrt(den);
  }
#pragma unroll
  for (int i = 0; i < KP; ++i)
    if (i < k) Ht[(size_t)j * k + i] = h[i];
}

// Overlap-averaged canvas from per-patch reconstructions (the running mean of image_reconstruction.py:389-392 and
// sklearn's reconstruct_from_patches_2d): patches of size p x p (x C channels) with top-left corners on the grid
// (gy*stride, gx*stride), gy < ny, gx < nx, grid patch j = gy*nx + gx.  One call adds the patches j0 <= j < j1, whose
// reconstructions are the rows R[(j - j0), (r*p + c)*C + ch].
// Gather form: one thread per canvas element sums its covering patches in ascending j -> deterministic, no atomics, and
// consecutive ranges give the bits of one call over [0, ny*nx): a pixel whose first covering patch is in the range starts
// from 0, any other continues the running sum an earlier call left in the canvas.  The covering patches of pixel (y, x)
// are the rectangle gy_lo..gy_hi x gx_lo..gx_hi; its last patch own = gy_hi*nx + gx_hi also names the owner of a pixel
// no patch covers (gy_hi = min(y / stride, ny - 1), likewise gx_hi), and only the call that holds `own` writes the final
// value (sum / count, or 0 and count 0) and the count.  Threads cover the canvas rows from y0 on that the range touches.
template <typename T>
__global__ void patch_grid_accumulate_kernel(const T* __restrict__ R, long long ldr, int ny, int nx, int p, int stride, int C,
                                             int Ww, long long j0, long long j1, int y0, long long tot, T* __restrict__ canvas,
                                             T* __restrict__ count) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= tot) return;
  const int ch = (int)(idx % C);
  const long long pix = idx / C + (long long)y0 * Ww;
  const long long out = pix * C + ch;
  const int x = (int)(pix % Ww), y = (int)(pix / Ww);
  // grid rows gy with gy*stride <= y < gy*stride + p
  int gy_hi = y / stride;
  if (gy_hi > ny - 1) gy_hi = ny - 1;
  int gy_lo = (y - p + stride) / stride;      // ceil((y - p + 1) / stride)
  if (y - p + 1 <= 0) gy_lo = 0;
  int gx_hi = x / stride;
  if (gx_hi > nx - 1) gx_hi = nx - 1;
  int gx_lo = (x - p + stride) / stride;
  if (x - p + 1 <= 0) gx_lo = 0;
  const long long own = (long long)gy_hi * nx + gx_hi;
  const bool owns = own >= j0 && own < j1;
  if (gy_lo > gy_hi || gx_lo > gx_hi) {       // no patch covers this pixel (below / right of the grid, or stride > p)
    if (owns) {
      canvas[out] = T(0);
      if (count != nullptr && ch == 0) count[pix] = T(0);
    }
    return;
  }
  const long long first = (long long)gy_lo * nx + gx_lo;
  if (first >= j1 || own < j0) return;        // no covering patch in this range
  T acc = first >= j0 ? T(0) : canvas[out];
  int gy_a = gy_lo, gy_b = gy_hi;
  if (gy_a < j0 / nx) gy_a = (int)(j0 / nx);
  if (gy_b > (j1 - 1) / nx) gy_b = (int)((j1 - 1) / nx);
  for (int gy = gy_a; gy <= gy_b; ++gy) {
    const long long row = (long long)gy * nx;
    const int r = y - gy * stride;
    int gx_a = gx_lo, gx_b = gx_hi;
    if (row + gx_a < j0) gx_a = (int)(j0 - row);
    if (row + gx_b >= j1) gx_b = (int)(j1 - 1 - row);
    for (int gx = gx_a; gx <= gx_b; ++gx) {
      const int c = x - gx * stride;
      acc += R[(size_t)(row + gx - j0) * ldr + ((size_t)r * p + c) * C + ch];
    }
  }
  if (owns) {
    const int cnt = (gy_hi - gy_lo + 1) * (gx_hi - gx_lo + 1);
    canvas[out] = acc / T(cnt);
    if (count != nullptr && ch == 0) count[pix] = T(cnt);
  } else {
    canvas[out] = acc;
  }
}

template <typename T>
static int pgd_t(const T* G, const T* Ct, long long n, int k, double alpha, int it, T* Ht, int q_begin, int q_end,
                 cudaStream_t st) {
  size_t smem = (size_t)k * k * sizeof(T);
  const int gsm = smem <= (size_t)max_smem_optin() ? 1 : 0;
  if (!gsm) smem = 0;
  const T scale = (T)sqrt((double)it + 10.0);
  int threads = 256;
  long long warps = n;
  int grid = (int)cdiv<long long>(warps * 32, threads);
  if (grid > 4 * num_sms()) grid = 4 * num_sms();
  if (grid < 1) grid = 1;
#define ONMF_PGD(NA)                                                                                 \
  {                                                                                                  \
    auto kern = pgd_sweep_kernel<T, NA>;                                                             \
    ONMF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));   \
    kern<<<grid, threads, smem, st>>>(G, Ct, n, k, (T)alpha, scale, Ht, q_begin, q_end, gsm);             \
  }
  if (k <= 32) ONMF_PGD(1)
  else if (k <= 64) ONMF_PGD(2)
  else if (k <= 128) ONMF_PGD(4)
  else if (k <= 256) ONMF_PGD(8)
  else if (k <= 512) ONMF_PGD(16)
  else return fail(ONMF_E_UNSUPPORTED, "pgd_sweep: n_components > 512");
#undef ONMF_PGD
  ONMF_LAUNCH_CHECK("pgd_sweep_kernel");
  return ONMF_OK;
}

template <typename TI, typename TO>
static int transpose_t(const void* src, long long rows, long long cols, void* dst, cudaStream_t st) {
  if (rows % 4 == 0 && cols % 4 == 0 && (reinterpret_cast<uintptr_t>(src) & 31) == 0 && (reinterpret_cast<uintptr_t>(dst) & 31) == 0 &&
      cdiv<long long>(rows, 64) <= 65535) {
    dim3 grid64((unsigned)cdiv<long long>(cols, 64), (unsigned)cdiv<long long>(rows, 64));
    transpose64_kernel<TI, TO><<<grid64, 256, 0, st>>>((const TI*)src, rows, cols, (TO*)dst);
    ONMF_LAUNCH_CHECK("transpose64_kernel");
    return ONMF_OK;
  }
  dim3 block(32, 8);
  dim3 grid((unsigned)cdiv<long long>(cols, 32), (unsigned)cdiv<long long>(rows, 32));
  if (grid.y > 65535) return fail(ONMF_E_UNSUPPORTED, "transpose: more than 2^21 rows; transpose the other way");
  transpose_kernel<TI, TO><<<grid, block, 0, st>>>((const TI*)src, rows, cols, (TO*)dst);
  ONMF_LAUNCH_CHECK("transpose_kernel");
  return ONMF_OK;
}

}  // namespace onmf

using namespace onmf;

extern "C" int onmf_gather_patches(int dtype, const void* img, int H, int Wd, int C, const int32_t* coords, int64_t n,
                                   int p, void* Xt, int64_t ld, void* stream) {
  if (!img || !coords || !Xt || H <= 0 || Wd <= 0 || C <= 0 || p <= 0 || n < 0 || p > H || p > Wd || ld < (int64_t)p * p * C)
    return fail(ONMF_E_ARG, "gather_patches: bad argument");
  if (n == 0) return ONMF_OK;
  cudaStream_t st = (cudaStream_t)stream;
  int threads = 256;
  {
    // vector path: 16 bytes of output per thread
    const int V = dtype == ONMF_F32 ? 4 : 2;
    const long long d = (long long)p * p * C;
    if ((dtype == ONMF_F32 || dtype == ONMF_F64) && d % V == 0 && ld % V == 0 && (reinterpret_cast<uintptr_t>(Xt) & 15) == 0 &&
        (reinterpret_cast<uintptr_t>(coords) & 7) == 0) {
      const int dv = (int)(d / V);
      if (dv <= 1024 && (long long)H * Wd * C < (1LL << 31)) {
        int py = 256 / dv;                                   // patches per CTA: about 256 threads
        if (py < 1) py = 1;
        dim3 block((unsigned)dv, (unsigned)py);
        long long gq = cdiv<long long>(n, py);
        const long long capq = (long long)num_sms() * (2048 / (dv * py)) * 4;
        const int gridq = (int)(gq > capq ? capq : gq);
        if (dtype == ONMF_F32) gather_patches_tile_kernel<float, float, 4><<<gridq, block, 0, st>>>((const float*)img, H, Wd, C, coords, n, nullptr, n, p, 1.f, (float*)Xt, ld);
        else gather_patches_tile_kernel<double, double, 2><<<gridq, block, 0, st>>>((const double*)img, H, Wd, C, coords, n, nullptr, n, p, 1.f, (double*)Xt, ld);
        ONMF_LAUNCH_CHECK("gather_patches_tile_kernel");
        return ONMF_OK;
      }
      const long long total = n * dv;
      long long g = cdiv<long long>(total, threads);
      const long long cap = 16LL * num_sms();
      const int grid = (int)(g > cap ? cap : g);
      const bool small = total + (long long)grid * threads < (1LL << 31);
      if (dtype == ONMF_F32) {
        if (small) gather_patches_vec_kernel<float, 4, unsigned><<<grid, threads, 0, st>>>((const float*)img, H, Wd, C, coords, n, p, (float*)Xt, ld, dv);
        else gather_patches_vec_kernel<float, 4, unsigned long long><<<grid, threads, 0, st>>>((const float*)img, H, Wd, C, coords, n, p, (float*)Xt, ld, dv);
      } else {
        if (small) gather_patches_vec_kernel<double, 2, unsigned><<<grid, threads, 0, st>>>((const double*)img, H, Wd, C, coords, n, p, (double*)Xt, ld, dv);
        else gather_patches_vec_kernel<double, 2, unsigned long long><<<grid, threads, 0, st>>>((const double*)img, H, Wd, C, coords, n, p, (double*)Xt, ld, dv);
      }
      ONMF_LAUNCH_CHECK("gather_patches_vec_kernel");
      return ONMF_OK;
    }
  }
  long long warps = n * p;
  int grid = (int)cdiv<long long>(warps * 32, threads);
  if (grid > 8 * num_sms()) grid = 8 * num_sms();
  if (dtype == ONMF_F32) gather_patches_kernel<float, float><<<grid, threads, 0, st>>>((const float*)img, H, Wd, C, coords, n, nullptr, n, p, 1.f, (float*)Xt, ld);
  else if (dtype == ONMF_F64) gather_patches_kernel<double, double><<<grid, threads, 0, st>>>((const double*)img, H, Wd, C, coords, n, nullptr, n, p, 1.f, (double*)Xt, ld);
  else return fail(ONMF_E_ARG, "gather_patches: bad dtype");
  ONMF_LAUNCH_CHECK("gather_patches_kernel");
  return ONMF_OK;
}

// the same two kernels on a patch minibatch: sample j is the patch at coords[idx[j]]
template <typename S, typename T>
static int gather_patches_mb(const onmf_patch_minibatch* pm, T* Xt, long long ld, cudaStream_t st) {
  const int H = pm->H, Wd = pm->W, C = pm->C, p = pm->p;
  const long long n = pm->n, d = (long long)p * p * C;
  const S* img = (const S*)pm->img;
  const float sc = (float)pm->scale;
  const long long* idx = (const long long*)pm->idx;
  constexpr int V = 16 / sizeof(T);
  if (d % V == 0 && ld % V == 0 && d / V <= 1024 && (reinterpret_cast<uintptr_t>(Xt) & 15) == 0 &&
      (reinterpret_cast<uintptr_t>(pm->coords) & 7) == 0 && (long long)H * Wd * C < (1LL << 31)) {
    const int dv = (int)(d / V);
    int py = 256 / dv;
    if (py < 1) py = 1;
    dim3 block((unsigned)dv, (unsigned)py);
    const long long gq = cdiv<long long>(n, py);
    const long long capq = (long long)num_sms() * (2048 / (dv * py)) * 4;
    gather_patches_tile_kernel<S, T, V><<<(int)(gq > capq ? capq : gq), block, 0, st>>>(img, H, Wd, C, pm->coords, pm->n_coords, idx,
                                                                                       n, p, sc, Xt, ld);
    ONMF_LAUNCH_CHECK("gather_patches_tile_kernel");
    return ONMF_OK;
  }
  int grid = (int)cdiv<long long>(n * p * 32, 256);
  if (grid > 8 * num_sms()) grid = 8 * num_sms();
  gather_patches_kernel<S, T><<<grid, 256, 0, st>>>(img, H, Wd, C, pm->coords, pm->n_coords, idx, n, p, sc, Xt, ld);
  ONMF_LAUNCH_CHECK("gather_patches_kernel");
  return ONMF_OK;
}

extern "C" int onmf_gather_patches_mb(const onmf_patch_minibatch* pm, int dtype_out, void* Xt, int64_t ld, void* stream) {
  if (!pm || !pm->img || !Xt || pm->H <= 0 || pm->W <= 0 || pm->C <= 0 || pm->p <= 0 || pm->p > pm->H || pm->p > pm->W || pm->n < 0 ||
      pm->n_coords < 0 || (pm->n_coords > 0 && !pm->coords) || ld < (int64_t)pm->p * pm->p * pm->C)
    return fail(ONMF_E_ARG, "gather_patches_mb: bad argument");
  if (!pm->idx && pm->n > pm->n_coords) return fail(ONMF_E_ARG, "gather_patches_mb: idx == NULL needs n <= n_coords");
  if (pm->n == 0) return ONMF_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (pm->kind == ONMF_F32 && dtype_out == ONMF_F32) return gather_patches_mb<float>(pm, (float*)Xt, ld, st);
  if (pm->kind == ONMF_F64 && dtype_out == ONMF_F64) return gather_patches_mb<double>(pm, (double*)Xt, ld, st);
  if (pm->kind == ONMF_STORE_U8 && dtype_out == ONMF_F32) return gather_patches_mb<unsigned char>(pm, (float*)Xt, ld, st);
  return fail(ONMF_E_ARG, "gather_patches_mb: storage / output kind must be F32 -> F32, F64 -> F64 or STORE_U8 -> F32");
}

extern "C" int onmf_gather_rows(int dtype, const void* pool, int64_t n_pool, int d, const int64_t* idx, int64_t n, void* Xt,
                                void* stream) {
  if (!pool || !idx || !Xt || d <= 0 || n < 0 || n_pool <= 0) return fail(ONMF_E_ARG, "gather_rows: bad argument");
  if (n == 0) return ONMF_OK;
  cudaStream_t st = (cudaStream_t)stream;
  int threads = 256;
  int grid = (int)cdiv<long long>(n * 32, threads);
  if (grid > 8 * num_sms()) grid = 8 * num_sms();
  if (dtype == ONMF_F32) gather_rows_kernel<float><<<grid, threads, 0, st>>>((const float*)pool, n_pool, d, (const long long*)idx, n, (float*)Xt);
  else if (dtype == ONMF_F64) gather_rows_kernel<double><<<grid, threads, 0, st>>>((const double*)pool, n_pool, d, (const long long*)idx, n, (double*)Xt);
  else return fail(ONMF_E_ARG, "gather_rows: bad dtype");
  ONMF_LAUNCH_CHECK("gather_rows_kernel");
  return ONMF_OK;
}

extern "C" int onmf_transpose(int dtype_in, int dtype_out, const void* src, int64_t rows, int64_t cols, void* dst,
                              void* stream) {
  if (!src || !dst || rows < 0 || cols < 0) return fail(ONMF_E_ARG, "transpose: bad argument");
  if (rows == 0 || cols == 0) return ONMF_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype_in == ONMF_F32 && dtype_out == ONMF_F32) return transpose_t<float, float>(src, rows, cols, dst, st);
  if (dtype_in == ONMF_F64 && dtype_out == ONMF_F32) return transpose_t<double, float>(src, rows, cols, dst, st);
  if (dtype_in == ONMF_F32 && dtype_out == ONMF_F64) return transpose_t<float, double>(src, rows, cols, dst, st);
  if (dtype_in == ONMF_F64 && dtype_out == ONMF_F64) return transpose_t<double, double>(src, rows, cols, dst, st);
  return fail(ONMF_E_ARG, "transpose: bad dtype");
}

extern "C" int onmf_pgd_sweep_rows(int dtype, const void* G, const void* Ct, int64_t n, int k, double alpha, int it, void* Ht,
                                   int q_begin, int q_end, void* stream) {
  if (!G || !Ct || !Ht || n < 0 || k <= 0 || it < 0 || q_begin < 0 || q_end > k || q_begin > q_end)
    return fail(ONMF_E_ARG, "pgd_sweep_rows: bad argument");
  if (n == 0 || q_begin == q_end) return ONMF_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == ONMF_F32) return pgd_t<float>((const float*)G, (const float*)Ct, n, k, alpha, it, (float*)Ht, q_begin, q_end, st);
  if (dtype == ONMF_F64) return pgd_t<double>((const double*)G, (const double*)Ct, n, k, alpha, it, (double*)Ht, q_begin, q_end, st);
  return fail(ONMF_E_ARG, "pgd_sweep_rows: bad dtype");
}

extern "C" int onmf_pgd_sweep(int dtype, const void* G, const void* Ct, int64_t n, int k, double alpha, int it, void* Ht,
                              void* stream) {
  if (!G || !Ct || !Ht || n < 0 || k <= 0 || it < 0) return fail(ONMF_E_ARG, "pgd_sweep: bad argument");
  if (n == 0) return ONMF_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == ONMF_F32) return pgd_t<float>((const float*)G, (const float*)Ct, n, k, alpha, it, (float*)Ht, 0, k, st);
  if (dtype == ONMF_F64) return pgd_t<double>((const double*)G, (const double*)Ct, n, k, alpha, it, (double*)Ht, 0, k, st);
  return fail(ONMF_E_ARG, "pgd_sweep: bad dtype");
}

extern "C" int onmf_pgd_code_columns(int dtype, const void* G, const void* Ct, int64_t n, int k, double alpha, int sub_iter,
                                     double stopping_diff, void* Ht, void* stream) {
  if (!G || !Ct || !Ht || n < 0 || k <= 0 || sub_iter < 0) return fail(ONMF_E_ARG, "pgd_code_columns: bad argument");
  if (n == 0) return ONMF_OK;
  cudaStream_t st = (cudaStream_t)stream;
  size_t tsz = dtype == ONMF_F64 ? 8 : 4;
  size_t smem = (size_t)k * k * tsz;
  const int gsm = smem <= (size_t)max_smem_optin() ? 1 : 0;
  if (!gsm) smem = 0;
  if (k <= 32 && n >= 16LL * num_sms()) {
    // large batch, small dictionary: one thread per sample (pgd_columns_tps_kernel)
    const unsigned g = (unsigned)cdiv<long long>(n, 128);
#define ONMF_TPS(TT, KP) pgd_columns_tps_kernel<TT, KP><<<g, 128, 0, st>>>((const TT*)G, (const TT*)Ct, n, k, (TT)alpha, sub_iter, (TT)stopping_diff, (TT*)Ht)
#define ONMF_TPS_K(TT)                   \
  if (k <= 8) ONMF_TPS(TT, 8);           \
  else if (k <= 12) ONMF_TPS(TT, 12);    \
  else if (k <= 16) ONMF_TPS(TT, 16);    \
  else if (k <= 20) ONMF_TPS(TT, 20);    \
  else if (k <= 24) ONMF_TPS(TT, 24);    \
  else if (k <= 28) ONMF_TPS(TT, 28);    \
  else ONMF_TPS(TT, 32);
    if (dtype == ONMF_F32) { ONMF_TPS_K(float) }
    else if (dtype == ONMF_F64) { ONMF_TPS_K(double) }
    else return fail(ONMF_E_ARG, "pgd_code_columns: bad dtype");
#undef ONMF_TPS_K
#undef ONMF_TPS
    ONMF_LAUNCH_CHECK("pgd_columns_tps_kernel");
    return ONMF_OK;
  }
  int threads = 256;
  int grid = (int)cdiv<long long>(n * 32, threads);
  if (grid > 4 * num_sms()) grid = 4 * num_sms();
#define ONMF_PGDC(TT, NA)                                                                              \
  {                                                                                                    \
    auto kern = pgd_columns_kernel<TT, NA>;                                                            \
    ONMF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));     \
    kern<<<grid, threads, smem, st>>>((const TT*)G, (const TT*)Ct, n, k, (TT)alpha, sub_iter, (TT)stopping_diff, (TT*)Ht, gsm); \
  }
#define ONMF_PGDC_K(TT)                                   \
  if (k <= 32) ONMF_PGDC(TT, 1)                           \
  else if (k <= 64) ONMF_PGDC(TT, 2)                      \
  else if (k <= 128) ONMF_PGDC(TT, 4)                     \
  else if (k <= 256) ONMF_PGDC(TT, 8)                     \
  else if (k <= 512) ONMF_PGDC(TT, 16)                    \
  else return fail(ONMF_E_UNSUPPORTED, "pgd_code_columns: n_components > 512");
  if (dtype == ONMF_F32) { ONMF_PGDC_K(float) }
  else if (dtype == ONMF_F64) { ONMF_PGDC_K(double) }
  else return fail(ONMF_E_ARG, "pgd_code_columns: bad dtype");
#undef ONMF_PGDC_K
#undef ONMF_PGDC
  ONMF_LAUNCH_CHECK("pgd_columns_kernel");
  return ONMF_OK;
}

extern "C" int onmf_patch_grid_accumulate(int dtype, const void* R, int64_t ldr, int ny, int nx, int p, int stride, int C, int H,
                                          int W, int64_t j0, int64_t j1, void* canvas, void* count, void* stream) {
  if (!R || !canvas || ny <= 0 || nx <= 0 || p <= 0 || stride <= 0 || C <= 0 || H <= 0 || W <= 0 || ldr < (int64_t)p * p * C ||
      j0 < 0 || j1 <= j0 || j1 > (int64_t)ny * nx)
    return fail(ONMF_E_ARG, "patch_grid_accumulate: bad argument");
  if (dtype != ONMF_F32 && dtype != ONMF_F64) return fail(ONMF_E_ARG, "patch_grid_accumulate: bad dtype");
  // canvas rows of this range: those of its covering patches, gy(j0)*stride .. gy(j1-1)*stride + p, and the uncovered rows it
  // owns: up to the next grid row's first row, or to the bottom of the canvas after the last grid row
  const long long gy0 = j0 / nx, gy1 = (j1 - 1) / nx;
  long long y0 = gy0 * stride, y1 = gy1 * stride + p;
  const long long own_end = gy1 == ny - 1 ? (long long)H : (gy1 + 1) * stride;
  if (y1 < own_end) y1 = own_end;
  if (y1 > H) y1 = H;
  if (y0 >= y1) return ONMF_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const long long tot = (y1 - y0) * W * C;
  unsigned grid = (unsigned)cdiv<long long>(tot, 256);
  if (dtype == ONMF_F32)
    patch_grid_accumulate_kernel<float><<<grid, 256, 0, st>>>((const float*)R, ldr, ny, nx, p, stride, C, W, j0, j1, (int)y0, tot,
                                                               (float*)canvas, (float*)count);
  else
    patch_grid_accumulate_kernel<double><<<grid, 256, 0, st>>>((const double*)R, ldr, ny, nx, p, stride, C, W, j0, j1, (int)y0, tot,
                                                                (double*)canvas, (double*)count);
  ONMF_LAUNCH_CHECK("patch_grid_accumulate_kernel");
  return ONMF_OK;
}

extern "C" int onmf_patch_grid_mean(int dtype, const void* R, int64_t ldr, int ny, int nx, int p, int stride, int C, int H, int W,
                                    void* canvas, void* count, void* stream) {
  if (ny <= 0 || nx <= 0) return fail(ONMF_E_ARG, "patch_grid_mean: bad argument");
  return onmf_patch_grid_accumulate(dtype, R, ldr, ny, nx, p, stride, C, H, W, 0, (int64_t)ny * nx, canvas, count, stream);
}

// ------------------------------------------------------------------------------------------------
// NDL motif-adjacency patches (SURVEY.md §8f.4): X[j, q*kk + r] = G.has_edge(emb[j, q], emb[j, r])
// (reference network_reconstruction_nx.py:302-305, one k x k patch per MCMC state).  The graph is a CSR adjacency
// with sorted neighbour lists (both directions stored for an undirected graph); one thread per patch entry does a
// binary search in the row of emb[j, q].  The MCMC walk that produces `emb` is sequential and stays on the host.
// ------------------------------------------------------------------------------------------------
namespace onmf {
template <typename T>
__global__ void motif_patches_kernel(const long long* __restrict__ rowptr, const int* __restrict__ colidx, int n_nodes,
                                     const int* __restrict__ emb, long long n, int kk, T* __restrict__ Xt) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long per = (long long)kk * kk;
  if (idx >= n * per) return;
  const long long j = idx / per;
  const int e = (int)(idx - j * per);
  const int q = e / kk, r = e - q * kk;
  const int u = emb[j * kk + q], v = emb[j * kk + r];
  T val = T(0);
  if (u >= 0 && u < n_nodes && v >= 0 && v < n_nodes) {
    long long lo = rowptr[u], hi = rowptr[u + 1];
    while (lo < hi) {
      long long mid = (lo + hi) >> 1;
      int c = colidx[mid];
      if (c < v) lo = mid + 1;
      else hi = mid;
    }
    if (lo < rowptr[u + 1] && colidx[lo] == v) val = T(1);
  }
  Xt[idx] = val;
}

// Tiled form (k*k <= 1024): blockDim.x = the k*k entries of ONE patch, blockDim.y = patches per CTA.  The flat kernel above is
// issue-bound (ncu: 70 % issue-active, 0.07 of the HBM rate -- two 64-bit divisions and a 64-bit search per entry); here a
// thread keeps its (q, r) for the whole grid-stride loop, and the search runs on 32-bit offsets inside the row.
template <typename T>
__global__ void __launch_bounds__(1024) motif_patches_tile_kernel(const long long* __restrict__ rowptr, const int* __restrict__ colidx,
                                                                  int n_nodes, const int* __restrict__ emb, long long n, int kk,
                                                                  T* __restrict__ Xt) {
  const int e = threadIdx.x;
  const int q = e / kk, r = e - q * kk;
  const int per = kk * kk;
  const long long step = (long long)gridDim.x * blockDim.y;
  for (long long j = (long long)blockIdx.x * blockDim.y + threadIdx.y; j < n; j += step) {
    const int* em = emb + j * kk;
    const int u = __ldg(em + q), v = __ldg(em + r);
    T val = T(0);
    if ((unsigned)u < (unsigned)n_nodes && (unsigned)v < (unsigned)n_nodes) {
      const long long base = __ldg(rowptr + u);
      const int* row = colidx + base;
      const int len = (int)(__ldg(rowptr + u + 1) - base);
      int lo = 0, hi = len;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(row + mid) < v) lo = mid + 1;
        else hi = mid;
      }
      if (lo < len && __ldg(row + lo) == v) val = T(1);
    }
    Xt[(size_t)j * per + e] = val;
  }
}
}  // namespace onmf

extern "C" int onmf_motif_patches(int dtype, const int64_t* rowptr, const int32_t* colidx, int n_nodes, const int32_t* emb,
                                  int64_t n, int kk, void* Xt, void* stream) {
  if (!rowptr || !colidx || !emb || !Xt || n_nodes <= 0 || n < 0 || kk <= 0) return fail(ONMF_E_ARG, "motif_patches: bad argument");
  if (n == 0) return ONMF_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype != ONMF_F32 && dtype != ONMF_F64) return fail(ONMF_E_ARG, "motif_patches: bad dtype");
  if (kk * kk <= 1024) {
    const int per = kk * kk;
    int py = 256 / per;
    if (py < 1) py = 1;
    dim3 block((unsigned)per, (unsigned)py);
    long long gq = cdiv<long long>(n, py);
    const long long capq = (long long)num_sms() * (2048 / (per * py)) * 8;
    const int gridq = (int)(gq > capq ? capq : gq);
    if (dtype == ONMF_F32) motif_patches_tile_kernel<float><<<gridq, block, 0, st>>>((const long long*)rowptr, colidx, n_nodes, emb, n, kk, (float*)Xt);
    else motif_patches_tile_kernel<double><<<gridq, block, 0, st>>>((const long long*)rowptr, colidx, n_nodes, emb, n, kk, (double*)Xt);
    ONMF_LAUNCH_CHECK("motif_patches_tile_kernel");
    return ONMF_OK;
  }
  long long tot = n * (long long)kk * kk;
  unsigned grid = (unsigned)cdiv<long long>(tot, 256);
  if (dtype == ONMF_F32) motif_patches_kernel<float><<<grid, 256, 0, st>>>((const long long*)rowptr, colidx, n_nodes, emb, n, kk, (float*)Xt);
  else if (dtype == ONMF_F64) motif_patches_kernel<double><<<grid, 256, 0, st>>>((const long long*)rowptr, colidx, n_nodes, emb, n, kk, (double*)Xt);
  else return fail(ONMF_E_ARG, "motif_patches: bad dtype");
  ONMF_LAUNCH_CHECK("motif_patches_kernel");
  return ONMF_OK;
}

// ------------------------------------------------------------------------------------------------
// Batched network reconstruction (SURVEY.md §8f.1, second half): running-mean edge weights of
// network_reconstruction_nx.py:475-491.  The reference codes ONE k x k patch per MCMC step and, for every (q, r), folds
// patch_recons[q, r] into the weight of the directed edge (emb[q], emb[r]) as a running mean ((j*w + x)/(j + 1), count
// j + 1 kept in a second DiGraph).  A running mean over a sequence is its arithmetic mean, so for a whole trajectory the
// result is sum / count per distinct (a, b): one thread per (state, q, r) entry adds into an open-addressing hash table
// keyed by (a << 32 | b) -- FP64 sums, integer counts.  The caller sizes the table (power of two, > 2x the entries is
// always enough), fills the keys with 0xFF bytes and zeroes sums / counts.
// A streamed reconstruction keeps one table across many calls (onmf_edge_table_add): the kernel then also counts the slots
// it claims, so that the caller knows the load and can move the table into a larger one (onmf_edge_table_grow) in time.
// ------------------------------------------------------------------------------------------------
#include <cooperative_groups.h>
namespace onmf {
__device__ __forceinline__ unsigned long long mix64(unsigned long long x) {    // splitmix64 finaliser
  x ^= x >> 30; x *= 0xbf58476d1ce4e5b9ULL;
  x ^= x >> 27; x *= 0x94d049bb133111ebULL;
  x ^= x >> 31;
  return x;
}

template <typename T>
__global__ void edge_scatter_kernel(const T* __restrict__ R, long long ldr, const int* __restrict__ emb, long long n, int kk,
                                    unsigned long long* __restrict__ keys, double* __restrict__ sums,
                                    unsigned int* __restrict__ cnts, unsigned long long mask, unsigned int* __restrict__ failed,
                                    unsigned long long* __restrict__ claimed) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long per = (long long)kk * kk;
  if (idx >= n * per) return;
  const long long j = idx / per;
  const int e = (int)(idx - j * per);
  const int q = e / kk, r = e - q * kk;
  const int a = emb[j * kk + q], b = emb[j * kk + r];
  if (a < 0 || b < 0) { atomicAdd(failed, 1u); return; }
  const unsigned long long key = ((unsigned long long)(unsigned)a << 32) | (unsigned long long)(unsigned)b;
  const double val = (double)R[(size_t)j * ldr + e];
  unsigned long long h = mix64(key) & mask;
  for (unsigned long long probe = 0; probe <= mask; ++probe) {
    const unsigned long long prev = atomicCAS(&keys[h], ~0ULL, key);
    if (prev == ~0ULL || prev == key) {
      atomicAdd(&sums[h], val);
      atomicAdd(&cnts[h], 1u);
      if (claimed != nullptr && prev == ~0ULL) {        // a new pair: one atomic per group of lanes that claimed together
        const cooperative_groups::coalesced_group g = cooperative_groups::coalesced_threads();
        if (g.thread_rank() == 0) atomicAdd(claimed, (unsigned long long)g.size());
      }
      return;
    }
    h = (h + 1) & mask;
  }
  atomicAdd(failed, 1u);                      // table full (caller sized it too small)
}

// One thread per old slot.  Keys are unique, so an occupied slot is moved whole into the first free slot of its probe
// sequence in the new table: the CAS that wins an empty key owns that slot, and its sum and count are stored, not added.
__global__ void edge_table_grow_kernel(const unsigned long long* __restrict__ keys, const double* __restrict__ sums,
                                       const unsigned int* __restrict__ cnts, long long capacity,
                                       unsigned long long* __restrict__ new_keys, double* __restrict__ new_sums,
                                       unsigned int* __restrict__ new_cnts, unsigned long long new_mask,
                                       unsigned int* __restrict__ failed) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= capacity) return;
  const unsigned long long key = keys[i];
  if (key == ~0ULL) return;
  unsigned long long h = mix64(key) & new_mask;
  for (unsigned long long probe = 0; probe <= new_mask; ++probe) {
    if (atomicCAS(&new_keys[h], ~0ULL, key) == ~0ULL) {
      new_sums[h] = sums[i];
      new_cnts[h] = cnts[i];
      return;
    }
    h = (h + 1) & new_mask;
  }
  atomicAdd(failed, 1u);                      // new table full (load above 1/2 is never asked for)
}
}  // namespace onmf

static int edge_scatter(const char* name, int dtype, const void* R, int64_t ldr, const int32_t* emb, int64_t n, int kk,
                        unsigned long long* keys, double* sums, unsigned int* counts, int64_t capacity, unsigned int* failed,
                        unsigned long long* claimed, void* stream) {
  char msg[96];
  if (!R || !emb || !keys || !sums || !counts || !failed || n < 0 || kk <= 0 || ldr < (int64_t)kk * kk) {
    snprintf(msg, sizeof(msg), "%s: bad argument", name);
    return fail(ONMF_E_ARG, msg);
  }
  if (capacity <= 0 || (capacity & (capacity - 1))) {
    snprintf(msg, sizeof(msg), "%s: capacity must be a power of two", name);
    return fail(ONMF_E_ARG, msg);
  }
  if (n == 0) return ONMF_OK;
  if (dtype != ONMF_F32 && dtype != ONMF_F64) {
    snprintf(msg, sizeof(msg), "%s: bad dtype", name);
    return fail(ONMF_E_ARG, msg);
  }
  cudaStream_t st = (cudaStream_t)stream;
  const long long tot = n * (long long)kk * kk;
  const unsigned grid = (unsigned)cdiv<long long>(tot, 256);
  const unsigned long long mask = (unsigned long long)capacity - 1;
  if (dtype == ONMF_F32)
    edge_scatter_kernel<float><<<grid, 256, 0, st>>>((const float*)R, ldr, emb, n, kk, keys, sums, counts, mask, failed, claimed);
  else
    edge_scatter_kernel<double><<<grid, 256, 0, st>>>((const double*)R, ldr, emb, n, kk, keys, sums, counts, mask, failed, claimed);
  ONMF_LAUNCH_CHECK("edge_scatter_kernel");
  return ONMF_OK;
}

extern "C" int onmf_edge_scatter_add(int dtype, const void* R, int64_t ldr, const int32_t* emb, int64_t n, int kk,
                                     unsigned long long* keys, double* sums, unsigned int* counts, int64_t capacity,
                                     unsigned int* failed, void* stream) {
  return edge_scatter("edge_scatter_add", dtype, R, ldr, emb, n, kk, keys, sums, counts, capacity, failed, nullptr, stream);
}

extern "C" int onmf_edge_table_add(int dtype, const void* R, int64_t ldr, const int32_t* emb, int64_t n, int kk,
                                   unsigned long long* keys, double* sums, unsigned int* counts, int64_t capacity,
                                   unsigned long long* claimed, unsigned int* failed, void* stream) {
  if (!claimed) return fail(ONMF_E_ARG, "edge_table_add: bad argument");
  return edge_scatter("edge_table_add", dtype, R, ldr, emb, n, kk, keys, sums, counts, capacity, failed, claimed, stream);
}

extern "C" int onmf_edge_table_grow(const unsigned long long* keys, const double* sums, const unsigned int* counts,
                                    int64_t capacity, unsigned long long* new_keys, double* new_sums, unsigned int* new_counts,
                                    int64_t new_capacity, unsigned int* failed, void* stream) {
  if (!keys || !sums || !counts || !new_keys || !new_sums || !new_counts || !failed)
    return fail(ONMF_E_ARG, "edge_table_grow: bad argument");
  if (capacity <= 0 || (capacity & (capacity - 1)) || new_capacity <= 0 || (new_capacity & (new_capacity - 1)))
    return fail(ONMF_E_ARG, "edge_table_grow: capacities must be powers of two");
  if (new_capacity <= capacity) return fail(ONMF_E_ARG, "edge_table_grow: the new capacity must be larger than the old one");
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned grid = (unsigned)cdiv<long long>(capacity, 256);
  edge_table_grow_kernel<<<grid, 256, 0, st>>>(keys, sums, counts, capacity, new_keys, new_sums, new_counts,
                                               (unsigned long long)new_capacity - 1, failed);
  ONMF_LAUNCH_CHECK("edge_table_grow_kernel");
  return ONMF_OK;
}

// ------------------------------------------------------------------------------------------------
// Narrow STORAGE formats for streamed minibatches (arithmetic stays fp32): image data is 8-bit before the reference divides
// it by 255 (image_reconstruction.py:88 `data = np.asarray(img) / 255`), so a host-resident stream of patches can cross PCIe
// as u8 (or fp16) -- 4x (2x) fewer bytes than fp32 -- and be widened on the device.  dst = (float)src * scale, optionally
// written directly as the TF32 hi/lo pair of the tensor-core path (hi = rna_tf32(x), lo = x - hi).
// ------------------------------------------------------------------------------------------------
#include <cuda_fp16.h>
namespace onmf {
template <typename S> __device__ __forceinline__ float widen(S v);
template <> __device__ __forceinline__ float widen<unsigned char>(unsigned char v) { return (float)v; }
template <> __device__ __forceinline__ float widen<__half>(__half v) { return __half2float(v); }

template <typename S, bool SPLIT>
__global__ void widen_kernel(const S* __restrict__ src, long long count, float scale, float* __restrict__ dst, float* __restrict__ lo) {
  // 4 elements per thread per iteration (count % 4 == 0; src 4-element aligned): one 4- or 8-byte load, float4 stores
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < count / 4; i += stride) {
    S v[4];
    if (sizeof(S) == 1) *reinterpret_cast<uint32_t*>(v) = reinterpret_cast<const uint32_t*>(src)[i];
    else *reinterpret_cast<uint2*>(v) = reinterpret_cast<const uint2*>(src)[i];
    float x[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) x[e] = widen<S>(v[e]) * scale;
    if (SPLIT) {
      float h[4], l[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        uint32_t t;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(t) : "f"(x[e]));
        h[e] = __uint_as_float(t);
        l[e] = x[e] - h[e];
      }
      reinterpret_cast<float4*>(dst)[i] = make_float4(h[0], h[1], h[2], h[3]);
      reinterpret_cast<float4*>(lo)[i] = make_float4(l[0], l[1], l[2], l[3]);
    } else {
      reinterpret_cast<float4*>(dst)[i] = make_float4(x[0], x[1], x[2], x[3]);
    }
  }
}
}  // namespace onmf

extern "C" int onmf_widen(int src_kind, const void* src, int64_t count, double scale, void* dst, void* lo, void* stream) {
  if (!src || !dst || count < 0 || count % 4) return fail(ONMF_E_ARG, "widen: bad argument (count must be a multiple of 4)");
  if (src_kind != ONMF_STORE_U8 && src_kind != ONMF_STORE_F16) return fail(ONMF_E_ARG, "widen: src_kind must be ONMF_STORE_U8 or ONMF_STORE_F16");
  if ((reinterpret_cast<uintptr_t>(src) & 7) || (reinterpret_cast<uintptr_t>(dst) & 15) || (lo && (reinterpret_cast<uintptr_t>(lo) & 15)))
    return fail(ONMF_E_ARG, "widen: pointers must be aligned (src 8 B, dst/lo 16 B)");
  if (count == 0) return ONMF_OK;
  cudaStream_t st = (cudaStream_t)stream;
  int grid = (int)cdiv<long long>(count / 4, 256);
  if (grid > 16 * num_sms()) grid = 16 * num_sms();
  const float sc = (float)scale;
  if (src_kind == ONMF_STORE_U8) {
    if (lo) widen_kernel<unsigned char, true><<<grid, 256, 0, st>>>((const unsigned char*)src, count, sc, (float*)dst, (float*)lo);
    else widen_kernel<unsigned char, false><<<grid, 256, 0, st>>>((const unsigned char*)src, count, sc, (float*)dst, nullptr);
  } else {
    if (lo) widen_kernel<__half, true><<<grid, 256, 0, st>>>((const __half*)src, count, sc, (float*)dst, (float*)lo);
    else widen_kernel<__half, false><<<grid, 256, 0, st>>>((const __half*)src, count, sc, (float*)dst, nullptr);
  }
  ONMF_LAUNCH_CHECK("widen_kernel");
  return ONMF_OK;
}
