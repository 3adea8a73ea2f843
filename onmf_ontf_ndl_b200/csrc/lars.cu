// K3 -- batched positive LARS-lasso sparse coder for sm_100a.
//
// Replaces SparseCoder(transform_algorithm='lasso_lars', positive_code=True).transform as called at
// reference src/ontf.py:79-86, i.e. the per-sample Python loop of LassoLars._fit
// (sklearn/linear_model/_least_angle.py:1136-1153) around _lars_path_solver (:415-917; Gram mode,
// method='lasso', positive=True, return_path=False).
//
// Mapping: one lane-group (LPC = 8/16/32 lanes) follows the homotopy path of one minibatch column; a
// warp carries 32/LPC columns, a CTA carries NW warps, columns are handed out through a global ticket
// counter.  The Gram matrix G = W^T W is staged once per CTA in shared memory when it fits (k <= 128 in
// fp32), otherwise read through L1/L2 with the row loads of a pass batched four rows deep.  Each group
// keeps the INVERSE CHOLESKY FACTOR V of its active Gram block (G_AA^-1 = V V^T, V upper triangular in join
// order) as packed FP64 columns in its own shared-memory tile.  A join appends one column after two read-only,
// lane-parallel sweeps t = V^T g, u = V t (pivot sigma = G_jj - |t|^2); a drop closes the slot gap and
// downdates V by Givens rotations of adjacent columns -- against sklearn's Cholesky append + two triangular
// solves (3 s dependent steps per knot).  The equiangular weights w = G_AA^-1 1 are maintained incrementally.
// V is FP64 also in the fp32 production mode, and is built from the FP64-accumulated Gram when the caller
// supplies it (onmf_lasso_lars_g64): the inverse amplifies the independent per-entry rounding of an fp32 Gram
// by cond(G) (~4e5 on the early online dictionaries), the exact Gram of the stored dictionary only sees
// cond(W) (DESIGN.md section 2).  Covariances, correlations, step lengths and coefficients are in the working
// precision T.  Cross-lane reductions are single REDUX instructions on order-preserving integer keys (fp32)
// or shuffle trees (fp64 / sums); the only barriers are __syncwarp().
//
// Path semantics reproduced from sklearn (so the result matches the reference also where sklearn is
// not at the exact lasso optimum, SURVEY.md §B.2):
//   - join: inactive atom with the largest covariance (ties: lowest index)
//   - recorded alpha of a knot = max INACTIVE covariance / d; stop when alpha <= alpha/d + eps32 and
//     interpolate linearly between the last two coefficient vectors (incl. the atom dropped by the last
//     step, which is still positive inside that segment)
//   - step gamma = min(min_pos((C-c_i)/(AA-a_i+tiny32)), C/AA); drop when a coefficient would cross 0
//     first (gamma = z_pos), no atom joins on the iteration after a drop, the dropped atom's covariance
//     is recomputed exactly.  fp32 only: an atom that ties EXACTLY with the joining one takes a zero-length
//     step and joins next (sklearn steps past it; in fp32 near-ties round to exact ones, see step 6)
//   - "alpha increasing" bail-out, degenerate-pivot rejection (cov := 0), max_iter.
// Columns whose active set outgrows a tier's slot count are queued (device-side list) and re-walked by the next tier.
// k <= 128: 32 -> 64 -> 128 slots, all in shared memory.  k > 128: a HYBRID first tier with 64 slots whose packed
// factor keeps columns 0..39 in shared memory (16 warps/SM) and columns 40..63 in an L2-resident global scratch, so the
// common case (active set <= 40) runs entirely out of shared memory and the occasional larger set costs a few global
// accesses instead of a re-walk; then 128 slots in shared memory, then k slots with V in global memory.
#include <math_constants.h>

#include <type_traits>

#include "common.cuh"

namespace onmf {

#ifndef LARS_EARLY
#define LARS_EARLY 1
#endif
#ifndef LARS_MAX_THREADS
#define LARS_MAX_THREADS 512     // 16 warps/SM at <= 128 registers per thread (20 warps at 96 registers measured no faster)
#endif

template <typename T>
struct LarsParams {
  const T* G;        // k x k   (working precision; may be null when G64 is given)
  const double* G64; // k x k FP64 Gram (exact Gram of the stored dictionary) feeding the active-block inverse, or null
  const T* Gp;       // k x KP zero-padded copy (workspace)
  const T* Ct;       // n x k
  T* Ht;             // n x k
  long long n;
  int k, d, max_iter;
  T amin;            // alpha / d
  unsigned long long* ticket;        // work counter (zeroed by the host wrapper)
  const long long* col_list;         // later tiers: columns to solve (else nullptr)
  const unsigned int* n_list;        // later tiers: device-side count
  long long* ovf_list;               // columns whose active set outgrew this tier
  unsigned int* ovf_count;
  double* Mscratch;                  // last tier: per-group M storage in global memory
  double* Mhyb;                      // hybrid tier: rows >= SPLIT of every resident group's packed M (global/L2)
  onmf_lars_stats* stats;
  int count_stats;                   // 1 on the first tier (overflow columns are counted once)
  unsigned int* over_thresh;         // counts finished columns whose active set exceeded `thresh` (scheduling feedback)
  int thresh;
  const unsigned int* hint;          // device-side scheduling state: the kernel runs only if *hint == run_if
  int run_if;
};

template <typename T> struct Num;
template <> struct Num<float> {
  static __device__ __forceinline__ float inf() { return CUDART_INF_F; }
  static __device__ __forceinline__ float big() { return 3.402823466e+38f; }
};
template <> struct Num<double> {
  static __device__ __forceinline__ double inf() { return CUDART_INF; }
  static __device__ __forceinline__ double big() { return 1.7976931348623157e+308; }
};

// ---- group reductions ------------------------------------------------------------------------------
template <int LPC>
__device__ __forceinline__ double gsum(double v) {
#pragma unroll
  for (int off = LPC / 2; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  return v;
}
template <int LPC>
__device__ __forceinline__ float gsum(float v) {
#pragma unroll
  for (int off = LPC / 2; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  return v;
}
__device__ __forceinline__ unsigned fkey(float f) {     // order-preserving float -> uint
  unsigned u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float fkey_inv(unsigned k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}
// (max value, lowest index attaining it)
template <int LPC>
__device__ __forceinline__ void gargmax(float& v, int& i, unsigned gmask) {
  unsigned key = fkey(v);
  unsigned kmax = __reduce_max_sync(gmask, key);
  int cand = (key == kmax) ? i : 0x7fffffff;
  i = __reduce_min_sync(gmask, cand);
  v = fkey_inv(kmax);
}
template <int LPC>
__device__ __forceinline__ void gargmax(double& v, int& i, unsigned) {
#pragma unroll
  for (int off = LPC / 2; off > 0; off >>= 1) {
    double ov = __shfl_xor_sync(0xffffffffu, v, off);
    int oi = __shfl_xor_sync(0xffffffffu, i, off);
    if (ov > v || (ov == v && oi < i)) { v = ov; i = oi; }
  }
}
// group maximum (fp32: one REDUX on the order-preserving key)
template <int LPC>
__device__ __forceinline__ float gmaxval(float v, unsigned gmask) {
  return fkey_inv(__reduce_max_sync(gmask, fkey(v)));
}
template <int LPC>
__device__ __forceinline__ double gmaxval(double v, unsigned) {
#pragma unroll
  for (int off = LPC / 2; off > 0; off >>= 1) {
    double o = __shfl_xor_sync(0xffffffffu, v, off);
    v = o > v ? o : v;
  }
  return v;
}
// min over strictly positive candidates (callers pass big() for "none")
template <int LPC>
__device__ __forceinline__ float gminpos(float v, unsigned gmask) {
  return __uint_as_float(__reduce_min_sync(gmask, __float_as_uint(v)));
}
template <int LPC>
__device__ __forceinline__ double gminpos(double v, unsigned) {
#pragma unroll
  for (int off = LPC / 2; off > 0; off >>= 1) {
    double o = __shfl_xor_sync(0xffffffffu, v, off);
    v = o < v ? o : v;
  }
  return v;
}
// (min positive value, highest slot attaining it)
template <int LPC>
__device__ __forceinline__ void gargminpos(float& v, int& s, unsigned gmask) {
  unsigned key = __float_as_uint(v);
  unsigned kmin = __reduce_min_sync(gmask, key);
  int cand = (key == kmin) ? s : -1;
  s = __reduce_max_sync(gmask, cand);
  v = __uint_as_float(kmin);
}
template <int LPC>
__device__ __forceinline__ void gargminpos(double& v, int& s, unsigned) {
#pragma unroll
  for (int off = LPC / 2; off > 0; off >>= 1) {
    double ov = __shfl_xor_sync(0xffffffffu, v, off);
    int os = __shfl_xor_sync(0xffffffffu, s, off);
    if (ov < v || (ov == v && os > s)) { v = ov; s = os; }
  }
}

// ---- fast FP64 reciprocal / reciprocal square root: fp32 seed + two Newton steps (rel. error < 1e-14) ----
__device__ __forceinline__ double fast_rcp(double x) {
  double y = (double)__frcp_rn((float)x);
  y = y * (2.0 - x * y);
  y = y * (2.0 - x * y);
  return y;
}
__device__ __forceinline__ double fast_rsqrt(double x) {
  double y = (double)rsqrtf((float)x);
  y = y * (1.5 - 0.5 * x * y * y);
  y = y * (1.5 - 0.5 * x * y * y);
  return y;
}
// one Newton step: ~1e-13 relative, enough where the result is rounded to fp32 anyway
__device__ __forceinline__ double fast_rsqrt1(double x) {
  double y = (double)rsqrtf((float)x);
  return y * (1.5 - 0.5 * x * y * y);
}
__device__ __forceinline__ float qdiv(float a, float b) {      // step-length candidates: a * rcp.approx(b), 2 instructions
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(b));
  return a * r;
}
__device__ __forceinline__ double qdiv(double a, double b) { return a / b; }

template <typename T> struct VecOf;
template <> struct VecOf<float> { typedef float4 type; static constexpr int N = 4; };
template <> struct VecOf<double> { typedef double2 type; static constexpr int N = 2; };

// vector load from a global address held as an integer (keeps LDG instead of a generic LD once the base is opaque)
__device__ __forceinline__ float4 ld_global_vec(const float4* p) {
  float4 v;
  asm("ld.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ double2 ld_global_vec(const double2* p) {
  double2 v;
  asm("ld.global.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p));
  return v;
}

// slot entry read by the correlation pass: (atom, normalised weight); free slots hold (0, 0)
template <typename T> struct SlotW;
template <> struct __align__(8) SlotW<float> { int atom; float w; };
template <> struct __align__(16) SlotW<double> { int atom; int pad; double w; };

// shared-memory words (4 B) one group needs: the FP64 factor V (packed columns; absent when it lives in global),
// g/t (FP64), slot entries, slot->atom
template <typename T, int LPC, int SMAX, bool MGLOB, int SPLIT = 0>
__host__ __device__ constexpr int group_words() {
  // SPLIT > 0: only the first SPLIT columns of the packed factor live in shared memory, the rest in global scratch
  int mwords = (SPLIT > 0) ? SPLIT * (SPLIT + 1) : SMAX * (SMAX + 1);
  int sv = (SMAX + LPC - 1) / LPC * LPC;
  int w = (MGLOB ? 0 : mwords) + 4 * sv + sv * (int)(sizeof(SlotW<T>) / 4) + sv;
  w = (w + 3) & ~3;                       // keep 16-byte alignment of the next group
  if (LPC < 32) {                         // start consecutive groups of a warp 2*LPC banks apart
    int r = w % 32;
    int want = (2 * LPC) % 32;
    w += (want - r + 32) % 32;
  }
  return w;
}
template <int LPC, int NA>
__host__ __device__ constexpr int gram_stride() {
  return LPC * NA + (LPC < 32 ? LPC : 0);
}

// G (k x k) -> Gp (k x KP) zero-padded rows, so that every Gram row read is an aligned, unpredicated vector load
template <typename T>
__global__ void pad_gram_kernel(const T* __restrict__ G, const double* __restrict__ G64, int k, int kp, T* __restrict__ Gp) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= k * kp) return;
  int a = idx / kp, i = idx - a * kp;
  Gp[idx] = (i < k) ? (G64 ? (T)G64[(size_t)a * k + i] : G[(size_t)a * k + i]) : T(0);
}

template <typename T, int LPC, int NA, int SMAX, bool GSM, bool MGLOB, int SPLIT>
__global__ void __launch_bounds__(LARS_MAX_THREADS, 1) lars_kernel(LarsParams<T> P) {
  typedef typename VecOf<T>::type VT;
  constexpr int VEC = VecOf<T>::N;
  constexpr int SA = (SMAX + LPC - 1) / LPC;   // active slots per lane
  constexpr int SV = SA * LPC;                 // length of the per-slot vectors (>= SMAX)
  constexpr int GPW = 32 / LPC;        // columns per warp
  constexpr int KP = LPC * NA;
  constexpr int GS = GSM ? gram_stride<LPC, NA>() : KP;   // row stride of the Gram copy this kernel reads
  constexpr int UQ = (NA >= 16 || sizeof(T) == 8) ? 2 : 4;  // Gram rows in flight per correlation-pass batch
  static_assert(NA % VEC == 0 && SMAX % 4 == 0, "bad tile shape");

  if (P.hint != nullptr && *P.hint != (unsigned)P.run_if) return;   // the other first-tier variant handles this call
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int k = P.k;
  T* Gs = reinterpret_cast<T*>(smem_raw);
  const size_t g_bytes = GSM ? round_up<size_t>((size_t)k * GS * sizeof(T), 128) : 0;
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int l = lane % LPC;
  const int gid = warp * GPW + lane / LPC;           // group id inside the CTA
  const unsigned gmask = (LPC == 32) ? 0xffffffffu : (((1u << (LPC & 31)) - 1u) << ((lane / LPC) * LPC));
  uint32_t* gbase = reinterpret_cast<uint32_t*>(smem_raw + g_bytes) +
                    (size_t)gid * group_words<T, LPC, SMAX, MGLOB, SPLIT>();
  static_assert(SPLIT == 0 || (SPLIT < SMAX && !MGLOB), "hybrid tiers keep the first SPLIT columns in shared memory");
  // V: the inverse Cholesky factor of the active Gram block, G_AA^-1 = V V^T, V upper triangular in join order.
  // Column i (the atom in slot i) is stored packed at [i(i+1)/2, i(i+1)/2 + i]: lanes reading one column touch
  // consecutive doubles, a lane walking down its own column touches offsets whose banks differ per half-warp.
  constexpr int MELEMS = SMAX * (SMAX + 1) / 2;
  constexpr int MSM = SPLIT > 0 ? SPLIT * (SPLIT + 1) / 2 : MELEMS;   // doubles of V kept in shared memory
  double* Mg;
  double* vecs;
  double* Mx = nullptr;                                // columns >= SPLIT of V (hybrid tiers)
  if (MGLOB) {
    Mg = P.Mscratch + ((size_t)blockIdx.x * (blockDim.x / LPC) + gid) * (size_t)MELEMS;
    vecs = reinterpret_cast<double*>(gbase);
  } else {
    Mg = reinterpret_cast<double*>(gbase);
    vecs = Mg + MSM;
    if (SPLIT > 0) Mx = P.Mhyb + ((size_t)blockIdx.x * (blockDim.x / LPC) + gid) * (size_t)(MELEMS - MSM);
  }
  double* gs = vecs;                                   // g = G[active, j]
  double* us = vecs + SV;                              // t = V^T g
  SlotW<T>* sw_ = reinterpret_cast<SlotW<T>*>(vecs + 2 * SV);     // (atom, normalised weight) by slot
  int* acts = reinterpret_cast<int*>(sw_ + SV);        // slot -> atom (-1 beyond the active count)

  // atom owned by (lane l, register m): VEC consecutive atoms per lane per vector load
  auto atom_of = [&](int m) -> int { return ((m / VEC) * LPC + l) * VEC + (m % VEC); };

  if (GSM) {
    for (int idx = threadIdx.x; idx < k * GS; idx += blockDim.x) {
      int a = idx / GS, i = idx - a * GS;
      Gs[idx] = (i < k) ? (P.G64 ? (T)P.G64[(size_t)a * k + i] : P.G[(size_t)a * k + i]) : T(0);
    }
    __syncthreads();
  }
  const T* Gr = GSM ? Gs : P.Gp;                       // padded rows, stride GS
  auto Gat = [&](int a, int i) -> T { return Gr[a * GS + i]; };
  // this lane's byte offset inside a Gram row, folded into the base once: a row address is one IMAD.WIDE
  // (kept opaque so that the compiler holds it in a register pair instead of re-deriving it from uniform registers)
  unsigned long long Grl = reinterpret_cast<unsigned long long>(Gr) + (unsigned long long)l * sizeof(VT);
  if (!GSM) asm volatile("" : "+l"(Grl));
  // Gram entries that enter the factor: FP64 when the caller supplies the FP64 Gram
  const double* __restrict__ G64 = P.G64;
  auto Gd = [&](int a, int i) -> double { return G64 ? G64[(size_t)a * k + i] : (double)Gat(a, i); };

  const T tiny = T(1.1754943508222875e-38);      // np.finfo(np.float32).tiny
  const T dT = T(P.d);
  // np.finfo(np.float32).eps (sklearn's equality_tolerance); fp32 coder: alpha and the tolerance in covariance units
  const T eps32 = (sizeof(T) == 4) ? T(1.1920928955078125e-07) * dT : T(1.1920928955078125e-07);
  const T amin = (sizeof(T) == 4) ? P.amin * dT : P.amin;

  int ci[SA];                                    // start of this lane's own columns in the packed factor
#pragma unroll
  for (int m = 0; m < SA; ++m) { const int i = l + LPC * m; ci[m] = i * (i + 1) / 2; }

  // ---- the two sweeps over the packed factor ----
  // Columns >= SPLIT of a hybrid tier live in the global tail (Mx); the sweeps are compiled twice and the
  // shared-memory-only version runs while the active set fits the shared part.
  // t_i = sum_{p <= i} V[p][i] src[p]   for the slots i < lim of the groups with `on`; src (shared) has nW valid entries
  auto sweep_t = [&](double (&t)[SA], const double* src, int nW, int lim, bool on) {
    int ie[SA];
#pragma unroll
    for (int m = 0; m < SA; ++m) { const int i = l + LPC * m; ie[m] = (on && i < lim) ? i : -1; }
    const int mMax = (nW + LPC - 1) / LPC;
    if (SPLIT > 0 && nW > SPLIT) {
      const double* colp[SA];                    // generic pointers: a lane's column is in shared or in global memory
#pragma unroll
      for (int m = 0; m < SA; ++m) colp[m] = (l + LPC * m >= SPLIT) ? (Mx + (ci[m] - MSM)) : (Mg + ci[m]);
#pragma unroll 2
      for (int p = 0; p < nW; ++p) {
        const double sp = src[p];
#pragma unroll
        for (int m = 0; m < SA; ++m)
          if (m < mMax && p <= ie[m]) t[m] += colp[m][p] * sp;
      }
    } else if (mMax <= 1) {                          // the common case: at most LPC active atoms, one slot register
#pragma unroll 4
      for (int p = 0; p < nW; ++p) {
        const double sp = src[p];
        if (p <= ie[0]) t[0] += Mg[ci[0] + p] * sp;
      }
    } else {
#pragma unroll 4
      for (int p = 0; p < nW; ++p) {
        const double sp = src[p];
#pragma unroll
        for (int m = 0; m < SA; ++m)
          if (m < mMax && p <= ie[m]) t[m] += Mg[ci[m] + p] * sp;
      }
    }
  };
  // u_p = sum_{p <= i < lim} V[p][i] src[i]; *ssq (when given) receives sum_i src[i]^2 in ascending order -- every lane
  // reads the whole source vector anyway, so |t|^2 of a join costs no cross-lane reduction (entries beyond a group's own
  // count are exact zeros)
  auto sweep_u = [&](double (&u)[SA], const double* src, int nW, int lim, bool on, double* ssq = nullptr) {
    double sq = 0.0;
    int pe[SA];
#pragma unroll
    for (int m = 0; m < SA; ++m) pe[m] = on ? (l + LPC * m) : 0x7fffffff;
    const int lim_e = (LPC == 32) ? nW : (on ? lim : 0);
    const int nS = (SPLIT > 0 && nW > SPLIT) ? SPLIT : nW;
    const double* rp = Mg + l;                     // &V[l][i] for the current column i
    const int nS1 = nS < LPC ? nS : LPC;           // columns < LPC only reach the first slot register
#pragma unroll 4
    for (int i = 0; i < nS1; ++i) {
      const double si = src[i];
      sq = fma(si, si, sq);
      if (pe[0] <= i && (LPC == 32 || i < lim_e)) u[0] += rp[0] * si;
      rp += i + 1;
    }
#pragma unroll 2
    for (int i = nS1; i < nS; ++i) {
      const double si = src[i];
      sq = fma(si, si, sq);
#pragma unroll
      for (int m = 0; m < SA; ++m)
        if (LPC * m <= i && pe[m] <= i && (LPC == 32 || i < lim_e)) u[m] += rp[LPC * m] * si;
      rp += i + 1;
    }
    if (SPLIT > 0 && nW > SPLIT) {
      rp = Mx + l;
#pragma unroll 2
      for (int i = SPLIT; i < nW; ++i) {
        const double si = src[i];
        sq = fma(si, si, sq);
#pragma unroll
        for (int m = 0; m < SA; ++m)
          if (LPC * m <= i && pe[m] <= i && (LPC == 32 || i < lim_e)) u[m] += rp[LPC * m] * si;
        rp += i + 1;
      }
    }
    if (ssq) *ssq = sq;
  };
  auto Vld = [&](int idx) -> double { return (SPLIT > 0 && idx >= MSM) ? Mx[idx - MSM] : Mg[idx]; };
  auto Vst = [&](int idx, double v) {
    if (SPLIT > 0 && idx >= MSM) Mx[idx - MSM] = v; else Mg[idx] = v;
  };
  // column `s` of the factor for the atom `a` joining the atoms in slots 0..s-1 (groups with `on`); sW = warp-wide
  // bound on s.  Returns the pivot sigma = G_aa - |t|^2; u = G_AA^-1 G[A, a] is left in u[], the column is NOT written.
  auto border = [&](int a, int s, int sW, bool on, double (&u)[SA]) -> double {
#pragma unroll
    for (int m = 0; m < SA; ++m) {
      if (LPC * m < sW) {
        const int p = l + LPC * m;
        double gv = 0.0;
        if (on && p < s) gv = Gd(a, acts[p]);      // row a of the (bitwise symmetric) Gram: one 8k-byte region for all lanes
        gs[p] = gv;
      }
    }
    __syncwarp();
    double t[SA];
#pragma unroll
    for (int m = 0; m < SA; ++m) { t[m] = 0.0; u[m] = 0.0; }
    sweep_t(t, gs, sW, s, on);
#pragma unroll
    for (int m = 0; m < SA; ++m)
      if (LPC * m < sW) us[l + LPC * m] = t[m];
    __syncwarp();
    double tt = 0.0;
    sweep_u(u, us, sW, s, on, &tt);
    return (on ? Gd(a, a) : 1.0) - tt;
  };

  unsigned long long st_knots = 0, st_s = 0, st_s2 = 0, st_drops = 0, st_flag = 0, st_cols = 0, st_ovf = 0;
  int st_maxact = 0;

  while (true) {
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(P.ticket, (unsigned long long)GPW);
    base = __shfl_sync(0xffffffffu, base, 0);
    const unsigned long long nwork = P.col_list ? (unsigned long long)(*P.n_list) : (unsigned long long)P.n;
    if (base >= nwork) break;
    const unsigned long long widx = base + lane / LPC;
    const bool valid = widx < nwork;
    const long long col = valid ? (P.col_list ? P.col_list[widx] : (long long)widx) : 0;
    const T* crow = P.Ct + (size_t)col * k;

    // ---- per-column state ----
    // active atoms (and the padding beyond k) carry cov = -inf: they never win the arg-max, their step-length
    // candidate is +inf or NaN (both fail "v < g1"), and -inf stays -inf under the covariance update -- no mask tests
    T cov[NA];
#pragma unroll
    for (int m = 0; m < NA; ++m) {
      int i = atom_of(m);
      bool ok = valid && i < k;
      cov[m] = ok ? crow[i] : -Num<T>::inf();
    }
    // per-slot registers; slots are compact (0..n_act-1 in join order), everything beyond n_act is zero
    T coef[SA], prev[SA];
    double wd[SA];                       // unnormalised equiangular weights G_AA^-1 1, maintained incrementally
#pragma unroll
    for (int m = 0; m < SA; ++m) {
      coef[m] = T(0); prev[m] = T(0); wd[m] = 0.0;
      SlotW<T> z; z.atom = 0; z.w = T(0);
      sw_[l + LPC * m] = z;
      acts[l + LPC * m] = -1;
    }
    double sw = 0.0;                     // sum of wd (group-uniform)
    int n_iter = 0, n_act = 0, status = 0, max_act = 0;
    unsigned kn_s = 0, kn_s2 = 0;        // per-column work counters (flushed to the 64-bit totals once per column)
    bool drop = false, done = !valid;
    int dslot = 0;
    T a_prev = T(0);
    // the atom dropped by the last step: inactive from now on, but sklearn's prev_coef still holds its value
    // at the previous knot, which matters when the path stops inside the segment that ended with the drop.
    int ghost_atom = -1;
    T ghost_prev = T(0), ghost_val = T(0);
    int banned = -1;                     // fp32: atom dropped by the most recent drop step (see the arg-max)

    while (!__all_sync(0xffffffffu, done)) {
      __syncwarp();
      // ---- 1. largest inactive covariance ----
      T best = -Num<T>::inf();
      int bi = 0x7fffffff;
      if (sizeof(T) == 4) {
        // value first (FMNMX + one REDUX), then the lowest atom attaining it (atom_of(m) increases with m)
#pragma unroll
        for (int m = 0; m < NA; ++m) best = cov[m] > best ? cov[m] : best;
        best = gmaxval<LPC>(best, gmask);
#pragma unroll
        for (int m = NA - 1; m >= 0; --m)
          if (cov[m] == best) bi = atom_of(m);
        bi = __reduce_min_sync(gmask, bi);
        // fp32 only: the atom dropped by the last drop step can never be the joiner of the first join knot after it -- in
        // exact arithmetic its covariance has fallen strictly below the active level by then (it left because its
        // correlation decays faster than the level).  When the drop and the next join are a near-tie (the step between
        // them shorter than one ulp of the covariances) its recomputed covariance can round to the level or one ulp above,
        // it wins the arg-max, re-enters with coefficient 0 and the path derails (one column's code off by 30 %, enough to
        // move the dictionary by 1e-3: tests/test_gpu_parity.py::test_cfg5_full_run_fp32_bars).  sklearn's float64 loop
        // has the same hazard at 1e-16 instead of 1e-7; the fp64 coder stays literal.
        const bool use_ban = (banned >= 0) && !drop && !done;
        if (__any_sync(0xffffffffu, use_ban && bi == banned)) {
          T b2 = -Num<T>::inf();
          int i2 = 0x7fffffff;
#pragma unroll
          for (int m = 0; m < NA; ++m) {
            const T cv = (use_ban && atom_of(m) == banned) ? -Num<T>::inf() : cov[m];
            b2 = cv > b2 ? cv : b2;
          }
          b2 = gmaxval<LPC>(b2, gmask);
#pragma unroll
          for (int m = NA - 1; m >= 0; --m)
            if (cov[m] == b2 && !(use_ban && atom_of(m) == banned)) i2 = atom_of(m);
          i2 = __reduce_min_sync(gmask, i2);
          if (use_ban && bi == banned && b2 > -Num<T>::inf()) { best = b2; bi = i2; }   // (no other candidate: keep it)
        }
        if (!drop) banned = -1;
      } else {
#pragma unroll
        for (int m = 0; m < NA; ++m) {
          const int i = atom_of(m);
          if (cov[m] > best || (cov[m] == best && i < bi)) { best = cov[m]; bi = i; }
        }
        gargmax<LPC>(best, bi, gmask);
      }
      const bool any_inact = best > -Num<T>::inf();
      const T C = any_inact ? best : T(0);
      // recorded alpha of the knot = C / d (sklearn divides by n_samples).  The fp32 coder keeps it in covariance units
      // (a = C, thresholds scaled by d): same decisions up to rounding, one division less per knot
      const T a_cur = (sizeof(T) == 4) ? C : C / dT;
      bool do_add = false, skip = false;
      if (!done) {
        if (a_cur <= amin + eps32) {
          T diff = a_cur - amin;
          if ((diff > eps32 || diff < -eps32) && n_iter > 0) {
            T ss = (a_prev - amin) / (a_prev - a_cur);
#pragma unroll
            for (int m = 0; m < SA; ++m) coef[m] = prev[m] + ss * (coef[m] - prev[m]);
            if (ghost_atom >= 0) ghost_val = ghost_prev - ss * ghost_prev;
          }
          done = true;
        } else if (n_iter >= P.max_iter || n_act >= k) {
          if (n_iter >= P.max_iter) status |= 4;
          done = true;
        } else {
          do_add = !drop;
        }
      }

      // ---- 2. atom j joins slot n_act: new column of the factor, w = G_AA^-1 1 updated incrementally ----
      if (__any_sync(0xffffffffu, do_add)) {
        const int j = bi;
        if (do_add && n_act >= SMAX) {       // active set outgrew this tier: hand the column to the next one
          status |= 8;
          done = true;
          do_add = false;
        }
        const int sW = __reduce_max_sync(0xffffffffu, do_add ? n_act : 0);
        double u[SA];
        const double sig = border(do_add ? j : 0, n_act, sW, do_add, u);
        // sklearn: diag = max(sqrt(|c - v|), eps); degenerate if diag < 1e-7  <=>  |sig| < 1e-14
        double asig = fabs(sig);
        asig = asig > 4.930380657631324e-32 ? asig : 4.930380657631324e-32;
        bool degen = asig < 1e-14;
        // an fp32 Gram cannot resolve a Schur complement below its own rounding noise
        if (sizeof(T) == 4 && G64 == nullptr) degen = degen || !(sig > 4.0 * 1.1920928955078125e-07 * Gd(do_add ? j : 0, do_add ? j : 0));
        // degenerate regressor (sklearn _least_angle.py:723-742): covariance zeroed, atom stays inactive;
        // otherwise the atom turns active (cov = -inf)
        if (do_add) {
          const T cnew = degen ? T(0) : -Num<T>::inf();
#pragma unroll
          for (int m = 0; m < NA; ++m)
            if (atom_of(m) == j) cov[m] = cnew;
        }
        if (do_add && degen) {
          status |= 1;
          do_add = false;
          skip = true;
        }
        double su = 0.0;
#pragma unroll
        for (int m = 0; m < SA; ++m) su += u[m];
        su = gsum<LPC>(su);
        if (do_add) {
          const double rs = fast_rsqrt(asig);
          const double tau = (1.0 - su) * rs * rs;         // new entry of G_AA^-1 1
          const int cs = n_act * (n_act + 1) / 2;
#pragma unroll
          for (int m = 0; m < SA; ++m) {
            const int p = l + LPC * m;
            if (p <= n_act) {
              Vst(cs + p, (p == n_act) ? rs : -u[m] * rs);
              wd[m] = (p == n_act) ? tau : wd[m] - tau * u[m];
              if (p == n_act) acts[p] = j;
            }
          }
          sw += tau * (1.0 - su);
          ++n_act;
          max_act = n_act > max_act ? n_act : max_act;
        }
        __syncwarp();
      }

#if LARS_EARLY
      // The Gram rows of the first correlation batch belong to slots 0..UQ-1, whose atoms are final once the join is
      // done: request them now, so that their L1/L2 latency overlaps the weight normalisation and the slot-table update
      constexpr bool EARLY = (!GSM && LPC == 32);
      VT gv0[EARLY ? UQ : 1][NA / VEC];
      if (EARLY) {
#pragma unroll
        for (int t = 0; t < UQ; ++t) {
          const int a0 = acts[t];
          const VT* row = reinterpret_cast<const VT*>(Grl + (unsigned long long)(unsigned)(a0 >= 0 ? a0 : 0) * (unsigned)(GS * sizeof(T)));
#pragma unroll
          for (int v = 0; v < NA / VEC; ++v) gv0[t][v] = ld_global_vec(row + v * LPC);
        }
      }
#endif
      // ---- 3. "alpha increasing" bail-out (sklearn _least_angle.py:752-765) ----
      if (!done && !skip && n_iter > 0 && a_prev < a_cur) {
        status |= 2;
        done = true;
      }
      bool live = !done && !skip;

      // ---- 4. normalise the equiangular weights: w = AA * G_AA^-1 1, AA = 1/sqrt(1^T G_AA^-1 1) ----
      if (live && !(sw > 0.0 && sw < 1e300)) {   // active Gram block numerically singular
        status |= 16;
        done = true;
        live = false;
      }
      const int hwL = __reduce_max_sync(0xffffffffu, live ? n_act : 0);
      const double AAd = live ? ((sizeof(T) == 4) ? fast_rsqrt1(sw) : fast_rsqrt(sw)) : 1.0;
      const T AA = (T)AAd;
      T w[SA];
#pragma unroll
      for (int m = 0; m < SA; ++m) {
        w[m] = (T)(wd[m] * AAd);
        if (LPC * m < hwL) {
          const int p = l + LPC * m;
          if (live && p < n_act) {
            SlotW<T> e; e.atom = acts[p]; e.w = w[m];
            sw_[p] = e;
          }
        }
      }
      __syncwarp();

      // ---- 5. correlation of every atom with the equiangular direction: G[:, A] w ----
      T corr[NA];
#pragma unroll
      for (int m = 0; m < NA; ++m) corr[m] = T(0);
#if LARS_EARLY
      if (EARLY && hwL > 0) {        // first batch: rows already requested (free slots carry weight 0, any row will do)
        SlotW<T> e[UQ];
#pragma unroll
        for (int t = 0; t < UQ; ++t) e[t] = sw_[t];
#pragma unroll
        for (int t = 0; t < UQ; ++t)
#pragma unroll
          for (int v = 0; v < NA / VEC; ++v) {
            const T* gp = reinterpret_cast<const T*>(&gv0[t][v]);
#pragma unroll
            for (int c = 0; c < VEC; ++c) corr[v * VEC + c] += gp[c] * e[t].w;
          }
      }
      for (int q0 = EARLY ? UQ : 0; q0 < hwL; q0 += UQ) {
#else
      for (int q0 = 0; q0 < hwL; q0 += UQ) {
#endif
        // slots beyond this group's active count hold (atom 0, weight 0): no masking needed
        SlotW<T> e[UQ];
#pragma unroll
        for (int t = 0; t < UQ; ++t) e[t] = sw_[q0 + t];
        VT gv[UQ][NA / VEC];
#pragma unroll
        for (int t = 0; t < UQ; ++t) {
          const VT* row = reinterpret_cast<const VT*>(Grl + (unsigned long long)(unsigned)e[t].atom * (unsigned)(GS * sizeof(T)));
#pragma unroll
          for (int v = 0; v < NA / VEC; ++v) gv[t][v] = GSM ? row[v * LPC] : ld_global_vec(row + v * LPC);
        }
#pragma unroll
        for (int t = 0; t < UQ; ++t)
#pragma unroll
          for (int v = 0; v < NA / VEC; ++v) {
            const T* gp = reinterpret_cast<const T*>(&gv[t][v]);
#pragma unroll
            for (int c = 0; c < VEC; ++c) corr[v * VEC + c] += gp[c] * e[t].w;
          }
      }
      if (sizeof(T) == 8) {
        // np.around(corr_eq_dir, decimals=15)  (sklearn _least_angle.py:806)
#pragma unroll
        for (int m = 0; m < NA; ++m) corr[m] = T(rint(double(corr[m]) * 1e15) / 1e15);
      }

      // ---- 6. step length ----
      T g1 = Num<T>::big();
#pragma unroll
      for (int m = 0; m < NA; ++m) {
        const T den = AA - corr[m] + tiny;
        // (fp32: an inactive covariance one ulp above C -- the just-dropped atom excluded from the arg-max -- is a tie)
        T v = qdiv((sizeof(T) == 4) ? (C - cov[m] > T(0) ? C - cov[m] : T(0)) : (C - cov[m]), den);
        // sklearn's min_pos takes strictly positive candidates.  C is the maximum, so the numerator is >= 0 and
        // v > 0 <=> den > 0 unless the atom TIES with the joining one (numerator exactly 0), where sklearn steps past
        // it.  In fp64 that is a structural (measure-zero) event and is reproduced literally; in fp32 a near-tie
        // rounds to an exact one now and then, and stepping past the atom changes the code by O(1) -- so the fp32
        // coder takes the zero-length step (the exact-arithmetic path: both atoms join).
        const bool ok = (sizeof(T) == 4) ? (den > T(0)) : (v > T(0));
        if (ok && v < g1) g1 = v;
      }
      g1 = gminpos<LPC>(g1, gmask);
      T gamma = qdiv(C, AA);
      gamma = g1 < gamma ? g1 : gamma;
      T zbest = Num<T>::big();
      int zs = -1;
#pragma unroll
      for (int m = 0; m < SA; ++m) {
        if (LPC * m < hwL) {
          int p = l + LPC * m;
          if (live && p < n_act) {
            T z = qdiv(-coef[m], w[m] + tiny);
            if (z > T(0) && z < zbest) { zbest = z; zs = p; }
          }
        }
      }
      gargminpos<LPC>(zbest, zs, gmask);
      if (live) {
        drop = false;
        if (zbest < gamma && zs >= 0) { gamma = zbest; drop = true; dslot = zs; }
        // ---- 7. move along the path ----
        ++n_iter;
        a_prev = a_cur;
        ghost_atom = -1;
#pragma unroll
        for (int m = 0; m < SA; ++m) {
          prev[m] = coef[m];
          coef[m] = prev[m] + gamma * w[m];
        }
#pragma unroll
        for (int m = 0; m < NA; ++m) cov[m] -= gamma * corr[m];
        kn_s += (unsigned)n_act;
        kn_s2 += (unsigned)(n_act * n_act);
      }

      // ---- 8. atom leaves slot p0: Givens downdate of the factor, Schur downdate of w, slots close up ----
      // With r = row p0 of V:  G'^-1 = V~ (I - r r^T / r^T r) V~^T  (V~ = V without row p0).  Rotating adjacent columns
      // p0, p0+1, ... so that r's weight moves into the running column leaves an upper-triangular factor of G'^-1 in
      // the first n_act-1 columns; the running column (parallel to V~ r) is discarded.  O(s (s - p0)) lane-parallel work.
      const bool dodrop = live && drop;
      if (__any_sync(0xffffffffu, dodrop)) {
        const int p0 = dodrop ? dslot : 0x7fffffff;
        const int a_d = dodrop ? acts[dslot] : 0;
        const int sD = __reduce_max_sync(0xffffffffu, dodrop ? n_act : 0);      // warp bound on the active count
        // r, and m = V r = column p0 of G_AA^-1
        double rr[SA], mv[SA], pre[SA];
        T gp = T(0);
        double wp0 = 0.0, rp0 = 0.0, mpp = 0.0;
#pragma unroll
        for (int m = 0; m < SA; ++m) {
          const int i = l + LPC * m;
          rr[m] = (dodrop && i >= p0 && i < n_act) ? Vld(ci[m] + p0) : 0.0;
          mv[m] = 0.0;
          if (LPC * m < sD) us[i] = rr[m];
          if (i == p0) { gp = prev[m]; wp0 = wd[m]; rp0 = rr[m]; }
          mpp += rr[m] * rr[m];
        }
        gp = gsum<LPC>(gp);
        wp0 = gsum<LPC>(wp0);
        rp0 = gsum<LPC>(rp0);
        mpp = gsum<LPC>(mpp);
        if (dodrop) { ghost_atom = a_d; ghost_prev = gp; banned = a_d; }
        __syncwarp();
        sweep_u(mv, us, sD, dodrop ? n_act : 0, dodrop);
        double sum_m = 0.0;
#pragma unroll
        for (int m = 0; m < SA; ++m) sum_m += mv[m];
        sum_m = gsum<LPC>(sum_m);
        const double fw = dodrop ? wp0 * fast_rcp(mpp) : 0.0;
        // inclusive prefix sums of r^2 over the slots (slot = l + LPC m: lanes first, then registers)
        {
          double run = 0.0;
#pragma unroll
          for (int m = 0; m < SA; ++m) {
            double x = rr[m] * rr[m];
#pragma unroll
            for (int off = 1; off < LPC; off <<= 1) {
              const double y = __shfl_up_sync(0xffffffffu, x, off, LPC);
              if (l >= off) x += y;
            }
            pre[m] = x + run;
            run += __shfl_sync(0xffffffffu, x, LPC - 1, LPC);
          }
        }
        __syncwarp();                    // sweep_u has finished reading us[]
        // rotation i (columns i, i+1 -> new column i) is parameterised by slot i+1: c = r_{i+1}/rho_{i+1},
        // sn = -a_i/rho_{i+1}, a_i = r_p0 for i = p0 and rho_i afterwards, rho_i^2 = sum_{q=p0..i} r_q^2
#pragma unroll
        for (int m = 0; m < SA; ++m) {
          const int i1 = l + LPC * m;                    // = i + 1
          if (LPC * m < sD) {
            double c = 1.0, sn = 0.0;
            if (dodrop && i1 > p0 && i1 < n_act) {
              const double rinv = fast_rsqrt(pre[m]);
              const double prev2 = pre[m] - rr[m] * rr[m];
              const double a = (i1 - 1 == p0) ? rp0 : prev2 * fast_rsqrt(prev2);
              c = rr[m] * rinv;
              sn = -a * rinv;
            }
            gs[i1] = c;
            us[i1] = sn;
          }
        }
        __syncwarp();
        {
          // running column R (lane = row): starts as old column p0
          double R[SA];
          int nrow[SA];                                   // row index after row p0 is removed (-1: this is row p0)
#pragma unroll
          for (int m = 0; m < SA; ++m) {
            const int p = l + LPC * m;
            R[m] = (dodrop && p <= p0) ? Vld(p0 * (p0 + 1) / 2 + p) : 0.0;
            nrow[m] = (p < p0) ? p : (p == p0 ? -1 : p - 1);
          }
          const int iB = __reduce_min_sync(0xffffffffu, p0);
          __syncwarp();
          for (int i = iB; i + 1 < sD; ++i) {
            const bool on = dodrop && i >= p0 && i + 1 < n_act;
            const double c = gs[i + 1], sn = us[i + 1];
            const int cn = (i + 1) * (i + 2) / 2, co = i * (i + 1) / 2;
#pragma unroll
            for (int m = 0; m < SA; ++m) {
              if (LPC * m <= i + 1) {
                const int p = l + LPC * m;
                if (on && p <= i + 1) {
                  const double X = Vld(cn + p);
                  const double nc = c * R[m] + sn * X;
                  R[m] = c * X - sn * R[m];
                  if (nrow[m] >= 0) Vst(co + nrow[m], nc);
                }
              }
            }
            __syncwarp();       // the next rotation overwrites the column this one has just read
          }
        }
        // w and its sum (Schur), then close the gap: slot p+1 -> slot p for p >= p0
        int nxt_act[SA];
#pragma unroll
        for (int m = 0; m < SA; ++m) {
          const int p = l + LPC * m;
          nxt_act[m] = (p + 1 < SV) ? acts[p + 1] : -1;
          if (dodrop) wd[m] = (p < n_act && p != p0) ? wd[m] - fw * mv[m] : 0.0;
          const T c_dn = __shfl_down_sync(0xffffffffu, coef[m], 1, LPC);
          const T p_dn = __shfl_down_sync(0xffffffffu, prev[m], 1, LPC);
          const double w_dn = __shfl_down_sync(0xffffffffu, wd[m], 1, LPC);
          const T c_wr = __shfl_sync(0xffffffffu, (m + 1 < SA) ? coef[m + 1 < SA ? m + 1 : m] : T(0), 0, LPC);
          const T p_wr = __shfl_sync(0xffffffffu, (m + 1 < SA) ? prev[m + 1 < SA ? m + 1 : m] : T(0), 0, LPC);
          // wd[m + 1] has not been downdated yet: apply the same formula to the wrapped value
          double w_nx = 0.0;
          if (m + 1 < SA) {
            const int pn = LPC * (m + 1);                 // slot of lane 0, register m + 1
            const double wv = wd[m + 1 < SA ? m + 1 : m], mvv = mv[m + 1 < SA ? m + 1 : m];
            w_nx = (dodrop && pn < n_act && pn != p0) ? wv - fw * mvv : (dodrop ? 0.0 : wv);
          }
          const double w_wr = __shfl_sync(0xffffffffu, w_nx, 0, LPC);
          if (p >= p0) {
            coef[m] = (l == LPC - 1) ? c_wr : c_dn;
            prev[m] = (l == LPC - 1) ? p_wr : p_dn;
            wd[m] = (l == LPC - 1) ? w_wr : w_dn;
          }
        }
        __syncwarp();
#pragma unroll
        for (int m = 0; m < SA; ++m) {
          const int p = l + LPC * m;
          if (p >= p0) acts[p] = nxt_act[m];
        }
        if (dodrop) {
          sw = sw - wp0 - fw * (sum_m - mpp);
          --n_act;
          ++st_drops;
          if (l == 0) { SlotW<T> z; z.atom = 0; z.w = T(0); sw_[n_act] = z; }
        }
        __syncwarp();
        const int i1 = __reduce_max_sync(0xffffffffu, dodrop ? n_act : 0);
        // exact covariance of the dropped atom (sklearn _least_angle.py:891)
        T part = T(0);
#pragma unroll
        for (int m = 0; m < SA; ++m) {
          if (LPC * m < i1) {
            const int p = l + LPC * m;
            if (dodrop && p < n_act) part += Gat(a_d, acts[p]) * coef[m];
          }
        }
        part = gsum<LPC>(part);
        if (dodrop) {
#pragma unroll
          for (int m = 0; m < NA; ++m)
            if (atom_of(m) == a_d) cov[m] = crow[a_d] - part;
        }
        __syncwarp();
      }
    }  // path loop

    // ---- write the code row ----
    const bool ovf = (status & 8) != 0;
    if (valid && !ovf) {
      T* hrow = P.Ht + (size_t)col * k;
#pragma unroll
      for (int m = 0; m < NA; ++m) {
        int i = atom_of(m);
        if (i < k) hrow[i] = T(0);
      }
    }
    __syncwarp();
    if (valid && !ovf) {
      T* hrow = P.Ht + (size_t)col * k;
#pragma unroll
      for (int m = 0; m < SA; ++m) {
        int p = l + LPC * m;
        if (p < n_act) hrow[acts[p]] = coef[m];
      }
      if (l == 0 && ghost_atom >= 0 && ghost_val != T(0)) hrow[ghost_atom] = ghost_val;
    }
    if (valid && l == 0) {
      if (ovf) {
        if (P.ovf_list) {
          unsigned slot = atomicAdd(P.ovf_count, 1u);
          P.ovf_list[slot] = col;
        }
        if (P.count_stats) ++st_ovf;
      } else {
        ++st_cols;
        if (status & ~8) ++st_flag;
        if (P.over_thresh != nullptr && max_act > P.thresh) atomicAdd(P.over_thresh, 1u);
      }
      st_maxact = max_act > st_maxact ? max_act : st_maxact;
    }
    st_knots += (unsigned)n_iter;
    st_s += kn_s;
    st_s2 += kn_s2;
    __syncwarp();
  }  // ticket loop

  if (P.stats && l == 0) {
    // knots / active-set sums are executed work (a column re-walked by a later tier counts again);
    // columns are counted once, by the tier that finishes them
    atomicAdd(&P.stats->columns, st_cols);
    atomicAdd(&P.stats->knots, st_knots);
    atomicAdd(&P.stats->sum_active, st_s);
    atomicAdd(&P.stats->sum_active2, st_s2);
    atomicAdd(&P.stats->drops, st_drops);
    atomicAdd(&P.stats->overflow, st_ovf);
    atomicAdd(&P.stats->flagged, st_flag);
    atomicMax(&P.stats->max_active, (unsigned long long)st_maxact);
  }
}

#include "lars_fast.cuh"

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------

struct LarsWs {           // header at the start of the caller's workspace
  unsigned long long ticket[5];   // per launch work counters                 (reset every call)
  unsigned int ovf_count[4];      // per tier overflow list lengths           (reset every call)
  unsigned int over_thresh;       // columns that needed more than tier-0 slots while run in tier 1 (reset every call)
  unsigned int hint;              // PERSISTS across calls: 0 = start columns in tier 0, 1 = start them in tier 1
};
static_assert(sizeof(LarsWs) == 64, "header size");
constexpr size_t LARS_WS_RESET_BYTES = 60;

// device-side scheduling feedback: columns that outgrow tier 0 are re-walked from the start by tier 1, so when more
// than 1/16 of a call's columns did (or would have), the next call starts every column in tier 1 directly.
__global__ void update_hint_kernel(LarsWs* hdr, long long n) {
  const unsigned int cur = hdr->hint;
  const unsigned long long big = cur == 0 ? hdr->ovf_count[0] : hdr->over_thresh;
  hdr->hint = (big * 16ull > (unsigned long long)n) ? 1u : 0u;
}

static int k_class(int k) { return k <= 32 ? 0 : k <= 64 ? 1 : k <= 128 ? 2 : k <= 256 ? 3 : k <= 512 ? 4 : -1; }
static int class_kp(int c) { static const int kp[5] = {32, 64, 128, 256, 512}; return kp[c]; }

static size_t ovf_scratch_groups(int kp) {
  size_t per = (size_t)kp * (kp + 1) / 2 * sizeof(double);
  size_t g = (96ull << 20) / per;
  if (g < 16) g = 16;
  if (g > 592) g = 592;
  return g;
}

// fast first tier: (threads per CTA, columns of V in shared memory, Gram rows in flight) variants
template <int NA, int SMAX, int SPLIT, int NT, int UQ, int LW = 4, bool NOAL = false, bool GSM = false>
static int launch_fast_variant(const LarsParams<float>& P, long long n_upper, cudaStream_t st) {
  auto kern = lars_fast_kernel<NA, SMAX, SPLIT, NT, UQ, LW, NOAL, GSM>;
  const size_t g_bytes = GSM ? round_up<size_t>((size_t)P.k * (32 * NA) * sizeof(float), 128) : 0;
  int nw = NT / 32;
  if (GSM) {                                            // as many warps as fit beside the staged Gram
    const long fit = ((long)max_smem_optin() - (long)g_bytes - 256) / (long)(fast_group_words<SMAX, SPLIT>() * 4);
    if (fit < nw) nw = (int)fit;
    if (nw < 1) return fail(ONMF_E_UNSUPPORTED, "lasso_lars: fast tier does not fit in shared memory");
  }
  const long long per_sm = cdiv<long long>(n_upper, num_sms());          // spread small minibatches over all SMs
  if (per_sm < nw) nw = per_sm < 1 ? 1 : (int)per_sm;
  const long long grid_ll = cdiv<long long>(n_upper, nw);
  int sms = num_sms() - g_lars_reserved_sms;
  if (sms < 1) sms = 1;
  const int grid = grid_ll > sms ? sms : (int)grid_ll;
  const size_t smem = g_bytes + (size_t)nw * fast_group_words<SMAX, SPLIT>() * 4;
  if ((long)smem > max_smem_optin()) return fail(ONMF_E_UNSUPPORTED, "lasso_lars: fast tier does not fit in shared memory");
  ONMF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<grid, nw * 32, smem, st>>>(P);
  ONMF_LAUNCH_CHECK("lars_fast_kernel");
  return ONMF_OK;
}
// k <= 128 (4 atoms per lane, Gram staged in shared memory): 32 slots, the whole factor in shared memory; the kernel needs few
// registers, and these minibatches are small enough to be latency-bound (a handful of columns per warp), so it runs
// with as many warps as the register file allows
template <int SMAX>
static int launch_fast_gsm(const LarsParams<float>& P, long long n_upper, cudaStream_t st) {
#ifdef LARS_FAST_EXPERIMENT
  static int cfg = -1;
  if (cfg < 0) { const char* e = getenv("ONMF_FAST_CFG"); cfg = e ? atoi(e) : 0; }
  switch (cfg) {
    case 1: return launch_fast_variant<4, SMAX, SMAX, 1024, 4, 4, true, true>(P, n_upper, st);
    case 2: return launch_fast_variant<4, SMAX, SMAX, 640, 4, 4, true, true>(P, n_upper, st);
    case 3: return launch_fast_variant<4, SMAX, SMAX, 512, 4, 4, true, true>(P, n_upper, st);
    case 4: return launch_fast_variant<4, SMAX, SMAX, 1024, 2, 4, true, true>(P, n_upper, st);
  }
#endif
  return launch_fast_variant<4, SMAX, SMAX, 768, 4, 4, true, true>(P, n_upper, st);     // (cfg4: 0.274 ms; 1024 / 640 / 512 threads: 0.286 / 0.277 / 0.290)
}

// k <= 64 on SMALL minibatches (at most one column per resident warp): these calls are latency-bound -- a handful of columns
// per SM, each a serial path of ~15-30 knots -- and one column per warp in the fast kernel (2 atoms per lane, Gram in shared
// memory) has the shorter knot than the general kernel's four / two columns per warp.  Larger minibatches stay with the
// general kernel, whose packing wins on throughput (measured: cfg2, k = 49, 27 columns per SM: 0.084 -> 0.065 ms; cfg3, k = 25,
// 68 columns per SM: 0.087 -> 0.104 ms -- hence one column per warp slot for k <= 32, two for k <= 64).
constexpr int FAST_SMALL_WARPS = 24;
static int launch_fast_small(const LarsParams<float>& P, long long n_upper, cudaStream_t st) {
  return launch_fast_variant<2, 32, 32, FAST_SMALL_WARPS * 32, 4, 2, true, true>(P, n_upper, st);
}

#ifdef LARS_FAST_EXPERIMENT
constexpr int FAST_MAX_WARPS = 32, FAST_MIN_SPLIT = 16;
#else
constexpr int FAST_MAX_WARPS = 20, FAST_MIN_SPLIT = 28;
#endif
template <int NA, int SMAX>
static int launch_fast(const LarsParams<float>& P, long long n_upper, cudaStream_t st) {
#ifdef LARS_FAST_EXPERIMENT
  static int cfg = -1;
  if (cfg < 0) { const char* e = getenv("ONMF_FAST_CFG"); cfg = e ? atoi(e) : 0; }
  switch (cfg) {
    case 1: return launch_fast_variant<NA, SMAX, 32, 640, 4, 4, false>(P, n_upper, st);
    case 2: return launch_fast_variant<NA, SMAX, 28, 640, 4, 4, true>(P, n_upper, st);
    case 3: return launch_fast_variant<NA, SMAX, 28, 640, 4, 2, true>(P, n_upper, st);
    case 4: return launch_fast_variant<NA, SMAX, 32, 640, 4, 2, false>(P, n_upper, st);
    case 5: return launch_fast_variant<NA, SMAX, 40, 512, 4, 2, true>(P, n_upper, st);
    case 6: return launch_fast_variant<NA, SMAX, 28, 640, 2, 2, true>(P, n_upper, st);
  }
#endif
  // measured at cfg5 (profiles/r2_lars_fast.md): 20 warps x 96 registers with 28 columns of V in shared memory (98 KB per CTA,
  // which leaves the larger L1 carve-out to the Gram rows) beat 16 warps x 128 registers / 40 columns by 5 %; 16 atoms per
  // lane (k <= 512) do not fit 96 registers
  if constexpr (NA <= 8) return launch_fast_variant<NA, SMAX, 28, 640, 4, 4, true>(P, n_upper, st);
  else return launch_fast_variant<NA, SMAX, 40, 512, 2, 4, true>(P, n_upper, st);
}

// *padded: whether the zero-padded global copy of G (P.Gp) has been written in this call; a tier that cannot stage G in
// shared memory writes it on first need (the small classes in fp32 never do: a launch less on their launch-bound steps)
template <typename T, int LPC, int NA, int SMAX, bool MGLOB, int SPLIT = 0>
static int launch_tier(LarsParams<T> P, long long n_upper, int max_warps, cudaStream_t st, bool* padded) {
  constexpr int GPW = 32 / LPC;
  const int k = P.k;
  const int smem_max = max_smem_optin();
  const size_t g_bytes = round_up<size_t>((size_t)k * gram_stride<LPC, NA>() * sizeof(T), 128);
  const size_t grp_bytes = (size_t)group_words<T, LPC, SMAX, MGLOB, SPLIT>() * 4;
  const bool gsm = !MGLOB && g_bytes <= 72 * 1024 && (smem_max - (long)g_bytes - 256) >= (long)(2 * GPW * grp_bytes);
  const size_t avail = smem_max - (gsm ? g_bytes : 0) - 256;
  int nw = (int)(avail / (GPW * grp_bytes));
  if (nw > max_warps) nw = max_warps;
  if (nw > LARS_MAX_THREADS / 32) nw = LARS_MAX_THREADS / 32;
  if (nw < 1) return fail(ONMF_E_UNSUPPORTED, "lasso_lars: shared memory too small for one warp");
  // spread small minibatches over all SMs instead of packing few CTAs
  long long groups = cdiv<long long>(n_upper, GPW);
  int nw_need = (int)cdiv<long long>(groups, num_sms());
  if (nw_need < nw) nw = nw_need < 1 ? 1 : nw_need;
  long long grid_ll = cdiv<long long>(groups, nw);
  // the kernel is persistent (one CTA per SM, full register file): optionally leave a few SMs free so that the
  // dictionary update running on another stream can be co-scheduled instead of queueing behind it
  int sms = num_sms() - g_lars_reserved_sms;
  if (sms < 1) sms = 1;
  int grid = grid_ll > sms ? sms : (int)grid_ll;
  if (MGLOB) {
    long long cap = (long long)ovf_scratch_groups(LPC * NA) / (nw * GPW);
    if (cap < 1) { nw = 1; cap = (long long)ovf_scratch_groups(LPC * NA) / GPW; }
    if (grid > cap) grid = (int)cap;
  }
  size_t smem = (gsm ? g_bytes : 0) + (size_t)nw * GPW * grp_bytes;
  if (!gsm && !*padded) {
    constexpr int KPAD = LPC * NA;
    pad_gram_kernel<T><<<cdiv(k * KPAD, 256), 256, 0, st>>>(P.G, P.G64, k, KPAD, const_cast<T*>(P.Gp));
    ONMF_LAUNCH_CHECK("pad_gram_kernel");
    *padded = true;
  }
  if constexpr (std::is_same<T, float>::value && LPC == 32 && SPLIT > 0 && !MGLOB) {
    // fp32 production path, k > 128: the warp-uniform fast tier walks the clean paths and hands everything else on
    if (!gsm && P.G64 != nullptr && P.ovf_list != nullptr && g_lars_fast && k > SMAX) return launch_fast<NA, SMAX>(P, n_upper, st);
  }
  if constexpr (std::is_same<T, float>::value && LPC == 32 && NA == 4 && SMAX == 32 && SPLIT == 0 && !MGLOB) {
    // fp32, 64 < k <= 128: first tier (32 slots) by the fast kernel with the Gram in shared memory
    if (gsm && P.G64 != nullptr && P.ovf_list != nullptr && g_lars_fast && P.col_list == nullptr) return launch_fast_gsm<SMAX>(P, n_upper, st);
  }
  if (gsm) {
    auto kern = lars_kernel<T, LPC, NA, SMAX, true, MGLOB, SPLIT>;
    ONMF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, nw * 32, smem, st>>>(P);
  } else {
    auto kern = lars_kernel<T, LPC, NA, SMAX, false, MGLOB, SPLIT>;
    ONMF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, nw * 32, smem, st>>>(P);
  }
  ONMF_LAUNCH_CHECK("lars_kernel");
  return ONMF_OK;
}

// workspace layout: [LarsWs | list1 (n x 8) | list2 (n x 8) | Gp (k x KP) | M scratch (last tier, k > 128)]
static size_t ws_list_bytes(long long n) { return round_up<size_t>((size_t)n * sizeof(long long), 256); }
static size_t ws_gp_bytes(int k, int kp) { return round_up<size_t>((size_t)k * kp * sizeof(double), 256); }
// hybrid first tier (k > 128): 64 slots, the first 40 rows of the packed inverse in shared memory, rows 40..63 here
#ifndef LARS_HYB_SPLIT
#define LARS_HYB_SPLIT 40
#endif
constexpr int HYB_SLOTS = 64, HYB_SPLIT = LARS_HYB_SPLIT;
static size_t ws_hyb_bytes(int kp) {
  if (kp <= 128) return 0;
  size_t per = (size_t)(HYB_SLOTS * (HYB_SLOTS + 1) / 2 - HYB_SPLIT * (HYB_SPLIT + 1) / 2) * sizeof(double);
  // (the fast first tier: padded columns, up to FAST_MAX_WARPS warps per SM -- expressed per general-kernel group)
  const size_t per_fast = (size_t)fast_tail_doubles<HYB_SLOTS, FAST_MIN_SPLIT>() * sizeof(double) * FAST_MAX_WARPS / (LARS_MAX_THREADS / 16) + 8;
  if (per_fast > per) per = per_fast;
  // resident groups per SM: one per LPC lanes; the k > 128 classes use LPC >= 16
  return round_up<size_t>((size_t)(num_sms() > 160 ? num_sms() : 160) * (LARS_MAX_THREADS / 16) * per, 256);
}

// tiers: S0 slots, then S1, S2, S3 (0 = none); the last non-zero tier keeps M in global scratch when GL
template <typename T, int LPC, int NA, int S0, int S1, int S2, int S3, bool GL, int SPLIT0 = 0>
static int launch_class(const T* G, const double* G64, const T* Ct, long long n, int k, int d, double alpha, int max_iter, T* Ht,
                        unsigned char* ws, onmf_lars_stats* stats, int first_tier, cudaStream_t st) {
  constexpr int KP = LPC * NA;
  LarsWs* hdr = reinterpret_cast<LarsWs*>(ws);
  const size_t lb = ws_list_bytes(n);
  long long* lists[2] = {reinterpret_cast<long long*>(ws + sizeof(LarsWs)),
                         reinterpret_cast<long long*>(ws + sizeof(LarsWs) + lb)};
  T* gp = reinterpret_cast<T*>(ws + sizeof(LarsWs) + 2 * lb);
  double* mhyb = reinterpret_cast<double*>(ws + sizeof(LarsWs) + 2 * lb + ws_gp_bytes(k, KP));
  double* mscr = reinterpret_cast<double*>(ws + sizeof(LarsWs) + 2 * lb + ws_gp_bytes(k, KP) + ws_hyb_bytes(KP));
  ONMF_CUDA(cudaMemsetAsync(hdr, 0, LARS_WS_RESET_BYTES, st));   // everything but the persistent hint
  bool padded = false;

  LarsParams<T> P;
  P.G = G; P.G64 = G64; P.Gp = gp; P.Ct = Ct; P.Ht = Ht; P.n = n; P.k = k; P.d = d; P.max_iter = max_iter;
  P.amin = T(alpha) / T(d);
  P.Mscratch = nullptr; P.Mhyb = mhyb; P.stats = stats;
  // tier t reads list (t-1)&1 and appends to list t&1.  first_tier: 0 / 1 = start every column in that tier,
  // -1 = adaptive (both first-tier variants are launched, the device-side hint decides which one does the work).
  const bool adaptive = (first_tier < 0) && S1 > 0;
  const int first = (first_tier > 0 && S1 > 0) ? 1 : 0;
  P.over_thresh = nullptr; P.thresh = S0; P.hint = nullptr; P.run_if = 0;
  auto tier_params = [&](int t, int ticket, bool from_list, bool has_next, bool glob) {
    LarsParams<T> Q = P;
    Q.ticket = &hdr->ticket[ticket];
    Q.col_list = from_list ? lists[(t - 1) & 1] : nullptr;
    Q.n_list = from_list ? &hdr->ovf_count[t - 1] : nullptr;
    Q.ovf_list = has_next ? lists[t & 1] : nullptr;
    Q.ovf_count = &hdr->ovf_count[t];
    Q.Mscratch = glob ? mscr : nullptr;
    Q.count_stats = !from_list;
    return Q;
  };
  int rc = ONMF_OK;
  if constexpr (std::is_same<T, float>::value && KP <= 64 && S0 == 32 && !GL) {
    if (G64 != nullptr && g_lars_fast && n <= (k <= 32 ? 1LL : 2LL) * num_sms() * FAST_SMALL_WARPS && k <= 64) {
      // fast tier over all columns, then the general kernel (the larger of its tiers) over the columns it handed on.
      // Taken for every first_tier: the fast kernel and the general kernel sum a join's FP64 terms in different orders, so
      // a first_tier that picked the general kernel here would change the codes in the last bits.  The hint is neither
      // read nor updated on this route.
      rc = launch_fast_small(tier_params(0, 0, false, true, false), n, st);
      if (rc) return rc;
      constexpr int NEXT = S1 > 0 ? S1 : S0;
      return launch_tier<T, LPC, NA, NEXT, false>(tier_params(1, 1, true, false, false), n, 32, st, &padded);
    }
  }
  if (adaptive || first == 0) {
    LarsParams<T> Q = tier_params(0, 0, false, S1 > 0, GL && S1 == 0);
    if (adaptive) { Q.hint = &hdr->hint; Q.run_if = 0; }
    rc = launch_tier<T, LPC, NA, S0, (GL && S1 == 0), SPLIT0>(Q, n, 32, st, &padded);
    if (rc) return rc;
  }
  if constexpr (S1 > 0) {
    if (adaptive || first == 1) {      // tier 1 over ALL columns
      LarsParams<T> Q = tier_params(1, 4, false, S2 > 0, GL && S2 == 0);
      if (adaptive) { Q.hint = &hdr->hint; Q.run_if = 1; Q.over_thresh = &hdr->over_thresh; }
      rc = launch_tier<T, LPC, NA, S1, (GL && S2 == 0)>(Q, n, (GL && S2 == 0) ? 2 : 32, st, &padded);
      if (rc) return rc;
    }
    if (adaptive || first == 0) {      // tier 1 over tier 0's overflow list
      rc = launch_tier<T, LPC, NA, S1, (GL && S2 == 0)>(tier_params(1, 1, true, S2 > 0, GL && S2 == 0), n, (GL && S2 == 0) ? 2 : 32, st, &padded);
      if (rc) return rc;
    }
  }
  if constexpr (S2 > 0) {
    rc = launch_tier<T, LPC, NA, S2, (GL && S3 == 0)>(tier_params(2, 2, true, S3 > 0, GL && S3 == 0), n, (GL && S3 == 0) ? 2 : 32, st, &padded);
    if (rc) return rc;
  }
  if constexpr (S3 > 0) {
    rc = launch_tier<T, LPC, NA, S3, GL>(tier_params(3, 3, true, false, GL), n, GL ? 2 : 32, st, &padded);
    if (rc) return rc;
  }
  if (adaptive) {
    update_hint_kernel<<<1, 1, 0, st>>>(hdr, n);
    ONMF_LAUNCH_CHECK("update_hint_kernel");
  }
  return ONMF_OK;
}

template <typename T>
static int lasso_lars_t(const void* G, const double* G64, const void* Ct, long long n, int k, int d, double alpha, int max_iter,
                        void* Ht, void* ws, onmf_lars_stats* stats, int first_tier, cudaStream_t st) {
  const T* g = (const T*)G; const T* c = (const T*)Ct; T* h = (T*)Ht; unsigned char* w = (unsigned char*)ws;
  switch (k_class(k)) {
    case 0: return launch_class<T, 8, 4, 32, 0, 0, 0, false>(g, G64, c, n, k, d, alpha, max_iter, h, w, stats, first_tier, st);
    case 1: return launch_class<T, 16, 4, 32, 64, 0, 0, false>(g, G64, c, n, k, d, alpha, max_iter, h, w, stats, first_tier, st);
    case 2: return launch_class<T, 32, 4, 32, 64, 128, 0, false>(g, G64, c, n, k, d, alpha, max_iter, h, w, stats, first_tier, st);
#if defined(LARS_K256_LPC16)
    case 3: return launch_class<T, 16, 16, HYB_SLOTS, 128, 256, 0, true, HYB_SPLIT>(g, G64, c, n, k, d, alpha, max_iter, h, w, stats, first_tier, st);
#else
    case 3: return launch_class<T, 32, 8, HYB_SLOTS, 128, 256, 0, true, HYB_SPLIT>(g, G64, c, n, k, d, alpha, max_iter, h, w, stats, first_tier, st);
#endif
    case 4: return launch_class<T, 32, 16, HYB_SLOTS, 128, 512, 0, true, HYB_SPLIT>(g, G64, c, n, k, d, alpha, max_iter, h, w, stats, first_tier, st);
  }
  return fail(ONMF_E_UNSUPPORTED, "lasso_lars: n_components > 512 not instantiated");
}

}  // namespace onmf

extern "C" size_t onmf_lasso_lars_workspace(int dtype, int k, int64_t n) {
  int c = onmf::k_class(k);
  if (c < 0 || n < 0) return 0;
  (void)dtype;
  int kp = onmf::class_kp(c);
  size_t bytes = sizeof(onmf::LarsWs) + 2 * onmf::ws_list_bytes(n) + onmf::ws_gp_bytes(k, kp) + onmf::ws_hyb_bytes(kp);
  if (kp > 128) bytes += onmf::ovf_scratch_groups(kp) * ((size_t)kp * (kp + 1) / 2) * sizeof(double);
  return bytes + 256;
}

static int lasso_lars_entry(int dtype, const void* G, const double* G64, const void* Ct, int64_t n, int k, int d,
                            double alpha, int max_iter, void* Ht, void* workspace, size_t workspace_bytes,
                            onmf_lars_stats* stats, int first_tier, void* stream) {
  using namespace onmf;
  if ((!G && !G64) || !Ct || !Ht || !workspace) return fail(ONMF_E_ARG, "lasso_lars: null pointer");
  if (n < 0 || k <= 0 || d <= 0 || max_iter < 0 || !(alpha >= 0.0)) return fail(ONMF_E_ARG, "lasso_lars: bad size/alpha");
  if (dtype != ONMF_F32 && dtype != ONMF_F64) return fail(ONMF_E_ARG, "lasso_lars: bad dtype");
  if (n == 0) return ONMF_OK;
  if (workspace_bytes < onmf_lasso_lars_workspace(dtype, k, n)) return fail(ONMF_E_WORKSPACE, "lasso_lars: workspace too small");
  if ((uintptr_t)workspace % 256) return fail(ONMF_E_ARG, "lasso_lars: workspace must be 256-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  // in FP64 working precision the FP64 Gram IS the working-precision Gram
  if (dtype == ONMF_F64) return lasso_lars_t<double>(G ? G : (const void*)G64, nullptr, Ct, n, k, d, alpha, max_iter, Ht, workspace, stats, first_tier, st);
  return lasso_lars_t<float>(G, G64, Ct, n, k, d, alpha, max_iter, Ht, workspace, stats, first_tier, st);
}

extern "C" int onmf_lasso_lars_ex(int dtype, const void* G, const void* Ct, int64_t n, int k, int d, double alpha,
                                  int max_iter, void* Ht, void* workspace, size_t workspace_bytes,
                                  onmf_lars_stats* stats, int first_tier, void* stream) {
  if (!G) return onmf::fail(ONMF_E_ARG, "lasso_lars: null pointer");
  return lasso_lars_entry(dtype, G, nullptr, Ct, n, k, d, alpha, max_iter, Ht, workspace, workspace_bytes, stats, first_tier, stream);
}

extern "C" int onmf_lasso_lars_g64(int dtype, const double* G64, const void* Ct, int64_t n, int k, int d, double alpha,
                                   int max_iter, void* Ht, void* workspace, size_t workspace_bytes,
                                   onmf_lars_stats* stats, int first_tier, void* stream) {
  if (!G64) return onmf::fail(ONMF_E_ARG, "lasso_lars: null pointer");
  return lasso_lars_entry(dtype, nullptr, G64, Ct, n, k, d, alpha, max_iter, Ht, workspace, workspace_bytes, stats, first_tier, stream);
}

extern "C" int onmf_lasso_lars(int dtype, const void* G, const void* Ct, int64_t n, int k, int d, double alpha,
                               int max_iter, void* Ht, void* workspace, size_t workspace_bytes,
                               onmf_lars_stats* stats, void* stream) {
  return onmf_lasso_lars_ex(dtype, G, Ct, n, k, d, alpha, max_iter, Ht, workspace, workspace_bytes, stats, -1, stream);
}
