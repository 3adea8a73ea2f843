/*
 * onmf_b200.h -- C ABI of libonmf_b200.so: hand-written sm_100a CUDA kernels for the online
 * NMF/NTF dictionary-learning hot path of HanbaekLyu/ONMF_ONTF_NDL.
 *
 * The reference has no FFI layer (it is pure Python: numpy + scikit-learn); the boundary a
 * maintainer would bind is its Python class API (src/onmf.py, src/ontf.py).  Each entry point
 * below replaces one numpy/sklearn call inside those classes and cites it.  INTEGRATION.md shows
 * the ctypes stub that goes into the reference's `Online_NTF` / `Online_NMF` methods.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless named `host_*`; the caller owns all buffers;
 *     nothing is allocated inside the library; `stream` is a cudaStream_t passed as void*.
 *   - dtype: ONMF_F32 (production) or ONMF_F64 (parity mode; the reference computes in float64).
 *   - "sample-major" layout: a minibatch is stored one sample per row,
 *         Xt (n x d), Ct = Xt W (n x k), Ht (n x k)       all row-major, leading dim = row length.
 *     (the reference's `joint_sparse_code_tensor` already returns H as n x r, src/ontf.py:86.)
 *     W is (d x k) row-major, A is (k x k), B is (k x d) row-major -- the reference's shapes.
 *   - every function returns 0 on success, a negative ONMF_E_* code otherwise;
 *     onmf_last_error() returns a thread-local message.
 *   - no function synchronises the stream; none is a CPU fallback.
 */
#ifndef ONMF_B200_H
#define ONMF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ONMF_F32 0
#define ONMF_F64 1

#define ONMF_OK 0
#define ONMF_E_ARG (-1)        /* bad argument (null pointer, unsupported size)            */
#define ONMF_E_CUDA (-2)       /* a CUDA runtime call failed; see onmf_last_error()       */
#define ONMF_E_UNSUPPORTED (-3)/* shape outside what the kernels were instantiated for    */
#define ONMF_E_WORKSPACE (-4)  /* workspace too small                                     */

/* options (kept per calling host thread, like the error string) */
#define ONMF_OPT_LARS_RESERVED_SMS 1  /* SMs the persistent LARS coder leaves free (default 0) so that kernels launched
                                         on other streams (the dictionary update) run concurrently with it */
#define ONMF_OPT_LARS_FAST_TIER 2     /* 1 (default): the fp32 coder for n_components > 128 walks clean homotopy paths in the
                                         warp-uniform fast first tier (csrc/lars_fast.cuh); 0: general kernel only */
int onmf_set_option(int key, int value);
int onmf_get_option(int key, int* value);

/* library / build identification */
int onmf_version(void);                      /* 100*major + minor                                   */
const char* onmf_last_error(void);
int onmf_built_arch(void);                   /* 100 => sm_100a                                      */
long long onmf_launch_count(void);           /* kernels launched so far by the calling host thread (every launch site of
                                                the library counts itself; graph replays count their kernel nodes) */

/* ---------------------------------------------------------------------------------------------
 * K1  patch gather / matricization
 * replaces: the np.append patch loops image_reconstruction.py:184-205,
 *           image_reconstruction_tensor.py:102-123, ising_reconstruction.py:56-65 and
 *           tl_unfold(...)[.T] + X_unfold[:, idx]  (src/ontf.py:203-208, :229-231)
 * ------------------------------------------------------------------------------------------- */

/* img: (H x Wd x C) row-major (C=1 gray / Ising lattice, C=3 colour); coords: n pairs (row, col) of
 * int32 top-left corners; out Xt (n x ld), Xt[j, (r*p + c)*C + ch] = img[a_j + r, b_j + c, ch]
 * -- the HWC feature order of the reference's reshape(k**2, 3) + mode-2 joint unfolding.  ld >= p*p*C is the row pitch of Xt in
 * elements (nothing is written beyond a patch's p*p*C features).  16-byte stores whenever p*p*C and ld are multiples of 16 bytes
 * and Xt is 16-byte aligned, scalar otherwise; same bytes either way. */
int onmf_gather_patches(int dtype, const void* img, int H, int Wd, int C, const int32_t* coords,
                        int64_t n, int p, void* Xt, int64_t ld, void* stream);

/* column gather of a resident sample-major data pool: out[j, :] = pool[idx[j], :]
 * (X_batch = X_unfold[:, idx], src/ontf.py:231; idx as int64 like numpy's randint).  An index outside [0, n_pool)
 * (numpy would raise IndexError) is never dereferenced: its output row is filled with NaN.  Likewise a patch corner
 * outside the image in onmf_gather_patches. */
int onmf_gather_rows(int dtype, const void* pool, int64_t n_pool, int d, const int64_t* idx,
                     int64_t n, void* Xt, void* stream);

/* storage formats of a streamed minibatch (arithmetic is always fp32 / fp64): the reference's image data is 8-bit before
 * `data / 255` (image_reconstruction.py:88), so host-resident patches can cross PCIe as u8 (4x fewer bytes) or fp16.
 * dst[i] = (float)src[i] * scale for i < count (count % 4 == 0); with lo != NULL the result is written as the TF32 hi/lo
 * pair of the tensor-core path (dst = hi). */
#define ONMF_STORE_U8 2
#define ONMF_STORE_F16 3
int onmf_widen(int src_kind, const void* src, int64_t count, double scale, void* dst, void* lo, void* stream);

/* elementwise precision change f32 <-> f64 (used to run the coder in FP64 on the covariances of the fp32 path for the one
 * minibatch that is coded against a raw, unnormalised initial dictionary; see OnmfEngine._code_wide) */
int onmf_convert(int dtype_in, int dtype_out, const void* src, int64_t count, void* dst, void* stream);

/* transpose/convert a (d x n) row-major matrix (the reference's X layout, any of f32/f64) into the
 * sample-major (n x d) layout in `dtype_out`.  Also used for H (k x n) <-> Ht. */
int onmf_transpose(int dtype_in, int dtype_out, const void* src, int64_t rows, int64_t cols,
                   void* dst, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K2  Gram and covariance products
 * replaces: gram = D D^T, cov = D X^T  (sklearn/decomposition/_dict_learning.py:422,426, reached
 *           from src/ontf.py:86) and A = W.T @ W, B = W.T @ X (src/onmf.py:242-243)
 * ------------------------------------------------------------------------------------------- */
int onmf_gram(int dtype, const void* W, int d, int k, void* G /* k x k */, void* stream);
/* same product with a workspace: the sum over d is split into up to 16 slices (fixed-order reduction) so the small
 * k x k output still fills the GPU */
size_t onmf_gram_workspace(int dtype, int d, int k);
int onmf_gram_ws(int dtype, const void* W, int d, int k, void* G, void* workspace, size_t workspace_bytes,
                 void* stream);
int onmf_cov(int dtype, const void* Xt, int64_t n, int d, const void* W, int k,
             void* Ct /* n x k */, void* stream);
/* FP64-accumulated Gram of an fp32 (dtype_in = ONMF_F32) or fp64 dictionary: G64 (k x k doubles), optional fp32 copy G32
 * (may be NULL).  This is the Gram the coder should be given (onmf_lasso_lars_g64): the active-block inverse amplifies
 * the independent per-entry rounding of an fp32 Gram by cond(G), while the exact Gram of the stored dictionary only
 * sees cond(W) = sqrt(cond(G)).  Sum over d split into up to 16 slices, fixed-order reduction (deterministic). */
size_t onmf_gram_f64_workspace(int d, int k);
int onmf_gram_f64(int dtype_in, const void* W, int d, int k, double* G64, float* G32, void* workspace,
                  size_t workspace_bytes, void* stream);

/* Spectral norm (largest singular value) of a sample-major n x k matrix M, written to the device double *out:
 * sqrt(lambda_max(M^T M)) -- FP64 Gram, then lambda_max by repeated squaring + Rayleigh quotient in one CTA (relative
 * error < 1e-5 for every spectrum).  replaces: np.linalg.norm(H1 - H1_old, 2) / np.linalg.norm(H1_old, 2), the stopping
 * test of update_code_within_radius (src/onmf.py:265). */
size_t onmf_spectral_norm_workspace(int64_t n, int k);
int onmf_spectral_norm(int dtype, const void* M, int64_t n, int k, double* out, void* workspace, size_t workspace_bytes,
                       void* stream);

/* ---------------------------------------------------------------------------------------------
 * K3  batched positive LARS-lasso (the sparse coder)
 * replaces: SparseCoder(..., 'lasso_lars', positive_code=True).transform (src/ontf.py:79-86), i.e.
 *           LassoLars.fit's per-sample loop sklearn/linear_model/_least_angle.py:1136-1153 over
 *           _lars_path_solver (:415-917, Gram mode, method='lasso', positive, return_path=False).
 * Per column: argmin_{h>=0} 0.5||x - W h||^2 + alpha*sum(h), following the same homotopy path and
 * the same stopping / last-segment interpolation rule (alpha_min = alpha/d, float32-eps equality
 * tolerance), so results agree with the reference also where sklearn is not at the exact optimum.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  unsigned long long columns;      /* columns solved                                   */
  unsigned long long knots;        /* LARS iterations executed (sum over columns)      */
  unsigned long long sum_active;   /* sum over knots of the active-set size s          */
  unsigned long long sum_active2;  /* sum over knots of s^2                            */
  unsigned long long drops;        /* lasso drop events                                */
  unsigned long long overflow;     /* columns re-solved by the large-active-set path   */
  unsigned long long flagged;      /* columns that hit degenerate / ill-conditioned / max_iter exits */
  unsigned long long max_active;   /* largest active set seen                          */
} onmf_lars_stats;

/* bytes of workspace onmf_lasso_lars needs for (dtype, k, n) */
size_t onmf_lasso_lars_workspace(int dtype, int k, int64_t n);

/* G (k x k), Ct (n x k) -> Ht (n x k).  d = number of features (enters only sklearn's alpha/d scaling
 * of the stopping rule).  stats may be NULL (device pointer to onmf_lars_stats, accumulated into). */
int onmf_lasso_lars(int dtype, const void* G, const void* Ct, int64_t n, int k, int d, double alpha,
                    int max_iter, void* Ht, void* workspace, size_t workspace_bytes,
                    onmf_lars_stats* stats, void* stream);
/* same, with explicit tier scheduling.  Columns whose active set outgrows a tier's slot count are re-walked from the
 * start by the next (larger, lower-occupancy) tier.  first_tier = 0 / 1 starts every column in that tier;
 * first_tier = -1 (what onmf_lasso_lars uses) is adaptive: a device-side flag kept in the first 64 bytes of the
 * workspace remembers whether more than 1/16 of the previous call's columns needed the larger tier.  The workspace
 * must therefore be zero-filled once before its first use and may be reused across calls.  Results are identical
 * for every setting. */
int onmf_lasso_lars_ex(int dtype, const void* G, const void* Ct, int64_t n, int k, int d, double alpha,
                       int max_iter, void* Ht, void* workspace, size_t workspace_bytes,
                       onmf_lars_stats* stats, int first_tier, void* stream);

/* same, Gram supplied in FP64 (onmf_gram_f64) while covariances / codes stay in `dtype`: the correlation passes run on
 * a working-precision copy, the active-block inverse is built from the FP64 entries.  The production fp32 path. */
int onmf_lasso_lars_g64(int dtype, const double* G64, const void* Ct, int64_t n, int k, int d, double alpha,
                        int max_iter, void* Ht, void* workspace, size_t workspace_bytes,
                        onmf_lars_stats* stats, int first_tier, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K4  surrogate aggregation
 * replaces: A1 = (1-w) A + w H^T H ; B1 = (1-w) B + w H^T X^T   (src/ontf.py:147-148,
 *           src/onmf.py:155-156), optional C1 = (1-w) C + w X X^T (src/onmf.py:157-158)
 * Two phases so that a multi-GPU run can all-reduce the packed partial sums in between:
 *   partial:  P = [ Ht^T Ht | Ht^T Xt ]   packed (k x (k+d)) row-major, THIS rank's columns only
 *   blend:    A = (1-w) A + w P[:, :k] ;  B = (1-w) B + w P[:, k:]
 * ------------------------------------------------------------------------------------------- */
size_t onmf_surrogate_workspace(int dtype, int64_t n, int k, int d);
int onmf_surrogate_partial(int dtype, const void* Ht, const void* Xt, int64_t n, int k, int d,
                           void* P /* k x (k+d) */, void* workspace, size_t workspace_bytes,
                           void* stream);
int onmf_surrogate_blend(int dtype, const void* P, int k, int d, double w, void* A, void* B,
                         void* stream);
/* same with the weight read from device memory (one double): the form a captured CUDA graph of the step replays */
int onmf_surrogate_blend_dev(int dtype, const void* P, int k, int d, const double* w_dev, void* A, void* B,
                             void* stream);
/* optional d x d aggregate: Cagg = (1-w) Cagg + w Xt^T Xt   (single rank; P2 is a d x d scratch) */
int onmf_xxt_partial(int dtype, const void* Xt, int64_t n, int d, void* P2, void* workspace,
                     size_t workspace_bytes, void* stream);
int onmf_axpby(int dtype, int64_t count, double a, const void* x, double b, void* y, void* stream);

/* surrogate loss read-out (SURVEY.md §8f.3; the error curve of ising_reconstruction.py:133,164 and
 * network_reconstruction_nx.py): out3[0] = tr(W A W^T) (as <G64, A> with the FP64 Gram of W), out3[1] = tr(W B),
 * out3[2] = tr(C) (0 when C is NULL); the loss is out3[0] - 2 out3[1] + out3[2].  out3: 3 device doubles. */
int onmf_surrogate_error(int dtype, const void* W, const double* G64, const void* A, const void* B, const void* C,
                         int d, int k, double* out3, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K2 / K4 on the tensor cores (fp32 only): TMA-fed tcgen05.mma kind::tf32 with TMEM accumulators and a
 * 3xTF32 operand split (hi = rna_tf32(x), lo = x - hi; hi*hi + hi*lo + lo*hi) for fp32-class accuracy.
 * Same products as onmf_cov / onmf_surrogate_partial above; operands are passed pre-split.
 * onmf_tc_supported(k, d) != 0 when the shapes satisfy TMA's 16-byte stride rule (k % 4 == 0, d % 4 == 0).
 * ------------------------------------------------------------------------------------------- */
int onmf_tc_supported(int k, int d);
int onmf_split_tf32(const void* src, void* hi, void* lo, int64_t count, void* stream);
/* fused minibatch gather + split: (hi, lo)[j, :] = split(pool[idx[j], :]) */
int onmf_gather_rows_split(const void* pool, int64_t n_pool, int d, const int64_t* idx, int64_t n, void* hi,
                           void* lo, void* stream);
int onmf_cov_tc(const void* Xt_hi, const void* Xt_lo, int64_t n, int d, const void* W_hi, const void* W_lo,
                int k, void* Ct, void* stream);
size_t onmf_surrogate_tc_workspace(int64_t n, int k, int d);
int onmf_surrogate_partial_tc(const void* Ht_hi, const void* Ht_lo, const void* Xt_hi, const void* Xt_lo,
                              int64_t n, int k, int d, void* P, void* workspace, size_t workspace_bytes,
                              void* stream);

/* ---------------------------------------------------------------------------------------------
 * K1 + K2 and K4 fused on the tensor cores (fp32, k <= 256): the minibatch is read ONCE per product, as stored.
 * Loader warps read the minibatch rows straight from the resident pool through the minibatch indices -- fp32, or the narrow
 * storage formats ONMF_STORE_U8 / ONMF_STORE_F16 (value = stored * scale) -- split them into TF32 hi / lo in registers and
 * write the swizzled UMMA operand tiles in shared memory; no hi/lo copy of the minibatch or of the codes ever exists in HBM.
 *   pool (n_pool x ld_pool, one sample per row), idx (n int64 row indices, or NULL for rows 0..n-1)
 *   onmf_cov_fused_tc       : Ct (n x k) = X[idx] W                                   (W_hi / W_lo: onmf_split_tf32 of W)
 *   onmf_surrogate_fused_tc : P (k x (k+d)) = [Ht^T Ht | Ht^T X[idx]]  (P may be NULL when blend != 0)
 *                             blend != 0 (single GPU): A <- (1-w) A + w P_A, B <- (1-w) B + w P_B in the same pass, w from
 *                             *w_dev (device double) when w_dev != NULL, else the host value w
 * Persistent CTAs (one per SM), FP32 accumulators in tensor memory, fixed-order reductions (deterministic).
 * ------------------------------------------------------------------------------------------- */
int onmf_fused_tc_supported(int k, int d);
int onmf_cov_fused_tc(int src_kind, const void* pool, int64_t n_pool, int64_t ld_pool, const int64_t* idx, int64_t n,
                      int d, double scale, const void* W_hi, const void* W_lo, int k, void* Ct, void* stream);
size_t onmf_surrogate_fused_tc_workspace(int64_t n, int k, int d);
int onmf_surrogate_fused_tc(const void* Ht, int src_kind, const void* pool, int64_t n_pool, int64_t ld_pool,
                            const int64_t* idx, int64_t n, int k, int d, double scale, void* P, int blend, double w,
                            const double* w_dev, void* A, void* B, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Patch minibatches by reference: the data matrix X (d x N), d = p*p*C, of the p x p patches of ONE resident image whose
 * top-left corners are coords[0..N), without materialising it:
 *     X[(r*p + c)*C + ch, j] = img[y_j + r, x_j + c, ch]        (the feature order of onmf_gather_patches)
 * A minibatch is idx[0..n) into [0, N) (NULL: columns 0..n-1).  An index outside [0, N), or a corner whose patch leaves
 * the image, yields a NaN row and is never dereferenced.  Storage: img is ONMF_F32, ONMF_F64 (fp64 engine, index gather
 * only) or ONMF_STORE_U8 (value = (float)stored * (float)scale).  Every product gives the same bits as the same call on
 * the materialised pool onmf_gather_patches(img, coords) (for u8: the pool of (float)u8 * scale, or the u8 pool on the
 * fused path) with the same idx: only the addressing differs.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  const void* img;          /* (H x W x C) row-major, device */
  int kind;                 /* ONMF_F32, ONMF_F64 or ONMF_STORE_U8 */
  int H, W, C, p;
  const int32_t* coords;    /* (n_coords x 2) int32 top-left corners (y, x), device */
  int64_t n_coords;         /* N */
  const int64_t* idx;       /* n indices into [0, n_coords), device, or NULL for 0..n-1 */
  int64_t n;                /* minibatch size (this rank's columns) */
  double scale;             /* ONMF_STORE_U8: value = (float)stored * (float)scale */
} onmf_patch_minibatch;

/* index gather: Xt[j, :] = patch(coords[idx[j]]) as dtype_out rows (pitch ld elements), widening u8 -> fp32.  dtype_out is the
 * image's dtype for ONMF_F32 / ONMF_F64 images and ONMF_F32 for ONMF_STORE_U8. */
int onmf_gather_patches_mb(const onmf_patch_minibatch* pm, int dtype_out, void* Xt, int64_t ld, void* stream);
/* onmf_cov_fused_tc / onmf_surrogate_fused_tc with the loaders reading patches of the image (fp32 or u8 image,
 * onmf_fused_tc_supported(k, p*p*C); ONMF_E_UNSUPPORTED when (p+32)*W*C >= 2^31).  Workspace: onmf_surrogate_fused_tc_workspace. */
int onmf_cov_fused_tc_patches(const onmf_patch_minibatch* pm, const void* W_hi, const void* W_lo, int k, void* Ct, void* stream);
int onmf_surrogate_fused_tc_patches(const void* Ht, const onmf_patch_minibatch* pm, int k, void* P, int blend, double w,
                                    const double* w_dev, void* A, void* B, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K5  dictionary update (one block-coordinate-descent sweep)
 * replaces: update_dict  src/ontf.py:91-115 == src/onmf.py:92-116
 *   for j in 0..k-1:  W[:,j] -= (W A[:,j] - B[j,:]^T) / (A[j,j] + 1);  W[:,j] = max(W[:,j], 0);
 *                     W[:,j] /= max(1, ||W[:,j]||_2)
 * W_in and W_out (d x k) may alias.  Three kernels, chosen by shape: one CTA (d <= 1024 and W, A within its shared memory),
 * one thread-block cluster of up to 16 CTAs (d*k up to ~0.9 M fp32 entries), a cooperative grid beyond that (onmf_update_dict_ws with a
 * workspace).  Each is deterministic and gives bit-identical results on every GPU of a data-parallel run; the three differ from
 * one another in summation order (last bits).
 * ------------------------------------------------------------------------------------------- */
int onmf_update_dict(int dtype, const void* W_in, const void* A, const void* B, int d, int k,
                     void* W_out, void* stream);
/* Dictionaries that fit one cluster's shared memory (up to 16 CTAs) (d*k up to ~0.9 M fp32 / 0.45 M fp64 entries: every BASELINE
 * config) are swept by one cluster with W resident in shared memory and need no workspace (the function returns 0).
 * Larger ones (joint unfoldings of big tensors) fall back to a cooperative grid with W in L2 and one grid-wide barrier
 * per atom; that path needs onmf_update_dict_workspace(dtype, d, k) bytes of scratch. */
size_t onmf_update_dict_workspace(int dtype, int d, int k);
int onmf_update_dict_ws(int dtype, const void* W_in, const void* A, const void* B, int d, int k,
                        void* W_out, void* workspace, size_t workspace_bytes, void* stream);
/* The kernel and launch shape onmf_update_dict[_ws] uses for (dtype, d, k), the same decision the launcher makes.  Host
 * only: launches nothing and needs no GPU (without one it assumes the B200's 227 KB of opt-in shared memory and 148 SMs).
 * Depends on the environment switches ONMF_BCD_SMALL, ONMF_BCD_TPR, ONMF_BCD_REGW and ONMF_BCD_MBAR as the launcher does.
 * ONMF_E_UNSUPPORTED when no kernel takes the shape. */
#define ONMF_BCD_KIND_SMALL 0    /* bcd_small_kernel: one CTA, one thread per row, W and A in shared memory */
#define ONMF_BCD_KIND_CLUSTER 1  /* bcd_kernel: a cluster of 1-16 CTAs, each with a row slab of W in shared memory */
#define ONMF_BCD_KIND_GRID 2     /* bcd_global_kernel: cooperative grid, W in global memory (needs the workspace) */
typedef struct {
  int kind;              /* ONMF_BCD_KIND_* */
  int ctas;              /* cluster size (CLUSTER), grid size (GRID), 1 (SMALL) */
  int rows_per_cta;      /* rows of W each CTA owns */
  int tpr;               /* lanes per row of W in the dot product (CLUSTER; 1 for SMALL, a warp for GRID) */
  int ks;                /* row pitch of W in shared memory, in elements (SMALL, CLUSTER) */
  int threads;           /* threads per CTA */
  int regw;              /* CLUSTER: 1 when each lane keeps its share of its row of W in registers (fp32) */
  int mbar;              /* CLUSTER: column-norm signalling, 0 barrier.cluster, 1 release-arrive, 2 st.async */
  size_t smem;           /* dynamic shared memory per CTA, bytes */
} onmf_bcd_plan;
int onmf_update_dict_plan(int dtype, int d, int k, onmf_bcd_plan* out);

/* ---------------------------------------------------------------------------------------------
 * secondary coder: row-wise projected gradient (shipped src/onmf.py:233-271 with r=None),
 * ONE outer iteration `it` (step 1/(sqrt(it+10) (G_qq+1))), in place on Ht (n x k).
 * The outer loop / stopping test stays on the host (it needs spectral norms).
 * ------------------------------------------------------------------------------------------- */
int onmf_pgd_sweep(int dtype, const void* G, const void* Ct, int64_t n, int k, double alpha,
                   int it, void* Ht, void* stream);
/* the same sweep restricted to the rows q_begin <= q < q_end of H (atoms): lets the host apply the reference's radius
 * projection (src/onmf.py:260-262), which -- because of the aliasing `H0 = H1` at :263 -- only ever acts after row 0 of
 * the first outer iteration. */
int onmf_pgd_sweep_rows(int dtype, const void* G, const void* Ct, int64_t n, int k, double alpha, int it, void* Ht,
                        int q_begin, int q_end, void* stream);

/* ---------------------------------------------------------------------------------------------
 * batched reconstruction (SURVEY.md §8f.1): replaces the per-patch Python loop
 * image_reconstruction.py:375-392 (one update_code_within_radius call + k*k python paints per patch)
 * ------------------------------------------------------------------------------------------- */
/* the complete projected-gradient coder per sample (outer loop + per-sample stopping test in-kernel), i.e. what the
 * reference computes when it calls update_code_within_radius on ONE patch at a time; Ht (n x k) holds H0 on entry.
 * One warp per sample; for k <= 32 and n >= 16 x SMs one thread per sample (same iteration and stopping test, dot products summed
 * in index order instead of butterfly order: results agree to rounding, not bit for bit). */
int onmf_pgd_code_columns(int dtype, const void* G, const void* Ct, int64_t n, int k, double alpha, int sub_iter,
                          double stopping_diff, void* Ht, void* stream);
/* overlap-averaged canvas (H x W x C) from the reconstructions R ((ny*nx) x ldr) of the p x p patches whose top-left
 * corners lie on the grid (gy*stride, gx*stride); count (H x W, may be NULL) receives the overlap counts.  Each pixel sums
 * its covering patches in ascending grid order j = gy*nx + gx; pixels no patch covers get 0 and count 0.  The whole-grid
 * call of onmf_patch_grid_accumulate. */
int onmf_patch_grid_mean(int dtype, const void* R, int64_t ldr, int ny, int nx, int p, int stride, int C, int H,
                         int W, void* canvas, void* count, void* stream);
/* the same mean, built from consecutive ranges of grid patches: this call adds the patches j0 <= j < j1, row j - j0 of R
 * being the reconstruction of grid patch j.  Calls over consecutive ranges that cover [0, ny*nx), in order, give the same
 * canvas and count bits as one onmf_patch_grid_mean call, with no memset: a pixel whose first covering patch lies in the
 * range starts from 0, every other one continues the running sum the earlier call left in the canvas; the call holding
 * the pixel's last covering patch divides by the count and writes it.  An uncovered pixel (y, x) is written (0, count
 * 0) by the call holding patch min(y / stride, ny - 1) * nx + min(x / stride, nx - 1).  A call touches only canvas rows
 * gy(j0)*stride .. gy(j1-1)*stride + p and the uncovered pixels it owns. */
int onmf_patch_grid_accumulate(int dtype, const void* R, int64_t ldr, int ny, int nx, int p, int stride, int C, int H,
                               int W, int64_t j0, int64_t j1, void* canvas, void* count, void* stream);

/* NDL motif-adjacency patches (SURVEY.md §8f.4): Xt[j, q*kk + r] = has_edge(emb[j, q], emb[j, r]) for a CSR graph with
 * sorted neighbour lists -- replaces the k*k python has_edge loop network_reconstruction_nx.py:302-305 for a batch of
 * MCMC states (onmf_motif_chain below produces them on the device). */
int onmf_motif_patches(int dtype, const int64_t* rowptr, const int32_t* colidx, int n_nodes, const int32_t* emb,
                       int64_t n, int kk, void* Xt, void* stream);

/* Batched network reconstruction (SURVEY.md §8f.1): the running-mean edge weights of network_reconstruction_nx.py:475-491
 * for a whole MCMC trajectory.  R (n x ldr) holds the patch reconstructions (R[j, q*kk + r] = (W h_j)[q*kk + r]), emb
 * (n x kk) the node index of every motif position; every entry is added to the directed pair (emb[j,q], emb[j,r]) in an
 * open-addressing hash table: keys (capacity x uint64, pre-filled with 0xFF bytes; key = a << 32 | b), sums (capacity
 * doubles, zeroed), counts (capacity uint32, zeroed).  capacity: a power of two > 2 n kk^2.  Mean weight = sum / count.
 * *failed (device uint32, zeroed) counts entries that could not be placed (negative node index, table full). */
int onmf_edge_scatter_add(int dtype, const void* R, int64_t ldr, const int32_t* emb, int64_t n, int kk,
                          unsigned long long* keys, double* sums, unsigned int* counts, int64_t capacity,
                          unsigned int* failed, void* stream);

/* NDL motif embeddings (the MCMC of network_reconstruction_nx.py: tree_sample, get_single_patch_glauber): n_chains independent
 * Glauber chains of homomorphisms x of the path 0 - 1 - ... - kk-1 into a graph (x[q] ~ x[q+1]), 2 <= kk <= 32.  The graph is
 * a CSR adjacency (rowptr n_nodes + 1 int64, colidx int32) with ascending rows, self-loops allowed; it must be symmetric.
 * state (n_chains x kk int32) holds node positions; chain c is the global chain chain0 + c (chain0 + n_chains <= 2^32).
 * Randomness: Philox4x32-10 (multipliers 0xD2511F53, 0xCD9E8D57, key increments 0x9E3779B9, 0xBB67AE85), key = seed (lo, hi);
 * mulhi32(u, m) = floor(u m / 2^32), a bias of at most m / 2^32 against the uniform draw from m items.
 *   init, draw q of chain c, counter (q, 0, c, 1):  x[0] = node mulhi32(word0, n_nodes), redrawn from counter (0, a, c, 1),
 *         a = 1, 2, ..., while it has no neighbour; x[q] = N(x[q-1])[mulhi32(word0, deg)] for q >= 1.
 *   Glauber step t of chain c, counter (t_lo, t_hi, c, 0):  site i = mulhi32(word0, kk); x[i] <- S[mulhi32(word1, |S|)] with
 *         S = N(x[i-1]) & N(x[i+1]) for 0 < i < kk-1, N(x[1]) for i = 0, N(x[kk-2]) for i = kk-1, in ascending order.  S holds
 *         the current x[i], so a step may leave the state unchanged.
 * A trajectory is a function of (seed, chain0 + c, t) only: launch shape, n_chains, steps_per_sample and the split of a run into
 * calls do not change it (oracle/motif_chain.py restates both entry points in numpy).
 * onmf_motif_chain_init writes state; it reads rowptr[n_nodes] and synchronises the stream once (ONMF_E_ARG for a graph
 * without an edge).
 * onmf_motif_chain runs the steps step0 + 1 ... step0 + n_samples * steps_per_sample and writes out[s, c, :] (n_samples x n_chains
 * x kk int32, row-major) = the state after step step0 + (s+1) * steps_per_sample; the final state is left in state.  It first
 * checks every state with one small kernel and synchronises the stream to read the result: ONMF_E_ARG, before any step, for
 * a node outside [0, n_nodes) or a consecutive pair that is not an edge.  Neither call can be captured in a CUDA graph.
 * ONMF_E_ARG: kk < 2, a non-positive count, n_nodes > INT32_MAX; ONMF_E_UNSUPPORTED: kk > 32. */
int onmf_motif_chain_init(const int64_t* rowptr, const int32_t* colidx, int64_t n_nodes, int kk, int64_t n_chains, int64_t chain0,
                          uint64_t seed, int32_t* state, void* stream);
int onmf_motif_chain(const int64_t* rowptr, const int32_t* colidx, int64_t n_nodes, int kk, int64_t n_chains, int64_t chain0,
                     uint64_t seed, uint64_t step0, int64_t n_samples, int64_t steps_per_sample, int32_t* state, int32_t* out,
                     void* stream);

/* Ising lattices (the trajectory of the Ising driver, ising_simulator.ising_update): n_chains independent checkerboard
 * heat-bath chains of P(sigma) ~ exp(beta sum_<ij> sigma_i sigma_j) on an H x W torus (J = 1, no field); H and W even and
 * >= 4 (a bipartite torus on which no neighbour repeats), H*W < 2^31.  state (n_chains x H x W int8, row-major) holds +-1;
 * chain c is the global chain chain0 + c (chain0 + n_chains <= 2^32).  colour(y, x) = (y + x) & 1; the sites of one colour
 * are numbered m = 0, 1, ... in row-major order.
 *   sweep t (t = 1, 2, ... counts sweeps globally): colour 0, then colour 1.  Site m of colour k draws word (m & 3) of
 *         Philox4x32-10 (the constants of onmf_motif_chain) at counter (t_lo, t_hi, chain0 + c, 2 (m >> 2) + k), key = seed
 *         (lo, hi), and becomes +1 iff that word < thr[(s + 4) / 2], s in {-4, -2, 0, 2, 4} the sum of its four neighbours.
 *   init: sweep t = 0 with every threshold 2^31 (independent uniform +-1).
 * A trajectory is a function of (seed, chain0 + c, t) only: the form the plan picks, the launch shape, n_chains,
 * sweeps_per_sample and the split of a run into calls do not change it (oracle/ising_chain.py restates both calls in numpy).
 * onmf_ising_chain runs the sweeps sweep0 + 1 ... sweep0 + n_samples * sweeps_per_sample and writes out[s, c, :, :]
 * (n_samples x n_chains x H x W, out_dtype ONMF_F32 or ONMF_F64, row-major) = +-1, the state after sweep
 * sweep0 + (s+1) * sweeps_per_sample; the final state is left in state.  No address depends on a spin value, so a state
 * that is not +-1 is not checked (its sites become +-1 as they are updated).
 * ONMF_E_ARG, before any launch: odd or too small sides, a non-positive count, chain0 out of range, a non-finite beta,
 * another out_dtype, or a last sweep beyond 2^64 - 1. */
int onmf_ising_chain_init(int H, int W, int64_t n_chains, int64_t chain0, uint64_t seed, int8_t* state, void* stream);
int onmf_ising_chain(int H, int W, int64_t n_chains, int64_t chain0, uint64_t seed, double beta, uint64_t sweep0, int64_t n_samples,
                     int64_t sweeps_per_sample, int8_t* state, void* out, int out_dtype, void* stream);
/* The heat-bath table thr[j] = min(floor(2^32 / (1 + exp(-2 beta (2j - 4)))), 2^32 - 1), j = 0..4: 2^32 P(+1 | s = 2j - 4);
 * thr[2] = 2^31.  Host only.  ONMF_E_ARG for a non-finite beta. */
int onmf_ising_thresholds(double beta, uint32_t thr[5]);
/* The form onmf_ising_chain uses for an H x W lattice, the same decision the launcher makes.  Host only: launches nothing and
 * needs no GPU (without one it assumes the B200's 227 KB of opt-in shared memory).  ONMF_E_ARG for a shape the chain refuses. */
#define ONMF_ISING_FORM_SMEM 0    /* one CTA per chain (grid-striding), the lattice in shared memory for every sweep of a call */
#define ONMF_ISING_FORM_GLOBAL 1  /* lattices above the opt-in shared memory: one launch per half-sweep over all chains */
typedef struct {
  int form;              /* ONMF_ISING_FORM_* */
  int threads;           /* threads per CTA (of the sweep kernel) */
  size_t smem;           /* dynamic shared memory per CTA, bytes (H * W for SMEM, 0 for GLOBAL) */
} onmf_ising_plan;
int onmf_ising_chain_plan(int H, int W, onmf_ising_plan* out);

/* ---------------------------------------------------------------------------------------------
 * The fused online step: ONE host call per minibatch
 * replaces: Online_NTF.step / Online_NMF.step  (src/ontf.py:117-154, src/onmf.py:119-167) -- sparse_code, the A/B
 *           recursion and update_dict with the OLD aggregates -- as a fixed schedule of the kernels above on two
 *           streams (DESIGN.md "Step schedule").  The plan owns the CUDA events that order the streams; the caller owns
 *           every buffer.  Nothing here allocates device memory or synchronises the host.
 *   single GPU : onmf_step(plan, buffers, Xt, NULL, n, w, cur)
 *   multi GPU  : onmf_step_launch(...);  all-reduce(sum) P[cur] (and P2) on side_stream;  onmf_step_finish(..., w, cur)
 * `cur` (0/1) selects the current dictionary W[cur] (with G[cur], Whi/Wlo[cur]) and the partial-sum buffer P[cur]; the
 * step writes the new dictionary to index cur^1 and the caller flips cur afterwards.  w = t^-beta.
 * Xt (n x d) are this rank's columns; Xt = NULL (tensor-core path): Xhi/Xlo already hold the split minibatch.
 * codes != NULL: externally computed codes (n x k) are aggregated instead of running the coder.
 * ------------------------------------------------------------------------------------------- */
typedef struct onmf_step_plan onmf_step_plan;
typedef struct {
  int dtype, d, k;
  int use_tc;            /* tensor-core products (fp32, onmf_tc_supported(k, d)) */
  int track_C;           /* also maintain C <- (1-w) C + w X X^T (src/onmf.py:157-158) */
  int max_iter;          /* LARS iteration cap (sklearn: 1000) */
  int reserve_sms;       /* SMs the coder leaves free for the dictionary update; -1 = automatic */
  int hold_coder;        /* 1: the coder waits for the previous step's blend (multi-GPU, see DESIGN.md) */
  double alpha;
  void* W[2];            /* d x k */
  double* G[2];          /* k x k, FP64 Gram of W[i] (always FP64) */
  void* Whi[2];          /* TF32 split of W[i] (tensor-core path) */
  void* Wlo[2];
  void* A;               /* k x k */
  void* B;               /* k x d */
  void* C;               /* d x d or NULL */
  void* P[2];            /* k x (k+d) packed partial sums, double-buffered */
  void* P2;              /* d x d partial sum for C or NULL */
  void* Ct;              /* n x k covariances */
  void* Ht;              /* n x k codes (output) */
  void* Xhi;             /* n x d TF32 split of the minibatch (tensor-core path) */
  void* Xlo;
  void* Hhi;             /* n x k TF32 split of the codes */
  void* Hlo;
  void* ws_lars;  size_t ws_lars_bytes;   /* onmf_lasso_lars_workspace, zero-filled once */
  void* ws_sur;   size_t ws_sur_bytes;    /* max(onmf_surrogate_workspace, onmf_surrogate_tc_workspace[, xxt]) */
  void* ws_gram;  size_t ws_gram_bytes;   /* onmf_gram_f64_workspace */
  onmf_lars_stats* stats;                 /* or NULL */
  void* main_stream;
  void* side_stream;
  double* w_dev;                          /* one device double (blend weight of onmf_step_graph) or NULL */
} onmf_step_buffers;

/* A minibatch by reference (fused tensor-core path, onmf_fused_tc_supported): rows idx[0..n) of a stored sample-major pool
 * in fp32 or a narrow storage format -- X_batch = X_unfold[:, idx] (src/ontf.py:231) without materialising it. */
typedef struct {
  int kind;              /* ONMF_F32, ONMF_STORE_U8 or ONMF_STORE_F16 */
  const void* base;      /* pool, one sample per row */
  int64_t n_pool;        /* rows in the pool */
  int64_t ld;            /* row pitch in elements */
  const int64_t* idx;    /* n row indices, or NULL for rows 0..n-1 */
  int64_t n;             /* minibatch size (this rank's columns) */
  double scale;          /* value = stored * scale (1/255 for 8-bit image data, image_reconstruction.py:88) */
} onmf_minibatch;

/* timing_slots > 0: the plan keeps a ring of event pairs around the coder launch (read with onmf_step_plan_lars_ms) */
int onmf_step_plan_create(onmf_step_plan** plan, int timing_slots);
int onmf_step_plan_destroy(onmf_step_plan* plan);
/* call after (re)setting W, A, B on main_stream: the first dictionary update must wait for those writes */
int onmf_step_plan_mark_state(onmf_step_plan* plan, void* main_stream);
long long onmf_step_plan_launches(const onmf_step_plan* plan);    /* kernels launched through the plan so far */
int onmf_step_plan_reset_timing(onmf_step_plan* plan);
/* elapsed ms of the coder launch of the last (up to timing_slots) steps; waits for those launches to finish */
int onmf_step_plan_lars_ms(onmf_step_plan* plan, float* out, int max_out, int* n_out);
int onmf_step_launch(onmf_step_plan* plan, const onmf_step_buffers* b, const void* Xt, const void* codes, int64_t n,
                     int cur);
int onmf_step_finish(onmf_step_plan* plan, const onmf_step_buffers* b, double w, int cur);
int onmf_step(onmf_step_plan* plan, const onmf_step_buffers* b, const void* Xt, const void* codes, int64_t n, double w,
              int cur);
/* onmf_step as ONE CUDA graph launch (single GPU; b->w_dev must be set).  The graph of a given (Xt, codes, n, cur,
 * buffers) is captured the second time that key is seen and replayed afterwards; anything a graph cannot express
 * (track_C, timing slots, hold_coder) and first sights fall through to onmf_step.  Same results, bit for bit. */
int onmf_step_graph(onmf_step_plan* plan, const onmf_step_buffers* b, const void* Xt, const void* codes, int64_t n, double w,
                    int cur);
long long onmf_step_plan_graph_steps(const onmf_step_plan* plan);   /* steps that ran as a graph replay */
/* the same four entry points for a minibatch passed by reference: cov and the partial sums read the pool rows in place
 * (gemm_fused.cu), and on a single GPU (onmf_step_mb / onmf_step_graph_mb) the blend is fused into the partial-sum
 * reduction.  ONMF_E_UNSUPPORTED unless use_tc, fp32 and onmf_fused_tc_supported(k, d); ws_sur must then hold
 * onmf_surrogate_fused_tc_workspace(n, k, d) bytes. */
int onmf_step_launch_mb(onmf_step_plan* plan, const onmf_step_buffers* b, const onmf_minibatch* mb, const void* codes, int cur);
int onmf_step_mb(onmf_step_plan* plan, const onmf_step_buffers* b, const onmf_minibatch* mb, const void* codes, double w,
                 int cur);
int onmf_step_graph_mb(onmf_step_plan* plan, const onmf_step_buffers* b, const onmf_minibatch* mb, const void* codes, double w,
                       int cur);
/* the same three forms for a patch minibatch (onmf_patch_minibatch, d = p*p*C): the fused kernels read the patches of the
 * image in place.  Same conditions as the _mb forms (use_tc, fp32, onmf_fused_tc_supported, no track_C) and an fp32 or u8
 * image; other engines gather the minibatch with onmf_gather_patches_mb and take the dense forms.  The graph of
 * onmf_step_graph_patches is keyed on the image, the corners, the geometry, the storage kind and the scale as well. */
int onmf_step_launch_patches(onmf_step_plan* plan, const onmf_step_buffers* b, const onmf_patch_minibatch* pm, const void* codes,
                             int cur);
int onmf_step_patches(onmf_step_plan* plan, const onmf_step_buffers* b, const onmf_patch_minibatch* pm, const void* codes,
                      double w, int cur);
int onmf_step_graph_patches(onmf_step_plan* plan, const onmf_step_buffers* b, const onmf_patch_minibatch* pm, const void* codes,
                            double w, int cur);

#ifdef __cplusplus
}
#endif
#endif /* ONMF_B200_H */
