"""CPU oracle for the online NMF/NTF dictionary-learning hot path.

TEST INFRASTRUCTURE ONLY -- never imported by the product package
(`onmf_ontf_ndl_b200`).  Only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s
`cpu_baseline` / `--impl reference` legs may import this file, and only as the
checker / the CPU baseline.

It is a numpy restatement (float64, like the reference) of

  * `Online_NTF.joint_sparse_code_tensor`   reference src/ontf.py:59-89
  * `Online_NTF.update_dict`                reference src/ontf.py:91-115 (== src/onmf.py:92-116)
  * `Online_NTF.step`                       reference src/ontf.py:117-154
  * `Online_NTF.train_dict_single` loop     reference src/ontf.py:156-244
  * `update_code_within_radius`             reference src/onmf.py:233-271
    (and its G / C form per sweep and per sample, `pgd_sweep_gc` / `pgd_columns_gc`)
  * tensor matricization (`tl_unfold`)      reference src/ontf.py:203-208
  * the drivers' patch gathers              reference image_reconstruction.py:173-206,
                                            image_reconstruction_tensor.py:87-124,
                                            ising_reconstruction.py:46-66

The sparse-coding arithmetic of the reference lives in a third-party dependency that
is not vendored in /root/reference: scikit-learn (unpinned by the reference; 1.9.0 in
this image) -- call chain src/ontf.py:79-86 -> sklearn/decomposition/_dict_learning.py
(`SparseCoder.transform` -> `_sparse_encode` -> `_sparse_encode_precomputed`, alpha /
n_features scaling at :119) -> sklearn/linear_model/_least_angle.py (`LassoLars._fit`
per-target loop :1136-1153 -> `_lars_path_solver` :415-917, Gram mode, method='lasso',
positive=True, return_path=False).  `lars_lasso_positive` below restates that published
algorithm (Efron et al. LARS, lasso modification with positivity, Gram mode) including
sklearn's stopping rule / last-segment interpolation; `sparse_code_sklearn` calls the
dependency itself exactly as the reference's call site does.

Parity pin: the reference ships no tests / golden vectors for this path (SURVEY.md §4),
so the pin is the reference itself run in the authoring container:
`oracle/make_golden.py` imports the unmodified reference (oracle/ref_loader.py) and
writes per-step (idx, H, A, B, W) fixtures to tests/golden/*.npz, and
tests/test_oracle.py checks every function here against those fixtures (and against
sklearn 1.9.0 directly).
"""
from __future__ import annotations

import numpy as np

_TINY32 = float(np.finfo(np.float32).tiny)
_EPS32 = float(np.finfo(np.float32).eps)
_EPS64 = float(np.finfo(np.float64).eps)


# --------------------------------------------------------------------------------------
# positive LARS-lasso, Gram mode, one target (sklearn/_least_angle.py:415-917 semantics)
# --------------------------------------------------------------------------------------

def _min_pos(v):
    """sklearn/utils/arrayfuncs.pyx `min_pos`: min over strictly positive entries, else DBL_MAX."""
    v = v[v > 0.0]
    return float(v.min()) if v.size else float(np.finfo(np.float64).max)


def _chol_append(L, s, g_row, g_diag):
    """Border the s x s lower Cholesky factor held in L[:s,:s] with a new variable.

    g_row = G[new, active], g_diag = G[new,new].  Returns the new diagonal pivot.
    (sklearn/_least_angle.py:686-720)
    """
    w = g_row.copy()
    for i in range(s):  # forward substitution L w = g_row
        w[i] = (w[i] - L[i, :i] @ w[:i]) / L[i, i]
    L[s, :s] = w
    piv = max(np.sqrt(abs(g_diag - w @ w)), _EPS64)
    L[s, s] = piv
    return piv


def _chol_solve(L, s, b):
    """Solve (L L^T) x = b with the s x s factor (LAPACK potrs semantics)."""
    y = b.astype(np.float64).copy()
    for i in range(s):
        y[i] = (y[i] - L[i, :i] @ y[:i]) / L[i, i]
    for i in range(s - 1, -1, -1):
        y[i] = (y[i] - L[i + 1:s, i] @ y[i + 1:s]) / L[i, i]
    return y


def _chol_delete(L, s, out):
    """Remove variable `out` from the s x s factor with Givens rotations
    (sklearn/utils/arrayfuncs.pyx `cholesky_delete`)."""
    for i in range(out, s - 1):          # shift rows up
        L[i, :i + 2] = L[i + 1, :i + 2]
    for i in range(out, s - 1):          # re-triangularise
        a, b = L[i, i], L[i, i + 1]
        r = np.hypot(a, b)
        if r == 0.0:
            c, sn = 1.0, 0.0
        else:
            c, sn = a / r, b / r
        L[i, i] = r
        L[i, i + 1] = 0.0
        for q in range(i + 1, s - 1):
            x, y = L[q, i], L[q, i + 1]
            L[q, i] = c * x + sn * y
            L[q, i + 1] = c * y - sn * x


def lars_lasso_positive(G, c, reg, n_features, max_iter=1000, return_info=False,
                        round_decimals=15):
    """argmin_{h>=0} 0.5*||x - W h||^2 + reg * sum(h) the way sklearn's positive lasso_lars does it.

    G = W^T W (k x k), c = W^T x (k,), n_features = d (sklearn scales alpha by 1/d,
    _dict_learning.py:119, and the LARS correlations by 1/n_samples=1/d,
    _least_angle.py:649).  Includes sklearn's termination rule: the path stops at the
    first knot whose recorded alpha (= max *inactive* covariance / d) is <= reg/d (+ float32
    eps) and linearly interpolates the last segment (_least_angle.py:651-663) -- which on
    the final (unregularised least-squares) segment lands at a slightly shifted alpha
    (SURVEY.md §B.2); that behaviour is reproduced here by construction.
    """
    G = np.asarray(G, dtype=np.float64)
    cov = np.array(c, dtype=np.float64)
    k = cov.shape[0]
    alpha_min = float(reg) / n_features
    coef = np.zeros(k)
    prev_coef = np.zeros(k)
    alpha_cur, alpha_prev = 0.0, 0.0
    active = []                 # ordered like the Cholesky factor
    inact = list(range(k))      # ordered like sklearn's shortened Cov (tie-breaking only)
    L = np.zeros((min(max_iter, k) + 1, min(max_iter, k) + 1))
    n_iter = 0
    drop = False
    max_active = 0
    n_drops = 0
    status = 0                  # 0 normal, 1 degenerate regressor seen, 2 alpha-increase bail-out, 3 max_iter
    while True:
        if inact:
            vals = cov[inact]
            pos = int(np.argmax(vals))
            C = float(vals[pos])
        else:
            pos, C = -1, 0.0
        alpha_cur = C / n_features
        if alpha_cur <= alpha_min + _EPS32:
            if abs(alpha_cur - alpha_min) > _EPS32 and n_iter > 0:
                ss = (alpha_prev - alpha_min) / (alpha_prev - alpha_cur)
                coef = prev_coef + ss * (coef - prev_coef)
            break
        if n_iter >= max_iter or len(active) >= k:
            status = 3 if n_iter >= max_iter else status
            break
        if not drop:
            s = len(active)
            inact[pos], inact[0] = inact[0], inact[pos]
            j = inact[0]
            piv = _chol_append(L, s, G[j, active], G[j, j])
            if piv < 1e-7:
                # degenerate regressor: sklearn zeroes its covariance and retries
                # (_least_angle.py:723-742); it stays inactive.
                cov[j] = 0.0
                inact[pos], inact[0] = inact[0], inact[pos]
                status = 1
                continue
            inact.pop(0)
            active.append(j)
            max_active = max(max_active, len(active))
        if n_iter > 0 and alpha_prev < alpha_cur:
            status = 2          # "alpha increasing" early stop (_least_angle.py:752-765)
            break
        s = len(active)
        w = _chol_solve(L, s, np.ones(s))
        AA = 1.0 / np.sqrt(w.sum())
        w = w * AA
        corr = G[np.ix_(inact, active)] @ w if inact else np.zeros(0)
        if round_decimals is not None:
            corr = np.around(corr, decimals=round_decimals)
        g1 = _min_pos((C - cov[inact]) / (AA - corr + _TINY32)) if inact else np.finfo(np.float64).max
        gamma = min(g1, C / AA)
        z = -coef[active] / (w + _TINY32)
        z_pos = _min_pos(z)
        drop = False
        drop_pos = []
        if z_pos < gamma:
            drop_pos = list(np.where(z == z_pos)[0][::-1])
            gamma = z_pos
            drop = True
        n_iter += 1
        prev_coef = coef
        alpha_prev = alpha_cur
        coef = np.zeros(k)
        coef[active] = prev_coef[active] + gamma * w
        cov[inact] -= gamma * corr
        if drop:
            n_drops += len(drop_pos)
            for p in drop_pos:
                _chol_delete(L, len(active), p)
                jd = active.pop(p)
                # exact covariance of the dropped variable (_least_angle.py:891)
                cov[jd] = c[jd] - G[jd] @ coef
                inact.insert(0, jd)
    if return_info:
        return coef, dict(n_iter=n_iter, max_active=max_active, n_drops=n_drops, status=status)
    return coef


def sparse_code_lars(X, W, alpha, return_info=False):
    """H (k x n) = per-column positive lasso_lars codes; restated solver (no sklearn)."""
    X = np.asarray(X, dtype=np.float64)
    W = np.asarray(W, dtype=np.float64)
    d, n = X.shape
    G = W.T @ W
    Cv = W.T @ X
    H = np.zeros((W.shape[1], n))
    infos = []
    for j in range(n):
        if return_info:
            H[:, j], info = lars_lasso_positive(G, Cv[:, j], alpha, d, return_info=True)
            infos.append(info)
        else:
            H[:, j] = lars_lasso_positive(G, Cv[:, j], alpha, d)
    return (H, infos) if return_info else H


def sparse_code_sklearn(X, W, alpha):
    """The dependency itself, called as the reference's call site does (src/ontf.py:79-86).
    Returns H transposed to k x n."""
    from sklearn.decomposition import SparseCoder
    coder = SparseCoder(dictionary=np.asarray(W).T, transform_n_nonzero_coefs=None,
                        transform_alpha=alpha, transform_algorithm='lasso_lars', positive_code=True)
    return coder.transform(np.asarray(X).T).T


# --------------------------------------------------------------------------------------
# surrogate aggregation + dictionary update + loop
# --------------------------------------------------------------------------------------

def update_dict(W, A, B):
    """One Gauss-Seidel sweep over atoms (reference src/ontf.py:91-115).
    W (d x k), A (k x k), B (k x d).  Step 1/(A_jj + 1), clamp at 0, shrink into the unit ball."""
    W1 = np.array(W, dtype=np.float64, copy=True)
    k = W1.shape[1]
    for j in range(k):
        col = W1[:, j] - (W1 @ A[:, j] - B[j, :]) / (A[j, j] + 1.0)
        col = np.maximum(col, 0.0)
        W1[:, j] = col / max(1.0, np.linalg.norm(col))
    return W1


def aggregate(A, B, H, X, t, beta=None):
    """A1 = (1-w) A + w H H^T ; B1 = (1-w) B + w H X^T ; w = t^-beta
    (reference src/ontf.py:141-148; H here is k x n)."""
    b = 1.0 if beta is None else beta
    w = float(t) ** (-b)
    return (1.0 - w) * A + w * (H @ H.T), (1.0 - w) * B + w * (H @ X.T)


def step(X, A, B, W, t, alpha, beta=None, coder="lars"):
    """reference src/ontf.py:117-154: code with W, aggregate, then update_dict with the OLD A, B."""
    a = 2 if alpha is None else alpha
    H = sparse_code_sklearn(X, W, a) if coder == "sklearn" else sparse_code_lars(X, W, a)
    A1, B1 = aggregate(A, B, H, X, t, beta)
    W1 = update_dict(W, A, B)
    return H, A1, B1, W1


def step_given_codes(X, H, W, A, B, C, t, beta=None):
    """`step` with the codes H (k x n) given: the coder drops out and the step is the update with the OLD aggregates and
    the blends.  C (d x d) or None follows C1 = (1-w) C + w X X^T (reference src/onmf.py:157-158).  Returns (W1, A1, B1, C1)."""
    X = np.asarray(X, dtype=np.float64)
    H = np.asarray(H, dtype=np.float64)
    W1 = update_dict(W, A, B)
    A1, B1 = aggregate(A, B, H, X, t, beta)
    C1 = None
    if C is not None:
        w = float(t) ** (-(1.0 if beta is None else beta))
        C1 = (1.0 - w) * C + w * (X @ X.T)
    return W1, A1, B1, C1


def run_given_codes(Xs, Hs, W0, A0, B0, ts, beta=None, C0=None):
    """step_given_codes over a sequence of minibatches Xs[i] (d x n_i) with codes Hs[i] (k x n_i) at steps ts[i].
    Returns the final (W, A, B, C)."""
    W, A, B, C = W0, A0, B0, C0
    for X, H, t in zip(Xs, Hs, ts):
        W, A, B, C = step_given_codes(X, H, W, A, B, C, t, beta)
    return W, A, B, C


def train(X, k, idx_seq, W0, A0=None, B0=None, history=0, alpha=1, beta=None, coder="lars",
          record=False):
    """reference src/ontf.py:224-236 with the minibatch indices given explicitly
    (idx_seq[i-1] is the `np.random.randint(n, size=batch)` draw of step i; None = all columns)."""
    d = X.shape[0]
    W = np.array(W0, dtype=np.float64)
    A = np.zeros((k, k)) if A0 is None else np.array(A0, dtype=np.float64)
    B = np.zeros((k, d)) if B0 is None else np.array(B0, dtype=np.float64)
    trace = []
    for i, idx in enumerate(idx_seq, start=1):
        Xb = X if idx is None else X[:, idx]
        H, A, B, W = step(Xb, A, B, W, history + i, alpha, beta, coder)
        if record:
            trace.append(dict(H=H, A=A, B=B, W=W))
    return (W, A, B, trace) if record else (W, A, B)


# --------------------------------------------------------------------------------------
# shipped-ONMF projected-gradient coder (reference src/onmf.py:233-271)
# --------------------------------------------------------------------------------------

def update_code_within_radius(X, W, H0, r=None, alpha=0, sub_iter=10, stopping_diff=0.1):
    """Row-wise projected gradient on 0.5||X-WH||^2 + alpha*sum(H), H>=0.  H0 must be given
    (the reference draws it from the global numpy RNG when None, src/onmf.py:245-246)."""
    G = W.T @ W
    Cv = W.T @ X
    H0 = np.array(H0, dtype=np.float64)
    H = H0.copy()
    it, dist = 0, 1.0
    while it < sub_iter and dist > stopping_diff:
        H_old = H.copy()
        for q in range(H.shape[0]):
            grad = G[q, :] @ H - Cv[q, :] + alpha
            H[q, :] = np.maximum(H[q, :] - grad / (np.sqrt(it + 10.0) * (G[q, q] + 1.0)), 0.0)
            if r is not None:
                dd = np.linalg.norm(H - H0, 2)
                H = H0 + (r / max(r, dd)) * (H - H0)
            H0 = H
        dist = np.linalg.norm(H - H_old, 2) / np.linalg.norm(H_old, 2)
        it += 1
    return H


def pgd_sweep_gc(G, Ct, Ht, alpha, it, q0=0, q1=None):
    """One outer iteration of the coder above in the kernels' G / C form (onmf_pgd_sweep_rows): for q0 <= q < q1, Gauss-Seidel
    in q, h_q <- max(h_q - (G[q, :] h - c_q + alpha) / (sqrt(it + 10) (G_qq + 1)), 0), independently per sample.
    G (k x k) is used as given (row q), so it need not be symmetric; Ct, Ht (n x k) are sample-major.  Returns the new Ht."""
    G = np.asarray(G, dtype=np.float64)
    Ct = np.asarray(Ct, dtype=np.float64)
    H = np.array(Ht, dtype=np.float64, copy=True)
    k = G.shape[0]
    q1 = k if q1 is None else q1
    scale = np.sqrt(it + 10.0)
    for q in range(q0, q1):
        grad = H @ G[q, :] - Ct[:, q] + alpha
        H[:, q] = np.maximum(H[:, q] - grad / (scale * (G[q, q] + 1.0)), 0.0)
    return H


def pgd_columns_gc(G, Ct, Ht, alpha, sub_iter, stopping_diff):
    """The whole coder per sample in the G / C form (onmf_pgd_code_columns): sweeps it = 0, 1, ... while it < sub_iter and
    dist > stopping_diff, dist = ||h - h_old|| / ||h_old|| of that sample alone (x / 0 = inf keeps going, 0 / 0 = NaN stops,
    like the reference's numpy division).  Returns (Ht, sweeps (n,), trail (n x sub_iter)): trail[j, i] is the dist after
    sweep i of sample j, valid for i < sweeps[j] (NaN beyond)."""
    G = np.asarray(G, dtype=np.float64)
    H = np.array(Ht, dtype=np.float64, copy=True)
    Ct = np.asarray(Ct, dtype=np.float64)
    n = H.shape[0]
    sweeps = np.zeros(n, dtype=np.int64)
    trail = np.full((n, max(int(sub_iter), 0)), np.nan)
    dist = np.ones(n)
    for it in range(int(sub_iter)):
        act = np.nonzero(dist > stopping_diff)[0]
        if act.size == 0:
            break
        h_old = H[act]
        h = pgd_sweep_gc(G, Ct[act], h_old, alpha, it)
        with np.errstate(divide="ignore", invalid="ignore"):
            dist[act] = np.linalg.norm(h - h_old, axis=1) / np.linalg.norm(h_old, axis=1)
        H[act] = h
        trail[act, it] = dist[act]
        sweeps[act] += 1
    return H, sweeps, trail


# --------------------------------------------------------------------------------------
# matricization and patch gathers
# --------------------------------------------------------------------------------------

def unfold(T, mode):
    """tensorly.unfold (numpy backend): mode-`mode` matricization, C order."""
    return np.reshape(np.moveaxis(T, mode, 0), (T.shape[mode], -1))


def matricize(T, mode, learn_joint_dict):
    """reference src/ontf.py:203-208 -> (d, n) data matrix."""
    U = unfold(T, mode)
    return U.T if learn_joint_dict else U


def gather_patches_gray(img, coords, k):
    """reference image_reconstruction.py:173-206 / ising_reconstruction.py:46-66:
    X[:, j] = img[a:a+k, b:b+k].reshape(-1) for (a, b) = coords[j]."""
    n = len(coords)
    X = np.empty((k * k, n))
    for j, (a, b) in enumerate(coords):
        X[:, j] = img[a:a + k, b:b + k].reshape(-1)
    return X


def gather_patches_color_tensor(img, coords, k):
    """reference image_reconstruction_tensor.py:87-124: tensor (k*k, C, N),
    T[:, :, j] = img[a:a+k, b:b+k, :].reshape(k*k, C)."""
    n = len(coords)
    C = img.shape[2]
    T = np.empty((k * k, C, n))
    for j, (a, b) in enumerate(coords):
        T[:, :, j] = img[a:a + k, b:b + k, :].reshape(k * k, C)
    return T


def surrogate_error(W, A, B, C):
    """tr(W A W^T) - 2 tr(W B) + tr(C)   (reference ising_reconstruction.py:133,164)."""
    return float(np.trace(W @ A @ W.T) - 2.0 * np.trace(W @ B) + np.trace(C))


# --------------------------------------------------------------------------------------
# patch-grid reconstruction loop (reference image_reconstruction.py:358-406)
# --------------------------------------------------------------------------------------

def reconstruct_image_loop(A, W, k, res, alpha, sub_iter, stopping_diff, H0, coder=None):
    """for every grid patch (i, j), i in range(0, H-k, res), j in range(0, W-k, res): code the flattened patch (HWC order)
    alone with update_code_within_radius(H0 = column of H0), reconstruct it with W and fold it into a running-mean canvas
    (image_reconstruction.py:375-392).  `coder`: optional callable (patch_column) -> code column, e.g. the reference's
    own update_code_within_radius.  Returns (canvas, overlap_count, codes (r x n))."""
    A3 = A[:, :, None] if A.ndim == 2 else A
    Hh, Ww, C = A3.shape
    rec = np.zeros(A3.shape)
    cnt = np.zeros((Hh, Ww))
    codes = []
    pidx = 0
    for i in range(0, Hh - k, res):
        for j in range(0, Ww - k, res):
            patch = A3[i:i + k, j:j + k, :].reshape((-1, 1))
            h0 = H0[:, pidx:pidx + 1]
            if coder is None:
                code = update_code_within_radius(patch, W, h0, r=None, alpha=alpha, sub_iter=sub_iter,
                                                 stopping_diff=stopping_diff)
            else:
                code = coder(patch, h0)
            codes.append(code[:, 0])
            pr = (W @ code).T.reshape(k, k, C)
            c = cnt[i:i + k, j:j + k]
            rec[i:i + k, j:j + k, :] = (c[:, :, None] * rec[i:i + k, j:j + k, :] + pr) / (c[:, :, None] + 1)
            cnt[i:i + k, j:j + k] += 1
            pidx += 1
    rec = rec[:, :, 0] if A.ndim == 2 else rec
    return rec, cnt, (np.stack(codes, 1) if codes else np.zeros((W.shape[1], 0)))


def motif_patches(adj_sets, emb):
    """network_reconstruction_nx.py:302-305 for a batch of embeddings: X[q*k + r, j] = has_edge(emb[j][q], emb[j][r]);
    adj_sets[u] = set of neighbours of u."""
    emb = np.asarray(emb)
    n, k = emb.shape
    X = np.zeros((k * k, n))
    for j in range(n):
        for q in range(k):
            for r in range(k):
                X[q * k + r, j] = 1.0 if emb[j, r] in adj_sets[emb[j, q]] else 0.0
    return X


def reconstruct_network_loop(adj_sets, W, embs, alpha=0.0, coder=None):
    """network_reconstruction_nx.py:464-491 restated: per MCMC state one k x k adjacency patch (has_edge of the embedded
    nodes, :302-305), coded with the positive lasso_lars at `alpha` (:466-473), patch_recons = W code (:474-475), every
    entry folded into a running mean per DIRECTED pair (emb[q], emb[r]) in loop order (:477-491).
    adj_sets: {node: set(neighbours)}; embs: (T x k) node labels.  Returns ({(a, b): weight}, {(a, b): count})."""
    embs = np.asarray(embs)
    kk = embs.shape[1]
    if coder is None:
        coder = lambda patch: sparse_code_lars(patch, W, alpha)
    weight, count = {}, {}
    for emb in embs.tolist():
        patch = np.zeros((kk * kk, 1))
        for q in range(kk):
            for r in range(kk):
                patch[q * kk + r, 0] = 1.0 if emb[r] in adj_sets.get(emb[q], ()) else 0.0
        code = coder(patch)                                   # (r x 1)
        rec = (W @ code).reshape(kk, kk)
        for q in range(kk):
            for r in range(kk):
                key = (emb[q], emb[r])
                j = count.get(key, 0)
                weight[key] = (j * weight[key] + rec[q, r]) / (j + 1) if j else rec[q, r]
                count[key] = j + 1
    return weight, count
