"""The projected-gradient coder (csrc/gather.cu) in every kernel form, against the fp64 G / C restatement
oracle.onmf_oracle.pgd_sweep_gc / pgd_columns_gc, and the spectral norm of its stopping test (csrc/gemm_simt.cu).

onmf_pgd_sweep(_rows) runs pgd_sweep_kernel<T, NA> and onmf_pgd_code_columns runs pgd_columns_kernel<T, NA>: one warp per
sample, NA = 1 / 2 / 4 / 8 / 16 for k <= 32 / 64 / 128 / 256 / 512, the Gram in shared memory while k^2 sizeof(T) fits the
opt-in limit and read from global memory above it; the warps stride over the samples beyond their grid of 4 x SMs CTAs of
8 warps.  onmf_pgd_code_columns takes pgd_columns_tps_kernel<T, KP> (one thread per sample, KP = k rounded up to a
multiple of 4) when k <= 32 and n >= 16 x SMs.  Every threshold is read from the device.

The kernels take G as given, so the cases use a NON-symmetric G (a Gram plus a skew-symmetric part; positive diagonal):
with G = W^T W a kernel that read G by column would pass.

Bars: fp64 1e-12 relative per sample after one sweep, 1e-10 after a whole code_columns run or ten chained sweeps; fp32
16 x the error of a numpy float32 emulation of the same iteration against the fp64 restatement, at least FLOOR32.  Runs with
a stopping test are compared where the kernel and the oracle take the same number of sweeps: stopping_diff is picked from
the oracle's dist trails, and a column whose trail comes within MARGIN64 / MARGIN32 (relative) of it is left out (at most
1 % of the columns; in fp64 none).  test_mutants_exceed_the_fp32_bar shows that these cases and bars tell a broken
kernel from rounding."""
import math
import os
import re

import numpy as np
import pytest
import torch

from onmf_ontf_ndl_b200 import _lib
from oracle import onmf_oracle as O

F32, F64 = torch.float32, torch.float64
ONMF_E_ARG, ONMF_E_UNSUPPORTED = -1, -3
FLOOR32 = 1e-6
MARGIN64, MARGIN32 = 1e-8, 1e-3
SWEEP_KS = [1, 7, 32, 33, 64, 65, 128, 129, 256, 257, 400, 512, "ks", "ks+1"]     # "ks": largest k with the Gram in shared memory
WARP_KS = [25, 64, 100, "ks", "ks+1", 256, 512]                                     # code_columns: every NA class, both Gram forms
TPS_KS = [1, 8, 9, 12, 13, 16, 17, 20, 21, 24, 25, 28, 29, 32]                      # every KP of the thread form
MUTANTS = ("jacobi", "sqrt_it_plus_11", "transposed_G", "no_clamp_from_atom_32", "new_h_in_denominator", "inclusive_q_end")


# --------------------------------------------------------------------------------------------------------- inputs, bars
def problem(k, n, seed, dt=F64):
    """G (k x k): the Gram of 2k + 3 Gaussian rows scaled to unit diagonal on average, plus a skew-symmetric part of the same
    order as the off-diagonal entries; Ct (n x k) in [-0.2, 1), so alpha = 0.3 clamps some atoms; H0 (n x k) in [0, 1).
    Rounded to dt and returned as float64."""
    rng = np.random.default_rng(seed)
    d = 2 * k + 3
    Wg = rng.standard_normal((d, k)) / math.sqrt(d)
    R = rng.standard_normal((k, k)) * (0.5 / math.sqrt(k))
    G = Wg.T @ Wg + (R - R.T)
    Ct = rng.random((n, k)) * 1.2 - 0.2
    H0 = rng.random((n, k))
    return tuple(rounded(x, dt) for x in (G, Ct, H0))


def rounded(x, dt):
    return np.asarray(x, dtype=np.float32 if dt == F32 else np.float64).astype(np.float64)


def sample_err(got, ref):
    """per sample ||got - ref|| / ||ref|| (a zero reference needs an exact zero)"""
    num = np.linalg.norm(got - ref, axis=1)
    den = np.linalg.norm(ref, axis=1)
    return np.where(num == 0, 0.0, num / np.maximum(den, 1e-300))


def bar(dt, emulated, ref, fp64_bar):
    if dt == F64:
        return fp64_bar
    return max(16 * float(sample_err(emulated, ref).max(initial=0.0)), FLOOR32)


# ------------------------------------------------------------------------- numpy variants of the restatement (emulation)
def sweep_np(G, Ct, H, alpha, it, q0, q1, dtype=np.float64, mutant=None):
    """the sweep in `dtype` with the kernels' operation order per coordinate (reciprocal step, then one multiply), or with
    one kernel bug (`mutant`)"""
    t = dtype
    G, Ct, H = np.asarray(G, t), np.asarray(Ct, t), np.array(H, t, copy=True)
    k = G.shape[0]
    Gr = np.ascontiguousarray(G.T) if mutant == "transposed_G" else G
    scale = t(math.sqrt(it + (11.0 if mutant == "sqrt_it_plus_11" else 10.0)))
    src = H.copy() if mutant == "jacobi" else H                          # Jacobi: every gradient from the old h
    end = min(q1 + 1, k) if mutant == "inclusive_q_end" else q1
    for q in range(q0, end):
        grad = src @ Gr[q] - Ct[:, q] + t(alpha)
        v = H[:, q] - (t(1) / (scale * (Gr[q, q] + t(1)))) * grad
        H[:, q] = v if (mutant == "no_clamp_from_atom_32" and q >= 32) else np.maximum(v, t(0))
    return H


def columns_np(G, Ct, H, alpha, sub_iter, stopping_diff, dtype=np.float64, mutant=None):
    t = dtype
    H = np.array(H, t, copy=True)
    dist = np.ones(H.shape[0], t)
    for it in range(sub_iter):
        act = np.nonzero(dist > t(stopping_diff))[0]
        if act.size == 0:
            break
        old = H[act]
        h = sweep_np(G, np.asarray(Ct)[act], old, alpha, it, 0, G.shape[0], t, mutant)
        den = h if mutant == "new_h_in_denominator" else old
        with np.errstate(divide="ignore", invalid="ignore"):
            dist[act] = np.sqrt(((h - old) ** 2).sum(1)) / np.sqrt((den ** 2).sum(1))
        H[act] = h
    return H


def pick_stopping_diff(trail, margin):
    """stopping_diff at the middle (in log) of the widest gap between the values of the oracle's dist trails (trail: from a
    run with stopping_diff = 0, whose prefix is every other run's trail) between their 10th and 90th percentiles, so that the columns stop
    after different numbers of sweeps.  Returns it and the mask of the columns whose trail comes within `margin` of it
    (their sweep counts may differ by rounding)."""
    v = trail[np.isfinite(trail) & (trail > 0)]
    lo, hi = np.quantile(v, [0.1, 0.9])
    v = np.log(np.unique(np.concatenate([[lo, hi], v[(v > lo) & (v < hi)]])))
    i = int(np.argmax(np.diff(v)))
    sd = float(np.exp(0.5 * (v[i] + v[i + 1])))
    with np.errstate(invalid="ignore"):
        near = (np.abs(trail / sd - 1.0) < margin).any(axis=1)
    return sd, near


def matrix_coder(G, Ct, Ht, alpha, sub_iter, stopping_diff, r=None):
    """update_code_within_radius in the G / C form for a whole matrix (sample-major Ht): the matrix stopping test (spectral
    norms) and the radius projection, which acts once, after row 0 of the first sweep (the reference's `H0 = H1`
    aliasing).  Returns (Ht, dist trail)."""
    H = np.array(Ht, dtype=np.float64, copy=True)
    k = G.shape[0]
    i, dist, trail = 0, 1.0, []
    while i < sub_iter and dist > stopping_diff:
        old = H.copy()
        if r is not None and i == 0:
            H = O.pgd_sweep_gc(G, Ct, H, alpha, 0, 0, 1)
            delta = H[:, 0] - old[:, 0]
            H[:, 0] = old[:, 0] + (r / max(r, np.linalg.norm(delta))) * delta
            H = O.pgd_sweep_gc(G, Ct, H, alpha, 0, 1, k)
        else:
            H = O.pgd_sweep_gc(G, Ct, H, alpha, i)
        dist = np.linalg.norm(H - old, 2) / np.linalg.norm(old, 2)
        trail.append(dist)
        i += 1
    return H, np.array(trail)


# ---------------------------------------------------------------------------------------------- CPU: the restatement
def test_sweep_gc_equals_update_code_within_radius_for_one_column():
    """with G = W^T W and Ct = X^T W, sub_iter sweeps of pgd_sweep_gc are update_code_within_radius(r = None) on a single
    column, and pgd_columns_gc is the same run with its stopping test (dist = vector 2-norm ratio)"""
    rng = np.random.default_rng(1)
    d, k = 30, 12
    W = rng.random((d, k))
    x = rng.random((d, 1))
    h0 = rng.random((k, 1))
    G, Ct = W.T @ W, (x.T @ W)
    for alpha, sub_iter, sd in ((0.3, 6, 0.0), (0.0, 10, 0.05), (2.0, 25, 0.01)):
        ref = O.update_code_within_radius(x, W, h0.copy(), None, alpha, sub_iter, sd)
        H, sweeps, trail = O.pgd_columns_gc(G, Ct, h0.T, alpha, sub_iter, sd)
        assert np.allclose(H.T, ref, rtol=1e-13, atol=1e-15), (alpha, sub_iter, sd)
        Hs = h0.T.copy()
        for it in range(sweeps[0]):
            Hs = O.pgd_sweep_gc(G, Ct, Hs, alpha, it)
        assert np.array_equal(Hs, H)
        assert sweeps[0] == np.isfinite(trail[0]).sum() and (sd == 0 or sweeps[0] == sub_iter or trail[0, sweeps[0] - 1] <= sd)


def test_matrix_form_equals_update_code_within_radius():
    """the matrix coder built from pgd_sweep_gc (the GPU tests' reference at large k) is update_code_within_radius on a
    whole matrix: spectral-norm stopping test, radius projection with the H0 = H1 aliasing"""
    rng = np.random.default_rng(2)
    d, k, n = 40, 20, 30
    W = rng.random((d, k)); W /= np.linalg.norm(W, axis=0)
    X = rng.random((d, n))
    H0 = rng.random((k, n))
    for r in (None, 0.5, 1e-3):
        for alpha, sub_iter, sd in ((0.3, 10, 0.01), (0.0, 4, 0.0)):
            ref = O.update_code_within_radius(X, W, H0.copy(), r, alpha, sub_iter, sd)
            H, trail = matrix_coder(W.T @ W, X.T @ W, H0.T, alpha, sub_iter, sd, r)
            assert np.allclose(H.T, ref, rtol=1e-12, atol=1e-14), (r, alpha, sub_iter, sd)
            assert len(trail) == sub_iter or trail[-1] <= sd


def test_columns_gc_special_columns():
    """inf on the first test of a zero start keeps a column going; 0 / 0 (a column clamped to zero twice) stops it; a
    fixed point stops after one sweep with dist 0"""
    k, alpha = 6, 0.25
    G, Ct, H0 = special_columns(*problem(k, 5, 3), alpha)
    H, sweeps, trail = O.pgd_columns_gc(G, Ct, H0, alpha, 10, 0.01)
    assert trail[0, 0] == np.inf and sweeps[0] >= 2
    assert sweeps[1] == 1 and trail[1, 0] == 0.0 and np.array_equal(H[1], H0[1])
    assert sweeps[2] == 1 and np.isnan(trail[2, 0]) and not H[2].any()
    assert sweeps[3] == 2 and trail[3, 0] == 1.0 and np.isnan(trail[3, 1]) and not H[3].any()


def special_columns(G, Ct, H0, alpha):
    """rows 0-3 of (Ct, H0) become: a zero start; the fixed point h = 2 e_0 (G_00 = 1.5 and c_0 = 3 + alpha, exact in both
    dtypes, every other atom clamps); a zero start whose atoms all clamp (0 / 0 on the first test); a start that clamps to
    zero in the first sweep (dist 1), then 0 / 0"""
    G, Ct, H0 = G.copy(), Ct.copy(), H0.copy()
    G[0, 0] = 1.5
    H0[0] = 0.0
    H0[1] = 0.0; H0[1, 0] = 2.0
    Ct[1] = 2.0 * G[:, 0] + alpha - 1.0; Ct[1, 0] = 3.0 + alpha
    H0[2] = 0.0; Ct[2] = alpha - 1.0
    Ct[3] = -50.0
    return G, Ct, H0


MUTANT_CASES = [("sweep", 65, 37, 7, 0.3, (0, 65)), ("sweep", 65, 37, 0, 0.3, (21, 43)), ("sweep", 257, 37, 7, 0.3, (85, 171)),
                ("columns", 64, 37, 10, 0.3, None), ("columns", 25, 200, 10, 0.3, None)]


def test_mutants_exceed_the_fp32_bar():
    """numpy variants of the restatement with one kernel bug each land >= 10x above the fp32 bar on at least one of the
    cases the GPU tests run"""
    sep = {m: 0.0 for m in MUTANTS}
    for kind, k, n, it, alpha, rows in MUTANT_CASES:
        G, Ct, H0 = problem(k, n, 1000 + k, F32)
        if kind == "sweep":
            ref = O.pgd_sweep_gc(G, Ct, H0, alpha, it, *rows)
            b = bar(F32, sweep_np(G, Ct, H0, alpha, it, *rows, np.float32), ref, 0)
            for m in MUTANTS:
                if m != "new_h_in_denominator":
                    sep[m] = max(sep[m], float(sample_err(sweep_np(G, Ct, H0, alpha, it, *rows, mutant=m), ref).max()) / b)
        else:
            _, _, trail = O.pgd_columns_gc(G, Ct, H0, alpha, it, 0.0)
            sd, near = pick_stopping_diff(trail, MARGIN32)
            ref = O.pgd_columns_gc(G, Ct, H0, alpha, it, sd)[0][~near]
            b = bar(F32, columns_np(G, Ct, H0, alpha, it, sd, np.float32)[~near], ref, 0)
            for m in MUTANTS:
                got = columns_np(G, Ct, H0, alpha, it, sd, mutant=m)[~near]
                sep[m] = max(sep[m], float(sample_err(got, ref).max()) / b)
    for m in MUTANTS:
        assert sep[m] >= 10, (m, sep)


# -------------------------------------------------------------------------------------- CPU: the spectral norm's bound
GEMM_SIMT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "onmf_ontf_ndl_b200", "csrc",
                         "gemm_simt.cu")
CLUSTER_CS = np.linspace(0.2, 3.0, 15)


def kernel_squarings():
    with open(GEMM_SIMT) as f:
        return int(re.search(r"constexpr int LMAX_SQUARINGS = (\d+);", f.read()).group(1))


def lambda_max_restated(G, squarings):
    """lambda_max_kernel in numpy: B = G / tr G, `squarings` times B <- B^2 / tr B^2, then sqrt of the Rayleigh quotient
    of G at the column of B with the largest diagonal entry"""
    B = G / np.trace(G)
    for _ in range(squarings):
        B = B @ B
        B /= np.trace(B)
    x = B[:, int(np.argmax(np.diag(B)))]
    return math.sqrt(x @ G @ x / (x @ x))


def clustered(k, c, seed=0):
    """M (k x k) with sigma_max(M) = 1: M^T M has the flat top eigenvector 1 / sqrt(k) and k - 1 eigenvalues at 1 - x,
    x = c ln k / 2^17, where the squarings leave the largest share of the near-top eigenspace"""
    rng = np.random.default_rng(seed)
    Q, _ = np.linalg.qr(np.column_stack([np.ones(k), rng.standard_normal((k, k - 1))]))
    x = c * math.log(k) / 2.0 ** 17
    ev = np.array([1.0] + [1.0 - x] * (k - 1))
    return np.sqrt(ev)[:, None] * Q.T


def test_restated_lambda_max_meets_the_bound_at_the_kernels_squaring_count():
    """at the kernel's squaring count the restatement's sigma_max is within 1e-5 (relative) on the clustered spectra at
    k = 256 and 512; with one squaring fewer it is not (the count is the least that keeps the bound)"""
    sq = kernel_squarings()
    worst = {}
    for k in (256, 512):
        Ms = [clustered(k, c) for c in CLUSTER_CS]
        Gs = [M.T @ M for M in Ms]
        worst[k] = max(abs(lambda_max_restated(G, sq) - 1.0) for G in Gs)
        assert worst[k] < 1e-5, (k, sq, worst[k])
    assert max(abs(lambda_max_restated(M.T @ M, sq - 1) - 1.0) for M in (clustered(512, c) for c in CLUSTER_CS)) > 1e-5


# ------------------------------------------------------------------------------------------------------------------ GPU
def _dev():
    return torch.device("cuda", 0)


def _limits():
    p = torch.cuda.get_device_properties(0)
    return p.multi_processor_count, p.shared_memory_per_block_optin


def k_shared(dt):
    """the largest k whose Gram fits the opt-in shared memory: the warp kernels' shared-memory form up to it"""
    return math.isqrt(_limits()[1] // (4 if dt == F32 else 8))


def resolve_k(k, dt):
    return k_shared(dt) + (k == "ks+1") if isinstance(k, str) else k


def tt(x, dt):
    return torch.from_numpy(np.ascontiguousarray(x)).to(_dev(), dt)


def host(t):
    return t.cpu().numpy().astype(np.float64)


def dev_sweep(G, Ct, H0, alpha, it, dt, rows=None):
    Ht = tt(H0, dt)
    if rows is None:
        _lib.pgd_sweep(tt(G, dt), tt(Ct, dt), alpha, it, Ht)
    else:
        _lib.pgd_sweep_rows(tt(G, dt), tt(Ct, dt), alpha, it, Ht, *rows)
    return host(Ht)


def dev_columns(G, Ct, H0, alpha, sub_iter, sd, dt):
    Ht = tt(H0, dt)
    _lib.pgd_code_columns(tt(G, dt), tt(Ct, dt), alpha, sub_iter, sd, Ht)
    return host(Ht)


def check_sweep(dt, got, G, Ct, H0, alpha, it, rows, what):
    q0, q1 = rows if rows is not None else (0, G.shape[0])
    ref = O.pgd_sweep_gc(G, Ct, H0, alpha, it, q0, q1)
    b = bar(dt, sweep_np(G, Ct, H0, alpha, it, q0, q1, np.float32) if dt == F32 else None, ref, 1e-12)
    err = float(sample_err(got, ref).max())
    assert err <= b, (what, err, b)
    return err


def check_columns(dt, G, Ct, H0, alpha, sub_iter, what, sd=None):
    """one code_columns run against the oracle; stopping_diff from the oracle's trails unless given"""
    near = np.zeros(H0.shape[0], dtype=bool)
    if sd is None:
        _, _, trail = O.pgd_columns_gc(G, Ct, H0, alpha, sub_iter, 0.0)
        sd, near = pick_stopping_diff(trail, MARGIN64 if dt == F64 else MARGIN32)
        assert near.mean() <= (0 if dt == F64 else 0.01), (what, sd, int(near.sum()))
    got = dev_columns(G, Ct, H0, alpha, sub_iter, sd, dt)
    ref, sweeps, _ = O.pgd_columns_gc(G, Ct, H0, alpha, sub_iter, sd)
    ok = ~near
    b = bar(dt, columns_np(G, Ct, H0, alpha, sub_iter, sd, np.float32)[ok] if dt == F32 else None, ref[ok], 1e-10)
    err = float(sample_err(got[ok], ref[ok]).max())
    assert err <= b, (what, sd, err, b)
    assert np.isfinite(got).all() and (got >= 0).all(), what
    return got, ref, sweeps


@pytest.mark.gpu
@pytest.mark.parametrize("kk", SWEEP_KS, ids=str)
@pytest.mark.parametrize("dt", [F32, F64], ids=["f32", "f64"])
def test_sweep_matches_restatement(dt, kk):
    """onmf_pgd_sweep, one sweep: n = 1, 37 and 4 x SMs x 8 warps + 123 (the grid-stride loop), it in {0, 7, 1000},
    alpha in {0, 0.3, 1e3} (1e3 clamps every atom)"""
    sms, _ = _limits()
    k = resolve_k(kk, dt)
    big = 4 * sms * 8 + 123
    runs = [(1, 0, 0.3)] + [(37, it, a) for it in (0, 7, 1000) for a in (0.0, 0.3, 1e3)] + [(big, 7, 0.3), (big, 0, 1e3)]
    worst = 0.0
    for i, (n, it, alpha) in enumerate(runs):
        G, Ct, H0 = problem(k, n, 10 * k + i, dt)
        got = dev_sweep(G, Ct, H0, alpha, it, dt)
        worst = max(worst, check_sweep(dt, got, G, Ct, H0, alpha, it, None, (k, n, it, alpha)))
        if alpha == 1e3:
            assert not got.any(), (k, n, it)
    gsm = k * k * (4 if dt == F32 else 8) <= _limits()[1]
    print("pgd_sweep %s k=%d (%s Gram): worst per-sample error %.2e" % (dt, k, "shared" if gsm else "global", worst))


@pytest.mark.gpu
@pytest.mark.parametrize("k", [7, 33, 129, 300])
@pytest.mark.parametrize("dt", [F32, F64], ids=["f32", "f64"])
def test_ten_chained_sweeps(dt, k):
    """sweeps it = 0..9 on the device, each against one oracle sweep of the device's previous state, and the tenth against
    ten oracle sweeps from H0"""
    G, Ct, H0 = problem(k, 37, 500 + k, dt)
    Gd, Cd, Ht = tt(G, dt), tt(Ct, dt), tt(H0, dt)
    ref, emu = H0, H0.astype(np.float32)
    for it in range(10):
        prev = host(Ht)
        _lib.pgd_sweep(Gd, Cd, 0.3, it, Ht)
        check_sweep(dt, host(Ht), G, Ct, prev, 0.3, it, None, (k, it))
        ref = O.pgd_sweep_gc(G, Ct, ref, 0.3, it)
        emu = sweep_np(G, Ct, emu, 0.3, it, 0, k, np.float32)
    err = float(sample_err(host(Ht), ref).max())
    assert err <= bar(dt, emu, ref, 1e-10), (k, err)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [7, 64, 100, 129, 400])
@pytest.mark.parametrize("dt", [F32, F64], ids=["f32", "f64"])
def test_sweep_rows(dt, k):
    """onmf_pgd_sweep_rows over (0, 1), (1, k), (k/3, 2k/3), (k - 1, k); an empty range (q, q) leaves Ht bit-unchanged"""
    sms, _ = _limits()
    for n in ((37, 4 * sms * 8 + 123) if k == 64 else (37,)):
        G, Ct, H0 = problem(k, n, 700 + k, dt)
        for rows in ((0, 1), (1, k), (k // 3, 2 * k // 3), (k - 1, k)):
            for it in (0, 7):
                got = dev_sweep(G, Ct, H0, 0.3, it, dt, rows)
                check_sweep(dt, got, G, Ct, H0, 0.3, it, rows, (k, n, rows, it))
                untouched = np.r_[0:rows[0], rows[1]:k]
                assert np.array_equal(got[:, untouched], H0[:, untouched]), (k, rows)
        for q in (0, k // 2, k):
            assert np.array_equal(dev_sweep(G, Ct, H0, 0.3, 3, dt, (q, q)), H0), (k, q)


@pytest.mark.gpu
@pytest.mark.parametrize("kk", WARP_KS, ids=str)
@pytest.mark.parametrize("dt", [F32, F64], ids=["f32", "f64"])
def test_code_columns_warp_form(dt, kk):
    """onmf_pgd_code_columns, one warp per sample, at every NA class and both Gram forms: stopping_diff from the trails,
    and stopping_diff = 0 (every column takes sub_iter sweeps); at k = 64 also past the grid (grid-stride loop)"""
    sms, optin = _limits()
    k = resolve_k(kk, dt)
    ns = (200,) if k <= 64 else (37,)
    if k == 64:
        ns += (4 * sms * 8 + 123,)
    for n in ns:
        assert not (k <= 32 and n >= 16 * sms)
        G, Ct, H0 = problem(k, n, 900 + k, dt)
        _, _, sweeps = check_columns(dt, G, Ct, H0, 0.3, 10, (k, n))
        assert sweeps.min() < 10 or n < 50, (k, n, np.bincount(sweeps))
        _, _, sweeps = check_columns(dt, G, Ct, H0, 0.3, 3, (k, n, 0.0), sd=0.0)
        assert (sweeps == 3).all()
    print("pgd_code_columns warp form %s k=%d (%s Gram)" % (dt, k, "shared" if k * k * (4 if dt == F32 else 8) <= optin else "global"))


@pytest.mark.gpu
@pytest.mark.parametrize("k", TPS_KS)
@pytest.mark.parametrize("dt", [F32, F64], ids=["f32", "f64"])
def test_code_columns_thread_form(dt, k):
    """one thread per sample (k <= 32 and n = 16 x SMs) at every KP; at k = 25 and 32 also n = 16 x SMs - 1 (warp form)"""
    sms, _ = _limits()
    for n in ((16 * sms - 1, 16 * sms) if k in (25, 32) else (16 * sms,)):
        G, Ct, H0 = problem(k, n, 1300 + k, dt)
        check_columns(dt, G, Ct, H0, 0.3, 10, (k, n))


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [F32, F64], ids=["f32", "f64"])
def test_code_columns_edges(dt):
    """sub_iter = 0 and stopping_diff >= 1 run no sweep (Ht bit-unchanged); the special columns (zero start: inf on the
    first test; a fixed point: dist 0; columns clamped to zero: 0 / 0) stop where the oracle stops, in both forms"""
    sms, _ = _limits()
    for k, n in ((25, 37), (25, 16 * sms), (64, 37), (300, 37)):
        G, Ct, H0 = problem(k, n, 1700 + k + n, dt)
        for sub_iter, sd in ((0, 0.01), (0, 0.0), (10, 1.0), (10, 5.0)):
            assert np.array_equal(dev_columns(G, Ct, H0, 0.3, sub_iter, sd, dt), H0), (k, n, sub_iter, sd)
        G, Ct, H0 = (rounded(x, dt) for x in special_columns(G, Ct, H0, 0.25))
        got, ref, sweeps = check_columns(dt, G, Ct, H0, 0.25, 10, (k, n, "special"))
        assert sweeps[0] >= 2 and sweeps[1] == 1 and sweeps[2] == 1 and sweeps[3] == 2, sweeps[:4]
        assert np.array_equal(got[1], H0[1]) and not got[2].any() and not got[3].any() and got[0].any()


@pytest.mark.gpu
def test_refusals_leave_ht_unchanged():
    """bad arguments -> ONMF_E_ARG, k > 512 -> ONMF_E_UNSUPPORTED; Ht is not touched"""
    lib = _lib.load()
    st = _lib._stream()
    n, k = 40, 8
    G, Ct, H0 = problem(k, n, 3)
    Gd, Cd, Ht = tt(G, F64), tt(Ct, F64), tt(H0, F64)
    p = _lib._ptr
    D = _lib.F64
    calls = {
        "rows q_end > k": lambda: lib.onmf_pgd_sweep_rows(D, p(Gd), p(Cd), n, k, 0.3, 0, p(Ht), 0, k + 1, st),
        "rows q_begin > q_end": lambda: lib.onmf_pgd_sweep_rows(D, p(Gd), p(Cd), n, k, 0.3, 0, p(Ht), 5, 4, st),
        "rows q_begin < 0": lambda: lib.onmf_pgd_sweep_rows(D, p(Gd), p(Cd), n, k, 0.3, 0, p(Ht), -1, 4, st),
        "rows it < 0": lambda: lib.onmf_pgd_sweep_rows(D, p(Gd), p(Cd), n, k, 0.3, -1, p(Ht), 0, k, st),
        "rows k = 0": lambda: lib.onmf_pgd_sweep_rows(D, p(Gd), p(Cd), n, 0, 0.3, 0, p(Ht), 0, 0, st),
        "rows n < 0": lambda: lib.onmf_pgd_sweep_rows(D, p(Gd), p(Cd), -1, k, 0.3, 0, p(Ht), 0, k, st),
        "rows bad dtype": lambda: lib.onmf_pgd_sweep_rows(7, p(Gd), p(Cd), n, k, 0.3, 0, p(Ht), 0, k, st),
        "rows null G": lambda: lib.onmf_pgd_sweep_rows(D, None, p(Cd), n, k, 0.3, 0, p(Ht), 0, k, st),
        "rows null Ct": lambda: lib.onmf_pgd_sweep_rows(D, p(Gd), None, n, k, 0.3, 0, p(Ht), 0, k, st),
        "rows null Ht": lambda: lib.onmf_pgd_sweep_rows(D, p(Gd), p(Cd), n, k, 0.3, 0, None, 0, k, st),
        "sweep it < 0": lambda: lib.onmf_pgd_sweep(D, p(Gd), p(Cd), n, k, 0.3, -1, p(Ht), st),
        "sweep k = 0": lambda: lib.onmf_pgd_sweep(D, p(Gd), p(Cd), n, 0, 0.3, 0, p(Ht), st),
        "sweep k < 0": lambda: lib.onmf_pgd_sweep(D, p(Gd), p(Cd), n, -3, 0.3, 0, p(Ht), st),
        "sweep bad dtype": lambda: lib.onmf_pgd_sweep(2, p(Gd), p(Cd), n, k, 0.3, 0, p(Ht), st),
        "sweep null G": lambda: lib.onmf_pgd_sweep(D, None, p(Cd), n, k, 0.3, 0, p(Ht), st),
        "sweep null Ct": lambda: lib.onmf_pgd_sweep(D, p(Gd), None, n, k, 0.3, 0, p(Ht), st),
        "sweep null Ht": lambda: lib.onmf_pgd_sweep(D, p(Gd), p(Cd), n, k, 0.3, 0, None, st),
        "columns sub_iter < 0": lambda: lib.onmf_pgd_code_columns(D, p(Gd), p(Cd), n, k, 0.3, -1, 0.01, p(Ht), st),
        "columns k = 0": lambda: lib.onmf_pgd_code_columns(D, p(Gd), p(Cd), n, 0, 0.3, 10, 0.01, p(Ht), st),
        "columns n < 0": lambda: lib.onmf_pgd_code_columns(D, p(Gd), p(Cd), -1, k, 0.3, 10, 0.01, p(Ht), st),
        "columns bad dtype": lambda: lib.onmf_pgd_code_columns(7, p(Gd), p(Cd), n, k, 0.3, 10, 0.01, p(Ht), st),
        "columns bad dtype, thread form": lambda: lib.onmf_pgd_code_columns(7, p(Gd), p(Cd), 1 << 20, k, 0.3, 10, 0.01, p(Ht), st),
        "columns null G": lambda: lib.onmf_pgd_code_columns(D, None, p(Cd), n, k, 0.3, 10, 0.01, p(Ht), st),
        "columns null Ct": lambda: lib.onmf_pgd_code_columns(D, p(Gd), None, n, k, 0.3, 10, 0.01, p(Ht), st),
        "columns null Ht": lambda: lib.onmf_pgd_code_columns(D, p(Gd), p(Cd), n, k, 0.3, 10, 0.01, None, st),
    }
    before = Ht.clone()
    for name, call in calls.items():
        rc = call()
        torch.cuda.synchronize()
        assert rc == ONMF_E_ARG, (name, rc)
        assert torch.equal(Ht, before), name
    kb = 513
    Gb, Cb, Hb = problem(kb, n, 4)
    for dt, D_ in ((F32, _lib.F32), (F64, _lib.F64)):
        Gd, Cd, Ht = tt(Gb, dt), tt(Cb, dt), tt(Hb, dt)
        before = Ht.clone()
        for name, call in {
            "sweep": lambda: lib.onmf_pgd_sweep(D_, p(Gd), p(Cd), n, kb, 0.3, 0, p(Ht), st),
            "rows": lambda: lib.onmf_pgd_sweep_rows(D_, p(Gd), p(Cd), n, kb, 0.3, 0, p(Ht), 0, kb, st),
            "columns": lambda: lib.onmf_pgd_code_columns(D_, p(Gd), p(Cd), n, kb, 0.3, 10, 0.01, p(Ht), st),
        }.items():
            rc = call()
            torch.cuda.synchronize()
            assert rc == ONMF_E_UNSUPPORTED and torch.equal(Ht, before), (name, dt, rc)


# ---------------------------------------------------------------------------------------------- GPU: the class level
def dictionary(d, k, seed):
    rng = np.random.default_rng(seed)
    W = rng.random((d, k))
    return W / np.linalg.norm(W, axis=0)


def stopping_diff_with_margin(trail, margin=1e-3):
    """a stopping_diff between two values of the matrix trail near its median, at the widest such gap, with no value within
    `margin` (relative) of it: the run stops before sub_iter, and the device's spectral norms (exact to 1e-5) take the
    same decisions"""
    v = np.log(np.unique(trail[1:]))
    mid = range(len(v) // 4, max(len(v) * 3 // 4, len(v) // 4 + 1))
    i = max((j for j in mid if j + 1 < len(v)), key=lambda j: v[j + 1] - v[j])
    sd = float(np.exp(0.5 * (v[i] + v[i + 1])))
    assert (np.abs(trail / sd - 1.0) > margin).all(), (trail, sd)
    return sd


@pytest.mark.gpu
@pytest.mark.parametrize("k", [50, 130, 300])
def test_update_code_within_radius_class_level(k):
    """update_code_within_radius (fp64) beyond k = 32, 400 columns, r = None, 0.5 and 1e-3 (the radius projection after
    row 0 of the first sweep), against the matrix coder of the restatement"""
    from onmf_ontf_ndl_b200 import update_code_within_radius
    rng = np.random.default_rng(k)
    d, n = 2 * k, 400
    W = dictionary(d, k, k)
    X = rng.random((d, n))
    H0 = rng.random((k, n))
    G, Ct = W.T @ W, X.T @ W
    for r in (None, 0.5, 1e-3):
        _, trail = matrix_coder(G, Ct, H0.T, 0.3, 10, 0.0, r)
        sd = stopping_diff_with_margin(trail)
        ref, trail = matrix_coder(G, Ct, H0.T, 0.3, 10, sd, r)
        assert len(trail) < 10
        got = update_code_within_radius(X, W, H0=H0, r=r, alpha=0.3, sub_iter=10, stopping_diff=sd, precision="fp64")
        err = float(sample_err(got.T, ref).max())
        assert err <= 1e-10, (k, r, sd, len(trail), err)


@pytest.mark.gpu
def test_online_nmf_pgd_sparse_code():
    """Online_NMF(coder="pgd").sparse_code at k = 64: H0 replayed from the global RNG, sub_iter 10, stopping_diff 0.01"""
    from onmf_ontf_ndl_b200 import Online_NMF
    k, d, n = 64, 100, 300
    rng = np.random.default_rng(64)
    W = dictionary(d, k, 65)
    X = rng.random((d, n))
    m = Online_NMF(X, n_components=k, iterations=2, batch_size=20, alpha=0.5, coder="pgd", precision="fp64")
    np.random.seed(64)
    got = m.sparse_code(X, W)
    np.random.seed(64)
    H0 = np.random.rand(k, n)
    ref, trail = matrix_coder(W.T @ W, X.T @ W, H0.T, 0.5, 10, 0.01)
    assert (np.abs(trail / 0.01 - 1.0) > 1e-3).all(), trail
    assert float(sample_err(got.T, ref).max()) <= 1e-10


@pytest.mark.gpu
@pytest.mark.parametrize("k", [49, 100])
@pytest.mark.parametrize("shape,p", [((26, 25), 8), ((20, 19, 3), 6)], ids=["grey", "colour"])
def test_reconstruct_image_pgd(shape, p, k):
    """reconstruct_image(coder="pgd") at k = 49 and 100 (the warp form, NA = 2 and 4) against the oracle's per-patch loop
    (update_code_within_radius on each patch, running overlap mean)"""
    from onmf_ontf_ndl_b200 import reconstruct_image
    rng = np.random.default_rng(k + len(shape))
    img = rng.random(shape)
    C = 1 if len(shape) == 2 else shape[2]
    W = dictionary(p * p * C, k, k)
    ys, xs = range(0, shape[0] - p), range(0, shape[1] - p)
    n = len(ys) * len(xs)
    H0 = rng.random((k, n))
    A3 = img.reshape(shape[0], shape[1], C)
    Xp = np.stack([A3[y:y + p, x:x + p, :].reshape(-1) for y in ys for x in xs], 1)
    _, _, trail = O.pgd_columns_gc(W.T @ W, Xp.T @ W, H0.T, 0.5, 10, 0.0)
    sd, near = pick_stopping_diff(trail, MARGIN64)
    assert not near.any()
    rec, cnt, code = reconstruct_image(img, W, p, 1, alpha=0.5, sub_iter=10, stopping_diff=sd, H0=H0, precision="fp64",
                                       return_code=True)
    ref_rec, ref_cnt, ref_code = O.reconstruct_image_loop(img, W, p, 1, 0.5, 10, sd, H0)
    assert np.array_equal(cnt, ref_cnt)
    assert float(sample_err(code.T, ref_code.T).max()) <= 1e-10
    assert np.abs(rec - ref_rec).max() <= 1e-10 * np.abs(ref_rec).max()


# ------------------------------------------------------------------------------------- GPU: the spectral norm's bound
@pytest.mark.gpu
@pytest.mark.parametrize("k", [256, 512])
def test_spectral_norm_clustered_spectrum(k):
    """onmf_spectral_norm within 1e-5 (the header's bound) on the clustered spectra the squarings resolve last: a flat
    top eigenvector and k - 1 eigenvalues at 1 - c ln k / 2^17, c in [0.2, 3]; fp64 and fp32 input"""
    worst = 0.0
    for c in CLUSTER_CS:
        M = clustered(k, c)
        for dt in (F64, F32):
            Mr = rounded(M, dt)
            ref = 1.0 if dt == F64 else float(np.linalg.norm(Mr, 2))
            out = torch.full((1,), float("nan"), dtype=torch.float64, device=_dev())
            ws = torch.empty(_lib.spectral_norm_workspace(k, k), dtype=torch.uint8, device=_dev())
            _lib.spectral_norm(tt(Mr, dt), out, ws)
            err = abs(float(out[0]) - ref) / ref
            worst = max(worst, err)
            assert err < 1e-5, (k, c, dt, err)
    print("spectral norm, clustered spectrum k=%d: worst relative error %.2e" % (k, worst))
