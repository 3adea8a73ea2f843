"""The batched positive LARS coder (csrc/lars.cu, csrc/lars_fast.cuh) in every dispatch form, against the C restatement
oracle.c_oracle.lars_columns (oracle_lars_positive in oracle/lars_oracle.c), column by column.

One call reaches: five k classes (k <= 32 / 64 / 128 / 256 / 512; lane groups of 8 / 16 / 32 lanes); active-set tiers
32 -> 64 -> 128 (k <= 128) or a 64-slot hybrid tier (V columns 40..63 in global scratch) -> 128 -> k with V in global
scratch (k > 128); the fp32 fast tiers (launch_fast: V columns 28..63 in an L2 tail; launch_fast_gsm at 64 < k <= 128;
launch_fast_small at k <= 64 on small minibatches); the Gram in shared memory or through the padded global copy; the fp64
coder, fp32 with the FP64 Gram (onmf_lasso_lars_g64) and fp32 with an fp32 Gram (onmf_lasso_lars_ex); first_tier 0 / 1 /
-1 with the workspace's persistent hint at 0 or 1; the reserved-SM and fast-tier options.

Inputs (CASES): a unit-norm U[0,1) dictionary with d >= k and one atom duplicated (a degenerate pivot), one k > d case per
class and a raw U[0,1) dictionary at k = 256.  Every case mixes random columns, exact nonnegative combinations of m atoms
with m on both sides of each slot boundary of its class (28/29, 32/33, 40/41, 64/65, 128/129; test_case_set_crosses_its_
boundaries checks the claim from the oracle's max_active), and the special columns: all-zero, all-negative, alpha above
every covariance, the duplicated atom itself, and an exact combination of min(k, 200) atoms.  The oracle runs once per
case; every form is compared with that one result.

Bars.  fp64: per column ||h - h_oracle|| / ||h_oracle|| <= max(1e-10, 64 eps64 cond(G_AA) sqrt(knots)) (bar64), G_AA the
Gram block of the oracle's final support; TIE64 = 1e-8 where the oracle's path has a near-tie within that bar (code_bar);
oracle-zero columns exactly zero; the path statistics (columns, flagged, max_active, overflow against the tier that
started, knots / drops) against the oracle's info on every column without a near-tie below NEAR_TIE (stat_exempt).
fp32: against the oracle run on the same fp32 covariances and the FP64 Gram, each column within 16 x its own float32
emulation's error (onmf_oracle.lars_lasso_positive(work_dtype=np.float32)), at least 16 FLOOR32 (bar32); where the
emulation ends on the oracle's support, the kernel does too.  test_mutants_exceed_the_fp64_bar shows that the cases and
bars tell a broken path from rounding.

Branch columns (branch_columns: a degenerate pivot, a nearly dependent join, the duplicated pair in the code) can take the
other branch of the 1e-7 pivot rule by rounding; in fp64 they are held with the pair summed (d >= k).  One is built on
purpose: the dup_atom column, 2 e + 0.5 w_0 with e the duplicated atom.  The fp32 coder, by its exact-tie rule, takes a
zero-length step for the twin, rejects the twin as degenerate at the next knot and stops with the level of w_0: 0 on the
pair where the answer is 2 - alpha.  test_fp32_duplicated_atom_column records that defect (expected to fail), as
test_global_tier_fp64_precision records the fp64 coder's shortfall on 400-knot paths."""
import contextlib
import functools
import math

import numpy as np
import pytest
import torch

from onmf_ontf_ndl_b200 import _lib
from oracle import c_oracle
from oracle import onmf_oracle as O

F32, F64 = torch.float32, torch.float64
ONMF_E_ARG, ONMF_E_UNSUPPORTED, ONMF_E_WORKSPACE = -1, -3, -4
EPS64 = float(np.finfo(np.float64).eps)
EPS32 = float(np.finfo(np.float32).eps)
BAR64 = 1e-10
# codes of a column whose path has a near-tie within its fp64 bar: the two branches of the tie end within 1e-8 (the numpy
# and C restatements, which take different branches on 4 to 12 columns of a case, agree to 1.5e-9 on them)
TIE64 = 1e-8
NEAR_TIE = 1e-10         # path statistics are compared on every column whose join / drop candidates are further apart
FLOOR32 = 1e-6
HINT_OFFSET = 60                        # LarsWs::hint (csrc/lars.cu): bytes 60..63 of the workspace, kept across calls
KS = [1, 2, 31, 32, 33, 64, 65, 72, 73, 128, 129, 256, 257, 512]
MUTANTS = ("tie_high", "no_interp", "no_drop_recompute", "join_after_drop", "alpha_unscaled", "max_iter_plus1", "no_eps_stop")


def tiers(k):
    """slot counts of the class's tiers (csrc/lars.cu lasso_lars_t); the last tier of k > 128 holds every atom"""
    return [32] if k <= 32 else [32, 64] if k <= 64 else [32, 64, 128] if k <= 128 else [64, 128, k]


def boundaries(k):
    """slot boundaries b (b active atoms fit, b + 1 do not) that a column can fall on either side of in this class"""
    if k <= 32:
        return []
    if k <= 128:
        return [b for b in (32, 64) if b < k]
    return [28, 32, 40, 64, 128]        # fast tier's shared part, 32, hybrid split, hybrid tier, 128-slot tier


# ------------------------------------------------------------------------------------------------------------- case set
ALPHA = {1: 0.2, 2: 0.0, 31: 1.0, 32: 0.0, 33: 0.2, 64: 1.0, 65: 0.2, 72: 0.0, 73: 1.0, 128: 0.0, 129: 0.2, 256: 1.0,
         257: 0.0, 512: 0.2}
CASES = ([(k, max(2 * k, 8), ALPHA[k], "unit") for k in KS] +
         [(24, 16, 0.2, "unit"), (60, 52, 0.0, "unit"), (100, 90, 1.0, "unit"), (200, 180, 0.2, "unit"),
          (400, 300, 0.0, "unit"), (256, 512, 1.0, "raw")])


def case_ids():
    return ["k%d_d%d_a%g_%s" % c for c in CASES]


@functools.lru_cache(maxsize=None)
def case(i):
    """(W (d x k), X (n x d), alpha, labels) of CASES[i]; labels[j] names column j.  For k >= 4 the last two atoms are the
    same unit vector e_{d-1}, orthogonal to every other atom; only the dup_atom column has a component along it, so the
    pair's covariance stays exactly 0 on every other path.  (A twin of an active atom rides at the active level: a near-tie
    at every knot, where rounding decides whether it wins an arg-max and is rejected as a degenerate pivot.  Kept to one
    column, that leaves the other columns' paths determined by their inputs.)"""
    k, d, alpha, kind = CASES[i]
    rng = np.random.default_rng(1000 + i)
    W = rng.random((d, k))
    pair = k >= 4
    if pair:
        W[d - 1, :] = 0.0
    if kind == "unit":
        W /= np.linalg.norm(W, axis=0)
    if pair:
        W[:, k - 2:] = 0.0
        W[d - 1, k - 2:] = 1.0
    pool = list(range(k - 2 if pair else k))
    cols, labels = [], []

    def add(x, lab):
        if pair and lab != "dup_atom":
            x[d - 1] = 0.0
        cols.append(x); labels.append(lab)

    for j in range(16):
        add(rng.random(d), "random")
    ms = sorted({m for b in boundaries(k) for m in (b - 2, b, b + 1, b + 3)} | {1, 2, 5, 12})
    for m in ms:
        if 1 <= m <= min(len(pool), d - 1, 200):
            for rep in range(2):
                h = np.zeros(k)
                h[rng.choice(pool, m, replace=False)] = rng.random(m) + 0.5
                add(W @ h, "comb%d" % m)
    # a combination plus noise has no structural tie at its last knot (an exact fit has one: an atom's coefficient reaches 0
    # together with the full step), so these keep columns past each boundary in the path-statistic checks
    for bb in boundaries(k):
        m = bb + 6
        if m <= min(len(pool), d - 1, 200):
            for rep in range(2):
                h = np.zeros(k)
                h[rng.choice(pool, m, replace=False)] = rng.random(m) + 0.5
                x = W @ h
                add(x + 1e-2 * np.linalg.norm(x) / math.sqrt(d) * rng.standard_normal(d), "noisy%d" % m)
    add(np.zeros(d), "zero")
    add(-rng.random(d), "negative")
    x = rng.random(d)
    x[d - 1] = 0.0
    add(x * (0.5 * alpha / max(float((W.T @ x).max()), 1e-300)) if alpha > 0 else -x, "below_alpha")
    # the pair ties exactly at the first knot (the lowest index joins); then the twin rides with atom 0
    add(2 * W[:, k - 2] + 0.5 * W[:, 0] if pair else 2 * W[:, 0], "dup_atom")
    m = min(len(pool), d - 1, 200)
    h = np.zeros(k)
    h[rng.choice(pool, m, replace=False)] = rng.random(m) + 0.5
    add(W @ h, "comb_all")
    return W, np.stack(cols), alpha, labels


def gram(W):
    G = W.T @ W
    return (G + G.T) / 2


@functools.lru_cache(maxsize=None)
def reference(i, dtype="f64", max_iter=1000):
    """the oracle on the case's covariances rounded to dtype, FP64 Gram; H (n x k), info, per-column fp64 bar"""
    W, X, alpha, _ = case(i)
    d, k = W.shape
    G = gram(W)
    Ct = X @ W
    if k >= 4:
        assert (G[:, k - 1] == G[:, k - 2]).all() and (Ct[:, k - 1] == Ct[:, k - 2]).all()
    if dtype == "f32":
        Ct = Ct.astype(np.float32).astype(np.float64)
    H, info = c_oracle.lars_columns(G, Ct, alpha, d, max_iter)
    return G, Ct, H, info, bar64(G, H, info)


def bar64(G, H, info):
    """per column max(1e-10, 64 eps64 cond(G_AA) sqrt(knots)): G_AA the Gram block of the oracle's final support, the
    rounding of each knot's update amplified by cond(G_AA) and accumulated over the path"""
    bar = np.full(H.shape[0], BAR64)
    for j in range(H.shape[0]):
        S = np.nonzero(H[j])[0]
        if S.size > 1:
            bar[j] = max(BAR64, 64 * EPS64 * np.linalg.cond(G[np.ix_(S, S)]) * math.sqrt(max(int(info["n_iter"][j]), 1)))
    return bar


@functools.lru_cache(maxsize=None)
def emulation(i, gram32):
    """every column of case i emulated in float32 (the kernel's working precision) for the fp32 form with the FP64 Gram
    (gram32=False) or the fp32 Gram"""
    G, Ct, H, info, _ = reference(i, "f32")
    W, X, alpha, labels = case(i)
    Gg = G.astype(np.float32).astype(np.float64) if gram32 else G
    return np.stack([O.lars_lasso_positive(Gg, c, alpha, W.shape[0], work_dtype=np.float32, gram32=gram32) for c in Ct])


def bar32(He, H):
    """per column 16 x the float32 emulation's error against the oracle, at least 16 FLOOR32"""
    return 16 * np.maximum(col_err(He, H), FLOOR32)


def branch_columns(i, H, info):
    """columns where rounding may pick the other branch of the degenerate-pivot rule: a degenerate pivot in the oracle, a
    join the oracle accepts with pivot^2 < 1e-8 G_jj (a nearly dependent atom, e.g. past d active atoms at k > d), or the
    duplicated pair in the code.  Their codes are held to nonnegativity, to exact zeros and to bit-identity across forms."""
    k = CASES[i][0]
    ex = ((info["status"] & 1) != 0) | (info["min_pivot"] < 1e-8)
    if k >= 4:
        ex |= (H[:, k - 2] > 0) | (H[:, k - 1] > 0)
    return ex


def code_bar(H, info, bar, br):
    """per column code bar: the fp64 bar, raised to TIE64 where the oracle's path has a near-tie within that bar (a join or a
    drop whose runner-up is that close: e.g. an exact combination's last knot, where an atom's coefficient reaches 0
    together with the full step)"""
    return np.where(info["min_gap"] < bar, np.maximum(bar, TIE64), bar)


def stat_exempt(i, H, info):
    """columns left out of the path-statistic checks: branch columns and columns whose oracle path has two join or drop
    candidates within NEAR_TIE relative at one knot"""
    return branch_columns(i, H, info) | (info["min_gap"] < NEAR_TIE)


def col_err(got, ref):
    num = np.linalg.norm(got - ref, axis=1)
    den = np.linalg.norm(ref, axis=1)
    return np.where(num == 0, 0.0, num / np.maximum(den, 1e-300))


# -------------------------------------------------------------------------------------------------------- CPU: oracle
def test_lars_columns_binding_matches_numpy_restatement():
    """c_oracle.lars_columns against onmf_oracle.lars_lasso_positive(return_info=True): equal knots, max_active, drop
    steps and status, codes to 1e-13, over a few hundred columns incl. degenerate pivots (a duplicated atom, k > d), drops,
    max_iter exits and the "alpha increasing" bail-out (mixed-sign dictionaries with a duplicated atom at k > d)."""
    rng = np.random.default_rng(5)
    sets = [(40, 30, 60, 0.2, 1000, "unit"), (12, 24, 60, 0.0, 1000, "unit"), (64, 48, 60, 0.0, 1000, "unit"),
            (50, 40, 40, 0.5, 3, "unit"), (100, 80, 40, 0.0, 7, "unit"), (30, 20, 40, 1.0, 1000, "raw")]
    seen = dict(degenerate=0, drops=0, max_iter=0, alpha_inc=0)
    total = 0
    for (d, k, n, alpha, max_iter, kind) in sets + [(7, 14, 50, 0.0, 1000, 31)]:
        if isinstance(kind, int):           # mixed signs, atoms 0 and 1 identical: degenerate pivots and bail-outs
            r = np.random.default_rng(kind)
            r.integers(3, 12); r.integers(4, 16)
            W = r.standard_normal((d, k))
            W[:, 1] = W[:, 0]
            X = r.standard_normal((n, d))
        else:
            W = rng.random((d, k))
            if kind == "unit":
                W /= np.linalg.norm(W, axis=0)
            X = rng.random((n, d)) - (0.0 if kind == "unit" else 0.45)
            X[0] = W[:, 2] + W[:, 3]            # ties at the first knot
        G = gram(W)
        Ct = X @ W
        H, info = c_oracle.lars_columns(G, Ct, alpha, d, max_iter)
        for j in range(n):
            h, inf = O.lars_lasso_positive(G, Ct[j], alpha, d, max_iter=max_iter, return_info=True)
            st = int(info["status"][j])
            assert int(info["n_iter"][j]) == inf["n_iter"] and int(info["max_active"][j]) == inf["max_active"], (d, k, j)
            assert int(info["drops"][j]) == inf["n_drops"], (d, k, j)
            # the numpy status keeps the last event (3 max_iter, 2 bail-out, 1 degenerate); the C status ORs bits 4 / 2 / 1.
            # With an atom and its exact twin the inactive twin rides at the active level (a near-tie at every knot): whether
            # it wins an arg-max and is rejected as degenerate is decided by rounding, so bit 1 is left out there
            twin = isinstance(kind, int)
            sn = 0 if twin and inf["status"] == 1 else inf["status"]
            stc = st & ~1 if twin else st
            assert {0: stc == 0, 1: stc == 1, 2: bool(stc & 2), 3: bool(stc & 4)}[sn], (d, k, j, st, inf["status"])
            assert np.abs(H[j] - h).max() <= 1e-13 * max(np.abs(h).max(), 1.0), (d, k, j)
            seen["degenerate"] += (st & 1) and inf["status"] == 1
            seen["drops"] += inf["n_drops"] > 0
            seen["max_iter"] += inf["status"] == 3
            seen["alpha_inc"] += inf["status"] == 2
            total += 1
    assert total >= 300 and all(v > 0 for v in seen.values()), seen


def test_float32_emulation_is_the_restatement_in_float64():
    """work_dtype=np.float64 takes none of the float32 rules: the default call, the explicit float64 call and the C
    restatement (untouched by the emulation) give the same path and the same codes (bit for bit between the two numpy
    calls, to 1e-13 against C); and the float32 emulation stays within float32 rounding of it on a clean path."""
    rng = np.random.default_rng(6)
    for (d, k, alpha) in [(60, 40, 0.2), (20, 30, 0.0), (100, 64, 1.0)]:
        W = rng.random((d, k)); W /= np.linalg.norm(W, axis=0)
        G = gram(W)
        for j in range(12):
            c = W.T @ rng.random(d)
            a, ia = O.lars_lasso_positive(G, c, alpha, d, return_info=True)
            b, ib = O.lars_lasso_positive(G, c, alpha, d, return_info=True, work_dtype=np.float64)
            assert np.array_equal(a, b) and ia == ib
            hc, ic = c_oracle.lars_columns(G, c[None], alpha, d)
            assert np.abs(hc[0] - a).max() <= 1e-13 * max(np.abs(a).max(), 1.0)
            assert (ia["n_iter"], ia["max_active"], ia["n_drops"]) == (ic["n_iter"][0], ic["max_active"][0], ic["drops"][0])
            e = O.lars_lasso_positive(G, c.astype(np.float32), alpha, d, work_dtype=np.float32)
            assert e.dtype == np.float64 and (e >= 0).all()
            if ia["status"] == 0 and ia["n_drops"] == 0:
                assert np.linalg.norm(e - a) <= 1e-3 * np.linalg.norm(a) + 1e-6, (d, k, j)


def test_case_set_crosses_its_boundaries():
    """Every case puts columns whose path statistics are checked (stat_exempt) on both sides of each slot boundary of its
    class (by the oracle's max_active); the column equal to the duplicated atom ends on the lower index of the pair (its
    first knot is an exact tie)."""
    for i, (k, d, alpha, kind) in enumerate(CASES):
        _, _, H, info, _ = reference(i)
        ma = info["max_active"][~stat_exempt(i, H, info)]
        for b in boundaries(k):
            if b + 1 <= min(k, d) - (1 if k >= 4 else 0):
                assert (ma <= b).any() and (ma > b).any(), (CASES[i], b, np.unique(ma))
        if k >= 4:
            j = case(i)[3].index("dup_atom")
            assert H[j, k - 2] > 0 and H[j, k - 1] == 0, CASES[i]


def test_mutants_exceed_the_fp64_bar():
    """numpy mutants of the restatement over the case set: each lands at least 10 x above the fp64 bar on some column, or
    changes a path statistic the GPU tests assert (knots, drops, flagged, max_active).  The unmutated restatement stays
    within the bar."""
    picks = {}
    for i, (k, d, alpha, kind) in enumerate(CASES):
        if k > 260:
            continue
        _, _, H, info, bar = reference(i)
        ex = stat_exempt(i, H, info)
        labels = case(i)[3]
        n = len(labels)
        sel = [j for j in range(n) if labels[j] in ("dup_atom", "zero", "below_alpha")]
        comb = [j for j in range(n) if labels[j].startswith("comb") and not ex[j]]
        sel += sorted(range(n), key=lambda j: -int(info["drops"][j]))[:3] + list(range(4)) + comb[-4:]
        picks[i] = sorted(set(sel))
    dist = {}
    for mutant in (None,) + MUTANTS:
        worst, stat_change = 0.0, False
        for i, sel in picks.items():
            W, X, alpha, _ = case(i)
            d = W.shape[0]
            for max_iter in (1000, 3):
                G, Ct, H, info, bar = reference(i, "f64", max_iter)
                ex = stat_exempt(i, H, info)
                for j in sel:
                    h, inf = O.lars_lasso_positive(G, Ct[j], alpha, d, max_iter=max_iter, return_info=True, mutant=mutant)
                    worst = max(worst, float(col_err(h[None], H[j][None])[0] / bar[j]))
                    stat_change |= not ex[j] and (inf["n_iter"] != info["n_iter"][j] or inf["n_drops"] != info["drops"][j] or
                                    inf["max_active"] != info["max_active"][j] or (inf["status"] != 0) != (info["status"][j] != 0))
        dist[mutant] = (worst, stat_change)
        if mutant is None:
            assert worst <= 1.0 and not stat_change, dist
        else:
            assert worst >= 10.0 or stat_change, (mutant, dist)
    print("mutant distance above the fp64 bar (ratio, path statistic changed):",
          {m: ("%.3g" % v[0], v[1]) for m, v in dist.items()})


# ------------------------------------------------------------------------------------------------------------ GPU runs
def dev():
    return torch.device("cuda", 0)


@contextlib.contextmanager
def options(**kw):
    keys = dict(fast=_lib.OPT_LARS_FAST_TIER, reserved=_lib.OPT_LARS_RESERVED_SMS)
    saved = {name: _lib.get_option(keys[name]) for name in kw}
    try:
        for name, v in kw.items():
            _lib.set_option(keys[name], v)
        yield
    finally:
        for name, v in saved.items():
            _lib.set_option(keys[name], v)


def new_ws(dtype, k, n):
    return torch.zeros(_lib.lasso_lars_workspace(dtype, k, max(n, 1)), dtype=torch.uint8, device=dev())


def hint_of(ws):
    return int(ws[HINT_OFFSET:HINT_OFFSET + 4].cpu().numpy().view(np.uint32)[0])


def code(G, Ct, d, alpha, first_tier=0, ws=None, max_iter=1000, fast=1, reserved=None):
    """one coder call on a NaN-filled Ht; returns (Ht, stats as a dict)"""
    n, k = Ct.shape
    Ht = torch.full((n, k), float("nan"), dtype=Ct.dtype, device=dev())
    ws = new_ws(Ct.dtype, k, n) if ws is None else ws
    stats = torch.zeros(8, dtype=torch.int64, device=dev())
    kw = dict(fast=fast) if reserved is None else dict(fast=fast, reserved=reserved)
    with options(**kw):
        _lib.lasso_lars(G, Ct, d, alpha, Ht, ws, max_iter=max_iter, stats=stats, first_tier=first_tier)
        torch.cuda.synchronize()
    s = stats.cpu().numpy()
    return Ht, dict(zip(("columns", "knots", "sum_active", "sum_active2", "drops", "overflow", "flagged", "max_active"),
                        (int(v) for v in s)))


def prime_rows():
    """a priming call's size: above the fast-small route's limit (48 x SMs), which neither reads nor updates the hint"""
    return 48 * torch.cuda.get_device_properties(0).multi_processor_count + 1


def overflowing_rows(i, first_slots, n):
    """n covariance rows of case i whose oracle path outgrows `first_slots` (repeated): primes the hint to 1; None when no
    column does (k = 33 with the duplicated pair: at most 32 atoms can be active)"""
    _, Ct, _, info, _ = reference(i)
    rows = np.nonzero(info["max_active"] > first_slots)[0]
    return Ct[np.resize(rows, n)] if rows.size else None


def forms(i, dtype, G, Ct, d, alpha):
    """every scheduling form of one call: (name, bit-identity group, tier that started, Ht, stats).  Forms in one group run
    the same kernels and must give the same bits: first_tier = t and the adaptive call under hint t; every form on the
    fp32 small-minibatch route (k <= 64, FP64 Gram, fast tier on), which runs whatever first_tier says.  Other forms are
    each held to the oracle: tiers with different slot counts keep the factor in different register layouts, and codes
    of columns they both finish agree to rounding (not bit for bit)."""
    k = Ct.shape[1]
    out = []
    fasts = (1, 0) if dtype == F32 and G.dtype == F64 else (1,)
    for fast in fasts:
        small = fast == 1 and dtype == F32 and G.dtype == F64 and k <= 64
        group = lambda t: (fast if k <= 64 else 1, "small" if small else t)
        for ft in (0, 1):
            t = ft if len(tiers(k)) > 1 else 0
            Ht, st = code(G, Ct, d, alpha, first_tier=ft, fast=fast)
            out.append(("first_tier=%d fast=%d" % (ft, fast), group(t), t, Ht, st))
        ws = new_ws(Ct.dtype, k, Ct.shape[0])
        Ht, st = code(G, Ct, d, alpha, first_tier=-1, ws=ws, fast=fast)
        out.append(("hint=0 fast=%d" % fast, group(0), 0, Ht, st))
        m = prime_rows()
        prime = overflowing_rows(i, tiers(k)[0], m) if len(tiers(k)) > 1 else None
        if prime is not None:
            ws = new_ws(Ct.dtype, k, m)
            code(G, torch.from_numpy(prime).to(dev(), Ct.dtype), d, alpha, first_tier=-1, ws=ws, fast=fast)
            assert hint_of(ws) == 1
            Ht, st = code(G, Ct, d, alpha, first_tier=-1, ws=ws, fast=fast)
            out.append(("hint=1 fast=%d" % fast, group(1), 1, Ht, st))
    return out


def check_stats(name, k, start, st, info, n):
    S = tiers(k)[start]
    ovf = int((info["max_active"] > S).sum())
    degen_at_S = int(((info["max_active"] == S) & (info["status"] & 1 != 0)).sum())
    assert st["columns"] == n and st["max_active"] == int(info["max_active"].max(initial=0)), (name, st)
    assert st["flagged"] == int((info["status"] != 0).sum()), (name, st, int((info["status"] != 0).sum()))
    assert ovf <= st["overflow"] <= ovf + degen_at_S, (name, st, ovf)
    if st["overflow"] == 0:
        assert st["knots"] == int(info["n_iter"].sum()) and st["drops"] == int(info["drops"].sum()), (name, st)
    else:   # a column handed on is re-walked from its start by the next tier and counts again
        assert st["knots"] >= int(info["n_iter"].sum()) and st["drops"] >= int(info["drops"].sum()), (name, st)


def pair_folded(H, k):
    """codes with the duplicated pair summed into its lower index (the pair's split is not determined, its sum is)"""
    H = np.array(H, dtype=np.float64, copy=True)
    if k >= 4:
        H[..., k - 2] += H[..., k - 1]
        H[..., k - 1] = 0.0
    return H


@pytest.mark.gpu
@pytest.mark.parametrize("i", range(len(CASES)), ids=case_ids())
def test_fp64_every_form_against_oracle(i):
    """fp64 coder in every scheduling form: every column within its code bar (code_bar; branch columns with the duplicated
    pair summed), oracle-zero columns exactly zero, forms of one group bit-identical; first_tier 0 against 1 recorded; path
    statistics against the oracle's info on the columns stat_exempt keeps, in a call of their own per starting tier"""
    k, d, alpha, kind = CASES[i]
    G, Ct, H, info, bar = reference(i)
    n = Ct.shape[0]
    Gd, Cd = torch.from_numpy(G).to(dev()), torch.from_numpy(Ct).to(dev())
    zero = ~H.any(1)
    br = branch_columns(i, H, info)
    # branch columns are held with the duplicated pair summed where the dictionary has full column rank (d >= k); at k > d the
    # nearly dependent joins leave even the sum to the branch taken
    cb = np.where(br, np.maximum(bar, TIE64) if d >= k else np.inf, code_bar(H, info, bar, br))
    tie = (info["min_gap"] < bar) & ~br
    ex = stat_exempt(i, H, info)
    Hf = pair_folded(H, k)
    worst = worst_tie = worst_branch = 0.0
    first, by_tier = {}, {}
    for name, group, start, Ht, st in forms(i, F64, Gd, Cd, d, alpha):
        Hk = Ht.cpu().numpy()
        assert not np.isnan(Hk).any() and (Hk >= 0).all(), name
        r = col_err(pair_folded(Hk, k), Hf) / cb
        worst = max(worst, float(r[~br & ~tie].max(initial=0.0)))
        worst_tie = max(worst_tie, float(r[tie].max(initial=0.0)))
        worst_branch = max(worst_branch, float(r[br].max(initial=0.0)))
        assert (r <= 1).all(), (CASES[i], name, np.nonzero(r > 1)[0], float(r.max()))
        assert (Hk[zero] == 0).all(), name
        # flagged may differ only by the branch columns; the other statistics below, on the columns stat_exempt keeps
        assert st["columns"] == n and st["max_active"] == int(info["max_active"].max()), (name, st)
        assert int((info["status"][~br] != 0).sum()) <= st["flagged"] <= int((info["status"] != 0).sum()) + int(br.sum()), (name, st)
        first.setdefault(group, Ht)
        assert torch.equal(Ht, first[group]), (CASES[i], name, group)
        by_tier.setdefault(start, Hk)
    clean = {key: v[~ex] for key, v in info.items()}
    rows = torch.from_numpy(np.nonzero(~ex)[0]).to(dev())
    for ft in (0, 1):
        _, st = code(Gd, Cd[rows].contiguous(), d, alpha, first_tier=ft)
        check_stats("clean columns first_tier=%d" % ft, k, ft if len(tiers(k)) > 1 else 0, st, clean, int((~ex).sum()))
    diff = ""
    if 1 in by_tier:
        dcol = (by_tier[0] != by_tier[1]).any(1)
        diff = "; first_tier 0 / 1 differ in %d columns (max_active %s), by at most %.3g of the code bar" % (
            int(dcol.sum()), sorted(set(info["max_active"][dcol].tolist()))[:6],
            float((col_err(pair_folded(by_tier[1], k), pair_folded(by_tier[0], k)) / cb).max()))
    print("fp64 %s: largest error / bar %.3g, near-tie columns %.3g, branch columns %.3g (%d branch, %d near-tie, %d "
          "statistic-exempt of %d)%s" % (case_ids()[i], worst, worst_tie, worst_branch, int(br.sum()), int(tie.sum()),
                                         int(ex.sum()), n, diff))


@pytest.mark.gpu
@pytest.mark.parametrize("gram32", [False, True], ids=["g64", "g32"])
@pytest.mark.parametrize("i", range(len(CASES)), ids=case_ids())
def test_fp32_every_form_against_oracle(i, gram32):
    """fp32 coder with the FP64 Gram (fast tier on and off) or an fp32 Gram, every scheduling form: each column within 16 x
    its own float32 emulation's error (bar32), nonnegative; where the emulation ends on the oracle's support the kernel
    does too, up to coefficients the column's bar cannot see; forms of one group bit-identical.  Branch columns are held
    to nonnegativity and bit-identity only (the dup_atom column: test_fp32_duplicated_atom_column)."""
    k, d, alpha, kind = CASES[i]
    G, Ct, H, info, _ = reference(i, "f32")
    br = branch_columns(i, H, info)
    He = emulation(i, gram32)
    b = bar32(He, H)
    nh = np.linalg.norm(H, axis=1)
    same_support = np.array([np.array_equal(He[j] > 0, H[j] > 0) and not br[j] for j in range(len(H))])
    Cd = torch.from_numpy(Ct).to(dev(), F32)
    Gd = torch.from_numpy(G).to(dev()) if not gram32 else torch.from_numpy(G).to(dev(), F32)
    first, worst = {}, 0.0
    for name, group, start, Ht, st in forms(i, F32, Gd, Cd, d, alpha):
        Hk = Ht.cpu().numpy().astype(np.float64)
        assert not np.isnan(Hk).any() and (Hk >= 0).all(), name
        assert st["columns"] == Ct.shape[0], (name, st)
        r = (col_err(Hk, H) / b)[~br]
        worst = max(worst, float(r.max()))
        assert (r <= 1).all(), (CASES[i], name, np.nonzero(~br)[0][r > 1], float(r.max()))
        for j in np.nonzero(same_support)[0]:
            differ = (Hk[j] > 0) != (H[j] > 0)
            assert (np.maximum(Hk[j], H[j])[differ] <= b[j] * nh[j]).all(), (CASES[i], name, j)
        first.setdefault(group, Ht)
        assert torch.equal(Ht, first[group]), (CASES[i], name, group, float((Ht - first[group]).abs().max()))
    labels = np.array(case(i)[3])
    rnd = (labels == "random") & ~br
    print("fp32 %s %s: largest error / bar %.3g; bars: random columns median %.3g max %.3g, all columns max %.3g" % (
        case_ids()[i], "g32" if gram32 else "g64", worst, float(np.median(b[rnd])), float(b[rnd].max()), float(b[~br].max())))


@pytest.mark.gpu
@pytest.mark.xfail(strict=True, reason="fp32 exact-tie rule: a zero-length step for the duplicated atom, which is then "
                                       "rejected as degenerate, and the path stops without moving (code 0 instead of 2 - alpha)")
@pytest.mark.parametrize("gram32", [False, True], ids=["g64", "g32"])
def test_fp32_duplicated_atom_column(gram32):
    """The dup_atom column (2 e + 0.5 w_0, e an atom with an exact twin) in fp32: the pair's summed coefficient should be
    the oracle's, 2 - alpha.  The fp32 coder returns 0 on the pair today; this test records that defect."""
    i = CASES.index((64, 128, 1.0, "unit"))
    k, d, alpha, kind = CASES[i]
    G, Ct, H, info, _ = reference(i, "f32")
    j = case(i)[3].index("dup_atom")
    Gd = torch.from_numpy(G).to(dev(), F32 if gram32 else F64)
    Hk, _ = code(Gd, torch.from_numpy(Ct[j:j + 1]).to(dev(), F32), d, alpha)
    got = float(Hk[0, k - 2:].sum())
    want = float(H[j, k - 2:].sum())
    assert abs(got - want) <= 1e-3 * want, (got, want)


@pytest.mark.gpu
def test_first_tier_settings_are_bit_identical_around_fast_small_threshold():
    """At k <= 32 (one tier) first_tier -1 / 0 / 1 give the same bits at any n; at k <= 64 on the fp32 small-minibatch
    route (FP64 Gram, n <= 48 x SMs) so do -1 / 0 / 1 and hint 0 / 1 -- before this route was taken for every first_tier,
    first_tier = 1 ran the general kernel there and differed in the last bits.  Elsewhere first_tier = t equals the
    adaptive call under hint t.  n on both sides of the route's limit (24 x SMs at k <= 32, 48 x SMs at k <= 64); fp64, fp32
    with the FP64 Gram and with an fp32 Gram."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    rng = np.random.default_rng(7)
    for (k, d, lim) in ((25, 100, 24 * sms), (49, 120, 48 * sms)):
        W = rng.random((d, k)); W /= np.linalg.norm(W, axis=0)
        G = gram(W)
        for n in (lim, lim + 1):
            X = rng.random((n, d))
            X[: n // 4] = W[:, rng.integers(0, k, (n // 4, 40))].sum(2).T  # long paths: some columns pass 32 atoms at k = 49
            Ct = X @ W
            for dtype, g in ((F64, F64), (F32, F64), (F32, F32)):
                Gd = torch.from_numpy(G).to(dev(), g)
                Cd = torch.from_numpy(Ct).to(dev(), dtype)
                H0, H1, Ha = (code(Gd, Cd, d, 0.1, first_tier=ft)[0] for ft in (0, 1, -1))
                assert torch.equal(Ha, H0), (k, n, dtype, g)
                small = dtype == F32 and g == F64 and n <= lim
                if k <= 32 or small:
                    assert torch.equal(H1, H0), (k, n, dtype, g, float((H1 - H0).abs().max()))
                if k > 32:
                    m = prime_rows()
                    ws = new_ws(dtype, k, m)
                    prime = Cd[torch.arange(m, device=dev()) % (n // 4)].contiguous()
                    code(Gd, prime, d, 0.0, first_tier=-1, ws=ws)    # alpha = 0 on the long paths: hint -> 1
                    assert hint_of(ws) == 1, (k, n, dtype, g)
                    Hh = code(Gd, Cd, d, 0.1, first_tier=-1, ws=ws)[0]
                    assert torch.equal(Hh, H0 if small else H1), (k, n, dtype, g)


@pytest.mark.gpu
def test_hint_state_machine():
    """k = 100 (three tiers), n = 1000 (not the fast-small route): exact combinations of 50 atoms at alpha = 0, > n/16
    columns outgrow 32 slots -> hint 1; then random columns at alpha = 5 (a few atoms each) -> hint 0; n = 0 -> untouched.  stats.overflow counts against the tier the
    hint starts (32 slots under hint 0, 64 under hint 1); every call bit-identical to first_tier = <the hint it ran under>."""
    rng = np.random.default_rng(8)
    k, d, n = 100, 200, 1000
    Wunit = rng.random((d, k))
    Wunit /= np.linalg.norm(Wunit, axis=0)
    Hc = np.zeros((n, k))
    for j in range(n):
        Hc[j, rng.choice(k, 50, replace=False)] = rng.random(50) + 0.5
    Xs = {0.0: Hc @ Wunit.T, 5.0: rng.random((n, d))}
    for dtype in (F64, F32):
        ws = new_ws(dtype, k, n)
        assert hint_of(ws) == 0
        seq = []
        for W, alpha in ((Wunit, 0.0), (Wunit, 0.0), (Wunit, 5.0), (Wunit, 5.0)):
            G = gram(W)
            Ct = Xs[alpha] @ W
            Gd, Cd = torch.from_numpy(G).to(dev()), torch.from_numpy(Ct).to(dev(), dtype)
            before = hint_of(ws)
            Ha, sa = code(Gd, Cd, d, alpha, first_tier=-1, ws=ws)
            H0, s0 = code(Gd, Cd, d, alpha, first_tier=0)
            H1, s1 = code(Gd, Cd, d, alpha, first_tier=1)
            assert torch.equal(Ha, H0 if before == 0 else H1), (dtype, alpha, before)
            assert sa["overflow"] == (s0 if before == 0 else s1)["overflow"], (before, sa, s0, s1)
            seq.append((before, hint_of(ws), sa["overflow"], s0["overflow"]))
        # the combinations at alpha = 0 outgrow 32 slots; the random columns at alpha = 5 do not
        assert seq[0][3] * 16 > n and seq[0][:2] == (0, 1) and seq[1][:2] == (1, 1), seq
        assert seq[2][3] * 16 <= n and seq[2][:2] == (1, 0) and seq[3][:2] == (0, 0), seq
        ws[HINT_OFFSET] = 1
        snapshot = ws.clone()
        p = _lib._ptr
        assert _lib.load().onmf_lasso_lars_g64(_lib.dt(Cd), p(Gd), p(Cd), 0, k, d, 1.0, 1000, p(Ha), p(ws), ws.numel(), None, -1,
                                               None) == 0
        torch.cuda.synchronize()
        assert torch.equal(ws, snapshot)


@pytest.mark.gpu
def test_column_independence():
    """A row permutation of Ct permutes Ht bit for bit; one column repeated gives identical rows; a column coded inside a
    full warp of other columns, alone among zero columns, or at every lane-group position, gives the same bits, in every
    lane-group size (LPC 8 / 16 / 32) and both dtypes."""
    rng = np.random.default_rng(9)
    for (k, d, n) in ((30, 64, 300), (60, 128, 300), (100, 200, 300), (256, 512, 300)):
        W = rng.random((d, k)); W /= np.linalg.norm(W, axis=0)
        G = gram(W)
        Ct = rng.random((n, d)) @ W
        for dtype, g in ((F64, F64), (F32, F64), (F32, F32)):
            Gd = torch.from_numpy(G).to(dev(), g)
            Cd = torch.from_numpy(Ct).to(dev(), dtype)
            H, _ = code(Gd, Cd, d, 0.3)
            perm = torch.from_numpy(rng.permutation(n)).to(dev())
            Hp, _ = code(Gd, Cd[perm].contiguous(), d, 0.3)
            assert torch.equal(Hp, H[perm]), (k, dtype, g)
            for j in (0, 7, 131):
                Hr, _ = code(Gd, Cd[j:j + 1].repeat(n, 1).contiguous(), d, 0.3)
                assert torch.equal(Hr, H[j:j + 1].repeat(n, 1)), (k, dtype, g, j)
                padded = torch.zeros_like(Cd)
                for pos in (0, 1, 3, 5, n - 1):
                    padded.zero_()
                    padded[pos] = Cd[j]
                    Hz, _ = code(Gd, padded, d, 0.3)
                    assert torch.equal(Hz[pos], H[j]) and int((Hz != 0).any(1).sum()) <= 1, (k, dtype, g, j, pos)


@pytest.mark.gpu
def test_grid_independence():
    """ONMF_OPT_LARS_RESERVED_SMS 0 / 17 / 64 and the fast tier on / off give the same bits (fp64, fp32 with each Gram)"""
    rng = np.random.default_rng(10)
    for (k, d, n) in ((49, 100, 500), (100, 200, 3000), (256, 512, 3000), (400, 800, 400)):
        W = rng.random((d, k)); W /= np.linalg.norm(W, axis=0)
        G = gram(W)
        Ct = rng.random((n, d)) @ W
        for dtype, g in ((F64, F64), (F32, F64), (F32, F32)):
            Gd = torch.from_numpy(G).to(dev(), g)
            Cd = torch.from_numpy(Ct).to(dev(), dtype)
            for fast in (1, 0):
                ref, _ = code(Gd, Cd, d, 0.5, first_tier=-1, reserved=0, fast=fast)
                if fast == 0 and k > 64:       # the fast tier gives the general kernel's bits above k = 64
                    assert torch.equal(ref, ref_fast), (k, dtype, g)
                ref_fast = ref
                for rsv in (17, 64):
                    H, _ = code(Gd, Cd, d, 0.5, first_tier=-1, reserved=rsv, fast=fast)
                    assert torch.equal(H, ref), (k, dtype, g, rsv, fast)


@functools.lru_cache(maxsize=None)
def scratch_problem(k, n):
    """d = 1024, n exact nonnegative combinations of 200 atoms each, alpha = 0: (G, Ct, H, info, Hk fp64 codes, stats)"""
    rng = np.random.default_rng(11)
    d = 1024
    W = rng.random((d, k)); W /= np.linalg.norm(W, axis=0)
    G = gram(W)
    Hs = np.zeros((n, k))
    for j in range(n):
        Hs[j, rng.choice(k, 200, replace=False)] = rng.random(200) + 0.5
    Ct = (Hs @ W.T) @ W
    H, info = c_oracle.lars_columns(G, Ct, 0.0, d)
    Hk, st = code(torch.from_numpy(G).to(dev()), torch.from_numpy(Ct).to(dev()), d, 0.0)
    return G, Ct, H, info, Hk.cpu().numpy(), st


# The fp64 coder on these 400-knot paths (200 active atoms, dozens of drops) ends up to 3e-7 from the restatement, while the
# numpy and C restatements agree to 1e-10 there and reach the generating codes to 1e-10: a precision shortfall of the kernel
# on long paths with many drops, recorded by test_global_tier_fp64_precision.  The reuse test holds the codes to LONG64.
LONG64 = 1e-6


@pytest.mark.gpu
@pytest.mark.xfail(strict=True, reason="fp64 coder on 400-knot paths with many drops: errors to 3e-7 where the restatements "
                                       "agree to 1e-10")
@pytest.mark.parametrize("k,n", [(300, 256), (256, 512)])
def test_global_tier_fp64_precision(k, n):
    """The scratch-reuse columns in fp64 held to their code bar (code_bar, at most 1e-8 here)."""
    G, Ct, H, info, Hk, st = scratch_problem(k, n)
    bar = bar64(G, H, info)
    ok = (info["status"] & 1 == 0) & (info["min_pivot"] >= 1e-8)
    r = (col_err(Hk, H) / code_bar(H, info, bar, ~ok))[ok]
    assert (r <= 1).all(), (float(r.max()), int((r > 1).sum()))


@pytest.mark.gpu
@pytest.mark.parametrize("k,n", [(300, 256), (256, 512)])
def test_global_tier_scratch_reuse(k, n):
    """More columns than the last tier's scratch holds groups (95 at k <= 512, 382 at k <= 256), every one past 128 active
    atoms: the scratch is reused across tickets.  fp64 within LONG64 (see there) on every column without a degenerate-pivot
    branch, fp32 (FP64 Gram) within 16 x each column's own float32 emulation error."""
    d = 1024
    G, Ct, H, info, Hk, st = scratch_problem(k, n)
    assert (info["max_active"] > 128).all(), np.unique(info["max_active"])
    # columns whose path the degenerate-pivot rule may branch on by rounding are held to nonnegativity only
    bar = bar64(G, H, info)
    ok = (info["status"] & 1 == 0) & (info["min_pivot"] >= 1e-8)
    cb = np.maximum(code_bar(H, info, bar, ~ok), LONG64)
    e = (col_err(Hk, H) / cb)[ok]
    assert ok.sum() >= n - n // 16 and (e <= 1).all() and st["columns"] == n and st["overflow"] == n, (
        int(ok.sum()), float(e.max()), st)
    assert (Hk >= 0).all()
    tie = info["min_gap"][ok] < bar[ok]
    print("scratch reuse k=%d fp64: largest error / bar %.3g (%.3g on %d near-tie columns) over %d columns" % (
        k, float(e[~tie].max(initial=0.0)), float(e[tie].max(initial=0.0)), int(tie.sum()), int(ok.sum())))
    C32 = Ct.astype(np.float32).astype(np.float64)
    H32, info32 = c_oracle.lars_columns(G, C32, 0.0, d)
    # a path with two candidates closer than eps32 (relative) at one knot is not resolved in float32: the kernel may take the
    # other branch (one of the 512 columns at k = 256 does, with a 3.5e-8 gap, and ends 0.5 away); those are held to
    # nonnegativity, every other column to its own bar
    ok32 = (info32["status"] & 1 == 0) & (info32["min_pivot"] >= 1e-8) & (info32["min_gap"] >= EPS32)
    idx = np.nonzero(ok32)[0]
    He = np.stack([O.lars_lasso_positive(G, C32[j], 0.0, d, work_dtype=np.float32) for j in idx])
    b = bar32(He, H32[idx])
    Hk32, st32 = code(torch.from_numpy(G).to(dev()), torch.from_numpy(C32).to(dev(), F32), d, 0.0)
    r32 = col_err(Hk32.cpu().numpy().astype(np.float64)[idx], H32[idx]) / b
    assert len(idx) >= n // 4 and (r32 <= 1).all() and st32["columns"] == n, (len(idx), idx[r32 > 1], float(r32.max()), st32)
    assert (Hk32 >= 0).all()
    print("scratch reuse k=%d fp32: largest error / bar %.3g over %d columns (bars median %.3g, max %.3g)" % (
        k, float(r32.max()), len(idx), float(np.median(b)), float(b.max())))


@pytest.mark.gpu
def test_max_iter_against_oracle():
    """max_iter 1, 3 and one below the longest path, fp64 and fp32: codes against the oracle run with the same max_iter,
    status-4 columns counted in flagged"""
    for i in (CASES.index((33, 66, 0.2, "unit")), CASES.index((129, 258, 0.2, "unit"))):
        k, d, alpha, _ = CASES[i]
        longest = int(reference(i)[3]["n_iter"].max())
        for max_iter in (1, 3, longest - 1):
            G, Ct, H, info, bar = reference(i, "f64", max_iter)
            Hk, st = code(torch.from_numpy(G).to(dev()), torch.from_numpy(Ct).to(dev()), d, alpha, max_iter=max_iter)
            br = branch_columns(i, H, info)
            e = col_err(Hk.cpu().numpy(), H)[~br]
            assert (e <= bar[~br]).all(), (k, max_iter, float((e / bar[~br]).max()))
            assert st["flagged"] == int((info["status"] != 0).sum()) and (info["status"] & 4).any(), (k, max_iter, st)
            G, C32, H32, info32, _ = reference(i, "f32", max_iter)
            Hk32, st32 = code(torch.from_numpy(G).to(dev()), torch.from_numpy(C32).to(dev(), F32), d, alpha, max_iter=max_iter)
            assert st32["flagged"] >= int(((info32["status"] & 4) != 0).sum()), (k, max_iter, st32)
            if max_iter <= 3:       # a few knots: the float32 emulation of every column is cheap
                ok = ~branch_columns(i, H32, info32)
                He = np.stack([O.lars_lasso_positive(G, C32[j], alpha, d, max_iter=max_iter, work_dtype=np.float32)
                               for j in np.nonzero(ok)[0]])
                bar32 = 16 * max(float(col_err(He, H32[ok]).max()), FLOOR32)
                e32 = col_err(Hk32.cpu().numpy().astype(np.float64), H32)[ok]
                assert e32.max() <= bar32, (k, max_iter, float(e32.max()), bar32)


@pytest.mark.gpu
def test_refusals_leave_codes_untouched():
    """a workspace one byte short, off its 256-byte alignment, k = 513, k = 0, alpha < 0 or NaN, max_iter < 0, a bad dtype:
    an error and Ht bit-untouched; n = 0 returns OK and touches nothing, not even the hint"""
    lib = _lib.load()
    k, n, d = 40, 16, 80
    G = torch.eye(k, dtype=F64, device=dev())
    Ct = torch.rand(n, k, dtype=F64, device=dev())
    Ht = torch.full((n, k), 7.0, dtype=F64, device=dev())
    need = _lib.lasso_lars_workspace(F64, k, n)
    big = torch.zeros(need + 512, dtype=torch.uint8, device=dev())
    p = _lib._ptr

    def call(dtype=1, G_=G, k_=k, n_=n, alpha=1.0, max_iter=1000, ws_ptr=None, ws_bytes=need):
        return lib.onmf_lasso_lars_ex(dtype, p(G_), p(Ct), n_, k_, d, alpha, max_iter, p(Ht),
                                      ws_ptr if ws_ptr is not None else p(big), ws_bytes, None, -1, None)
    dt64 = _lib.dt(Ct)
    snap = Ht.clone()
    assert call(dt64, ws_bytes=need - 1) == ONMF_E_WORKSPACE
    assert call(dt64, ws_ptr=big.data_ptr() + 8) == ONMF_E_ARG
    G513 = torch.eye(513, dtype=F64, device=dev())
    assert call(dt64, G_=G513, k_=513, ws_bytes=need + 512) == ONMF_E_UNSUPPORTED
    assert call(dt64, k_=0) == ONMF_E_ARG
    assert call(dt64, alpha=-1.0) == ONMF_E_ARG
    assert call(dt64, alpha=float("nan")) == ONMF_E_ARG
    assert call(dt64, max_iter=-1) == ONMF_E_ARG
    assert call(7) == ONMF_E_ARG
    torch.cuda.synchronize()
    assert torch.equal(Ht, snap)
    big[HINT_OFFSET] = 1
    before = big.clone()
    assert call(dt64, n_=0) == 0
    torch.cuda.synchronize()
    assert torch.equal(big, before) and torch.equal(Ht, snap)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [F64, F32], ids=["fp64", "fp32"])
def test_engine_sparse_code_equals_direct_call(dtype):
    """OnmfEngine.sparse_code at one k per class equals the direct coder call on the engine's covariances and Gram, bit
    for bit; fp32 also on a raw dictionary (the FP64 coder on fp32 covariances, _lars_wide)"""
    from onmf_ontf_ndl_b200 import OnmfEngine
    rng = np.random.default_rng(12)
    for (k, d) in ((20, 50), (50, 100), (100, 200), (200, 400), (300, 600)):
        for raw in ((False, True) if dtype == F32 else (False,)):
            W = rng.random((d, k))
            if not raw:
                W /= np.linalg.norm(W, axis=0)
            n = 400
            X = rng.random((n, d))
            eng = OnmfEngine(d, k, alpha=0.5, dtype=dtype, device=dev())
            eng.set_state(W)
            Xt = torch.from_numpy(X).to(dev(), dtype)
            Hs = eng.sparse_code(Xt).clone()
            Ct = eng.Ct[:n].clone()
            f = eng.derive_foreign(torch.from_numpy(W).to(dev(), dtype))
            assert f.wide == raw
            G64 = f.G.clone()
            torch.cuda.synchronize()
            if raw:
                H64, _ = code(G64, Ct.double(), d, 0.5, first_tier=-1)
                Hd = H64.float()
            else:
                Hd, _ = code(G64, Ct, d, 0.5, first_tier=-1)
            assert torch.equal(Hs, Hd), (k, dtype, raw)
