"""Inputs, fp32 emulation and bug restatements of the dictionary-update tests (tests/test_update_dict_variants.py), and
the subprocess entry that runs onmf_update_dict under one setting of the ONMF_BCD_* switches (they are read once per
process): `python _bcd_worker.py cases.json out.npz` writes every case's output dictionary and the plan it ran with."""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")

FAMILIES = ("golden", "learned", "mixed", "zero")


def _unit(W):
    return W / np.maximum(np.linalg.norm(W, axis=0), 1e-300)


def _learned(d, k, rng, steps=20, n=32):
    """unit columns; A, B blended over `steps` minibatches of sparse nonnegative codes of data near the dictionary
    (A = (1-w) A + w H H^T, B = (1-w) B + w H X^T, w = 1/t: the reference's recursion)"""
    W = _unit(np.abs(rng.standard_normal((d, k))) * (rng.random((d, k)) < 0.7) + 1e-3)
    A, B = np.zeros((k, k)), np.zeros((k, d))
    dens = min(0.3, 4.0 / k) if k > 1 else 1.0
    for t in range(1, steps + 1):
        H = rng.random((k, n)) * (rng.random((k, n)) < dens)
        X = W @ H + 0.05 * rng.random((d, n))
        w = 1.0 / t
        A, B = (1 - w) * A + w * (H @ H.T), (1 - w) * B + w * (H @ X.T)
    return W, A, B


def state(family, d, k, seed=0):
    """(W, A, B) in float64 for one input family at shape (d, k)"""
    rng = np.random.default_rng(1000003 * d + 7919 * k + seed)
    if family == "golden":
        # the reference's own final state: full_cfg1..4 at their shapes, otherwise rows / atoms of full_cfg5 (cycled
        # beyond 1024 rows or 256 atoms: the state of a dictionary with repeated features / atoms)
        for i in (1, 2, 3, 4, 5):
            g = np.load(os.path.join(GOLDEN, "full_cfg%d.npz" % i))
            if g["W"].shape == (d, k):
                return g["W"].copy(), g["A"].copy(), g["B"].copy()
        ri, ai = np.arange(d) % 1024, np.arange(k) % 256
        return g["W"][np.ix_(ri, ai)], g["A"][np.ix_(ai, ai)], g["B"][np.ix_(ai, ri)]
    W, A, B = _learned(d, k, rng)
    if family == "learned":
        return W, A, B
    if family == "zero":                       # the first update of a run: clamp and shrink only
        return 3.0 * rng.random((d, k)) / np.sqrt(max(d, 1)) + W, np.zeros((k, k)), np.zeros((k, d))
    assert family == "mixed"
    # unused atoms (zero row and column of A, zero row of B), columns that must shrink, entries and whole columns that clamp
    at = rng.permutation(k)
    unused, grow, clamp, dead = at[0::5], at[1::5], at[2::5], at[3::10]
    W[:, grow] *= 2.5                          # updated norm > 1: shrink
    B[clamp] *= 0.3                            # many entries below zero: clamp
    diag = float(np.mean(np.diag(A))) if k else 0.0
    for z in dead:                             # B row zero and strong coupling: the whole column clamps to zero
        B[z] = 0.0
        A[z, :] += 0.5 * diag
        A[:, z] += 0.5 * diag
        A[z, z] -= 0.5 * diag
        W[:, z] *= 0.01
    A[unused, :] = 0.0
    A[:, unused] = 0.0
    B[unused] = 0.0
    return W, A, B


def rounded(x, dtype):
    """the values a device tensor of `dtype` ("float32" / "float64") holds, as float64"""
    return np.asarray(x, dtype=np.float32).astype(np.float64) if dtype == "float32" else np.asarray(x, dtype=np.float64)


def emulate_fp32(W, A, B):
    """the fp32 sweep as the kernels form it: fp32 dot products, difference with B and the step in FP64, fp32 norm"""
    W1 = np.array(W, dtype=np.float32)
    A32, B32 = np.asarray(A, dtype=np.float32), np.asarray(B, dtype=np.float32)
    for j in range(W1.shape[1]):
        dot = (W1 @ A32[:, j]).astype(np.float64)
        v = W1[:, j].astype(np.float64) - (1.0 / (float(A32[j, j]) + 1.0)) * (dot - B32[j].astype(np.float64))
        wn = np.maximum(v, 0.0).astype(np.float32)
        nrm = np.sqrt(np.sum(wn * wn, dtype=np.float32))
        W1[:, j] = (np.float32(1.0) / max(nrm, np.float32(1.0))) * wn
    return W1.astype(np.float64)


MUTANTS = ("no_exchange", "stale_regw", "step_1_over_ajj", "norm_missing_last_cta", "b_wrong_row")


def sweep(W, A, B, mutant=None, cut_rows=1):
    """the FP64 sweep (== oracle.onmf_oracle.update_dict) with one plausible kernel bug:
    no_exchange           : atom j's dot product keeps the OLD entry of column j-1 (the pipelined exchange term dropped)
    stale_regw            : the register copy of W is never refreshed (dot product with the sweep's input W, only the
                            exchange term of column j-1 applied)
    step_1_over_ajj       : step 1 / A_jj instead of 1 / (A_jj + 1)
    norm_missing_last_cta : the column norm leaves out the last `cut_rows` rows (the last CTA's slab)
    b_wrong_row           : B[j-1, :] instead of B[j, :] (the B pipeline one atom late)"""
    W0 = np.array(W, dtype=np.float64)
    W1 = W0.copy()
    d, k = W1.shape
    for j in range(k):
        dot = W1 @ A[:, j]
        if mutant == "no_exchange" and j > 0:
            dot = dot - (W1[:, j - 1] - W0[:, j - 1]) * A[j - 1, j]
        elif mutant == "stale_regw":
            dot = W0 @ A[:, j]
            if j > 0:
                dot = dot + (W1[:, j - 1] - W0[:, j - 1]) * A[j - 1, j]
        b = B[j - 1] if (mutant == "b_wrong_row" and j > 0) else B[j]
        c = 1.0 / (A[j, j] + 1.0)
        if mutant == "step_1_over_ajj" and A[j, j] > 0:
            c = 1.0 / A[j, j]
        col = np.maximum(W1[:, j] - c * (dot - b), 0.0)
        nrm = np.linalg.norm(col[:max(d - cut_rows, 0)] if mutant == "norm_missing_last_cta" else col)
        W1[:, j] = col / max(1.0, nrm)
    return W1


def atom_err(W, Wref):
    """largest per-atom (column) error, absolute: every column of an updated dictionary lies in the unit ball"""
    return float(np.max(np.linalg.norm(np.asarray(W, dtype=np.float64) - Wref, axis=0))) if W.size else 0.0


def run_cases(cases):
    """cases: [(dtype name, d, k, family)] -> {key: W_out}, {key: plan}"""
    import torch
    from onmf_ontf_ndl_b200 import _lib
    outs, plans = {}, {}
    dev = torch.device("cuda", 0)
    for dt, d, k, fam in cases:
        tdt = getattr(torch, dt)
        W, A, B = state(fam, d, k)
        Wd = torch.from_numpy(np.ascontiguousarray(W)).to(dev, tdt)
        out = torch.empty_like(Wd)
        _lib.update_dict(Wd, torch.from_numpy(np.ascontiguousarray(A)).to(dev, tdt),
                         torch.from_numpy(np.ascontiguousarray(B)).to(dev, tdt), out)
        key = "%s_%d_%d_%s" % (dt, d, k, fam)
        outs[key] = out.cpu().numpy().astype(np.float64)
        plans[key] = _lib.update_dict_plan(tdt, d, k)
    torch.cuda.synchronize()
    return outs, plans


if __name__ == "__main__":
    with open(sys.argv[1]) as f:
        cases = [tuple(c) for c in json.load(f)]
    outs, plans = run_cases(cases)
    np.savez(sys.argv[2], plans=json.dumps(plans), **outs)
