"""ctypes loader of oracle/liblars_oracle.so (the plain-C restatement in lars_oracle.c).
TEST INFRASTRUCTURE ONLY -- see the header of lars_oracle.c."""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "liblars_oracle.so")
_lib = None


def build():
    src = os.path.join(_HERE, "lars_oracle.c")
    if not os.path.isfile(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-o", _SO, src, "-lm"])
    return _SO


def load():
    global _lib
    if _lib is None:
        build()
        _lib = ctypes.CDLL(_SO)
        dp = ctypes.POINTER(ctypes.c_double)
        _lib.oracle_sparse_code.restype = ctypes.c_int
        _lib.oracle_sparse_code.argtypes = [dp, dp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double,
                                            ctypes.c_int, dp]
        _lib.oracle_update_dict.restype = None
        _lib.oracle_update_dict.argtypes = [dp, dp, dp, ctypes.c_int, ctypes.c_int]
        _lib.oracle_aggregate.restype = None
        _lib.oracle_aggregate.argtypes = [dp, dp, dp, dp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double]
        ip = ctypes.POINTER(ctypes.c_int)
        _lib.oracle_lars_positive.restype = ctypes.c_int
        _lib.oracle_lars_positive.argtypes = [dp, dp, ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_int, dp, ip, dp, ip,
                                              dp]
    return _lib


def _p(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))


def sparse_code(X, W, alpha, max_iter=1000):
    """H (k x n), positive lasso_lars codes (C restatement)."""
    X = np.ascontiguousarray(X, dtype=np.float64)
    W = np.ascontiguousarray(W, dtype=np.float64)
    d, n = X.shape
    k = W.shape[1]
    H = np.zeros((k, n))
    load().oracle_sparse_code(_p(X), _p(W), d, n, k, float(alpha), int(max_iter), _p(H))
    return H


def lars_columns(G, Ct, alpha, d, max_iter=1000):
    """Positive lasso_lars codes of the rows of Ct (n x k covariances W^T x) against the Gram G (k x k), one
    oracle_lars_positive path per row.  Returns H (n x k) and a dict of per-row arrays: n_iter (knots), max_active,
    drops (drop steps), status (bits 1 degenerate pivot, 2 "alpha increasing" bail-out, 4 max_iter), min_gap (the
    smallest relative gap between the joining covariance and the runner-up, or between a drop and the step it competes
    with: a near-tie) and min_pivot (the smallest pivot^2 / G_jj of an accepted join)."""
    G = np.ascontiguousarray(G, dtype=np.float64)
    Ct = np.ascontiguousarray(Ct, dtype=np.float64)
    n, k = Ct.shape
    lib = load()
    H = np.zeros((n, k))
    info = np.zeros((n, 4), dtype=np.int32)
    gaps = np.zeros((n, 2))
    gap = np.zeros(2)
    work = np.empty((k + 1) * (k + 1) + 6 * k)
    iwork = np.empty(2 * k, dtype=np.int32)
    one = np.zeros(3, dtype=np.int32)
    h = np.empty(k)
    ip = ctypes.POINTER(ctypes.c_int)
    for j in range(n):
        c = Ct[j]
        info[j, 3] = lib.oracle_lars_positive(_p(G), _p(c), k, int(d), float(alpha), int(max_iter), _p(h),
                                              one.ctypes.data_as(ip), _p(work), iwork.ctypes.data_as(ip), _p(gap))
        gaps[j] = gap
        info[j, :3] = one
        H[j] = h
    return H, dict(n_iter=info[:, 0].copy(), max_active=info[:, 1].copy(), drops=info[:, 2].copy(), status=info[:, 3].copy(),
                 min_gap=gaps[:, 0].copy(), min_pivot=gaps[:, 1].copy())


def update_dict(W, A, B):
    W1 = np.array(W, dtype=np.float64, order="C", copy=True)
    A = np.ascontiguousarray(A, dtype=np.float64)
    B = np.ascontiguousarray(B, dtype=np.float64)
    d, k = W1.shape
    load().oracle_update_dict(_p(W1), _p(A), _p(B), d, k)
    return W1


def step(X, A, B, W, t, alpha, beta=None):
    """reference src/ontf.py:117-154 with the C restatement: returns H (k x n), A1, B1, W1."""
    X = np.ascontiguousarray(X, dtype=np.float64)
    a = 2 if alpha is None else alpha
    H = sparse_code(X, W, a)
    w = float(t) ** (-(1.0 if beta is None else beta))
    A1 = np.array(A, dtype=np.float64, order="C", copy=True)
    B1 = np.array(B, dtype=np.float64, order="C", copy=True)
    d, n = X.shape
    load().oracle_aggregate(_p(A1), _p(B1), _p(H), _p(X), d, n, W.shape[1], w)
    W1 = update_dict(W, A, B)
    return H, A1, B1, W1
