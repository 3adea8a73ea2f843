"""ctypes binding of libonmf_b200.so (the C ABI declared in include/onmf_b200.h).

There is no CPU fallback: importing the kernels without the built library raises, and every
wrapper raises `OnmfKernelError` on a non-zero status.  PyTorch is used only as the owner of
device memory and streams (tensors are passed as raw `data_ptr()`s).
"""
from __future__ import annotations

import ctypes
import os

import torch

F32, F64 = 0, 1
_HERE = os.path.dirname(os.path.abspath(__file__))
# ONMF_B200_LIB: alternative build of the same library (kernel experiments); never a different implementation
LIB_PATH = os.environ.get("ONMF_B200_LIB") or os.path.join(_HERE, "libonmf_b200.so")


class OnmfKernelError(RuntimeError):
    pass


class LarsStats(ctypes.Structure):
    _fields_ = [(n, ctypes.c_ulonglong) for n in
                ("columns", "knots", "sum_active", "sum_active2", "drops", "overflow", "flagged",
                 "max_active")]


STATS_FIELDS = [f[0] for f in LarsStats._fields_]

_vp, _i, _i64, _dbl, _sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_double, ctypes.c_size_t
_u64 = ctypes.c_uint64

# name -> (restype, argtypes); must list every symbol include/onmf_b200.h declares
SIGNATURES = {
    "onmf_version": (_i, []),
    "onmf_last_error": (ctypes.c_char_p, []),
    "onmf_built_arch": (_i, []),
    "onmf_launch_count": (ctypes.c_longlong, []),
    "onmf_gather_patches": (_i, [_i, _vp, _i, _i, _i, _vp, _i64, _i, _vp, _i64, _vp]),
    "onmf_gather_rows": (_i, [_i, _vp, _i64, _i, _vp, _i64, _vp, _vp]),
    "onmf_transpose": (_i, [_i, _i, _vp, _i64, _i64, _vp, _vp]),
    "onmf_convert": (_i, [_i, _i, _vp, _i64, _vp, _vp]),
    "onmf_widen": (_i, [_i, _vp, _i64, _dbl, _vp, _vp, _vp]),
    "onmf_gram": (_i, [_i, _vp, _i, _i, _vp, _vp]),
    "onmf_gram_workspace": (_sz, [_i, _i, _i]),
    "onmf_gram_ws": (_i, [_i, _vp, _i, _i, _vp, _vp, _sz, _vp]),
    "onmf_set_option": (_i, [_i, _i]),
    "onmf_get_option": (_i, [_i, ctypes.POINTER(_i)]),
    "onmf_gram_f64_workspace": (_sz, [_i, _i]),
    "onmf_gram_f64": (_i, [_i, _vp, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "onmf_lasso_lars_g64": (_i, [_i, _vp, _vp, _i64, _i, _i, _dbl, _i, _vp, _vp, _sz, _vp, _i, _vp]),
    "onmf_cov": (_i, [_i, _vp, _i64, _i, _vp, _i, _vp, _vp]),
    "onmf_spectral_norm_workspace": (_sz, [_i64, _i]),
    "onmf_spectral_norm": (_i, [_i, _vp, _i64, _i, _vp, _vp, _sz, _vp]),
    "onmf_lasso_lars_workspace": (_sz, [_i, _i, _i64]),
    "onmf_lasso_lars": (_i, [_i, _vp, _vp, _i64, _i, _i, _dbl, _i, _vp, _vp, _sz, _vp, _vp]),
    "onmf_lasso_lars_ex": (_i, [_i, _vp, _vp, _i64, _i, _i, _dbl, _i, _vp, _vp, _sz, _vp, _i, _vp]),
    "onmf_surrogate_workspace": (_sz, [_i, _i64, _i, _i]),
    "onmf_surrogate_partial": (_i, [_i, _vp, _vp, _i64, _i, _i, _vp, _vp, _sz, _vp]),
    "onmf_surrogate_blend": (_i, [_i, _vp, _i, _i, _dbl, _vp, _vp, _vp]),
    "onmf_surrogate_blend_dev": (_i, [_i, _vp, _i, _i, _vp, _vp, _vp, _vp]),
    "onmf_xxt_partial": (_i, [_i, _vp, _i64, _i, _vp, _vp, _sz, _vp]),
    "onmf_axpby": (_i, [_i, _i64, _dbl, _vp, _dbl, _vp, _vp]),
    "onmf_tc_supported": (_i, [_i, _i]),
    "onmf_split_tf32": (_i, [_vp, _vp, _vp, _i64, _vp]),
    "onmf_gather_rows_split": (_i, [_vp, _i64, _i, _vp, _i64, _vp, _vp, _vp]),
    "onmf_cov_tc": (_i, [_vp, _vp, _i64, _i, _vp, _vp, _i, _vp, _vp]),
    "onmf_surrogate_tc_workspace": (_sz, [_i64, _i, _i]),
    "onmf_surrogate_partial_tc": (_i, [_vp, _vp, _vp, _vp, _i64, _i, _i, _vp, _vp, _sz, _vp]),
    "onmf_fused_tc_supported": (_i, [_i, _i]),
    "onmf_cov_fused_tc": (_i, [_i, _vp, _i64, _i64, _vp, _i64, _i, _dbl, _vp, _vp, _i, _vp, _vp]),
    "onmf_surrogate_fused_tc_workspace": (_sz, [_i64, _i, _i]),
    "onmf_surrogate_fused_tc": (_i, [_vp, _i, _vp, _i64, _i64, _vp, _i64, _i, _i, _dbl, _vp, _i, _dbl, _vp, _vp, _vp, _vp, _sz, _vp]),
    "onmf_update_dict": (_i, [_i, _vp, _vp, _vp, _i, _i, _vp, _vp]),
    "onmf_update_dict_workspace": (_sz, [_i, _i, _i]),
    "onmf_update_dict_ws": (_i, [_i, _vp, _vp, _vp, _i, _i, _vp, _vp, _sz, _vp]),
    "onmf_update_dict_plan": (_i, [_i, _i, _i, _vp]),
    "onmf_pgd_sweep": (_i, [_i, _vp, _vp, _i64, _i, _dbl, _i, _vp, _vp]),
    "onmf_pgd_sweep_rows": (_i, [_i, _vp, _vp, _i64, _i, _dbl, _i, _vp, _i, _i, _vp]),
    "onmf_surrogate_error": (_i, [_i, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp]),
    "onmf_pgd_code_columns": (_i, [_i, _vp, _vp, _i64, _i, _dbl, _i, _dbl, _vp, _vp]),
    "onmf_patch_grid_mean": (_i, [_i, _vp, _i64, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "onmf_patch_grid_accumulate": (_i, [_i, _vp, _i64, _i, _i, _i, _i, _i, _i, _i, _i64, _i64, _vp, _vp, _vp]),
    "onmf_motif_patches": (_i, [_i, _vp, _vp, _i, _vp, _i64, _i, _vp, _vp]),
    "onmf_edge_scatter_add": (_i, [_i, _vp, _i64, _vp, _i64, _i, _vp, _vp, _vp, _i64, _vp, _vp]),
    "onmf_motif_chain_init": (_i, [_vp, _vp, _i64, _i, _i64, _i64, _u64, _vp, _vp]),
    "onmf_motif_chain": (_i, [_vp, _vp, _i64, _i, _i64, _i64, _u64, _u64, _i64, _i64, _vp, _vp, _vp]),
    "onmf_ising_chain_init": (_i, [_i, _i, _i64, _i64, _u64, _vp, _vp]),
    "onmf_ising_chain": (_i, [_i, _i, _i64, _i64, _u64, _dbl, _u64, _i64, _i64, _vp, _vp, _i, _vp]),
    "onmf_ising_thresholds": (_i, [_dbl, ctypes.POINTER(ctypes.c_uint32)]),
    "onmf_ising_chain_plan": (_i, [_i, _i, _vp]),
    "onmf_step_plan_create": (_i, [ctypes.POINTER(_vp), _i]),
    "onmf_step_plan_destroy": (_i, [_vp]),
    "onmf_step_plan_mark_state": (_i, [_vp, _vp]),
    "onmf_step_plan_launches": (ctypes.c_longlong, [_vp]),
    "onmf_step_plan_reset_timing": (_i, [_vp]),
    "onmf_step_plan_lars_ms": (_i, [_vp, ctypes.POINTER(ctypes.c_float), _i, ctypes.POINTER(_i)]),
    "onmf_step_launch": (_i, [_vp, _vp, _vp, _vp, _i64, _i]),
    "onmf_step_finish": (_i, [_vp, _vp, _dbl, _i]),
    "onmf_step": (_i, [_vp, _vp, _vp, _vp, _i64, _dbl, _i]),
    "onmf_step_graph": (_i, [_vp, _vp, _vp, _vp, _i64, _dbl, _i]),
    "onmf_step_plan_graph_steps": (ctypes.c_longlong, [_vp]),
    "onmf_step_launch_mb": (_i, [_vp, _vp, _vp, _vp, _i]),
    "onmf_step_mb": (_i, [_vp, _vp, _vp, _vp, _dbl, _i]),
    "onmf_step_graph_mb": (_i, [_vp, _vp, _vp, _vp, _dbl, _i]),
    "onmf_gather_patches_mb": (_i, [_vp, _i, _vp, _i64, _vp]),
    "onmf_cov_fused_tc_patches": (_i, [_vp, _vp, _vp, _i, _vp, _vp]),
    "onmf_surrogate_fused_tc_patches": (_i, [_vp, _vp, _i, _vp, _i, _dbl, _vp, _vp, _vp, _vp, _sz, _vp]),
    "onmf_step_launch_patches": (_i, [_vp, _vp, _vp, _vp, _i]),
    "onmf_step_patches": (_i, [_vp, _vp, _vp, _vp, _dbl, _i]),
    "onmf_step_graph_patches": (_i, [_vp, _vp, _vp, _vp, _dbl, _i]),
}



class StepBuffers(ctypes.Structure):
    """onmf_step_buffers (include/onmf_b200.h)."""
    _fields_ = [("dtype", _i), ("d", _i), ("k", _i), ("use_tc", _i), ("track_C", _i), ("max_iter", _i),
                ("reserve_sms", _i), ("hold_coder", _i), ("alpha", _dbl),
                ("W", _vp * 2), ("G", _vp * 2), ("Whi", _vp * 2), ("Wlo", _vp * 2),
                ("A", _vp), ("B", _vp), ("C", _vp), ("P", _vp * 2), ("P2", _vp),
                ("Ct", _vp), ("Ht", _vp), ("Xhi", _vp), ("Xlo", _vp), ("Hhi", _vp), ("Hlo", _vp),
                ("ws_lars", _vp), ("ws_lars_bytes", _sz), ("ws_sur", _vp), ("ws_sur_bytes", _sz),
                ("ws_gram", _vp), ("ws_gram_bytes", _sz), ("stats", _vp), ("main_stream", _vp), ("side_stream", _vp),
                ("w_dev", _vp)]


class Minibatch(ctypes.Structure):
    """onmf_minibatch (include/onmf_b200.h): a minibatch by reference -- rows idx[0..n) of a stored pool."""
    _fields_ = [("kind", _i), ("base", _vp), ("n_pool", _i64), ("ld", _i64), ("idx", _vp), ("n", _i64), ("scale", _dbl)]


def make_minibatch(pool, idx, n, scale=1.0):
    _req(pool, "pool")
    if idx is not None:
        _req(idx, "idx", torch.int64)
    mb = Minibatch()
    mb.kind = _store_kind(pool)
    mb.base = pool.data_ptr()
    mb.n_pool, mb.ld = pool.shape[0], pool.stride(0)
    mb.idx = idx.data_ptr() if idx is not None else None
    mb.n = int(n)
    mb.scale = float(scale)
    return mb


class PatchMinibatch(ctypes.Structure):
    """onmf_patch_minibatch (include/onmf_b200.h): the patches at corners coords[idx[0..n)] of a resident image."""
    _fields_ = [("img", _vp), ("kind", _i), ("H", _i), ("W", _i), ("C", _i), ("p", _i), ("coords", _vp), ("n_coords", _i64),
                ("idx", _vp), ("n", _i64), ("scale", _dbl)]


def make_patch_minibatch(img, p, coords, idx, n, scale=1.0):
    """img (H x W) or (H x W x C) float32 / float64 / uint8, coords (N x 2) int32, idx int64 (n) or None (0..n-1)"""
    _req(img, "img"); _req(coords, "coords", torch.int32)
    if idx is not None:
        _req(idx, "idx", torch.int64)
    if img.dim() not in (2, 3) or coords.dim() != 2 or coords.shape[1] != 2:
        raise OnmfKernelError("img must be (H x W [x C]) and coords (N x 2)")
    pm = PatchMinibatch()
    pm.img = img.data_ptr()
    pm.kind = F64 if img.dtype == torch.float64 else _store_kind(img)
    pm.H, pm.W = img.shape[0], img.shape[1]
    pm.C = img.shape[2] if img.dim() == 3 else 1
    pm.p = int(p)
    pm.coords = coords.data_ptr()
    pm.n_coords = coords.shape[0]
    pm.idx = idx.data_ptr() if idx is not None else None
    pm.n = int(n)
    pm.scale = float(scale)
    return pm


_lib = None


def load():
    """Load libonmf_b200.so (built in-tree by `make` / `__graft_entry__.build()`)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise OnmfKernelError(
            "libonmf_b200.so is not built (%s). Run `make` or `python -c 'import __graft_entry__ as g; "
            "g.build()'` at the repo root; there is no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)      # AttributeError if a declared symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _check(rc, what):
    if rc != 0:
        msg = load().onmf_last_error().decode(errors="replace")
        raise OnmfKernelError("%s failed (status %d): %s" % (what, rc, msg))


def dt(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.float64:
        return F64
    raise OnmfKernelError("unsupported dtype %s (float32 / float64 only)" % t.dtype)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream(stream=None):
    s = stream if stream is not None else torch.cuda.current_stream()
    return ctypes.c_void_p(s.cuda_stream)


def _req(t, name, dtype=None):
    if not t.is_cuda:
        raise OnmfKernelError("%s must be a CUDA tensor (no CPU path)" % name)
    if not t.is_contiguous():
        raise OnmfKernelError("%s must be contiguous" % name)
    if dtype is not None and t.dtype != dtype:
        raise OnmfKernelError("%s must have dtype %s" % (name, dtype))


# ---- thin wrappers (shapes documented in include/onmf_b200.h) --------------------------------

def gather_patches(img, coords, p, out, stream=None):
    _req(img, "img"); _req(coords, "coords", torch.int32)
    if not out.is_cuda or out.dtype != img.dtype or out.dim() != 2 or (out.shape[0] > 1 and out.stride(1) != 1):
        raise OnmfKernelError("out must be a CUDA (n x d) tensor of the image's dtype with unit column stride (rows may be pitched)")
    H, Wd = img.shape[0], img.shape[1]
    C = img.shape[2] if img.dim() == 3 else 1
    n = coords.shape[0]
    _check(load().onmf_gather_patches(dt(img), _ptr(img), H, Wd, C, _ptr(coords), n, p, _ptr(out),
                                      out.stride(0) if n else p * p * C, _stream(stream)), "onmf_gather_patches")
    return out


def gather_rows(pool, idx, out, stream=None):
    _req(pool, "pool"); _req(idx, "idx", torch.int64); _req(out, "out", pool.dtype)
    if idx.shape[0] == 0:
        return out
    _check(load().onmf_gather_rows(dt(pool), _ptr(pool), pool.shape[0], pool.shape[1], _ptr(idx), idx.shape[0],
                                   _ptr(out), _stream(stream)), "onmf_gather_rows")
    return out


def transpose(src, out, stream=None):
    _req(src, "src"); _req(out, "out")
    rows, cols = src.shape
    _check(load().onmf_transpose(dt(src), dt(out), _ptr(src), rows, cols, _ptr(out), _stream(stream)), "onmf_transpose")
    return out


STORE_U8, STORE_F16 = 2, 3


def convert(src, dst, stream=None):
    """elementwise f32 <-> f64"""
    _req(src, "src"); _req(dst, "dst")
    _check(load().onmf_convert(dt(src), dt(dst), _ptr(src), src.numel(), _ptr(dst), _stream(stream)), "onmf_convert")
    return dst


def widen(src, scale, dst, lo=None, stream=None):
    """dst (float32) = float(src) * scale for a uint8 / float16 device tensor; with lo: the TF32 (hi, lo) pair."""
    _req(src, "src"); _req(dst, "dst", torch.float32)
    if lo is not None:
        _req(lo, "lo", torch.float32)
    if src.dtype == torch.uint8:
        kind = STORE_U8
    elif src.dtype == torch.float16:
        kind = STORE_F16
    else:
        raise OnmfKernelError("widen: source must be uint8 or float16")
    _check(load().onmf_widen(kind, _ptr(src), src.numel(), float(scale), _ptr(dst), _ptr(lo), _stream(stream)), "onmf_widen")
    return dst


OPT_LARS_RESERVED_SMS = 1
OPT_LARS_FAST_TIER = 2
MAX_COMPONENTS = 512          # largest n_components the LARS coder is instantiated for (csrc/lars.cu k_class)


def set_option(key, value):
    _check(load().onmf_set_option(int(key), int(value)), "onmf_set_option")


def launch_count():
    """kernels launched so far by this host thread through the library (graph replays count their kernel nodes)"""
    return int(load().onmf_launch_count())


def get_option(key):
    v = _i(0)
    _check(load().onmf_get_option(int(key), ctypes.byref(v)), "onmf_get_option")
    return int(v.value)


def gram_workspace(dtype, d, k):
    return int(load().onmf_gram_workspace(F64 if dtype == torch.float64 else F32, d, k))


def gram(W, G, stream=None, workspace=None):
    _req(W, "W"); _req(G, "G", W.dtype)
    d, k = W.shape
    if workspace is not None:
        _req(workspace, "workspace", torch.uint8)
        _check(load().onmf_gram_ws(dt(W), _ptr(W), d, k, _ptr(G), _ptr(workspace), workspace.numel(), _stream(stream)),
               "onmf_gram_ws")
    else:
        _check(load().onmf_gram(dt(W), _ptr(W), d, k, _ptr(G), _stream(stream)), "onmf_gram")
    return G


def gram_f64_workspace(d, k):
    return int(load().onmf_gram_f64_workspace(d, k))


def gram_f64(W, G64, workspace, G32=None, stream=None):
    """G64 (k x k, float64) = W^T W accumulated in FP64 from a float32 / float64 W; optional float32 copy."""
    _req(W, "W"); _req(G64, "G64", torch.float64); _req(workspace, "workspace", torch.uint8)
    if G32 is not None:
        _req(G32, "G32", torch.float32)
    d, k = W.shape
    _check(load().onmf_gram_f64(dt(W), _ptr(W), d, k, _ptr(G64), _ptr(G32), _ptr(workspace), workspace.numel(),
                                _stream(stream)), "onmf_gram_f64")
    return G64


def spectral_norm_workspace(n, k):
    return int(load().onmf_spectral_norm_workspace(int(n), int(k)))


def spectral_norm(M, out, workspace, stream=None):
    """out (one device float64) = largest singular value of the sample-major matrix M (n x k)"""
    _req(M, "M"); _req(out, "out", torch.float64); _req(workspace, "workspace", torch.uint8)
    n, k = M.shape
    _check(load().onmf_spectral_norm(dt(M), _ptr(M), n, k, _ptr(out), _ptr(workspace), workspace.numel(), _stream(stream)),
           "onmf_spectral_norm")
    return out


def cov(Xt, W, Ct, stream=None):
    _req(Xt, "Xt"); _req(W, "W", Xt.dtype); _req(Ct, "Ct", Xt.dtype)
    n, d = Xt.shape
    _check(load().onmf_cov(dt(Xt), _ptr(Xt), n, d, _ptr(W), W.shape[1], _ptr(Ct), _stream(stream)), "onmf_cov")
    return Ct


def lasso_lars_workspace(dtype, k, n):
    return int(load().onmf_lasso_lars_workspace(F64 if dtype == torch.float64 else F32, k, n))


def lasso_lars(G, Ct, d, alpha, Ht, workspace, max_iter=1000, stats=None, stream=None, first_tier=-1):
    """G may be in the working precision of Ct / Ht, or float64 next to float32 covariances (the production path)."""
    _req(G, "G"); _req(Ct, "Ct"); _req(Ht, "Ht", Ct.dtype); _req(workspace, "workspace", torch.uint8)
    n, k = Ct.shape
    if G.dtype != Ct.dtype:
        _req(G, "G", torch.float64)
        _check(load().onmf_lasso_lars_g64(dt(Ct), _ptr(G), _ptr(Ct), n, k, d, float(alpha), int(max_iter), _ptr(Ht),
                                          _ptr(workspace), workspace.numel(), _ptr(stats), int(first_tier), _stream(stream)),
               "onmf_lasso_lars_g64")
        return Ht
    _check(load().onmf_lasso_lars_ex(dt(G), _ptr(G), _ptr(Ct), n, k, d, float(alpha), int(max_iter), _ptr(Ht),
                                     _ptr(workspace), workspace.numel(), _ptr(stats), int(first_tier), _stream(stream)),
           "onmf_lasso_lars")
    return Ht


def surrogate_workspace(dtype, n, k, d):
    return int(load().onmf_surrogate_workspace(F64 if dtype == torch.float64 else F32, n, k, d))


def surrogate_partial(Ht, Xt, P, workspace, stream=None):
    _req(Ht, "Ht"); _req(Xt, "Xt", Ht.dtype); _req(P, "P", Ht.dtype); _req(workspace, "workspace", torch.uint8)
    n, k = Ht.shape
    d = Xt.shape[1]
    _check(load().onmf_surrogate_partial(dt(Ht), _ptr(Ht), _ptr(Xt), n, k, d, _ptr(P), _ptr(workspace),
                                         workspace.numel(), _stream(stream)), "onmf_surrogate_partial")
    return P


def surrogate_blend(P, w, A, B, stream=None):
    _req(P, "P"); _req(A, "A", P.dtype); _req(B, "B", P.dtype)
    k, d = B.shape
    _check(load().onmf_surrogate_blend(dt(P), _ptr(P), k, d, float(w), _ptr(A), _ptr(B), _stream(stream)),
           "onmf_surrogate_blend")


def xxt_partial(Xt, P2, workspace, stream=None):
    _req(Xt, "Xt"); _req(P2, "P2", Xt.dtype)
    n, d = Xt.shape
    _check(load().onmf_xxt_partial(dt(Xt), _ptr(Xt), n, d, _ptr(P2), _ptr(workspace),
                                   workspace.numel() if workspace is not None else 0, _stream(stream)), "onmf_xxt_partial")
    return P2


def axpby(a, x, b, y, stream=None):
    _req(x, "x"); _req(y, "y", x.dtype)
    _check(load().onmf_axpby(dt(x), x.numel(), float(a), _ptr(x), float(b), _ptr(y), _stream(stream)), "onmf_axpby")


def update_dict_workspace(dtype, d, k):
    return int(load().onmf_update_dict_workspace(F64 if dtype == torch.float64 else F32, d, k))


class BcdPlan(ctypes.Structure):
    """onmf_bcd_plan (include/onmf_b200.h): the kernel and launch shape of the dictionary update for one (dtype, d, k)."""
    _fields_ = [("kind", _i), ("ctas", _i), ("rows_per_cta", _i), ("tpr", _i), ("ks", _i), ("threads", _i), ("regw", _i),
                ("mbar", _i), ("smem", _sz)]


BCD_KINDS = ("small", "cluster", "grid")


def update_dict_plan(dtype, d, k):
    """what onmf_update_dict launches for this shape, as a dict (kind: "small" / "cluster" / "grid"); host only"""
    p = BcdPlan()
    _check(load().onmf_update_dict_plan(F64 if dtype == torch.float64 else F32, int(d), int(k), ctypes.byref(p)),
           "onmf_update_dict_plan")
    out = {f: int(getattr(p, f)) for f, _ in BcdPlan._fields_}
    out["kind"] = BCD_KINDS[p.kind]
    return out


def update_dict(W, A, B, W_out, stream=None, workspace=None):
    _req(W, "W"); _req(A, "A", W.dtype); _req(B, "B", W.dtype); _req(W_out, "W_out", W.dtype)
    d, k = W.shape
    if workspace is None:
        nb = update_dict_workspace(W.dtype, d, k)
        if nb:          # large dictionaries only: the cooperative-grid fallback exchanges column norms through this scratch
            workspace = torch.empty(nb, dtype=torch.uint8, device=W.device)
    _check(load().onmf_update_dict_ws(dt(W), _ptr(W), _ptr(A), _ptr(B), d, k, _ptr(W_out), _ptr(workspace),
                                      workspace.numel() if workspace is not None else 0, _stream(stream)), "onmf_update_dict")
    return W_out


def surrogate_error(W, G64, A, B, C, out3, stream=None):
    """out3 (3 float64 on the device) = [tr(W A W^T), tr(W B), tr(C)]."""
    _req(W, "W"); _req(G64, "G64", torch.float64); _req(A, "A", W.dtype); _req(B, "B", W.dtype)
    _req(out3, "out3", torch.float64)
    if C is not None:
        _req(C, "C", W.dtype)
    d, k = W.shape
    _check(load().onmf_surrogate_error(dt(W), _ptr(W), _ptr(G64), _ptr(A), _ptr(B), _ptr(C), d, k, _ptr(out3),
                                       _stream(stream)), "onmf_surrogate_error")
    return out3


def pgd_sweep_rows(G, Ct, alpha, it, Ht, q_begin, q_end, stream=None):
    _req(G, "G"); _req(Ct, "Ct", G.dtype); _req(Ht, "Ht", G.dtype)
    n, k = Ct.shape
    _check(load().onmf_pgd_sweep_rows(dt(G), _ptr(G), _ptr(Ct), n, k, float(alpha), int(it), _ptr(Ht), int(q_begin),
                                      int(q_end), _stream(stream)), "onmf_pgd_sweep_rows")
    return Ht


def pgd_sweep(G, Ct, alpha, it, Ht, stream=None):
    _req(G, "G"); _req(Ct, "Ct", G.dtype); _req(Ht, "Ht", G.dtype)
    n, k = Ct.shape
    _check(load().onmf_pgd_sweep(dt(G), _ptr(G), _ptr(Ct), n, k, float(alpha), int(it), _ptr(Ht), _stream(stream)),
           "onmf_pgd_sweep")
    return Ht


# ---- tensor-core (3xTF32) path ---------------------------------------------------------------

def tc_supported(k, d):
    return bool(load().onmf_tc_supported(int(k), int(d)))


def split_tf32(src, hi, lo, stream=None):
    _req(src, "src", torch.float32); _req(hi, "hi", torch.float32); _req(lo, "lo", torch.float32)
    _check(load().onmf_split_tf32(_ptr(src), _ptr(hi), _ptr(lo), src.numel(), _stream(stream)), "onmf_split_tf32")


def gather_rows_split(pool, idx, hi, lo, stream=None):
    _req(pool, "pool", torch.float32); _req(idx, "idx", torch.int64); _req(hi, "hi", torch.float32); _req(lo, "lo", torch.float32)
    if idx.shape[0] == 0:
        return
    _check(load().onmf_gather_rows_split(_ptr(pool), pool.shape[0], pool.shape[1], _ptr(idx), idx.shape[0], _ptr(hi), _ptr(lo),
                                         _stream(stream)), "onmf_gather_rows_split")


def cov_tc(Xhi, Xlo, Whi, Wlo, Ct, stream=None):
    for t, nm in ((Xhi, "Xhi"), (Xlo, "Xlo"), (Whi, "Whi"), (Wlo, "Wlo"), (Ct, "Ct")):
        _req(t, nm, torch.float32)
    n, d = Xhi.shape
    _check(load().onmf_cov_tc(_ptr(Xhi), _ptr(Xlo), n, d, _ptr(Whi), _ptr(Wlo), Whi.shape[1], _ptr(Ct), _stream(stream)), "onmf_cov_tc")
    return Ct


def surrogate_tc_workspace(n, k, d):
    return int(load().onmf_surrogate_tc_workspace(n, k, d))


def surrogate_partial_tc(Hhi, Hlo, Xhi, Xlo, P, workspace, stream=None):
    for t, nm in ((Hhi, "Hhi"), (Hlo, "Hlo"), (Xhi, "Xhi"), (Xlo, "Xlo"), (P, "P")):
        _req(t, nm, torch.float32)
    _req(workspace, "workspace", torch.uint8)
    n, k = Hhi.shape
    d = Xhi.shape[1]
    _check(load().onmf_surrogate_partial_tc(_ptr(Hhi), _ptr(Hlo), _ptr(Xhi), _ptr(Xlo), n, k, d, _ptr(P), _ptr(workspace),
                                            workspace.numel(), _stream(stream)), "onmf_surrogate_partial_tc")
    return P


# ---- fused tensor-core path (csrc/gemm_fused.cu): minibatch read once, as stored ---------------------

def fused_tc_supported(k, d):
    return bool(load().onmf_fused_tc_supported(int(k), int(d)))


def _store_kind(t):
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.uint8:
        return STORE_U8
    if t.dtype == torch.float16:
        return STORE_F16
    raise OnmfKernelError("minibatch storage must be float32, uint8 or float16 (got %s)" % t.dtype)


def cov_fused_tc(pool, idx, n, Whi, Wlo, Ct, scale=1.0, stream=None):
    """Ct (n x k) = pool[idx] @ W; pool (n_pool x d) float32 / uint8 / float16, idx int64 (n) or None (rows 0..n-1)."""
    _req(pool, "pool"); _req(Whi, "Whi", torch.float32); _req(Wlo, "Wlo", torch.float32); _req(Ct, "Ct", torch.float32)
    if idx is not None:
        _req(idx, "idx", torch.int64)
    d, k = Whi.shape
    _check(load().onmf_cov_fused_tc(_store_kind(pool), _ptr(pool), pool.shape[0], pool.stride(0), _ptr(idx), int(n), d,
                                    float(scale), _ptr(Whi), _ptr(Wlo), k, _ptr(Ct), _stream(stream)), "onmf_cov_fused_tc")
    return Ct


def surrogate_fused_tc_workspace(n, k, d):
    return int(load().onmf_surrogate_fused_tc_workspace(int(n), int(k), int(d)))


def surrogate_fused_tc(Ht, pool, idx, n, d, P, workspace, scale=1.0, blend=None, stream=None):
    """P (k x (k+d)) = [Ht^T Ht | Ht^T pool[idx]]; blend = (w or a device float64 tensor, A, B) also applies the A/B recursion."""
    _req(Ht, "Ht", torch.float32); _req(pool, "pool"); _req(workspace, "workspace", torch.uint8)
    if P is not None:
        _req(P, "P", torch.float32)
    if idx is not None:
        _req(idx, "idx", torch.int64)
    k = Ht.shape[1]
    w, w_dev, A, B = 0.0, None, None, None
    if blend is not None:
        wv, A, B = blend
        _req(A, "A", torch.float32); _req(B, "B", torch.float32)
        if isinstance(wv, torch.Tensor):
            _req(wv, "w_dev", torch.float64)
            w_dev = wv
        else:
            w = float(wv)
    _check(load().onmf_surrogate_fused_tc(_ptr(Ht), _store_kind(pool), _ptr(pool), pool.shape[0], pool.stride(0), _ptr(idx), int(n),
                                          k, int(d), float(scale), _ptr(P), 1 if blend is not None else 0, w, _ptr(w_dev),
                                          _ptr(A), _ptr(B), _ptr(workspace), workspace.numel(), _stream(stream)),
           "onmf_surrogate_fused_tc")
    return P


def gather_patches_mb(pm, out, stream=None):
    """out (n x d, float32 / float64, rows may be pitched) = the patches of a PatchMinibatch, widening uint8 to float32"""
    if not out.is_cuda or out.dim() != 2 or (out.shape[0] > 1 and out.stride(1) != 1):
        raise OnmfKernelError("out must be a CUDA (n x d) tensor with unit column stride")
    _check(load().onmf_gather_patches_mb(ctypes.byref(pm), dt(out), _ptr(out), out.stride(0) if out.shape[0] else out.shape[1],
                                         _stream(stream)), "onmf_gather_patches_mb")
    return out


def cov_fused_tc_patches(pm, Whi, Wlo, Ct, stream=None):
    """Ct (n x k) = (patch minibatch) @ W on the fused tensor-core path"""
    _req(Whi, "Whi", torch.float32); _req(Wlo, "Wlo", torch.float32); _req(Ct, "Ct", torch.float32)
    _check(load().onmf_cov_fused_tc_patches(ctypes.byref(pm), _ptr(Whi), _ptr(Wlo), Whi.shape[1], _ptr(Ct), _stream(stream)),
           "onmf_cov_fused_tc_patches")
    return Ct


def surrogate_fused_tc_patches(Ht, pm, P, workspace, blend=None, stream=None):
    """P (k x (k+d)) = [Ht^T Ht | Ht^T X] for a patch minibatch X; blend = (w or a device float64 tensor, A, B)"""
    _req(Ht, "Ht", torch.float32); _req(workspace, "workspace", torch.uint8)
    if P is not None:
        _req(P, "P", torch.float32)
    w, w_dev, A, B = 0.0, None, None, None
    if blend is not None:
        wv, A, B = blend
        _req(A, "A", torch.float32); _req(B, "B", torch.float32)
        if isinstance(wv, torch.Tensor):
            _req(wv, "w_dev", torch.float64)
            w_dev = wv
        else:
            w = float(wv)
    _check(load().onmf_surrogate_fused_tc_patches(_ptr(Ht), ctypes.byref(pm), Ht.shape[1], _ptr(P), 1 if blend is not None else 0, w,
                                                  _ptr(w_dev), _ptr(A), _ptr(B), _ptr(workspace), workspace.numel(), _stream(stream)),
           "onmf_surrogate_fused_tc_patches")
    return P


# ---- batched reconstruction ---------------------------------------------------------------------

def pgd_code_columns(G, Ct, alpha, sub_iter, stopping_diff, Ht, stream=None):
    _req(G, "G"); _req(Ct, "Ct", G.dtype); _req(Ht, "Ht", G.dtype)
    n, k = Ct.shape
    _check(load().onmf_pgd_code_columns(dt(G), _ptr(G), _ptr(Ct), n, k, float(alpha), int(sub_iter), float(stopping_diff),
                                        _ptr(Ht), _stream(stream)), "onmf_pgd_code_columns")
    return Ht


def patch_grid_mean(R, ny, nx, p, stride, C, H, W, canvas, count=None, stream=None):
    _req(R, "R"); _req(canvas, "canvas", R.dtype)
    if count is not None:
        _req(count, "count", R.dtype)
    _check(load().onmf_patch_grid_mean(dt(R), _ptr(R), R.stride(0), ny, nx, p, stride, C, H, W, _ptr(canvas), _ptr(count),
                                       _stream(stream)), "onmf_patch_grid_mean")
    return canvas


def patch_grid_accumulate(R, j0, j1, ny, nx, p, stride, C, H, W, canvas, count=None, stream=None):
    """add grid patches j0 <= j < j1 (reconstructions R[j - j0]) to the overlap mean; consecutive ranges covering the grid,
    in order, give the bits of one patch_grid_mean call (include/onmf_b200.h)"""
    _req(R, "R"); _req(canvas, "canvas", R.dtype)
    if count is not None:
        _req(count, "count", R.dtype)
    _check(load().onmf_patch_grid_accumulate(dt(R), _ptr(R), R.stride(0), ny, nx, p, stride, C, H, W, int(j0), int(j1),
                                             _ptr(canvas), _ptr(count), _stream(stream)), "onmf_patch_grid_accumulate")
    return canvas


def coder_band_floor(device=None):
    """Fewest columns per band when a coder call is split into bands that must give the bits of one call.  The coders pick a
    kernel variant from the number of columns n, and the variants agree only to rounding: the LARS coder takes its
    one-column-per-warp fast tier for k <= 32 when n <= 24 x SMs and for k <= 64 when n <= 48 x SMs (csrc/lars.cu
    launch_class, FAST_SMALL_WARPS), onmf_pgd_code_columns one thread per sample for k <= 32 when n >= 16 x SMs
    (csrc/gather.cu).  Bands of more than 48 x SMs columns fall on the same side of all three as any larger call."""
    return 48 * torch.cuda.get_device_properties(device).multi_processor_count + 1


def motif_patches(rowptr, colidx, emb, out, stream=None):
    _req(rowptr, "rowptr", torch.int64); _req(colidx, "colidx", torch.int32); _req(emb, "emb", torch.int32); _req(out, "out")
    n, kk = emb.shape
    _check(load().onmf_motif_patches(dt(out), _ptr(rowptr), _ptr(colidx), rowptr.shape[0] - 1, _ptr(emb), n, kk, _ptr(out),
                                     _stream(stream)), "onmf_motif_patches")
    return out


def edge_scatter_add(R, emb, keys, sums, counts, failed, stream=None):
    _req(R, "R"); _req(emb, "emb", torch.int32); _req(keys, "keys", torch.int64); _req(sums, "sums", torch.float64)
    _req(counts, "counts", torch.int32); _req(failed, "failed", torch.int32)
    n, kk = emb.shape
    _check(load().onmf_edge_scatter_add(dt(R), _ptr(R), R.stride(0) if n else kk * kk, _ptr(emb), n, kk, _ptr(keys),
                                        _ptr(sums), _ptr(counts), keys.numel(), _ptr(failed), _stream(stream)),
           "onmf_edge_scatter_add")


def _csr_args(rowptr, colidx, state):
    _req(rowptr, "rowptr", torch.int64); _req(colidx, "colidx", torch.int32); _req(state, "state", torch.int32)
    if state.dim() != 2:
        raise OnmfKernelError("state must be (n_chains x kk)")
    return _ptr(rowptr), _ptr(colidx), rowptr.shape[0] - 1, state.shape[1], state.shape[0]


def motif_chain_init(rowptr, colidx, state, chain0, seed, stream=None):
    """state (n_chains x kk int32) <- the initial path homomorphisms of chains chain0 .. chain0 + n_chains - 1"""
    rp, ci, n_nodes, kk, n_chains = _csr_args(rowptr, colidx, state)
    _check(load().onmf_motif_chain_init(rp, ci, n_nodes, kk, n_chains, int(chain0), int(seed), _ptr(state), _stream(stream)),
           "onmf_motif_chain_init")
    return state


def motif_chain(rowptr, colidx, state, chain0, seed, step0, steps_per_sample, out, stream=None):
    """out (n_samples x n_chains x kk int32) <- the states after steps step0 + (s+1) * steps_per_sample; state advanced in place"""
    rp, ci, n_nodes, kk, n_chains = _csr_args(rowptr, colidx, state)
    _req(out, "out", torch.int32)
    if out.numel() % max(n_chains * kk, 1):
        raise OnmfKernelError("out must hold n_samples x n_chains x kk entries")
    _check(load().onmf_motif_chain(rp, ci, n_nodes, kk, n_chains, int(chain0), int(seed), int(step0),
                                   out.numel() // (n_chains * kk), int(steps_per_sample), _ptr(state), _ptr(out), _stream(stream)),
           "onmf_motif_chain")
    return out


def ising_thresholds(beta):
    """the heat-bath table thr[0..4] (list of ints) of onmf_ising_chain at inverse temperature beta; host only"""
    thr = (ctypes.c_uint32 * 5)()
    _check(load().onmf_ising_thresholds(float(beta), thr), "onmf_ising_thresholds")
    return [int(v) for v in thr]


class IsingPlan(ctypes.Structure):
    """onmf_ising_plan (include/onmf_b200.h): the form onmf_ising_chain uses for one lattice shape."""
    _fields_ = [("form", _i), ("threads", _i), ("smem", _sz)]


ISING_FORMS = ("smem", "global")


def ising_chain_plan(H, W):
    """what onmf_ising_chain launches for an H x W lattice, as a dict (form: "smem" / "global"); host only"""
    p = IsingPlan()
    _check(load().onmf_ising_chain_plan(int(H), int(W), ctypes.byref(p)), "onmf_ising_chain_plan")
    return dict(form=ISING_FORMS[p.form], threads=int(p.threads), smem=int(p.smem))


def _lattice_args(state):
    _req(state, "state", torch.int8)
    if state.dim() != 3:
        raise OnmfKernelError("state must be (n_chains x H x W)")
    return state.shape[0], state.shape[1], state.shape[2]


def ising_chain_init(state, chain0, seed, stream=None):
    """state (n_chains x H x W int8) <- the uniform +-1 initial lattices of chains chain0 .. chain0 + n_chains - 1"""
    C, H, W = _lattice_args(state)
    _check(load().onmf_ising_chain_init(H, W, C, int(chain0), int(seed), _ptr(state), _stream(stream)), "onmf_ising_chain_init")
    return state


def ising_chain(state, chain0, seed, beta, sweep0, sweeps_per_sample, out, stream=None):
    """out (n_samples x n_chains x H x W, float32 / float64) <- the lattices after sweeps sweep0 + (s+1) * sweeps_per_sample;
    state advanced in place"""
    C, H, W = _lattice_args(state)
    _req(out, "out")
    if out.numel() % max(C * H * W, 1):
        raise OnmfKernelError("out must hold n_samples x n_chains x H x W entries")
    _check(load().onmf_ising_chain(H, W, C, int(chain0), int(seed), float(beta), int(sweep0), out.numel() // (C * H * W),
                                   int(sweeps_per_sample), _ptr(state), _ptr(out), dt(out), _stream(stream)),
           "onmf_ising_chain")
    return out


# ---- fused step (csrc/step.cu) ---------------------------------------------------------------------

class StepPlan:
    """Owner of an onmf_step_plan (CUDA events ordering the two streams of the fused step)."""

    def __init__(self, timing_slots=0):
        self._h = _vp()
        _check(load().onmf_step_plan_create(ctypes.byref(self._h), int(timing_slots)), "onmf_step_plan_create")
        self.timing_slots = int(timing_slots)

    def __del__(self):
        try:
            if self._h:
                load().onmf_step_plan_destroy(self._h)
                self._h = _vp()
        except Exception:
            pass

    def mark_state(self, main_stream):
        _check(load().onmf_step_plan_mark_state(self._h, _stream(main_stream)), "onmf_step_plan_mark_state")

    def launches(self):
        return int(load().onmf_step_plan_launches(self._h))

    def reset_timing(self):
        _check(load().onmf_step_plan_reset_timing(self._h), "onmf_step_plan_reset_timing")

    def lars_ms(self):
        if self.timing_slots <= 0:
            return []
        buf = (ctypes.c_float * self.timing_slots)()
        n = _i(0)
        _check(load().onmf_step_plan_lars_ms(self._h, buf, self.timing_slots, ctypes.byref(n)), "onmf_step_plan_lars_ms")
        return [float(buf[i]) for i in range(n.value)]

    def launch(self, bufs, Xt, codes, n, cur):
        _check(load().onmf_step_launch(self._h, ctypes.byref(bufs), _ptr(Xt), _ptr(codes), int(n), int(cur)), "onmf_step_launch")

    def finish(self, bufs, w, cur):
        _check(load().onmf_step_finish(self._h, ctypes.byref(bufs), float(w), int(cur)), "onmf_step_finish")

    def step(self, bufs, Xt, codes, n, w, cur):
        _check(load().onmf_step(self._h, ctypes.byref(bufs), _ptr(Xt), _ptr(codes), int(n), float(w), int(cur)), "onmf_step")

    def step_graph(self, bufs, Xt, codes, n, w, cur):
        _check(load().onmf_step_graph(self._h, ctypes.byref(bufs), _ptr(Xt), _ptr(codes), int(n), float(w), int(cur)),
               "onmf_step_graph")

    def graph_steps(self):
        return int(load().onmf_step_plan_graph_steps(self._h))

    def launch_mb(self, bufs, mb, codes, cur):
        _check(load().onmf_step_launch_mb(self._h, ctypes.byref(bufs), ctypes.byref(mb), _ptr(codes), int(cur)), "onmf_step_launch_mb")

    def step_mb(self, bufs, mb, codes, w, cur, graph=False):
        fn = load().onmf_step_graph_mb if graph else load().onmf_step_mb
        _check(fn(self._h, ctypes.byref(bufs), ctypes.byref(mb), _ptr(codes), float(w), int(cur)), "onmf_step_mb")

    def launch_patches(self, bufs, pm, codes, cur):
        _check(load().onmf_step_launch_patches(self._h, ctypes.byref(bufs), ctypes.byref(pm), _ptr(codes), int(cur)),
               "onmf_step_launch_patches")

    def step_patches(self, bufs, pm, codes, w, cur, graph=False):
        fn = load().onmf_step_graph_patches if graph else load().onmf_step_patches
        _check(fn(self._h, ctypes.byref(bufs), ctypes.byref(pm), _ptr(codes), float(w), int(cur)), "onmf_step_patches")
