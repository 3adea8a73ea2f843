"""Online_NMF and update_code_within_radius -- drop-ins for the reference's src/onmf.py on B200.

The reference tree ships three mutually incompatible generations of this class (SURVEY.md §A.4); this
class accepts the union of their constructor arguments:

    Online_NMF(X, n_components=100, iterations=500, batch_size=20,
               ini_dict=None, ini_A=None, ini_B=None, ini_C=None,     # what ALL shipped drivers pass
               ini_agg=None,                                          # shipped src/onmf.py:28
               history=0, alpha=None, beta=None, subsample=False)
      .train_dict(full_code=False)
            -> (W, At, Bt, Ct, H)        driver style (image_reconstruction.py:298, ising_reconstruction.py:127,
                                         network_reconstruction_nx.py:364)   [default]
            -> (W, [A, B(, C)], code)    shipped style (src/onmf.py:226)     [when ini_agg is given or
                                                                              compat="shipped_onmf"]
      .sparse_code(X, W) -> H (r x n)    src/onmf.py:51-90
      .update_dict(W, A, B) -> W1        src/onmf.py:92-116
      .step(X, aggregates, W, t) -> (H1, aggregates1, W1)            src/onmf.py:119-167
      .history, .code

Default semantics are the `ontf.py` / paper recursion (aggregates accumulate across steps; sparse coding
is the positive lasso -- BASELINE.json north_star: "a batched nonnegative-lasso kernel replaces
sparse_code").  `compat="shipped_onmf"` reproduces the literal shipped file instead: random-H0
projected-gradient coder (src/onmf.py:87, :233-271) and the aggregate re-binding of src/onmf.py:217.

alpha=None follows the coder, as in the reference: every lasso_lars call site there uses transform_alpha=2 for None
(src/ontf.py:79-81 and the lasso variant kept as a string literal in src/onmf.py:71-80), the projected-gradient coder
uses 0 (src/onmf.py:82-84).  All shipped drivers pass alpha=None.

Extra keywords (not in the reference): precision ("fp32" | "fp64"), coder ("lasso_lars" | "pgd"),
compat (None | "shipped_onmf"), track_C (maintain the d x d aggregate C even without full_code),
process_group (data-parallel training over several GPUs, see Online_NTF; lasso_lars coder, subsample=True or False),
keep_code (False: no (r x N) `code` matrix is kept or copied back; the code slot of train_dict's result is None).

X may also be a patches.ImagePatches: the patches of one resident image by reference (lasso_lars coder only).  train_dict
then trains on the patches at the drawn indices without ever writing the (d x N) matrix out, with the same results, bit for
bit, and the same draws from the global RNG as on X = ImagePatches.to_matrix().  X may also be a patches.SamplePool: a data
matrix already on the device in the sample-major layout, trained on in place with the results of the host matrix.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _host, _lib
from .engine import OnmfEngine
from .patches import ImagePatches, SamplePool
from .parallel import default_group, shard_range

DEBUG = False


class Online_NMF():

    def __init__(self,
                 X,
                 n_components=100,
                 iterations=500,
                 batch_size=20,
                 ini_dict=None,
                 ini_A=None,
                 ini_B=None,
                 ini_C=None,
                 ini_agg=None,
                 history=0,
                 alpha=None,
                 beta=None,
                 subsample=False,
                 precision=None,
                 coder=None,
                 compat=None,
                 track_C=None,
                 process_group=None,
                 keep_code=True):
        self.X = X
        self.n_components = n_components
        self.batch_size = batch_size
        self.iterations = iterations
        self.subsample = subsample
        self.initial_dict = ini_dict
        self.initial_agg = ini_agg
        if ini_agg is None and (ini_A is not None or ini_B is not None):
            agg = [ini_A, ini_B]
            if ini_C is not None:
                agg.append(ini_C)
            self.initial_agg = agg
        self._shipped_return = (ini_agg is not None) or (compat == "shipped_onmf")
        self.history = history
        self.alpha = alpha
        self.beta = beta
        self.keep_code = bool(keep_code)
        self.code = np.zeros(shape=(n_components, X.shape[1])) if self.keep_code else None
        if compat not in (None, "shipped_onmf"):
            raise ValueError("compat must be None or 'shipped_onmf'")
        self.compat = compat
        self.coder = coder if coder is not None else ("pgd" if compat == "shipped_onmf" else "lasso_lars")
        if self.coder not in ("lasso_lars", "pgd"):
            raise ValueError("coder must be 'lasso_lars' or 'pgd'")
        if isinstance(X, ImagePatches):
            if self.coder != "lasso_lars" or compat is not None:
                raise ValueError("training on ImagePatches uses the lasso_lars coder with accumulating aggregates")
            if precision is None:
                precision = X.precision
            elif _host.torch_dtype(precision) != X.engine_dtype:
                raise ValueError("precision %r differs from the ImagePatches' %r" % (precision, X.precision))
        if isinstance(X, SamplePool):
            if precision is None:
                precision = X.precision
            elif _host.torch_dtype(precision) != X.Xt.dtype:
                raise ValueError("precision %r differs from the SamplePool's %r" % (precision, X.precision))
        self.precision = precision
        self._dtype = _host.torch_dtype(precision)
        self.track_C = track_C
        self.lars_stats = None
        self.process_group = process_group
        self._engines = {}

    def _alpha(self):
        if self.alpha is None:
            return 2 if self.coder == "lasso_lars" else 0     # src/ontf.py:79-81 (lasso) / src/onmf.py:82-84 (PGD)
        return self.alpha

    def _engine(self, d, r, track_C=False, group=None):
        """one engine per (d, r, track_C, group) kept on the object (drivers call sparse_code / step per patch or epoch)"""
        key = (int(d), int(r), bool(track_C), id(group) if group is not None else None)
        eng = self._engines.get(key)
        if eng is None or eng.alpha != float(self._alpha()) or eng.beta != (1.0 if self.beta is None else float(self.beta)):
            eng = OnmfEngine(d, r, alpha=self._alpha(), beta=self.beta, dtype=self._dtype, device=_host.device(),
                             track_C=track_C, collect_stats=True, process_group=group)
            self._engines[key] = eng
        eng.stats.zero_()
        return eng

    # -- coders ----------------------------------------------------------------------------------
    def _code_device(self, eng, Xt, Wd):
        """Ht (n x r) on device with the configured coder."""
        if self.coder == "lasso_lars":
            return eng.sparse_code(Xt, Wd, alpha=self._alpha())
        n, r = Xt.shape[0], Wd.shape[1]
        H0 = np.random.rand(r, n)                              # src/onmf.py:245-246 (global host RNG)
        Ht = _host.to_sample_major(H0, self._dtype, Xt.device)    # uploaded as drawn, transposed on the device
        return _pgd_device(Xt, Wd, Ht, self._alpha(), 10, 0.01)   # src/onmf.py:87

    def sparse_code(self, X, W):
        """H (r x n) for data X (d x n) and dictionary W (d x r)."""
        dev = _host.device()
        Xt = _host.to_sample_major(X, self._dtype, dev)
        Wd = _host.to_device(W, self._dtype, dev)
        eng = self._engine(Wd.shape[0], Wd.shape[1])
        Ht = self._code_device(eng, Xt, Wd)
        self.lars_stats = eng.read_stats()
        return _host.from_sample_major(Ht)

    def update_dict(self, W, A, B):
        dev = _host.device()
        Wd = _host.to_device(W, self._dtype, dev)
        out = torch.empty_like(Wd)
        _lib.update_dict(Wd, _host.to_device(A, self._dtype, dev), _host.to_device(B, self._dtype, dev), out)
        return _host.to_numpy(out)

    def step(self, X, aggregates, W, t):
        """src/onmf.py:119-167 on host arrays: returns (H1 (r x n), [A1, B1(, C1)], W1)."""
        dev = _host.device()
        d, r = np.shape(W)
        has_C = len(aggregates) == 3
        eng = self._engine(d, r, track_C=has_C)
        eng.set_state(W, aggregates[0], aggregates[1], aggregates[2] if has_C else None)
        Xt = _host.to_sample_major(X, self._dtype, dev)
        H1 = self._step_device(eng, Xt, float(t))
        Wd, Ad, Bd, Cd = eng.state()
        out = [_host.to_numpy(Ad), _host.to_numpy(Bd)]
        if has_C:
            out.append(_host.to_numpy(Cd))
        self.history = np.float64(t) + 1
        return _host.from_sample_major(H1), out, _host.to_numpy(Wd)

    def _step_device(self, eng, Xt, t):
        if self.coder == "lasso_lars":
            return eng.step(Xt, t)
        Ht = self._code_device(eng, Xt, eng.W)
        return eng.step(Xt, t, codes=Ht)

    def surrogate_error(self):
        """tr(W A W^T) - 2 tr(W B) + tr(C) of the state the last train_dict left on the device, read there (the surrogate loss
        the Ising and network drivers plot, ising_reconstruction.py:133,164; tr(C) is 0 when C was not tracked)"""
        if getattr(self, "_trained", None) is None:
            raise RuntimeError("surrogate_error() reads the state of train_dict(); call train_dict() first")
        return self._trained.surrogate_error()

    # -- training loop ---------------------------------------------------------------------------
    def train_dict(self, full_code=False):
        dev = _host.device()
        patches = isinstance(self.X, ImagePatches)
        resident = isinstance(self.X, SamplePool)
        X = self.X if patches or resident else np.asarray(self.X)
        d, n = X.shape
        r = self.n_components
        code = self.code
        agg0 = self.initial_agg
        want_C = bool(full_code) or (self.track_C if self.track_C is not None else not self._shipped_return) \
            or (agg0 is not None and len(agg0) == 3)

        if self.initial_dict is None:
            W = np.random.rand(d, r)                    # src/onmf.py:190
            A0 = B0 = C0 = None
        else:
            W = self.initial_dict
            A0 = agg0[0] if agg0 is not None else None
            B0 = agg0[1] if agg0 is not None else None
            C0 = agg0[2] if (agg0 is not None and len(agg0) == 3) else None
        t0 = self.history

        if resident:
            pool = X.Xt if X.Xt.device == dev else X.Xt.to(dev)                        # (n x d), already sample-major
        else:
            pool = None if patches else _host.to_sample_major(X, self._dtype, dev)    # (n x d)
        group, world, rank = default_group(self.process_group)
        if world > 1:
            if self.coder != "lasso_lars" or self.compat == "shipped_onmf":
                raise ValueError("multi-GPU training uses the lasso_lars coder with accumulating aggregates")
            W, A0, B0, _ = _host.broadcast_run_inputs(group, dev, d, r, W, A0, B0, None)
        eng = self._engine(d, r, track_C=want_C, group=group)
        eng.set_state(W, A0, B0, C0)
        shipped = self.compat == "shipped_onmf"
        if shipped:
            A_init, B_init = eng.A.clone(), eng.B.clone()
            C_init = eng.C.clone() if want_C else None
        m = self.batch_size if self.subsample else n
        lo, hi = shard_range(m, world, rank)
        Xb = torch.empty(hi - lo, d, dtype=self._dtype, device=dev) if self.subsample and not patches else None
        # lasso coder: nothing but the minibatch draw touches the global RNG inside the loop, so all steps' indices are
        # drawn up front (same stream as src/onmf.py:212 step by step) and uploaded once; the PGD coder interleaves its
        # H0 = np.random.rand(r, n) draws (src/onmf.py:245-246) and keeps the per-step order.
        idx_all = idx_dev = None
        if self.subsample and self.coder == "lasso_lars" and self.iterations > 1:
            idx_all = np.stack([np.random.randint(n, size=self.batch_size) for _ in range(int(self.iterations) - 1)])
            if world > 1:
                idx_all = _host.broadcast_indices(group, dev, idx_all)
            idx_dev = _host.upload_indices(idx_all[:, lo:hi], dev)
        # ImagePatches without subsampling: every column each step (this rank's range of them)
        cols = torch.arange(lo, hi, dtype=torch.int64, device=dev) if patches and not self.subsample and world > 1 else None
        for i in np.arange(1, self.iterations):
            idx = np.arange(n)
            if patches:
                # the patches at the drawn corners, read out of the image by the kernels (or gathered into the engine's buffer)
                if self.subsample:
                    idx = idx_all[i - 1]
                Ht = eng.step_patches(X, idx_dev[i - 1] if self.subsample else cols, float(t0 + i))
                self.history = np.float64(t0 + i) + 1
                if code is not None:
                    code[:, idx[lo:hi]] += _host.from_sample_major(Ht)
                continue
            if self.subsample:
                if idx_all is not None:
                    idx = idx_all[i - 1]
                    if self.coder == "lasso_lars" and not shipped:
                        # X_batch = X[:, idx] (src/onmf.py:213) by reference: the kernels read the pool rows in place
                        Ht = eng.step_pool(pool, idx_dev[i - 1], float(t0 + i))
                        self.history = np.float64(t0 + i) + 1
                        if code is not None:
                            code[:, idx[lo:hi]] += _host.from_sample_major(Ht)    # src/onmf.py:221 (this rank's columns)
                        continue
                    _lib.gather_rows(pool, idx_dev[i - 1], Xb)
                else:
                    idx = np.random.randint(n, size=self.batch_size)      # src/onmf.py:212
                    _lib.gather_rows(pool, _host.upload_indices(idx, dev), Xb)
                Xt = Xb
            else:
                Xt = pool[lo:hi]
            if shipped:
                # src/onmf.py:217 re-binds the aggregates to the arrays fixed before the loop.  reset_aggregates orders the
                # copies behind the previous step's blend AND the next dictionary update behind the copies.
                eng.reset_aggregates(A_init, B_init, C_init)
            Ht = self._step_device(eng, Xt, float(t0 + i))
            self.history = np.float64(t0 + i) + 1
            if code is not None:
                code[:, idx[lo:hi]] += _host.from_sample_major(Ht)    # src/onmf.py:221 (this rank's columns)
        Wd, Ad, Bd, Cd = eng.state()
        self.lars_stats = eng.read_stats()
        self._trained = eng
        Wn, An, Bn = _host.to_numpy(Wd), _host.to_numpy(Ad), _host.to_numpy(Bd)
        Cn = _host.to_numpy(Cd) if want_C else None
        if self._shipped_return:
            aggregates = [An, Bn]
            if Cn is not None and (full_code or (agg0 is not None and len(agg0) == 3)):
                aggregates.append(Cn)
            return Wn, aggregates, code
        return Wn, An, Bn, Cn, code


####################################
# custom sparsecoder

def _pgd_device(Xt, Wd, Ht, alpha, sub_iter, stopping_diff, r=None):
    """Outer loop of the reference's projected-gradient coder (src/onmf.py:252-268) around the onmf_pgd_sweep
    kernel.  The stopping test needs two spectral norms per outer iteration (np.linalg.norm(., 2),
    src/onmf.py:265): onmf_spectral_norm (FP64 Gram + largest eigenvalue by repeated squaring, csrc/gemm_simt.cu).

    Radius mode (r is not None, src/onmf.py:260-263): the reference projects H1 back to within spectral distance r of
    H0 after every row update and then executes `H0 = H1`, which ALIASES the two arrays -- from the second row on the
    in-place row updates change H0 as well, the distance is 0 and the projection is the identity.  So the projection
    acts exactly once: after row 0 of the first outer iteration, where H1 - H0 has a single non-zero row and its
    spectral norm is that row's 2-norm.  Reproduced literally (golden vector tests/golden/pgd_coder.npz:H_radius)."""
    k = Wd.shape[1]
    G = torch.empty(k, k, dtype=Wd.dtype, device=Wd.device)
    Ct = torch.empty(Xt.shape[0], k, dtype=Wd.dtype, device=Wd.device)
    _lib.gram(Wd, G)
    _lib.cov(Xt, Wd, Ct)
    i, dist = 0, 1.0
    n = Ht.shape[0]
    ws_n = torch.empty(_lib.spectral_norm_workspace(max(n, 1), k), dtype=torch.uint8, device=Wd.device)
    norms = torch.zeros(2, dtype=torch.float64, device=Wd.device)
    H_old = torch.empty_like(Ht)
    while i < sub_iter and dist > stopping_diff:
        H_old.copy_(Ht)
        if r is not None and i == 0:
            h_before = Ht[:, 0].clone()                          # row 0 of H = column 0 of the sample-major Ht
            _lib.pgd_sweep_rows(G, Ct, alpha, i, Ht, 0, 1)
            delta = Ht[:, 0] - h_before
            _lib.spectral_norm(delta.contiguous().view(-1, 1), norms[:1], ws_n)      # 2-norm of the one changed row
            dd = float(norms[0])
            Ht[:, 0] = h_before + (r / max(r, dd)) * delta
            _lib.pgd_sweep_rows(G, Ct, alpha, i, Ht, 1, k)
        else:
            _lib.pgd_sweep(G, Ct, alpha, i, Ht)
        if n > 0:
            _lib.spectral_norm(H_old, norms[1:], ws_n)
            _lib.axpby(1.0, Ht, -1.0, H_old)                     # H_old <- H1 - H1_old
            _lib.spectral_norm(H_old, norms[:1], ws_n)
            nn = norms.tolist()
            dist = nn[0] / nn[1] if nn[1] > 0 else float("inf") if nn[0] > 0 else float("nan")
        i += 1
    return Ht


def update_code_within_radius(X, W, H0=None, r=None, alpha=0, sub_iter=10, stopping_diff=0.1, precision=None):
    """Row-wise projected gradient descent for argmin_H |X - WH|^2/2 + alpha|H|_1, H >= 0
    (reference src/onmf.py:233-271).  Returns H (r x n) as numpy float64."""
    if r is not None and not (r > 0):
        raise ValueError("r must be positive (the reference divides by max(r, distance) and returns NaN for r = 0)")
    dev = _host.device()
    dtype = _host.torch_dtype(precision)
    X = np.asarray(X)
    W = np.asarray(W)
    if H0 is None:
        H0 = np.random.rand(W.shape[1], X.shape[1])              # src/onmf.py:245-246
    Xt = _host.to_sample_major(X, dtype, dev)
    Wd = _host.to_device(W, dtype, dev)
    Ht = _host.to_device(np.ascontiguousarray(np.asarray(H0).T), dtype, dev)
    Ht = _pgd_device(Xt, Wd, Ht, alpha, sub_iter, stopping_diff, r=r)
    return _host.from_sample_major(Ht)
