"""Device-resident engine for the online NMF/NTF dictionary-learning step.

One `OnmfEngine` owns the replicated state (W, A, B[, C]) of one rank and runs, per minibatch,

    main stream :  G = W^T W ; Ct = Xt W ; Ht = lasso_lars(G, Ct) ; P = [Ht^T Ht | Ht^T Xt]
    side stream :  (all-reduce P of the PREVIOUS step) ; A,B <- (1-w) A,B + w P ; W' = BCD(W; A_prev, B_prev)

which is the reference's `step` (src/ontf.py:117-154): code with the current dictionary, update the
aggregates, and update the dictionary with the OLD aggregates (src/ontf.py:151).  That one-step lag is
what lets the side stream (and, across GPUs, the NCCL all-reduce of the k x (k+d) partial sums) overlap
the next minibatch's sparse coding.  Minibatch columns are sharded across ranks; W, A, B are replicated
and stay bit-identical because every rank runs the same deterministic dictionary update on the same
all-reduced aggregates.

All arithmetic is in the hand-written kernels of libonmf_b200.so (see _lib.py); torch only owns
memory, streams, events and the process group.
"""
from __future__ import annotations

import os
from typing import Optional

import torch

from . import _lib


RAW_NORM = 1.5      # a dictionary with a column norm beyond this counts as raw (unnormalised): see OnmfEngine.set_state


class OnmfEngine:
    def __init__(self, d: int, k: int, alpha: float = 1.0, beta: Optional[float] = None,
                 dtype: torch.dtype = torch.float32, device=None, max_iter: int = 1000,
                 process_group=None, track_C: bool = False, collect_stats: bool = False, use_tc=None,
                 reserve_sms: Optional[int] = None, fused: bool = True, lars_timing: bool = False,
                 graph: Optional[bool] = None):
        if not torch.cuda.is_available():
            raise _lib.OnmfKernelError("OnmfEngine needs a CUDA device (there is no CPU path)")
        _lib.load()
        self.d, self.k = int(d), int(k)
        if self.d <= 0 or self.k <= 0:
            raise _lib.OnmfKernelError("OnmfEngine: d and k must be positive")
        if self.k > _lib.MAX_COMPONENTS:
            # fail before any training starts (the coder's atom classes stop at 512; see INTEGRATION.md "Limits")
            raise _lib.OnmfKernelError("OnmfEngine: n_components = %d > %d is not instantiated in the LARS coder"
                                       % (self.k, _lib.MAX_COMPONENTS))
        self.alpha = float(alpha)
        self.beta = 1.0 if beta is None else float(beta)
        self.dtype = dtype
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.max_iter = int(max_iter)
        self.pg = process_group
        self.world = 1
        if process_group is not None:
            import torch.distributed as dist
            self.world = dist.get_world_size(process_group)
        self.track_C = bool(track_C)
        dev, dt_ = self.device, dtype
        self.W = torch.zeros(d, k, dtype=dt_, device=dev)
        self.W_next = torch.zeros(d, k, dtype=dt_, device=dev)
        self.A = torch.zeros(k, k, dtype=dt_, device=dev)
        self.B = torch.zeros(k, d, dtype=dt_, device=dev)
        self.C = torch.zeros(d, d, dtype=dt_, device=dev) if track_C else None
        # Gram of self.W (kept in step with it): always FP64, accumulated in FP64 from the stored dictionary -- the coder
        # inverts active blocks of it, and an fp32 Gram's per-entry rounding is amplified by cond(G) (csrc/gemm_simt.cu)
        self.G = torch.empty(k, k, dtype=torch.float64, device=dev)
        self.G_next = torch.empty(k, k, dtype=torch.float64, device=dev)
        self._G_scratch = torch.empty(k, k, dtype=torch.float64, device=dev)  # for sparse_code() against a foreign W
        self.P = [torch.zeros(k, k + d, dtype=dt_, device=dev) for _ in range(2)]
        self.P2 = torch.zeros(d, d, dtype=dt_, device=dev) if track_C else None
        self._cap = 0
        self.Ct = self.Ht = self._ws_lars = self._ws_sur = None
        # tensor-core (tcgen05, 3xTF32) path for the three large products; fp32 + TMA-friendly shapes only
        self.use_tc = bool(use_tc if use_tc is not None else True) and dtype == torch.float32 and _lib.tc_supported(k, d)
        if self.use_tc:
            self.Whi = torch.empty(d, k, dtype=dt_, device=dev)
            self.Wlo = torch.empty(d, k, dtype=dt_, device=dev)
            self.Whi_next = torch.empty(d, k, dtype=dt_, device=dev)
            self.Wlo_next = torch.empty(d, k, dtype=dt_, device=dev)
            self._Whi_s = torch.empty(d, k, dtype=dt_, device=dev)
            self._Wlo_s = torch.empty(d, k, dtype=dt_, device=dev)
        # minibatch-by-reference kernels (csrc/gemm_fused.cu): gather + widening + TF32 split inside the tensor-core kernels
        self.fused_tc = self.use_tc and _lib.fused_tc_supported(k, d) and os.environ.get("ONMF_B200_FUSED_TC", "1") != "0"
        self.Xhi = self.Xlo = self.Hhi = self.Hlo = None
        self.stats = torch.zeros(len(_lib.STATS_FIELDS), dtype=torch.int64, device=dev)   # in-kernel work counters
        self._collect = bool(collect_stats)
        self.main = torch.cuda.current_stream(dev)
        self.side = torch.cuda.Stream(dev, priority=-1)     # dictionary update / all-reduce: short kernels, scheduled first
        self._ws_gram = torch.empty(max(_lib.gram_f64_workspace(d, k), _lib.update_dict_workspace(dt_, d, k)),
                                    dtype=torch.uint8, device=dev)
        self._ws_gram_s = torch.empty(_lib.gram_f64_workspace(d, k), dtype=torch.uint8, device=dev)  # sparse_code(foreign W)
        if reserve_sms is None and os.environ.get("ONMF_RESERVE_SMS"):
            reserve_sms = int(os.environ["ONMF_RESERVE_SMS"])
        self.reserve_sms = reserve_sms
        self._ev_P = torch.cuda.Event()        # P[cur] complete on main
        self._ev_W = torch.cuda.Event()        # W (for the next coding) complete on side
        self._ev_code = torch.cuda.Event()     # main finished reading W / Xt of the current step
        self._ev_AB = torch.cuda.Event()       # A, B of the previous step blended on side (the next dictionary update follows)
        self._cur = 0
        # fused step (csrc/step.cu): one C call per minibatch enqueues the whole schedule; the Python-composed schedule
        # below (same kernels, same ordering, torch events) remains for analysis (bench.py --timeline)
        self.fused = bool(fused)
        # the coder-launch timing ring (two timed events per step) is only created when somebody reads it (bench.py)
        self._plan = _lib.StepPlan(timing_slots=256 if lars_timing else 0) if self.fused else None
        self._pairs = None
        self._sb = None
        # CUDA-graph replay of the fused step (single GPU): default on; ONMF_B200_GRAPH=0 disables
        if graph is None:
            graph = os.environ.get("ONMF_B200_GRAPH", "1") != "0"
        self.graph = bool(graph) and self.fused and self.world == 1
        self._w_dev = torch.zeros(1, dtype=torch.float64, device=dev)

    @property
    def launches(self):
        """kernels launched so far by this host thread through libonmf_b200.so (every launch site of the library counts
        itself; a CUDA-graph replay counts its kernel nodes).  Use differences."""
        return _lib.launch_count()

    def _make_bufs(self):
        """(re)build the onmf_step_buffers descriptor of the fused step from the engine's tensors"""
        if self._pairs is None:      # fixed order of the double buffers: index == self._cur
            tc = self.use_tc
            self._pairs = dict(W=[self.W, self.W_next], G=[self.G, self.G_next],
                               Whi=[self.Whi, self.Whi_next] if tc else [None, None],
                               Wlo=[self.Wlo, self.Wlo_next] if tc else [None, None])
        p = lambda t: t.data_ptr() if t is not None else None
        sb = _lib.StepBuffers()
        sb.dtype = _lib.F64 if self.dtype == torch.float64 else _lib.F32
        sb.d, sb.k = self.d, self.k
        sb.use_tc, sb.track_C, sb.max_iter = int(self.use_tc), int(self.track_C), self.max_iter
        sb.reserve_sms = -1 if self.reserve_sms is None else int(self.reserve_sms)
        sb.hold_coder = int(self.world > 1)
        sb.alpha = self.alpha
        for name in ("W", "G", "Whi", "Wlo"):
            arr = getattr(sb, name)
            arr[0], arr[1] = p(self._pairs[name][0]), p(self._pairs[name][1])
        sb.A, sb.B, sb.C = p(self.A), p(self.B), p(self.C)
        sb.P[0], sb.P[1] = p(self.P[0]), p(self.P[1])
        sb.P2 = p(self.P2)
        sb.Ct, sb.Ht = p(self.Ct), p(self.Ht)
        sb.Xhi, sb.Xlo, sb.Hhi, sb.Hlo = p(self.Xhi), p(self.Xlo), p(self.Hhi), p(self.Hlo)
        sb.ws_lars = p(self._ws_lars); sb.ws_lars_bytes = self._ws_lars.numel() if self._ws_lars is not None else 0
        sb.ws_sur = p(self._ws_sur); sb.ws_sur_bytes = self._ws_sur.numel() if self._ws_sur is not None else 0
        sb.ws_gram = p(self._ws_gram); sb.ws_gram_bytes = self._ws_gram.numel()
        sb.stats = p(self.stats)
        sb.main_stream, sb.side_stream = self.main.cuda_stream, self.side.cuda_stream
        sb.w_dev = p(self._w_dev)
        self._sb = sb

    def reset_lars_timing(self):
        if self._plan is not None:
            self._plan.reset_timing()

    def read_lars_ms(self):
        """elapsed ms of the coder launch of the last steps (fused path; waits for them)"""
        return self._plan.lars_ms() if self._plan is not None else []

    # ------------------------------------------------------------------ state
    def set_state(self, W, A=None, B=None, C=None):
        self.flush()
        self.W.copy_(torch.as_tensor(W).to(self.device, self.dtype))
        for dst, src in ((self.A, A), (self.B, B), (self.C, C)):
            if dst is None:
                continue
            if src is None:
                dst.zero_()
            else:
                dst.copy_(torch.as_tensor(src).to(self.device, self.dtype))
        self._derive(self.W, self.G, getattr(self, "Whi", None), getattr(self, "Wlo", None), self.main)
        # A raw initial dictionary (the reference's W0 = np.random.rand(d, r), src/ontf.py:213, columns of norm ~sqrt(d/3))
        # makes the covariances O(d/4) while the path is decided by differences of O(1e-5): beyond fp32 resolution.  The
        # dictionary update puts every column into the unit ball, so only the FIRST minibatch after set_state is coded
        # against such a dictionary; the fp32 engine codes that one minibatch with the FP64 coder (see _code_wide).
        self._raw_W = False
        if self.dtype == torch.float32:
            Wn = W if isinstance(W, torch.Tensor) else None
            if Wn is None:
                import numpy as _np
                self._raw_W = bool(_np.max(_np.linalg.norm(_np.asarray(W, dtype=_np.float64), axis=0)) > RAW_NORM)
            else:
                self._raw_W = bool(float(torch.diagonal(self.G).max().item()) > RAW_NORM ** 2)
        # the first dictionary update (side stream) reads W, A, B and shares the Gram workspace with the derive above
        if self._plan is not None:
            self._plan.mark_state(self.main)
        else:
            self._ev_code.record(self.main)

    def reset_aggregates(self, A=None, B=None, C=None):
        """Overwrite the aggregates (device tensors or arrays; None = keep) between steps.  The copies run on the main
        stream AFTER everything the side stream still has in flight (the previous step's blend), and the next dictionary
        update -- which reads A, B on the side stream -- is ordered behind them (the plan's state event is re-recorded)."""
        self.flush()
        for dst, src in ((self.A, A), (self.B, B), (self.C, C)):
            if dst is None or src is None:
                continue
            dst.copy_(torch.as_tensor(src).to(self.device, self.dtype))
        if self._plan is not None:
            self._plan.mark_state(self.main)
        else:
            self._ev_code.record(self.main)

    def _derive(self, W, G, Whi, Wlo, stream, use_ws=True):
        """Everything the coder needs that depends on the dictionary only: Gram matrix and (tensor-core path)
        the TF32 hi/lo split of W.  Runs right after the dictionary update, off the minibatch's critical path."""
        _lib.gram_f64(W, G, self._ws_gram if use_ws else self._ws_gram_s, stream=stream)
        if self.use_tc:
            _lib.split_tf32(W, Whi, Wlo, stream=stream)

    def _reserve(self, n):
        if n <= self._cap:
            return
        dev, dt_ = self.device, self.dtype
        self._cap = int(n)
        self.Ct = torch.empty(self._cap, self.k, dtype=dt_, device=dev)
        self.Ht = torch.empty(self._cap, self.k, dtype=dt_, device=dev)
        self._ws_lars = torch.zeros(_lib.lasso_lars_workspace(dt_, self.k, self._cap), dtype=torch.uint8, device=dev)
        nbytes = _lib.surrogate_workspace(dt_, self._cap, self.k, self.d)
        if self.track_C:
            nbytes = max(nbytes, 64 * self.d * self.d * self.W.element_size() + 256)
        if self.use_tc:
            nbytes = max(nbytes, _lib.surrogate_tc_workspace(self._cap, self.k, self.d))
            self.Xhi = self.Xlo = self.Hhi = self.Hlo = None      # pre-split copies: only the non-fused tensor-core path
        if self.fused_tc:
            nbytes = max(nbytes, _lib.surrogate_fused_tc_workspace(self._cap, self.k, self.d))
        self._ws_sur = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        self._sb = None                       # the fused step's descriptor points at the old buffers

    def _need_split_buffers(self):
        """TF32 hi/lo copies of the minibatch and the codes (pre-split tensor-core kernels: k > 256, or the Python-composed
        schedule); the fused kernels never need them."""
        if self.use_tc and self.Xhi is None:
            dev, dt_ = self.device, self.dtype
            self.Xhi = torch.empty(self._cap, self.d, dtype=dt_, device=dev)
            self.Xlo = torch.empty(self._cap, self.d, dtype=dt_, device=dev)
            self.Hhi = torch.empty(self._cap, self.k, dtype=dt_, device=dev)
            self.Hlo = torch.empty(self._cap, self.k, dtype=dt_, device=dev)
            self._sb = None

    def _stats_ptr(self):
        return self.stats

    # ------------------------------------------------------------------ coding only
    def _cov_into(self, Xt, pool, idx, scale, n, W, Whi, Wlo, Ct, stream):
        """Ct = minibatch @ W for a dense minibatch Xt or a minibatch by reference (pool, idx, scale); a patch minibatch
        by reference comes as pool = _Patches."""
        if isinstance(pool, _Patches) and Xt is None:
            _lib.cov_fused_tc_patches(pool.pm, Whi, Wlo, Ct, stream=stream)
            return
        if self.fused_tc:
            src = Xt if Xt is not None else pool
            _lib.cov_fused_tc(src, idx if Xt is None else None, n, Whi, Wlo, Ct, scale=scale if Xt is None else 1.0, stream=stream)
            return
        if Xt is None:
            Xt = self._dense(pool, idx, scale, n, stream)
        if self.use_tc:
            self._need_split_buffers()
            _lib.split_tf32(Xt, self.Xhi[:n], self.Xlo[:n], stream=stream)
            _lib.cov_tc(self.Xhi[:n], self.Xlo[:n], Whi, Wlo, Ct, stream=stream)
        else:
            _lib.cov(Xt, W, Ct, stream=stream)

    def _dense(self, pool, idx, scale, n, stream):
        """materialise a minibatch by reference (engines without the fused kernels): K1 gather (+ widening)"""
        if pool.dtype in (torch.uint8, torch.float16):
            if idx is not None:
                raise _lib.OnmfKernelError("narrow storage with an index needs the fused tensor-core path")
            if getattr(self, "_wide", None) is None or self._wide.shape[0] < n:
                self._wide = torch.empty(max(n, 1), self.d, dtype=torch.float32, device=self.device)
            if n:
                _lib.widen(pool[:n], scale, self._wide[:n], stream=stream)
            return self._wide[:n]
        if idx is None:
            return pool[:n]
        if getattr(self, "_Xg", None) is None or self._Xg.shape[0] < n:
            self._Xg = torch.empty(max(n, 1), self.d, dtype=self.dtype, device=self.device)
        if n:
            _lib.gather_rows(pool, idx, self._Xg[:n], stream=stream)
        return self._Xg[:n]

    def _dense_patches(self, pm, stream):
        """materialise a patch minibatch (engines without the fused kernels, track_C): K1 index gather (+ widening)"""
        n = int(pm.n)
        if getattr(self, "_Xg", None) is None or self._Xg.shape[0] < n:
            self._Xg = torch.empty(max(n, 1), self.d, dtype=self.dtype, device=self.device)
        if n:
            _lib.gather_patches_mb(pm, self._Xg[:n], stream=stream)
        return self._Xg[:n]

    def sparse_code(self, Xt: torch.Tensor, W: Optional[torch.Tensor] = None, alpha=None, out=None):
        """Ht (n x k) = positive lasso_lars codes of the rows of Xt (n x d) against W (default: current)."""
        n = Xt.shape[0]
        self._reserve(max(n, 1))
        Ct = self.Ct[:n]
        Ht = self.Ht[:n] if out is None else out
        if n == 0:
            return Ht
        if W is None:
            self.flush()
            f = _Dictionary(self.W, self.G, getattr(self, "Whi", None), getattr(self, "Wlo", None), self._raw_W)
        else:
            f = self.derive_foreign(W)
        self._cov_into(Xt, None, None, 1.0, n, f.W, f.Whi, f.Wlo, Ct, torch.cuda.current_stream(self.device))
        self._lars(f, Ct, alpha, Ht, -1)
        return Ht

    def derive_foreign(self, W: torch.Tensor):
        """Everything the coder needs from a dictionary W (d x k, the engine's dtype) other than the engine's own: its FP64
        Gram and, on the tensor-core path, its TF32 split, in the engine's scratch buffers; and whether it is raw (fp32
        engine: coded in FP64, see set_state).  Returns the handle sparse_code_patches takes; it stays valid until the
        next derive_foreign or sparse_code(Xt, W) call, which reuse the same buffers."""
        G = self._G_scratch
        Whi, Wlo = (self._Whi_s, self._Wlo_s) if self.use_tc else (None, None)
        self._derive(W, G, Whi, Wlo, torch.cuda.current_stream(self.device), use_ws=False)
        wide = self.dtype == torch.float32 and float(torch.diagonal(G).max().item()) > RAW_NORM ** 2
        return _Dictionary(W, G, Whi, Wlo, wide)

    def sparse_code_patches(self, pm, f, alpha=None, out=None, first_tier=-1):
        """Ht (n x k) = positive lasso_lars codes of a patch minibatch BY REFERENCE (an onmf_patch_minibatch descriptor, see
        _lib.make_patch_minibatch) against the dictionary of the handle f = derive_foreign(W).  Fused tensor-core engines
        read the patches out of the image in the covariance kernel; every other engine gathers them into its dense buffer
        first.  Same bits as sparse_code(<the gathered patches>, W).  first_tier: the coder's first active-set tier (0 / 1),
        or -1 for the workspace's adaptive hint, which an earlier call may have moved."""
        n = int(pm.n)
        self._reserve(max(n, 1))
        Ct = self.Ct[:n]
        Ht = self.Ht[:n] if out is None else out
        if n == 0:
            return Ht
        st = torch.cuda.current_stream(self.device)
        if self.fused_tc:
            self._cov_into(None, _Patches(pm), None, 1.0, n, f.W, f.Whi, f.Wlo, Ct, st)
        else:
            self._cov_into(self._dense_patches(pm, st), None, None, 1.0, n, f.W, f.Whi, f.Wlo, Ct, st)
        self._lars(f, Ct, alpha, Ht, first_tier)
        return Ht

    def _lars(self, f, Ct, alpha, Ht, first_tier):
        a = self.alpha if alpha is None else alpha
        if f.wide:
            self._lars_wide(f.G, Ct, a, Ht, torch.cuda.current_stream(self.device), first_tier)
        else:
            _lib.lasso_lars(f.G, Ct, self.d, a, Ht, self._ws_lars, max_iter=self.max_iter, stats=self._stats_ptr(),
                            first_tier=first_tier)

    def _lars_wide(self, G64, Ct, alpha, Ht, stream, first_tier=-1):
        """fp32 engine, raw dictionary: the coder in FP64 on the fp32 covariances (FP64 Gram as always), codes rounded to
        fp32.  Temporary FP64 copies of Ct / Ht live only for this call."""
        n = Ct.shape[0]
        with torch.cuda.stream(stream):
            Ct64 = torch.empty(n, self.k, dtype=torch.float64, device=self.device)
            Ht64 = torch.empty(n, self.k, dtype=torch.float64, device=self.device)
            ws = torch.zeros(_lib.lasso_lars_workspace(torch.float64, self.k, n), dtype=torch.uint8, device=self.device)
            _lib.convert(Ct, Ct64, stream=stream)
            _lib.lasso_lars(G64, Ct64, self.d, alpha, Ht64, ws, max_iter=self.max_iter, stats=self._stats_ptr(), stream=stream,
                            first_tier=first_tier)
            _lib.convert(Ht64, Ht, stream=stream)
            for t_ in (Ct64, Ht64, ws):
                t_.record_stream(stream)

    # ------------------------------------------------------------------ one online step
    def step_with_codes(self, Xt, Ht, t):
        """Same as step() but with externally computed codes Ht (n x k), e.g. from the PGD coder."""
        return self.step(Xt, t, codes=Ht)

    def split_buffers(self, n):
        """(Xhi, Xlo) views of the engine-owned pre-split minibatch buffers (pre-split tensor-core kernels): a producer such
        as _lib.gather_rows_split can write the minibatch straight into them and then call step(None, t, n=n)."""
        self._reserve(max(n, 1))
        self._need_split_buffers()
        return self.Xhi[:n], self.Xlo[:n]

    def step_pool(self, pool: torch.Tensor, idx: Optional[torch.Tensor], t: float, n: Optional[int] = None, scale: float = 1.0,
                  codes: Optional[torch.Tensor] = None):
        """One minibatch BY REFERENCE: rows idx (int64, device; None = rows 0..n-1) of a resident sample-major pool, which
        may be stored as float32 or -- fp32 engine on the fused tensor-core path -- uint8 / float16 (value = stored *
        scale).  X_batch = X_unfold[:, idx] (src/ontf.py:231) is never materialised: the covariance and partial-sum
        kernels read the pool rows in place."""
        n = int(idx.shape[0] if idx is not None else (pool.shape[0] if n is None else n))
        return self._step(None, (pool, idx, float(scale)), t, codes, n)

    def step_patches(self, src, idx: Optional[torch.Tensor], t: float, codes: Optional[torch.Tensor] = None):
        """One minibatch of image patches BY REFERENCE: columns idx (int64, device; None = columns 0..N-1) of an
        ImagePatches `src` (patches.py).  On the fused tensor-core path (fp32, k <= 256, no track_C) the covariance and
        partial-sum kernels read the patches straight out of the image; every other engine gathers the minibatch into its
        dense buffer first.  Same results, bit for bit, as step_pool on the materialised pool of the same patches."""
        if src.d != self.d:
            raise _lib.OnmfKernelError("step_patches: the patches have d = %d, the engine %d" % (src.d, self.d))
        if src.engine_dtype != self.dtype:
            raise _lib.OnmfKernelError("step_patches: %s image for a %s engine" % (src.dtype, self.dtype))
        n = int(idx.shape[0]) if idx is not None else src.N
        return self._step(None, _Patches(src.minibatch(idx, n), idx), t, codes, n)

    def step(self, Xt: Optional[torch.Tensor], t: float, codes: Optional[torch.Tensor] = None, n: Optional[int] = None):
        """One minibatch: Xt (n_local x d) are THIS rank's columns of the minibatch, t the step index
        (w = t^-beta).  Returns the local codes Ht (view, valid until the next call).
        Xt=None (pre-split tensor-core kernels only): the minibatch is already in split_buffers(n)."""
        if Xt is None and not self.use_tc:
            raise _lib.OnmfKernelError("step(None, ...) needs the tensor-core path")
        n = Xt.shape[0] if Xt is not None else int(n)
        return self._step(Xt, None, t, codes, n)

    def _step(self, Xt, ref, t, codes, n):
        main, side = self.main, self.side
        pend = getattr(self, "_d2h_pending", None)
        if pend:
            # step_host copy-backs run on their own stream: this step's dictionary update overwrites W_next -- wait for the
            # copy that read that buffer (issued two steps ago, long finished)
            ev = pend.pop(self.W_next.data_ptr(), None)
            if ev is not None:
                side.wait_event(ev)
                main.wait_event(ev)
        presplit = Xt is None and ref is None
        self._reserve(max(n, 1))
        w = float(t) ** (-self.beta)
        cur = self._cur
        patches = isinstance(ref, _Patches)
        pool, idx, scale = (ref, ref.idx, 1.0) if patches else ref if ref is not None else (None, None, 1.0)
        by_ref = ref is not None and self.fused_tc and self.fused and not self.track_C      # kernels read the pool in place
        if ref is not None and not by_ref:
            Xt = self._dense_patches(ref.pm, main) if patches else self._dense(pool, idx, scale, n, main)
            ref = None
        if self._raw_W and codes is None:
            # first minibatch against a raw initial dictionary (fp32 engine): code it with the FP64 coder, then run the
            # normal step on those codes (aggregation + dictionary update are unaffected)
            self._raw_W = os.environ.get("ONMF_B200_WIDE_ALWAYS") == "1"      # (analysis switch: FP64 coder at every step)
            if n > 0:
                Ct, Ht = self.Ct[:n], self.Ht[:n]
                if presplit:
                    _lib.cov_tc(self.Xhi[:n], self.Xlo[:n], self.Whi, self.Wlo, Ct, stream=main)
                else:
                    self._cov_into(Xt, pool, idx, scale, n, self.W, getattr(self, "Whi", None), getattr(self, "Wlo", None), Ct, main)
                self._lars_wide(self.G, Ct, self.alpha, Ht, main)
                codes = Ht
        if os.environ.get("ONMF_B200_WIDE_ALWAYS") != "1":
            self._raw_W = False
        if self.fused:
            return self._step_fused(Xt, ref, codes, n, w, cur)
        # ---- Python-composed schedule (analysis: bench.py --timeline; same kernels as the pre-split C path) ----
        if self.use_tc:
            self._need_split_buffers()
        # side stream: dictionary update for this step with the OLD aggregates (src/ontf.py:151).  It is
        # queued behind the previous step's all-reduce + blend (same stream), and must not overwrite the
        # buffer the previous coding was still reading.
        with torch.cuda.stream(side):
            side.wait_event(self._ev_code)
            _lib.update_dict(self.W, self.A, self.B, self.W_next, stream=side, workspace=self._ws_gram)
            self._derive(self.W_next, self.G_next, getattr(self, "Whi_next", None), getattr(self, "Wlo_next", None), side)
            self._ev_W.record(side)
        # main stream: code this minibatch with W_{t-1}
        Ht = self.Ht[:n] if codes is None else codes
        if self.track_C:
            main.wait_stream(side)                  # P2 is single-buffered
        if n > 0:
            if self.use_tc:
                Xhi, Xlo = self.Xhi[:n], self.Xlo[:n]
                if not presplit:
                    _lib.split_tf32(Xt, Xhi, Xlo, stream=main)
            if codes is None:
                Ct = self.Ct[:n]
                if self.use_tc:
                    _lib.cov_tc(Xhi, Xlo, self.Whi, self.Wlo, Ct, stream=main)
                else:
                    _lib.cov(Xt, self.W, Ct, stream=main)
                if self.world > 1:
                    # The dictionary update is one thread-block cluster: it can only be placed while a whole group of SMs
                    # in one GPC is free, i.e. BEFORE the persistent coder has spread over the GPU.  On one GPU it is queued
                    # at the start of the step and wins that race; across GPUs it waits for the all-reduce of the previous
                    # partial sums, so hold the coder back until that has landed: both become runnable together and the
                    # high-priority side stream is placed first (the coder's last CTAs start when the update retires).
                    main.wait_event(self._ev_AB)
                rsv = self.reserve_sms if self.reserve_sms is not None else 0
                saved = _lib.get_option(_lib.OPT_LARS_RESERVED_SMS)
                _lib.set_option(_lib.OPT_LARS_RESERVED_SMS, rsv)
                try:
                    _lib.lasso_lars(self.G, Ct, self.d, self.alpha, Ht, self._ws_lars, max_iter=self.max_iter,
                                    stats=self._stats_ptr(), stream=main)
                finally:
                    _lib.set_option(_lib.OPT_LARS_RESERVED_SMS, saved)
            if self.use_tc:
                _lib.split_tf32(Ht, self.Hhi[:n], self.Hlo[:n], stream=main)
                _lib.surrogate_partial_tc(self.Hhi[:n], self.Hlo[:n], Xhi, Xlo, self.P[cur], self._ws_sur, stream=main)
            else:
                _lib.surrogate_partial(Ht, Xt, self.P[cur], self._ws_sur, stream=main)
            if self.track_C:
                if presplit:
                    raise _lib.OnmfKernelError("track_C needs the unsplit minibatch")
                _lib.xxt_partial(Xt, self.P2, self._ws_sur, stream=main)
        else:
            with torch.cuda.stream(main):
                self.P[cur].zero_()
                if self.track_C:
                    self.P2.zero_()
        self._ev_P.record(main)
        self._ev_code.record(main)
        # side stream: all-reduce the packed partial sums and blend them into A, B.  Nothing on the main
        # stream waits for this: it overlaps the NEXT minibatch's coding and is only consumed by the next
        # dictionary update (queued behind it on this stream).
        with torch.cuda.stream(side):
            side.wait_event(self._ev_P)
            if self.world > 1:
                import torch.distributed as dist
                dist.all_reduce(self.P[cur], group=self.pg)
                if self.track_C:
                    dist.all_reduce(self.P2, group=self.pg)
            _lib.surrogate_blend(self.P[cur], w, self.A, self.B, stream=side)
            self._ev_AB.record(side)
            if self.track_C:
                _lib.axpby(w, self.P2, 1.0 - w, self.C, stream=side)
        # the next coding needs W_t (= W_next): wait for the dictionary update only
        main.wait_event(self._ev_W)
        self.W, self.W_next = self.W_next, self.W
        self.G, self.G_next = self.G_next, self.G
        if self.use_tc:
            self.Whi, self.Whi_next = self.Whi_next, self.Whi
            self.Wlo, self.Wlo_next = self.Wlo_next, self.Wlo
        self._cur ^= 1
        return Ht

    def _step_fused(self, Xt, ref, codes, n, w, cur):
        """the same schedule through ONE call into libonmf_b200.so (onmf_step[_mb] / onmf_step_launch[_mb] + onmf_step_finish)"""
        for t_, nm in ((Xt, "Xt"), (codes, "codes")):
            if t_ is not None:
                _lib._req(t_, nm, self.dtype)
        if codes is not None and tuple(codes.shape) != (n, self.k):
            raise _lib.OnmfKernelError("codes must be (n x k)")
        if Xt is not None and Xt.shape[1] != self.d:
            raise _lib.OnmfKernelError("Xt must be (n x d)")
        mb = pm = None
        if isinstance(ref, _Patches):
            pm = ref.pm
        elif ref is not None:
            pool, idx, scale = ref
            if pool.shape[1] != self.d:
                raise _lib.OnmfKernelError("pool must be (n_pool x d)")
            mb = _lib.make_minibatch(pool, idx, n, scale)
        elif Xt is not None and self.fused_tc and not self.track_C:
            mb = _lib.make_minibatch(Xt, None, n, 1.0)          # a dense minibatch is a pool read front to back
            Xt = None
        elif self.use_tc:
            self._need_split_buffers()                           # pre-split tensor-core kernels (k > 256, track_C)
        if self._sb is None:
            self._make_bufs()
        if self.world > 1:
            import torch.distributed as dist
            if pm is not None:
                self._plan.launch_patches(self._sb, pm, codes, cur)
            elif mb is not None:
                self._plan.launch_mb(self._sb, mb, codes, cur)
            else:
                self._plan.launch(self._sb, Xt, codes, n, cur)
            with torch.cuda.stream(self.side):
                dist.all_reduce(self.P[cur], group=self.pg)
                if self.track_C:
                    dist.all_reduce(self.P2, group=self.pg)
            self._plan.finish(self._sb, w, cur)
        elif pm is not None:
            self._plan.step_patches(self._sb, pm, codes, w, cur, graph=self.graph)
        elif mb is not None:
            self._plan.step_mb(self._sb, mb, codes, w, cur, graph=self.graph)
        elif self.graph:
            self._plan.step_graph(self._sb, Xt, codes, n, w, cur)
        else:
            self._plan.step(self._sb, Xt, codes, n, w, cur)
        self.W, self.W_next = self.W_next, self.W
        self.G, self.G_next = self.G_next, self.G
        if self.use_tc:
            self.Whi, self.Whi_next = self.Whi_next, self.Whi
            self.Wlo, self.Wlo_next = self.Wlo_next, self.Wlo
        self._cur ^= 1
        return self.Ht[:n] if codes is None else codes

    # ------------------------------------------------------------------ host-buffer entry (end-to-end path)
    def step_host(self, Xt_host: torch.Tensor, t: float, W_out_host: Optional[torch.Tensor] = None, scale: Optional[float] = None):
        """step() for a minibatch that lives in (pinned) HOST memory, sample-major (n x d).

        Xt_host may be float32 / float64 (the engine's dtype), or a narrower STORAGE format -- uint8 (scale defaults to
        1/255, the reference's `data / 255`, image_reconstruction.py:88) or float16 (scale 1) -- which crosses PCIe at a
        quarter / half of the bytes; on the fused tensor-core path the kernels read the staged bytes as they are (widening
        inside the loaders), otherwise onmf_widen expands them once.  Arithmetic is fp32 either way.

        The host->device copy runs on a copy stream into one of two staging buffers, so the copy of minibatch t+1 overlaps
        the coding of minibatch t; if W_out_host (pinned, d x k) is given the updated dictionary is copied back
        asynchronously after the step's dictionary update.  Nothing blocks the host; call flush()+synchronize (or
        read_back()) before touching W_out_host."""
        if Xt_host.is_cuda:
            raise _lib.OnmfKernelError("step_host expects a host tensor")
        n = Xt_host.shape[0]
        sdt = Xt_host.dtype
        narrow = sdt in (torch.uint8, torch.float16)
        if not narrow and sdt != self.dtype:
            raise _lib.OnmfKernelError("step_host: minibatch dtype %s (engine %s; uint8 / float16 storage also accepted)" % (sdt, self.dtype))
        if narrow and (self.dtype != torch.float32 or self.d % 4):
            raise _lib.OnmfKernelError("step_host: uint8 / float16 storage needs the fp32 engine and d % 4 == 0")
        if not hasattr(self, "_stage") or self._stage[0].shape[0] < n or self._stage[0].dtype != sdt:
            self._stage = [torch.empty(max(n, 1), self.d, dtype=sdt, device=self.device) for _ in range(2)]
            self._stage_ev = [torch.cuda.Event(), torch.cuda.Event()]
            self._stage_i = 0
            self._copy = torch.cuda.Stream(self.device)
            self._ev_h2d = torch.cuda.Event()
        i = self._stage_i
        self._stage_i ^= 1
        buf = self._stage[i][:n]
        with torch.cuda.stream(self._copy):
            self._copy.wait_event(self._stage_ev[i])       # the step that last used this buffer is done with it
            buf.copy_(Xt_host, non_blocking=True)
            self._ev_h2d.record(self._copy)
        self.main.wait_event(self._ev_h2d)
        if narrow:
            sc = (1.0 / 255.0 if sdt == torch.uint8 else 1.0) if scale is None else float(scale)
            Ht = self.step_pool(self._stage[i], None, t, n=n, scale=sc)
        else:
            Ht = self.step(buf, t)
        self._stage_ev[i].record(self.main)
        if W_out_host is not None:
            # Copy-back on its own stream, after the whole step: on the side stream it sat between this step's blend and the
            # next step's dictionary update, whose cluster then reached the GPU after the persistent coder had taken every
            # SM and ran behind it instead of under it (N = 8, uint8 storage: 2.7 instead of 1.9 ms per step).
            if getattr(self, "_d2h", None) is None:
                self._d2h = torch.cuda.Stream(self.device)
                self._d2h_events = {}
                self._d2h_pending = {}
            self._d2h.wait_stream(self.main)
            self._d2h.wait_stream(self.side)
            key = self.W.data_ptr()
            done = self._d2h_events.setdefault(key, torch.cuda.Event())
            with torch.cuda.stream(self._d2h):
                W_out_host.copy_(self.W, non_blocking=True)     # self.W is the dictionary this step produced
                done.record(self._d2h)
            self._d2h_pending[key] = done
        return Ht

    def flush(self):
        """Make W, A, B (C) visible to the current stream / host."""
        self.main.wait_stream(self.side)
        if getattr(self, "_d2h", None) is not None:
            self.main.wait_stream(self._d2h)                     # (copy-backs of step_host)

    def state(self):
        self.flush()
        return self.W, self.A, self.B, self.C

    def surrogate_error(self):
        """tr(W A W^T) - 2 tr(W B) + tr(C): the surrogate loss the Ising / network drivers plot
        (ising_reconstruction.py:133,164); tr(C) is included when the engine tracks C.  Returns a float."""
        self.flush()
        out = torch.empty(3, dtype=torch.float64, device=self.device)
        _lib.surrogate_error(self.W, self.G, self.A, self.B, self.C, out)
        t = out.cpu().tolist()
        return t[0] - 2.0 * t[1] + t[2]

    def read_stats(self):
        torch.cuda.synchronize(self.device)
        vals = self.stats.cpu().tolist()
        return dict(zip(_lib.STATS_FIELDS, vals))


class _Patches:
    """a patch minibatch by reference inside OnmfEngine: the C descriptor and the index tensor it points at"""

    def __init__(self, pm, idx=None):
        self.pm, self.idx = pm, idx


class _Dictionary:
    """what the coder reads of one dictionary: W, its FP64 Gram G, the TF32 split (Whi, Wlo; None off the tensor-core
    path) and whether the fp32 engine codes against it in FP64 (wide)"""

    def __init__(self, W, G, Whi, Wlo, wide):
        self.W, self.G, self.Whi, self.Wlo, self.wide = W, G, Whi, Wlo, bool(wide)
