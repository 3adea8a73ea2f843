#!/usr/bin/env python
"""bench.py -- ONMF samples/s (code + surrogate + dictionary update) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg5] [--dump-outputs DIR]

Workload (BASELINE.json configs[4], the one the metric is quoted on): synthetic nonnegative data,
d=1024 (32x32 patches), k=256 atoms, global minibatch 262,144 columns sharded by columns over the N GPUs
(strong scaling: the global minibatch is fixed), alpha=1, beta=1, fp32 production mode.  A "step" is one
pass of the hot path over one minibatch: K1 gather of a freshly resampled minibatch from the resident
pool, K2 Gram+covariance, K3 LARS-lasso coding, K4 surrogate partial sums (+ NCCL all-reduce of the packed
k x (k+d) buffer at N>1) + blend, K5 dictionary update.

Prints ONE JSON line (rank 0).  `value` = device-timed throughput with inputs resident in HBM; `e2e` = the
same steps fed from pinned HOST memory through OnmfEngine.step_host (H2D of every minibatch and D2H of the
updated dictionary inside the timed region).  `roofline` describes the dominant kernel (the LARS coder,
timed live with CUDA events on its launch stream), `cpu_baseline` the reference CPU path (numpy + sklearn
lasso_lars, the oracle port) on a bounded column sample on this box's host cores.

--dump-outputs DIR writes what the last timed step returned (its codes) and left behind (W, A, B) as .npy files.
The pool, W0 and the minibatch indices come from fixed seeds, so two builds run with the same arguments can be
compared array by array.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (d, k, global minibatch, alpha)
    "cfg1": (100, 25, 1000, 1.0),
    "cfg2": (300, 49, 4000, 1.0),
    "cfg3": (441, 25, 10000, 1.0),
    "cfg4": (400, 100, 16384, 1.0),
    "cfg5": (1024, 256, 262144, 1.0),
}
METRIC = "ONMF samples/sec (code+surrogate+dict update)"
UNIT = "samples/s"
LARS_DRAM_BYTES = 4.92e8     # ncu dram bytes of one first-tier coder launch at cfg5, N=1 (profiles/r2_lars_fast.md)


def workload_name(name, d, k, n_global, alpha):
    """the SAME string in both arms (the driver compares config.workload); per-arm detail goes into other config keys"""
    return "%s: synthetic U[0,1) d=%d k=%d global minibatch %d alpha=%g" % (name, d, k, n_global, alpha)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        try:
            j = json.load(open(p))
            return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_CODE_ROWS = 16384       # code rows kept by --dump-outputs: 16 MB at k=256, about 18 MB with W, A and B


def timed_outputs(eng, codes):
    """What a caller of the timed path holds after its last step, as host arrays: that step's codes (this rank's
    n x k; a fixed, seeded sample of DUMP_CODE_ROWS rows in ascending order when n is larger) and the dictionary and
    aggregates the step left behind."""
    import torch
    W, A, B, _ = eng.state()
    n = codes.shape[0]
    if n > DUMP_CODE_ROWS:
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_CODE_ROWS, replace=False))
        codes = codes.index_select(0, torch.from_numpy(rows).to(codes.device))
    return {name: x.cpu().numpy() for name, x in (("codes", codes), ("W", W), ("A", A), ("B", B))}


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU during the timed region (NVML; same fields as the
    nvidia-smi line of B200_PROFILING.md)."""

    def __init__(self, index, period=0.02):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            self._stop_evt.wait(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------ reference arm
def _cpu_worker_init():
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(1)                       # one BLAS thread per worker process: the workers are the parallelism
    except Exception:
        pass
    import warnings
    warnings.filterwarnings("ignore")


def _cpu_code_chunk(task):
    Xc, W, alpha = task
    from oracle import onmf_oracle as O
    return O.sparse_code_sklearn(Xc, W, alpha)


def cpu_reference_step(d, k, alpha, cols, seed=0, steps=1, warmup=0, procs=1):
    """The reference's CPU step (numpy + scikit-learn positive lasso_lars + A,B recursion + update_dict) via the
    oracle port (oracle/onmf_oracle.py, coder='sklearn' = the dependency called like src/ontf.py:79-86) on a
    bounded sample of `cols` columns of the same synthetic workload.  The reference itself codes the minibatch in one
    single-threaded sklearn loop; with procs > 1 the columns are additionally split over `procs` worker processes (the
    columns are independent), i.e. the most the host cores can give this algorithm.  Returns (samples/s, s/step)."""
    import warnings
    warnings.filterwarnings("ignore")
    from oracle import onmf_oracle as O
    rng = np.random.RandomState(seed)
    X = rng.rand(d, cols)
    W = rng.rand(d, k)
    A, B = np.zeros((k, k)), np.zeros((k, d))
    # one untimed dictionary sweep so the timed steps see a unit-ball dictionary like every step after the first
    W = O.update_dict(W, A, B)
    pool = None
    if procs > 1:
        import multiprocessing as mp
        pool = mp.get_context("spawn").Pool(procs, initializer=_cpu_worker_init)
        pool.map(_cpu_code_chunk, [(X[:, :2].copy(), W, alpha)] * procs)      # start the workers (imports) untimed
        bounds = np.linspace(0, cols, procs * 4 + 1).astype(int)
    times = []
    for t in range(1, warmup + steps + 1):
        t0 = time.perf_counter()
        if pool is None:
            H, A, B, W = O.step(X, A, B, W, float(t), alpha, None, coder="sklearn")
        else:
            parts = pool.map(_cpu_code_chunk, [(np.ascontiguousarray(X[:, a:b]), W, alpha)
                                               for a, b in zip(bounds[:-1], bounds[1:]) if b > a])
            H = np.concatenate(parts, axis=1)
            A1, B1 = O.aggregate(A, B, H, X, float(t), None)
            W = O.update_dict(W, A, B)
            A, B = A1, B1
        el = time.perf_counter() - t0
        if t > warmup:
            times.append(el)
    if pool is not None:
        pool.close()
        pool.join()
    sec = float(np.mean(times))
    return cols / sec, sec


def host_cores():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


PER_COL_MS = {"cfg5": 7.6, "cfg4": 3.2, "cfg3": 2.1, "cfg2": 2.2, "cfg1": 1.05}   # one host core, sklearn lasso_lars


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    d, k, n_global, alpha = WORKLOADS[args.workload]
    procs = args.cpu_procs or host_cores()
    # bounded sample: ~PER_COL_MS per column per core -> keep the whole run near two minutes
    cols = args.cpu_cols or int(max(64 * procs, min(n_global, 110e3 * procs / PER_COL_MS[args.workload] / (args.steps + args.warmup))))
    val, sec = cpu_reference_step(d, k, alpha, cols, steps=args.steps, warmup=args.warmup, procs=procs)
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args.workload, d, k, n_global, alpha), "d": d, "k": k, "global_batch": n_global,
                   "detail": "CPU arm: %d-column sample of the minibatch per step" % cols},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": procs, "kind": "port",
                         "sample": "%d of %d columns per step; numpy + scikit-learn lasso_lars (the reference's CPU path via the "
                                   "oracle port), columns split over %d worker processes with one BLAS thread each (the "
                                   "reference itself runs this loop on one core); host cpus=%s"
                                   % (cols, n_global, procs, os.cpu_count())},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------ our arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    from onmf_ontf_ndl_b200 import OnmfEngine, _lib
    from onmf_ontf_ndl_b200.parallel import init_from_env, shard_range

    rank, world, local = init_from_env("nccl")
    if world != args.gpus and world > 1:
        args.gpus = world
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    d, k, n_global, alpha = WORKLOADS[args.workload]
    if args.batch:
        n_global = args.batch
    lo, hi = shard_range(n_global, world, rank)
    n = hi - lo
    dt = torch.float32
    K, Wm = args.steps, args.warmup

    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    pool = torch.rand(n, d, dtype=dt, device=dev, generator=gen)       # this rank's resident column pool
    gw = torch.Generator(device=dev)
    gw.manual_seed(0)                                                   # same W0 on every rank
    W0 = torch.rand(d, k, dtype=dt, device=dev, generator=gw)
    # Small configurations (BASELINE configs[0..3]) are launch-latency bound: their steps replay as ONE CUDA graph
    # (onmf_step_graph); the per-launch coder time of the roofline object is then measured in a separate pass after the
    # timed region (event pairs cannot be read out of a graph).  cfg5 keeps the stream schedule with the coder timed live.
    graph_mode = (args.graph == "on") or (args.graph == "auto" and args.workload != "cfg5" and world == 1 and not args.timeline)
    pg = dist.group.WORLD if world > 1 else None
    eng = OnmfEngine(d, k, alpha=alpha, dtype=dt, device=dev, process_group=pg, collect_stats=True, fused=not args.timeline,
                     lars_timing=not graph_mode, graph=graph_mode)
    eng.set_state(W0)
    main = eng.main

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # fresh minibatch per step: the pool resampled with replacement.  Like the reference-facing classes (which draw every
    # step's np.random.randint up front, src/ontf.py:230), the index sequence of the whole run is drawn before the timed
    # region; two index buffers alternate so that a step's (pool, idx) key is stable for the CUDA-graph replay.
    n_seq = Wm + K + 64
    idx_all = torch.randint(0, n, (n_seq, n), device=dev, generator=gen)
    idx_buf = [torch.empty(n, dtype=torch.int64, device=dev) for _ in range(2)]

    def one_step(t, eng=eng):
        # the step takes the minibatch BY REFERENCE (pool + indices): on the fused tensor-core path K1 (gather) happens
        # inside the covariance / partial-sum kernels, otherwise the engine runs the K1 gather kernel first
        if graph_mode:
            idx = idx_buf[t & 1]
            idx.copy_(idx_all[t % n_seq])
        else:
            idx = idx_all[t % n_seq]
        return eng.step_pool(pool, idx, float(t))

    # The end-to-end loops below re-run the SAME steps as the device-timed loop (the coder's work per step depends on how far
    # the dictionary has come: +4 % per 13 steps at cfg5, profiles/r2_steps.md): the state two steps before the end of the
    # warm-up is kept, restored before each end-to-end loop, and the loop's two pipeline-fill steps replay t = W-1, W.
    t = 0
    snap = None
    for _ in range(Wm):
        if not graph_mode and t == Wm - 2:
            with torch.cuda.stream(main):                       # (clones ordered on the engine's main stream)
                snap = tuple(x.clone() for x in eng.state()[:3]) + (t,)
        t += 1
        one_step(t)
    barrier()
    if eng.stats is not None:
        eng.stats.zero_()
    launches0 = eng.launches
    sampler = ClockSampler(local)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    lars_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    # wrap the LARS launch with events on its launch stream (the engine's main stream)
    orig_lars = _lib.lasso_lars
    counter = {"i": 0}

    def timed_lars(*a, **kw):
        i = counter["i"]
        if i < K:
            lars_ev[i][0].record(main)
        r = orig_lars(*a, **kw)
        if i < K:
            lars_ev[i][1].record(main)
        counter["i"] = i + 1
        return r

    if not eng.fused:
        _lib.lasso_lars = timed_lars
    eng.reset_lars_timing()
    # optional timeline (analysis only): device timestamps of the side-stream kernels relative to the timed region start
    tl = []
    if args.timeline:
        import torch.distributed as _d

        def wrap(mod, name, label, stream_of):
            orig = getattr(mod, name)

            def f(*a, **kw):
                st = stream_of(kw)
                e0_, e1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0_.record(st)
                r = orig(*a, **kw)
                e1_.record(st)
                tl.append((label, e0_, e1_))
                return r
            setattr(mod, name, f)
            return orig
        cur = lambda kw: kw.get("stream") or torch.cuda.current_stream(dev)
        origs = [(_lib, "update_dict", wrap(_lib, "update_dict", "bcd", cur)),
                 (_lib, "gram_f64", wrap(_lib, "gram_f64", "gram", cur)),
                 (_lib, "surrogate_blend", wrap(_lib, "surrogate_blend", "blend", cur)),
                 (_lib, "cov_tc", wrap(_lib, "cov_tc", "cov", cur)),
                 (_lib, "surrogate_partial_tc", wrap(_lib, "surrogate_partial_tc", "surrogate", cur))]
        if world > 1:
            origs.append((_d, "all_reduce", wrap(_d, "all_reduce", "allreduce", lambda kw: torch.cuda.current_stream(dev))))
    barrier()
    ev0.record(main)
    for _ in range(K):
        t += 1
        codes = one_step(t)
    eng.flush()
    ev1.record(main)
    barrier()
    _lib.lasso_lars = orig_lars
    if args.timeline:
        for mod, name, orig in origs:
            setattr(mod, name, orig)
        torch.cuda.synchronize(dev)
        if rank == 0:
            rows = [(lab, ev0.elapsed_time(a_), ev0.elapsed_time(b_)) for lab, a_, b_ in tl]
            rows += [("lars", ev0.elapsed_time(a_), ev0.elapsed_time(b_)) for a_, b_ in lars_ev]
            rows.sort(key=lambda r: r[1])
            sys.stderr.write("timeline (ms from the start of the timed region): label start end\n")
            for lab, t0_, t1_ in rows[:80]:
                sys.stderr.write("  %-10s %8.3f %8.3f\n" % (lab, t0_, t1_))
    clocks = sampler.stop()
    # copied now: the passes below step the same engine again
    outputs = timed_outputs(eng, codes) if (args.dump_outputs and rank == 0) else None
    elapsed_ms = ev0.elapsed_time(ev1)
    launches = eng.launches - launches0
    stats = eng.read_stats()
    graph_steps = eng._plan.graph_steps() if eng._plan is not None else 0
    if graph_mode:
        # separate pass (outside the timed region): same state, stream schedule with event pairs around the coder launch
        eng_t = OnmfEngine(d, k, alpha=alpha, dtype=dt, device=dev, collect_stats=False, lars_timing=True, graph=False)
        Wc, Ac, Bc, _ = eng.state()
        eng_t.set_state(Wc, Ac, Bc)
        kt = max(3, min(K, 20))
        for _ in range(3):
            t += 1
            one_step(t, eng_t)
        eng_t.reset_lars_timing()
        for _ in range(kt):
            t += 1
            one_step(t, eng_t)
        eng_t.flush()
        torch.cuda.synchronize(dev)
        lars_ms = float(np.mean(eng_t.read_lars_ms()[-kt:]))
        del eng_t
    elif eng.fused:
        lars_ms = float(np.mean(eng.read_lars_ms()[-K:]))       # event pairs around the coder launch, recorded by the plan
    else:
        lars_ms = float(np.mean([a.elapsed_time(b) for a, b in lars_ev]))
    tmax = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    elapsed_ms = float(tmax.item())
    value = n_global * K / (elapsed_ms * 1e-3)

    # ---------------- end-to-end: pinned host minibatches through OnmfEngine.step_host -----------------------
    host = [torch.empty(n, d, dtype=dt).pin_memory() for _ in range(2)]
    for hbuf in host:
        hbuf.copy_(pool)                                   # synthetic host-resident minibatches
    W_host = torch.empty(d, k, dtype=dt).pin_memory()
    e2e_steps = max(3, min(K, 20))
    e2e_warm = 6 if graph_mode else 2          # graph mode: every (staging buffer, parity) key is captured on its second sight
    if snap is not None:
        with torch.cuda.stream(main):
            eng.set_state(snap[0], snap[1], snap[2])
        t = snap[3]
    e2e_t_first = t + e2e_warm + 1
    for i in range(e2e_warm):
        t += 1
        eng.step_host(host[i & 1], float(t), W_host)
    eng.flush()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(main)
    for i in range(e2e_steps):
        t += 1
        eng.step_host(host[i & 1], float(t), W_host)
    eng.flush()
    e1.record(main)
    barrier()
    e2e_ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_value = n_global * e2e_steps / (float(e2e_ms.item()) * 1e-3)
    e2e_coder_ms = float(np.mean(eng.read_lars_ms()[-e2e_steps:])) if (eng.fused and not graph_mode) else None
    checksum = float(W_host.double().sum())
    assert np.isfinite(checksum)

    # ---------------- the same end-to-end loop with the minibatch STORED as uint8 on the host (8-bit image data, the form
    # the reference's drivers hold before `data / 255`, image_reconstruction.py:88): a quarter of the PCIe bytes, widened to
    # fp32 on the device (onmf_widen fused with the TF32 split); arithmetic unchanged.  Reported beside the fp32 line.
    e2e_u8 = None
    if d % 4 == 0:
        del host
        # the same minibatches as the fp32 line, quantised to 8 bits (pixel data)
        q8 = torch.clamp(torch.round(pool * 255.0), 0, 255).to(torch.uint8).cpu()
        host8 = [q8.clone().pin_memory() for _ in range(2)]
        del q8
        if snap is not None:
            with torch.cuda.stream(main):
                eng.set_state(snap[0], snap[1], snap[2])
            t = snap[3]
        for i in range(e2e_warm):
            t += 1
            eng.step_host(host8[i & 1], float(t), W_host)
        eng.flush()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(main)
        for i in range(e2e_steps):
            t += 1
            eng.step_host(host8[i & 1], float(t), W_host)
        eng.flush()
        e1.record(main)
        barrier()
        u8_ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(u8_ms, op=dist.ReduceOp.MAX)
        assert np.isfinite(float(W_host.double().sum()))
        e2e_u8 = {"value": n_global * e2e_steps / (float(u8_ms.item()) * 1e-3), "unit": UNIT, "h2d_bytes_per_step": n * d,
                  "d2h_bytes_per_step": d * k * 4, "steps": e2e_steps,
                  "coder_ms_per_launch": float(np.mean(eng.read_lars_ms()[-e2e_steps:])) if (eng.fused and not graph_mode) else None,
                  "ms_per_step": float(u8_ms.item()) / e2e_steps,
                  "api": "OnmfEngine.step_host(pinned uint8 Xt, t, W_out_host)  # storage u8, x/255 widened on the device, fp32 arithmetic"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---------------- roofline of the dominant kernel (LARS coder) -------------------------------------------
    hbm_peak, peak_src = measured_peaks()
    tsz = 4
    alg_bytes = (2.0 * n * k + k * k) * tsz                 # read Ct (n x k) + G (k x k), write Ht (n x k), once
    achieved = alg_bytes / (lars_ms * 1e-3) / 1e9
    cols = max(stats["columns"] + stats["overflow"], 1)
    # executed work of the solver, counted in-kernel: per knot with active size s the kernel does one k x s
    # correlation pass (2ks flop, 4ks bytes of Gram rows through L1/shared memory) and, on the FP64 packed inverse,
    # u = M g (2 s^2 flop, 8 s^2 bytes) + the rank-1 update of the lower triangle (s^2 flop, 8 s^2 bytes)
    flop = 2.0 * k * stats["sum_active"] + 3.0 * stats["sum_active2"]
    smem_bytes = 4.0 * k * stats["sum_active"] + 16.0 * stats["sum_active2"]
    lars_total_s = lars_ms * 1e-3 * K
    sm_clock = (clocks.get("sm_mhz") or 1900.0) * 1e6
    fp32_peak = 148 * 128 * 2 * sm_clock / 1e12               # TFLOP/s at the observed clock
    smem_peak = 148 * 128 * sm_clock / 1e9                    # GB/s  (128 B/clk/SM)
    fp32_ach = flop / lars_total_s / 1e12
    smem_ach = smem_bytes / lars_total_s / 1e9
    # The dominant kernel is the LARS coder.  Its binding roof is the FP32 FMA pipe / the L1-shared-memory data pipe
    # (SURVEY.md §8d: "FMA/shared-memory throughput for the lasso solver"), not HBM -- algorithmic HBM bytes per launch
    # (read Ct, write Ht, read G once) would take 0.08 ms.  `achieved` = executed solver work counted in-kernel (per
    # knot with active size s: one k x s correlation pass = 2ks flop, FP64 factor sweeps = 3 s^2 flop) / launch time;
    # `peak` = 148 SMs x 128 FMA lanes x 2 at the SM clock observed during the timed region.  The HBM and
    # shared-memory views are kept beside it.
    # What the profiler shows to be the binding unit (profiles/r2_lars_fast.md) is the L1 data pipe: the Gram rows of the
    # correlation pass (4ks bytes per knot, the algorithmic minimum of a path-following coder), the FP64 factor sweeps,
    # gathers and shuffles all pass through it; ncu: 78 % of its peak in every version of the kernel.  `l1_data_pipe`
    # reports the algorithmic part (Gram-row bytes only) live, the profiler's total utilisation as the recorded constant.
    gram_bytes = 4.0 * k * stats["sum_active"]
    l1_pipe = {"algorithmic_gram_row_gbs": gram_bytes / lars_total_s / 1e9, "peak_gbs_at_clock": smem_peak,
               "frac_algorithmic": gram_bytes / lars_total_s / 1e9 / smem_peak,
               "ncu_total_utilisation": 0.78 if (args.workload == "cfg5" and not args.batch) else None,
               "source": "profiles/r2_lars_fast.md (l1tex__data_pipe_lsu_wavefronts, pct of peak)"}
    roofline = {"bound": "fp32_fma", "kernel": "lars_fast_kernel / lars_kernel (K3 sparse coder)", "achieved": fp32_ach, "peak": fp32_peak,
                "unit": "TFLOP/s", "frac": fp32_ach / fp32_peak,
                "peak_source": "148 SMs x 128 lanes x 2 flop x observed SM clock (%.0f MHz)" % (sm_clock / 1e6),
                # dram__bytes_read.sum + dram__bytes_write.sum of one first-tier launch at cfg5, N=1 (ncu --set full,
                # profiles/); only valid for that workload
                "traffic": LARS_DRAM_BYTES if (args.workload == "cfg5" and world == 1 and not args.batch) else None,
                "ms_per_launch": lars_ms, "share_of_step": lars_ms * K / elapsed_ms,
                "hbm": {"algorithmic_bytes": alg_bytes, "achieved_gbs": achieved, "peak_gbs": hbm_peak,
                        "frac": achieved / hbm_peak, "peak_source": peak_src},
                "smem": {"achieved_gbs": smem_ach, "peak_gbs_at_clock": smem_peak, "frac": smem_ach / smem_peak},
                "l1_data_pipe": l1_pipe,
                "work": {"knots_per_column": stats["knots"] / cols, "mean_active": stats["sum_active"] / max(stats["knots"], 1),
                         "max_active": stats["max_active"], "drops_per_column": stats["drops"] / cols,
                         "overflow_columns": stats["overflow"], "flagged_columns": stats["flagged"],
                         "executed_gflop_per_launch": flop / K / 1e9}}

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        procs = args.cpu_procs or host_cores()
        ccols = args.cpu_cols or int(min(n_global, max(64 * procs, 12e3 * procs / PER_COL_MS[args.workload])))   # ~12 s
        cval, csec = cpu_reference_step(d, k, alpha, ccols, steps=1, warmup=0, procs=procs)
        cpu = {"value": cval, "unit": UNIT, "cores": procs, "kind": "port",
               "sample": "%d of %d columns, 1 step (%.1f s), numpy + scikit-learn lasso_lars via the oracle port, columns "
                         "split over %d worker processes (the reference runs this loop on one core: ~%.0f samples/s per "
                         "core); host cpus=%s" % (ccols, n_global, csec, procs, cval / procs, os.cpu_count())}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": elapsed_ms / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.workload, d, k, n_global, alpha), "d": d, "k": k, "global_batch": n_global,
                   "detail": "%d columns/GPU; fresh minibatch per step resampled from a resident pool; inputs (%.2f GB/GPU) "
                             "larger than L2" % (n, n * d * 4 / 1e9),
                   "parallelism": "dp%d (column shards, all-reduce of k x (k+d))" % world},
        "clocks": clocks, "gpu_launches": launches,
        "schedule": ("CUDA graph replay of the fused step (%d of %d timed steps); coder time of the roofline object from a "
                     "separate stream-scheduled pass" % (graph_steps, K)) if graph_mode else "two streams + events (onmf_step)",
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": n * d * 4, "d2h_bytes_per_step": d * k * 4,
                "steps": e2e_steps, "t_first": e2e_t_first, "coder_ms_per_launch": e2e_coder_ms,
                "api": "OnmfEngine.step_host(pinned float32 Xt, t, W_out_host)", "u8_storage": e2e_u8},
        "roofline": roofline, "cpu_baseline": cpu,
    }
    if outputs is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg5", choices=sorted(WORKLOADS) + ["next"],
                    help="cfgN: BASELINE.json configs; next: per-kernel lines of the K1 gathers, K5 and the SURVEY 8(f) rows (bench_next.py)")
    ap.add_argument("--quick", action="store_true", help="--workload next: smaller shapes")
    ap.add_argument("--only", default="", help="--workload next: comma-separated kernel names")
    ap.add_argument("--cpu-cols", type=int, default=0)
    ap.add_argument("--cpu-procs", type=int, default=0, help="worker processes of the CPU baseline (default: all host cores)")
    ap.add_argument("--batch", type=int, default=0, help="override the global minibatch size (analysis only; the line says so)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--timeline", action="store_true", help="print device timestamps of the step's kernels (analysis only)")
    ap.add_argument("--graph", default="auto", choices=["auto", "on", "off"],
                    help="replay the fused step as a CUDA graph (auto: the small workloads cfg1..cfg4 on one GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the last timed step's outputs to DIR/<name>.npy (float32): codes (rank 0's rows, at most "
                         "%d of them, a fixed seeded sample), W, A, B" % DUMP_CODE_ROWS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload == "next"):
        ap.error("--dump-outputs needs --impl ours and a cfgN workload")
    if args.workload == "next":
        import bench_next
        return bench_next.main((["--quick"] if args.quick else []) + (["--only", args.only] if args.only else []))
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "ours" and args.workload != "cfg5" and args.graph != "off" and args.warmup < 5:
        args.warmup = 5          # a step's graph is captured the second time its (buffer, parity) key is seen
    if args.impl == "reference":
        return run_reference(args)
    if args.gpus > 1 and "RANK" not in os.environ:
        # convenience: relaunch under torchrun on one node
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
