"""Network reconstruction from device motif chains: the one-pass reconstruct_network(G, W, chains.sample(n)) against the
streamed reconstruct_network_chains(chains, W, n), on the graph of prof_motif_chain.py (seeded, 10^6 nodes, mean degree about
20, 5 hubs of degree about 10^4), kk = 21, r = 25, a unit-norm random W, pivot chains, fp32, alpha = 0.
    1. Both forms at a size both fit (CHAINS x SAMPLES states), alternated REPS times, each on a fresh chain object of the
       same seed.  states_per_s: states over the host clock around the whole call (sampling, coding, scatter, the copy of
       the table to the host and its sort), after a warm-up call of each form.  peak_bytes: torch.cuda.max_memory_allocated
       during the call, less what was allocated before it (the graph and the chain states).  Both forms must give the same
       pairs and counts (equal = true).
    2. One more call of each form with CUDA events around every kernel wrapper (a run of its own: the events cost host
       time): device seconds per stage -- sample (chain kernel), patches, cov (X W), coder (LARS), product (H W^T), scatter
       (edge_scatter_add / edge_table_add), grow (edge_table_grow).
    3. The streamed form alone at LARGE_CHAINS x LARGE_SAMPLES states: distinct pairs, peak bytes, states/s.
One JSON line per measurement, each with the GPU name and power limit read in the same run.
    python profiles/tools/prof_recons_network.py [large_chains large_samples]"""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np  # noqa: E402
import scipy.sparse as sp  # noqa: E402
import torch  # noqa: E402

from onmf_ontf_ndl_b200 import _lib, patches, reconstruct  # noqa: E402
from prof_motif_chain import gpu_info, make_graph  # noqa: E402

KK, R, SEED, MCMC, PREC = 21, 25, 1, "pivot", "fp32"
CHAINS, SAMPLES, REPS = 10_000, 100, 3
STAGES = ("sample", "patches", "cov", "coder", "product", "scatter", "grow")


class StageEvents:
    """CUDA events around every call of the kernel wrappers the two forms use, summed per stage"""

    def __init__(self):
        self.ev = {s: [] for s in STAGES}
        self.saved = []

    def _wrap(self, owner, name, stage, setter):
        fn = owner[name] if isinstance(owner, dict) else getattr(owner, name)

        def timed(*a, **k):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn(*a, **k)
            e1.record()
            self.ev[stage(*a) if callable(stage) else stage].append((e0, e1))
            return out
        self.saved.append((owner, name, fn, setter))
        setter(owner, name, timed)

    def __enter__(self):
        seta, seti = setattr, dict.__setitem__
        self._wrap(patches._MOTIF_STEPS, MCMC, "sample", seti)
        self._wrap(_lib, "motif_patches", "patches", seta)
        self._wrap(_lib, "cov", lambda X, W, *_: "product" if X.shape[1] == R else "cov", seta)
        self._wrap(_lib, "lasso_lars", "coder", seta)
        for name in ("edge_scatter_add", "edge_table_add"):
            self._wrap(_lib, name, "scatter", seta)
        self._wrap(_lib, "edge_table_grow", "grow", seta)
        return self

    def __exit__(self, *exc):
        for owner, name, fn, setter in reversed(self.saved):
            setter(owner, name, fn)

    def seconds(self):
        torch.cuda.synchronize()
        return {s: round(sum(a.elapsed_time(b) for a, b in ev) / 1e3, 4) for s, ev in self.ev.items()}


def run(form, csr, M, W, n_chains, n_samples):
    ch = patches.MotifChains(csr, KK, n_chains, SEED, mcmc=MCMC)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    t = time.perf_counter()
    if form == "one_pass":
        res = reconstruct.reconstruct_network(M, W, ch.sample(n_samples), alpha=0, precision=PREC)
    else:
        res = reconstruct.reconstruct_network_chains(ch, W, n_samples, alpha=0, precision=PREC)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t
    peak = torch.cuda.max_memory_allocated() - base
    del ch
    torch.cuda.empty_cache()
    return res, dt, peak


def main():
    large_chains = int(sys.argv[1]) if len(sys.argv) > 1 else 100_000
    large_samples = int(sys.argv[2]) if len(sys.argv) > 2 else 200
    name, power = gpu_info()
    rp, ci = make_graph()
    csr = (rp, ci)
    n_nodes = len(rp) - 1
    M = sp.csr_matrix((np.ones(len(ci), dtype=np.int8), ci, rp), shape=(n_nodes, n_nodes))
    W = np.random.RandomState(0).rand(KK * KK, R)
    W /= np.linalg.norm(W, axis=0)
    base = dict(gpu=name, power_limit=power, nodes=n_nodes, kk=KK, r=R, mcmc=MCMC, precision=PREC)
    n = CHAINS * SAMPLES

    for form in ("one_pass", "streamed"):                                   # warm-up: module load, allocator
        run(form, csr, M, W, 1000, 10)
    ref = None
    for rep in range(REPS):
        for form in ("one_pass", "streamed"):
            (p, w, c), dt, peak = run(form, csr, M, W, CHAINS, SAMPLES)
            key = (p.astype(np.int64), c)
            if ref is None:
                ref = key
            equal = bool(np.array_equal(key[0], ref[0]) and np.array_equal(key[1], ref[1]))
            print(json.dumps(dict(base, what="compare", form=form, rep=rep, chains=CHAINS, samples=SAMPLES, states=n,
                                  seconds=round(dt, 3), states_per_s=n / dt, peak_bytes=int(peak), distinct_pairs=len(c),
                                  equal=equal)), flush=True)
            del p, w, c
    del ref, key

    for form in ("one_pass", "streamed"):
        with StageEvents() as ev:
            _, dt, peak = run(form, csr, M, W, CHAINS, SAMPLES)
        print(json.dumps(dict(base, what="stages", form=form, chains=CHAINS, samples=SAMPLES, states=n, seconds=round(dt, 3),
                              stage_seconds=ev.seconds())), flush=True)

    nl = large_chains * large_samples
    (p, w, c), dt, peak = run("streamed", csr, M, W, large_chains, large_samples)
    print(json.dumps(dict(base, what="large", form="streamed", chains=large_chains, samples=large_samples, states=nl,
                          seconds=round(dt, 3), states_per_s=nl / dt, peak_bytes=int(peak), distinct_pairs=len(c),
                          count_sum=int(c.sum()), expected_count_sum=nl * KK * KK)), flush=True)


if __name__ == "__main__":
    main()
