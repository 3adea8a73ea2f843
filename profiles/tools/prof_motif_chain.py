"""Device motif chains (patches.MotifChains, csrc/motif_chain.cu) against the host walk.

Graph: seeded, 10^6 nodes, about 10^7 uniformly random undirected edges (average degree about 20) plus 5 hubs joined to
10^4 random nodes each; symmetric CSR, 2.1e7 stored entries (84 MB of colidx, inside the 126 MB L2 with rowptr's 8 MB).
    1. Glauber states per second on the device (chains x steps / time): kk = 21 and kk = 6, 10^4, 10^5 and 10^6 chains.  The
       timed call is MotifChains.sample(1, steps_per_sample=S) (validation kernel + S steps + one output slice), CUDA events
       around it, S chosen from a probe so that each run lasts about 2 s.
    2. The same count from the numpy oracle (oracle/motif_chain.run_chain) on one host core: one chain at a time, as the
       reference walks, for about 5 s per kk.
    3. One NDL epoch at the cfg3 shape (kk = 21, d = 441, r = 25, sample_size = batch = 10,000, Online_NMF with iterations=11,
       i.e. 10 steps over the whole sample, lasso coder, fp32): device chains (100 chains x 100 states, the ndl.train_dict
       default, and 10^4 chains x 1 state; the one-time MotifChains construction is reported apart) with the patches trained
       on in place, against the host walk (the oracle chain,
       10^4 consecutive states of one chain) followed by host patches and Online_NMF on the host matrix.  Host clock around
       each stage, each stage ending in a device synchronise.
One JSON line per measurement, each with the GPU name and power limit read in the same run.
    python profiles/tools/prof_motif_chain.py"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import scipy.sparse as sp  # noqa: E402
import torch  # noqa: E402

from onmf_ontf_ndl_b200 import Online_NMF, patches  # noqa: E402
from oracle import motif_chain as mc  # noqa: E402


def gpu_info():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True)
        name, power = [s.strip() for s in out.splitlines()[0].split(",")]
    except Exception:
        name, power = torch.cuda.get_device_name(0), "unknown"
    return name, power


def make_graph(n=1_000_000, m=10_000_000, hubs=5, hub_deg=10_000, seed=0):
    rs = np.random.RandomState(seed)
    a = rs.randint(0, n, size=m)
    b = rs.randint(0, n, size=m)
    ha = np.repeat(np.arange(hubs), hub_deg)
    hb = rs.randint(hubs, n, size=hubs * hub_deg)
    r = np.concatenate([a, b, ha, hb])
    c = np.concatenate([b, a, hb, ha])
    keep = r != c
    M = sp.csr_matrix((np.ones(int(keep.sum()), dtype=np.int8), (r[keep], c[keep])), shape=(n, n))
    M.sum_duplicates()
    M.sort_indices()
    return M.indptr.astype(np.int64), M.indices.astype(np.int32)


def timed_sample(ch, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    ch.sample(1, steps_per_sample=steps)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3


def main():
    name, power = gpu_info()
    t = time.time()
    rp, ci = make_graph()
    csr = (rp, ci)
    deg = np.diff(rp)
    base = dict(gpu=name, power_limit=power, nodes=len(rp) - 1, entries=int(rp[-1]), max_degree=int(deg.max()),
                mean_degree=round(float(deg.mean()), 2))
    print(json.dumps(dict(base, what="graph", build_s=round(time.time() - t, 1))), flush=True)

    for kk in (21, 6):
        for n_chains in (10_000, 100_000, 1_000_000):
            ch = patches.MotifChains(csr, kk, n_chains, seed=1)
            timed_sample(ch, 5)                                        # warm-up (module load, L2)
            probe = 50
            dt = timed_sample(ch, probe)
            steps = max(probe, int(probe * 2.0 / max(dt, 1e-6)))
            dt = timed_sample(ch, steps)
            print(json.dumps(dict(base, what="device_chain", kk=kk, chains=n_chains, steps=steps, seconds=round(dt, 3),
                                  states_per_s=n_chains * steps / dt)), flush=True)
            del ch
            torch.cuda.empty_cache()

    for kk in (21, 6):
        x0 = mc.chain_init(rp, ci, kk, 1, 0, 1)
        steps, t0 = 0, time.time()
        while time.time() - t0 < 5.0:
            x0 = mc.run_chain(rp, ci, x0, 0, 1, steps, 1, 500)[1]
            steps += 500
        dt = time.time() - t0
        print(json.dumps(dict(base, what="host_oracle_chain", kk=kk, chains=1, steps=steps, seconds=round(dt, 3),
                              states_per_s=steps / dt, host_cores=1)), flush=True)

    kk, r, sample, iters = 21, 25, 10_000, 11
    for n_chains in (100, 10_000):
        torch.cuda.synchronize()
        tc = time.time()
        ch = patches.MotifChains(csr, kk, n_chains, seed=2)            # once per graph: CSR check, upload, init
        torch.cuda.synchronize()
        setup_ms = round(1e3 * (time.time() - tc), 2)
        for rep in range(2):                                           # first pass warms the engine up
            np.random.seed(5)
            torch.cuda.synchronize()
            t0 = time.time()
            X = patches.SamplePool(ch.patches(sample // n_chains))
            torch.cuda.synchronize()
            t1 = time.time()
            Online_NMF(X, r, iterations=iters, batch_size=sample, precision="fp32").train_dict()
            torch.cuda.synchronize()
            t2 = time.time()
        print(json.dumps(dict(base, what="ndl_epoch_device", kk=kk, r=r, sample_size=sample, batch=sample, chains=n_chains,
                              nmf_steps=iters - 1, chains_setup_ms=setup_ms, sample_ms=round(1e3 * (t1 - t0), 2), train_ms=round(1e3 * (t2 - t1), 2),
                              epoch_ms=round(1e3 * (t2 - t0), 2))), flush=True)
    np.random.seed(5)
    t0 = time.time()
    x0 = mc.chain_init(rp, ci, kk, 1, 0, 2)
    out, _ = mc.run_chain(rp, ci, x0, 0, 2, 0, sample)
    t1 = time.time()
    X = patches.motif_patches(csr, out[:, 0, :])
    torch.cuda.synchronize()
    t2 = time.time()
    Online_NMF(X, r, iterations=iters, batch_size=sample, precision="fp32").train_dict()
    torch.cuda.synchronize()
    t3 = time.time()
    print(json.dumps(dict(base, what="ndl_epoch_host_walk", kk=kk, r=r, sample_size=sample, batch=sample, chains=1,
                          nmf_steps=iters - 1, walk_ms=round(1e3 * (t1 - t0), 2), patches_ms=round(1e3 * (t2 - t1), 2),
                          train_ms=round(1e3 * (t3 - t2), 2), epoch_ms=round(1e3 * (t3 - t0), 2))), flush=True)


if __name__ == "__main__":
    main()
