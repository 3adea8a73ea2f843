"""Device Ising chains (patches.IsingChains, csrc/ising_chain.cu) against a host sampler.

    1. Site updates per second on the device (chains x H x W x sweeps / time), beta = 0.44: 200 x 200 with 1 chain (the
       Ising driver's case; the shared-memory form runs one CTA, so one SM), 10^3 and 10^4 chains; 1024 x 1024 with 16
       chains (the global form, one launch per half-sweep).  The timed call is IsingChains.sample(1, sweeps_per_sample=S)
       (S sweeps + one fp32 frame per chain), CUDA events around it, S chosen from a probe so that each run lasts about 1 s.
    2. The same rate from the numpy oracle (oracle/ising_chain.run_chain) on one host core, one 200 x 200 chain, about 3 s.
    3. One Ising-driver epoch (200 x 200 lattice, one sweep, 20 x 20 patches, r = 100, 1000 patches, batch 50, Online_NMF
       with iterations = 20, subsample, lasso coder, fp32): the device chain with the patches read out of the frame by
       reference (ising.train_dict's epoch), against the host sampler (the oracle's sweep) followed by host patches and
       Online_NMF on the host matrix.  Host clock around each stage, each stage ending in a device synchronise; the median of
       5 epochs after one warm-up epoch.
One JSON line per measurement, each with the GPU name and power limit read in the same run.
    python profiles/tools/prof_ising.py"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from onmf_ontf_ndl_b200 import Online_NMF, _lib  # noqa: E402
from onmf_ontf_ndl_b200.patches import ImagePatches, IsingChains, frame_patch_coords, gather_patches  # noqa: E402
from oracle import ising_chain as ic  # noqa: E402

BETA = 0.44


def gpu_info():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True)
        name, power = [s.strip() for s in out.splitlines()[0].split(",")]
    except Exception:
        name, power = torch.cuda.get_device_name(0), "unknown"
    return name, power


def timed_sample(ch, sweeps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    ch.sample(1, sweeps_per_sample=sweeps)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / 1e3


def device_rate(shape, n_chains):
    ch = IsingChains(shape, BETA, n_chains, 1)
    timed_sample(ch, 2)                                          # warm-up (module load, attribute, occupancy query)
    S = 4
    while timed_sample(ch, S) < 0.05:
        S *= 4
    S = max(1, int(S * 1.0 / timed_sample(ch, S)))
    dt = timed_sample(ch, S)
    return dict(form=_lib.ising_chain_plan(*shape)["form"], sweeps=S, seconds=round(dt, 4),
                site_updates_per_s=float(n_chains) * shape[0] * shape[1] * S / dt)


def oracle_rate(shape=(200, 200), budget=3.0):
    x = ic.chain_init(shape[0], shape[1], 1, 0, 1)
    thr = ic.thresholds(BETA)
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < budget:
        _, x = ic.run_chain(x, thr, 0, 1, n, 1)
        n += 1
    dt = time.perf_counter() - t0
    return dict(sweeps=n, seconds=round(dt, 3), site_updates_per_s=shape[0] * shape[1] * n / dt)


def epoch_times(reps=5):
    shape, p, r, N, bs, it = (200, 200), 20, 100, 1000, 50, 20
    kw = dict(iterations=it, batch_size=bs, subsample=True, precision="fp32")
    dev, host = [], []
    ch = IsingChains(shape, BETA, 1, 2)
    x = ic.chain_init(shape[0], shape[1], 1, 0, 2)
    thr = ic.thresholds(BETA)
    for rep in range(reps + 1):
        # device: one sweep, corners, Online_NMF on the frame by reference
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        frames = ch.sample(1, 1)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        X = ImagePatches(frames.reshape(shape), p, frame_patch_coords(1, shape, p, N))
        Online_NMF(X, r, keep_code=False, **kw).train_dict()
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        # host: the oracle's sweep, host patches, Online_NMF on the host matrix
        _, x = ic.run_chain(x, thr, 0, 2, rep, 1)
        t3 = time.perf_counter()
        Xh = gather_patches(x[0].astype(np.float64), frame_patch_coords(1, shape, p, N), p)
        t4 = time.perf_counter()
        Online_NMF(Xh, r, **kw).train_dict()
        torch.cuda.synchronize()
        t5 = time.perf_counter()
        if rep:
            dev.append((t1 - t0, t2 - t1))
            host.append((t3 - t2, t4 - t3, t5 - t4))
    med = lambda rows, i: float(np.median([row[i] for row in rows])) * 1e3
    return dict(device_ms=dict(sample=med(dev, 0), train=med(dev, 1), total=med([(a + b,) for a, b in dev], 0)),
                host_ms=dict(sample=med(host, 0), patches=med(host, 1), train=med(host, 2),
                             total=med([(a + b + c,) for a, b, c in host], 0)))


def main():
    assert torch.cuda.is_available(), "prof_ising.py measures on the GPU"
    name, power = gpu_info()
    emit = lambda rec: print(json.dumps(dict(rec, gpu=name, power_limit=power)), flush=True)
    for shape, n in (((200, 200), 1), ((200, 200), 1000), ((200, 200), 10000), ((1024, 1024), 16)):
        emit(dict(what="device", shape=list(shape), n_chains=n, **device_rate(shape, n)))
    emit(dict(what="oracle_one_core", shape=[200, 200], n_chains=1, **oracle_rate()))
    emit(dict(what="driver_epoch", **epoch_times()))


if __name__ == "__main__":
    main()
