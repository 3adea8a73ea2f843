"""Patch minibatches by reference vs the materialised pool at the cfg5 shape (32 x 32 grey patches, d = 1024, k = 256).

All 4,068,289 patch positions of one 2048 x 2048 grey image; 262,144-column minibatches drawn from them (one seeded index
sequence shared by every variant).  Three variants see the same values:
    u8    ImagePatches of the uint8 image (value = float(u8) * float(1/255), widened inside the loaders)
    f32   ImagePatches of the fp32 image float(u8) * float(1/255)
    pool  the fp32 pool of all 4,068,289 patches materialised from that fp32 image (16.7 GB), read through step_pool
Each run: a fresh engine, the same initial dictionary, 5 warm-up and 20 device-timed steps (CUDA events around the steps
on the engine's main stream, as bench.py does); variants alternate and the whole set repeats to show the spread.  Then the
fused covariance and surrogate kernels alone, CUDA-event timed over 10 launches each on the same minibatch.
One JSON line per variant (the GPU name and power limit read in the same run), with the final W compared bitwise to the
pool variant's.
    python profiles/tools/prof_patches.py [repeats]"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from onmf_ontf_ndl_b200 import OnmfEngine, _lib, patches  # noqa: E402

P, K, HW, N_MB, WARM, TIMED = 32, 256, 2048, 262144, 5, 20
D = P * P


def gpu_info():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True)
        name, power = [s.strip() for s in out.splitlines()[0].split(",")]
    except Exception:
        name, power = torch.cuda.get_device_name(0), "unknown"
    return name, power


def ev():
    return torch.cuda.Event(enable_timing=True)


def run(variant, srcs, idx_all, W0):
    dev = torch.device("cuda", 0)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    eng = OnmfEngine(D, K, alpha=1.0, dtype=torch.float32, device=dev)
    assert eng.fused_tc
    eng.set_state(W0)

    def step(t):
        idx = idx_all[t - 1]
        if variant == "pool":
            eng.step_pool(srcs["pool"], idx, float(t))
        else:
            eng.step_patches(srcs[variant], idx, float(t))
    for t in range(1, WARM + 1):
        step(t)
    torch.cuda.synchronize()
    e0, e1 = ev(), ev()
    e0.record(eng.main)
    for t in range(WARM + 1, WARM + TIMED + 1):
        step(t)
    eng.flush()
    e1.record(eng.main)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / TIMED
    peak = torch.cuda.max_memory_allocated() - base
    # the two fused tensor-core products alone, on the last minibatch, with the final dictionary
    idx = idx_all[WARM + TIMED - 1]
    Ct, Ht = eng.Ct[:N_MB], eng.Ht[:N_MB]
    P_ = eng.P[0]
    if variant == "pool":
        cov = lambda: _lib.cov_fused_tc(srcs["pool"], idx, N_MB, eng.Whi, eng.Wlo, Ct, stream=eng.main)
        sur = lambda: _lib.surrogate_fused_tc(Ht, srcs["pool"], idx, N_MB, D, P_, eng._ws_sur, stream=eng.main)
    else:
        pm = srcs[variant].minibatch(idx)
        cov = lambda: _lib.cov_fused_tc_patches(pm, eng.Whi, eng.Wlo, Ct, stream=eng.main)
        sur = lambda: _lib.surrogate_fused_tc_patches(Ht, pm, P_, eng._ws_sur, stream=eng.main)
    kern = {}
    for name, fn in (("cov_fused_ms", cov), ("sur_fused_ms", sur)):
        fn()
        a, b = ev(), ev()
        a.record(eng.main)
        for _ in range(10):
            fn()
        b.record(eng.main)
        torch.cuda.synchronize()
        kern[name] = a.elapsed_time(b) / 10
    W = eng.state()[0].clone()
    del eng
    torch.cuda.empty_cache()
    return ms, peak, kern, W


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 3
    name, power = gpu_info()
    dev = torch.device("cuda", 0)
    rs = np.random.RandomState(0)
    img8 = rs.randint(0, 256, size=(HW, HW)).astype(np.uint8)
    co = patches.all_patch_coords(img8.shape, P)
    n_pos = co.shape[0]
    t8 = torch.from_numpy(img8).to(dev)
    f32 = t8.float() * torch.tensor(1.0 / 255.0, dtype=torch.float32)
    srcs = {"u8": patches.ImagePatches(img8, P, co), "f32": patches.ImagePatches(f32, P, co)}
    pool = torch.empty(n_pos, D, dtype=torch.float32, device=dev)
    _lib.gather_patches(f32.reshape(HW, HW, 1).contiguous(), srcs["f32"].coords, P, pool)
    srcs["pool"] = pool
    resident = {"u8": img8.nbytes + co.nbytes, "f32": f32.numel() * 4 + co.nbytes, "pool": pool.numel() * 4}
    idx_all = torch.from_numpy(rs.randint(0, n_pos, size=(WARM + TIMED, N_MB))).to(dev)
    W0 = torch.from_numpy(rs.rand(D, K).astype(np.float32)).to(dev)
    res = {v: dict(ms=[], peak=[], cov=[], sur=[], W=None) for v in ("u8", "f32", "pool")}
    for _ in range(reps):
        for v in ("u8", "f32", "pool"):
            ms, peak, kern, W = run(v, srcs, idx_all, W0)
            r = res[v]
            r["ms"].append(ms); r["peak"].append(peak); r["cov"].append(kern["cov_fused_ms"]); r["sur"].append(kern["sur_fused_ms"])
            if r["W"] is None:
                r["W"] = W
            r["W_repeats"] = bool(torch.equal(r["W"].view(torch.int32), W.view(torch.int32)))
    pool_ms = float(np.median(res["pool"]["ms"]))
    for v in ("u8", "f32", "pool"):
        r = res[v]
        med = float(np.median(r["ms"]))
        print(json.dumps(dict(
            variant=v, gpu=name, power_limit=power, positions=n_pos, minibatch=N_MB, d=D, k=K, warmup=WARM, timed_steps=TIMED,
            ms_per_step=[round(x, 4) for x in r["ms"]], ms_per_step_median=round(med, 4),
            samples_per_s=round(N_MB / (med / 1e3), 1), vs_pool=round(med / pool_ms, 4),
            cov_fused_ms=[round(x, 4) for x in r["cov"]], sur_fused_ms=[round(x, 4) for x in r["sur"]],
            peak_device_mb_above_baseline=round(max(r["peak"]) / 2 ** 20, 1), resident_data_mb=round(resident[v] / 2 ** 20, 1),
            W_bitwise_equal_to_pool=bool(torch.equal(r["W"].view(torch.int32), res["pool"]["W"].view(torch.int32))),
            W_repeats=r["W_repeats"])), flush=True)


if __name__ == "__main__":
    main()
