"""Whole-image reconstruction: banded by reference (reconstruct.reconstruct_image) against the materialised one-pass form.

Settings: grey image, 32 x 32 patches (d = 1024), k = 256 atoms cut from the image and normalised, fp32, the lasso coder,
stride 1, every position (include_last=True).  The image is a smooth field plus uniform noise, from a fixed seed.
    1024 x 1024 (986,049 patches): materialised vs banded (default max_band), alternated, `repeats` times each.  Each run
        reports ms from the host image to the host canvas (host clock around the call, which ends in a device-to-host copy)
        and the peak device bytes above what was allocated before the call.  A second, staged pass of the same calls
        splits the device time into covariances, coder, product Ht W^T and overlap mean (CUDA events around each stage,
        summed over bands).  The canvases of the two forms are compared bit for bit.
    4096 x 4096 (16,524,225 patches): banded only, time and peak memory.
One JSON line per measurement, each with the GPU name and power limit read in the same run.
    python profiles/tools/prof_recons.py [repeats]"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from onmf_ontf_ndl_b200 import OnmfEngine, _host, _lib, patches, reconstruct  # noqa: E402
from onmf_ontf_ndl_b200.engine import _Patches  # noqa: E402

P, K, ALPHA = 32, 256, 1.0
D = P * P
STAGES = ("gather_cov", "coder", "product", "overlap")


def gpu_info():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True)
        name, power = [s.strip() for s in out.splitlines()[0].split(",")]
    except Exception:
        name, power = torch.cuda.get_device_name(0), "unknown"
    return name, power


def image_and_dictionary(H, seed=0):
    rs = np.random.RandomState(seed)
    yy, xx = np.meshgrid(np.linspace(0, 12, H), np.linspace(0, 9, H), indexing="ij")
    img = (0.5 + 0.25 * np.sin(yy) * np.cos(xx) + 0.1 * rs.rand(H, H)).astype(np.float32)
    co = rs.randint(0, H - P + 1, size=(K, 2))
    W = np.stack([img[a:a + P, b:b + P].reshape(-1) for a, b in co], 1).astype(np.float64)
    return img, W / np.linalg.norm(W, axis=0)


class Stages:
    """CUDA events at stage boundaries on the current stream; elapsed ms per stage summed over bands"""

    def __init__(self):
        self.marks = []

    def mark(self, name):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        self.marks.append((name, e))

    def split(self):
        torch.cuda.synchronize()
        out = {s: 0.0 for s in STAGES}
        for (_, a), (name, b) in zip(self.marks, self.marks[1:]):
            out[name] += a.elapsed_time(b)
        return {s: round(v, 3) for s, v in out.items()}


def staged(img, W, bands):
    """the calls of reconstruct_image (lasso coder, fp32), CUDA events between the stages.  bands = [(0, n)] is the
    materialised form: one gather of the whole patch matrix and one dense coder call, as before banding."""
    dev = _host.device()
    H = img.shape[0]
    ny = nx = H - P + 1
    ys = np.arange(ny)
    t_img = torch.from_numpy(img).to(dev).reshape(H, H, 1)
    Wd = torch.from_numpy(W.astype(np.float32)).to(dev)
    Wt = torch.empty(K, D, device=dev)
    _lib.transpose(Wd, Wt)
    canvas = torch.empty(H, H, 1, device=dev)
    count = torch.empty(H, H, device=dev)
    eng = OnmfEngine(D, K, alpha=ALPHA, dtype=torch.float32, device=dev)
    f = eng.derive_foreign(Wd)
    one = len(bands) == 1
    mmax = max(j1 - j0 for j0, j1 in bands)
    R = torch.empty(mmax, D, device=dev)
    Xt = torch.empty(mmax, D, device=dev) if one else None
    st = torch.cuda.current_stream()
    s = Stages()
    s.mark("start")
    for j0, j1 in bands:
        m = j1 - j0
        jj = np.arange(j0, j1)
        corners = torch.from_numpy(np.stack([ys[jj // nx], ys[jj % nx]], 1).astype(np.int32)).to(dev)
        pm = _lib.make_patch_minibatch(t_img, P, corners, None, m, 1.0)
        eng._reserve(m)
        Ct, Ht = eng.Ct[:m], eng.Ht[:m]
        if one:
            _lib.gather_patches(t_img, corners, P, Xt[:m])
            eng._cov_into(Xt[:m], None, None, 1.0, m, f.W, f.Whi, f.Wlo, Ct, st)
        else:
            eng._cov_into(None, _Patches(pm), None, 1.0, m, f.W, f.Whi, f.Wlo, Ct, st)
        s.mark("gather_cov")
        eng._lars(f, Ct, ALPHA, Ht, -1 if one else 0)
        s.mark("coder")
        _lib.cov(Ht, Wt, R[:m])
        s.mark("product")
        _lib.patch_grid_accumulate(R[:m], j0, j1, ny, nx, P, 1, 1, H, H, canvas, count)
        s.mark("overlap")
    out = canvas.cpu().numpy()[:, :, 0]
    return out, s.split()


def materialised(img, W):
    """the one-pass form: whole patch matrix, codes and reconstructions resident at once"""
    dev = _host.device()
    H = img.shape[0]
    n = (H - P + 1) ** 2
    t_img = torch.from_numpy(img).to(dev).reshape(H, H, 1)
    coords = torch.from_numpy(patches.all_patch_coords(img.shape, P)).to(dev)
    Xt = torch.empty(n, D, device=dev)
    _lib.gather_patches(t_img, coords, P, Xt)
    Wd = torch.from_numpy(W.astype(np.float32)).to(dev)
    eng = OnmfEngine(D, K, alpha=ALPHA, dtype=torch.float32, device=dev)
    Ht = eng.sparse_code(Xt, Wd, alpha=ALPHA).clone()
    Wt = torch.empty(K, D, device=dev)
    _lib.transpose(Wd, Wt)
    R = torch.empty(n, D, device=dev)
    _lib.cov(Ht, Wt, R)
    canvas = torch.zeros(H, H, 1, device=dev)
    count = torch.zeros(H, H, device=dev)
    _lib.patch_grid_mean(R, H - P + 1, H - P + 1, P, 1, 1, H, H, canvas, count)
    return canvas.cpu().numpy()[:, :, 0].astype(np.float64)         # what reconstruct_image returns


def banded(img, W):
    return reconstruct.reconstruct_image(img, W, P, 1, alpha=ALPHA, coder="lasso_lars", precision="fp32", include_last=True)[0]


def timed(fn, *a):
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    out = fn(*a)
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3
    return out, ms, torch.cuda.max_memory_allocated() - base


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 3
    name, power = gpu_info()
    img, W = image_and_dictionary(1024)
    n = (1024 - P + 1) ** 2
    bands = reconstruct._band_plan(n, 262144, _lib.coder_band_floor())
    for fn in (materialised, banded):                                  # warm-up: module loads, allocator pools
        fn(img, W)
    res = {v: dict(ms=[], peak=[]) for v in ("materialised", "banded")}
    outs = {}
    for _ in range(reps):
        for v, fn in (("materialised", materialised), ("banded", banded)):
            out, ms, peak = timed(fn, img, W)
            res[v]["ms"].append(ms)
            res[v]["peak"].append(peak)
            outs[v] = out
    split = {"materialised": staged(img, W, [(0, n)])[1], "banded": staged(img, W, bands)[1]}
    for v in ("materialised", "banded"):
        r = res[v]
        print(json.dumps(dict(
            image="1024x1024", variant=v, gpu=name, power_limit=power, patches=n, d=D, k=K, dtype="fp32", coder="lasso_lars",
            bands=len(bands) if v == "banded" else 1, ms=[round(x, 2) for x in r["ms"]], ms_median=round(float(np.median(r["ms"])), 2),
            peak_device_mb=round(max(r["peak"]) / 2 ** 20, 1), stage_ms=split[v],
            canvas_bitwise_equal=bool(np.array_equal(outs["materialised"].view(np.int64), outs["banded"].view(np.int64))))),
            flush=True)
    del outs
    img4, W4 = image_and_dictionary(4096, seed=1)
    n4 = (4096 - P + 1) ** 2
    out, ms, peak = timed(banded, img4, W4)
    print(json.dumps(dict(image="4096x4096", variant="banded", gpu=name, power_limit=power, patches=n4, d=D, k=K, dtype="fp32",
                          coder="lasso_lars", bands=len(reconstruct._band_plan(n4, 262144, _lib.coder_band_floor())),
                          ms=round(ms, 2), peak_device_mb=round(peak / 2 ** 20, 1), canvas_finite=bool(np.isfinite(out).all()))),
          flush=True)


if __name__ == "__main__":
    main()
