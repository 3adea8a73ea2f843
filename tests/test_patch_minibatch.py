"""Patch minibatches by reference (ImagePatches, OnmfEngine.step_patches, the *_patches entry points): every product and
every training step must give the same bits as the same call on the materialised pool of the same patches with the same
indices -- only the addressing differs.  NaN rows (an index outside [0, N), a corner whose patch leaves the image) are
compared as int bit patterns."""
import ctypes
import os
import socket
import subprocess

import numpy as np
import pytest
import torch

from onmf_ontf_ndl_b200 import _lib
from onmf_ontf_ndl_b200.patches import ImagePatches

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu
SCALE = 1.0 / 255.0


# ---------------------------------------------------------------------------------------------------------------- helpers
def bits(t):
    """int view of a float tensor: equal bits, NaN payloads included"""
    t = t.detach().contiguous()
    return t.view(torch.int64 if t.dtype == torch.float64 else torch.int32).cpu()


def assert_bits_equal(a, b, what=""):
    assert a.shape == b.shape, (what, a.shape, b.shape)
    ba, bb = bits(a), bits(b)
    if not torch.equal(ba, bb):
        bad = (ba != bb).nonzero()
        raise AssertionError("%s: %d of %d entries differ, first at %s" % (what, bad.shape[0], ba.numel(), bad[0].tolist()))


def make_image(rs, H, W, C, kind):
    """uint8 image and the device image of the requested kind: uint8, or float(u8) * float(1/255) in fp32 / fp64"""
    u8 = rs.randint(0, 256, size=(H, W, C)).astype(np.uint8)
    dev = torch.device("cuda")
    t8 = torch.from_numpy(u8).to(dev)
    if kind == "u8":
        return u8, t8
    f32 = t8.float() * torch.tensor(SCALE, dtype=torch.float32)
    return u8, (f32 if kind == "f32" else f32.double())


def corners(rs, H, W, p, N):
    return np.stack([rs.randint(0, H - p + 1, size=N), rs.randint(0, W - p + 1, size=N)], 1).astype(np.int32)


def pool_of(img, coords_dev, p, dtype):
    """the materialised (N x d) pool of the patches, with the pre-existing K1 gather; a uint8 image gives the pool of
    float(u8) * float(scale) (the values the kernels widen to)"""
    if img.dtype == torch.uint8:
        img = img.float() * torch.tensor(SCALE, dtype=torch.float32)
    img = img.to(dtype)
    C = img.shape[2]
    out = torch.empty(coords_dev.shape[0], p * p * C, dtype=dtype, device=img.device)
    return _lib.gather_patches(img.contiguous(), coords_dev, p, out)


def u8_pool_of(img8, coords, p):
    """the uint8 pool of the patches (valid corners only), by plain tensor indexing"""
    H, W, C = img8.shape
    c = torch.from_numpy(coords.astype(np.int64)).to(img8.device)
    r = torch.arange(p, device=img8.device)
    ys = (c[:, 0, None] + r[None, :])[:, :, None].expand(-1, p, p)
    xs = (c[:, 1, None] + r[None, :])[:, None, :].expand(-1, p, p)
    return img8[ys, xs].reshape(c.shape[0], p * p * C).contiguous()


def split(W):
    hi, lo = torch.empty_like(W), torch.empty_like(W)
    _lib.split_tf32(W, hi, lo)
    return hi, lo


# ------------------------------------------------------------------------------------------------------------- CPU tests
def test_patch_minibatch_struct_layout_matches_header(tmp_path):
    """ctypes mirror of onmf_patch_minibatch vs the C definition: same size and field offsets (compiled with gcc)."""
    fields = [f[0] for f in _lib.PatchMinibatch._fields_]
    src = tmp_path / "layout.c"
    body = "\n".join('  printf("%s %%zu\\n", offsetof(onmf_patch_minibatch, %s));' % (f, f) for f in fields)
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "onmf_b200.h"\nint main(void) {\n'
                   '  printf("sizeof %zu\\n", sizeof(onmf_patch_minibatch));\n' + body + "\n  return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    out = dict(l.split() for l in subprocess.check_output([str(exe)], text=True).splitlines())
    assert int(out["sizeof"]) == ctypes.sizeof(_lib.PatchMinibatch)
    for f in fields:
        assert int(out[f]) == getattr(_lib.PatchMinibatch, f).offset, f


@pytest.mark.parametrize("case", ["ndim", "coords_shape", "u8_fp64", "p_too_large", "coords_float"])
def test_image_patches_validates_before_touching_the_device(case, monkeypatch):
    from onmf_ontf_ndl_b200 import _host

    def no_device():
        raise AssertionError("device touched before validation")
    monkeypatch.setattr(_host, "device", no_device)
    img = np.zeros((20, 30), dtype=np.float32)
    co = np.zeros((5, 2), dtype=np.int32)
    with pytest.raises(ValueError):
        if case == "ndim":
            ImagePatches(np.zeros((2, 20, 30, 3)), 4, co)
        elif case == "coords_shape":
            ImagePatches(img, 4, np.zeros((5, 3), dtype=np.int32))
        elif case == "u8_fp64":
            ImagePatches(img.astype(np.uint8), 4, co, precision="fp64")
        elif case == "p_too_large":
            ImagePatches(img, 21, co)
        else:
            ImagePatches(img, 4, co.astype(np.float64))


def test_image_patches_rejects_pgd_and_shipped_compat_without_device():
    from onmf_ontf_ndl_b200 import Online_NMF
    src = ImagePatches.__new__(ImagePatches)          # shape / precision are all Online_NMF looks at before training
    src.d, src.N, src.precision, src.dtype = 16, 10, "fp32", torch.float32
    for kw in (dict(coder="pgd"), dict(compat="shipped_onmf")):
        with pytest.raises(ValueError):
            Online_NMF(src, n_components=4, **kw)


# ------------------------------------------------------------------------------------------------------------- GPU tests
FUSED_SHAPES = [(32, 1, 256), (16, 3, 64), (10, 1, 32), (6, 3, 36)]      # (p, C, k): cfg5, colour, straddling chunks x2


@gpu
@pytest.mark.parametrize("kind", ["f32", "u8"])
@pytest.mark.parametrize("p,C,k", FUSED_SHAPES)
def test_fused_kernels_patches_equal_pool(p, C, k, kind):
    rs = np.random.RandomState(p * 100 + C * 10 + k)
    H, W = p + 37, p + 29
    u8, img = make_image(rs, H, W, C, kind)
    N = 700
    co = corners(rs, H, W, p, N)
    co[N - 1] = (H - p + 1, 0)                          # patch leaves the image: NaN column
    src = ImagePatches(img, p, co, precision="fp32")
    d = p * p * C
    assert _lib.fused_tc_supported(k, d)
    pool = pool_of(img, src.coords, p, torch.float32)
    dev = img.device
    Wd = torch.from_numpy(rs.rand(d, k).astype(np.float32)).to(dev)
    Whi, Wlo = split(Wd)
    idx_clean = rs.randint(0, N - 1, size=300)
    idx_clean[5:9] = idx_clean[0]                       # duplicates
    idx_nan = idx_clean.copy()
    idx_nan[7] = N + 5                                  # out of range
    idx_nan[200] = N - 1                                # the corner outside the image
    ws = torch.empty(_lib.surrogate_fused_tc_workspace(300, k, d), dtype=torch.uint8, device=dev)
    for name, idx_np in (("clean", idx_clean), ("nan", idx_nan), ("empty", idx_clean[:0]), ("none", None)):
        idx = torch.from_numpy(idx_np).to(dev) if idx_np is not None else None
        n = len(idx_np) if idx_np is not None else 300
        pm = src.minibatch(idx, n)
        Ct_a = torch.full((max(n, 1), k), 7.0, device=dev)
        Ct_b = Ct_a.clone()
        _lib.cov_fused_tc(pool, idx, n, Whi, Wlo, Ct_a)
        _lib.cov_fused_tc_patches(pm, Whi, Wlo, Ct_b)
        assert_bits_equal(Ct_a, Ct_b, "cov %s" % name)
        if name == "nan":
            assert torch.isnan(Ct_b[7]).all() and torch.isnan(Ct_b[200]).all() and not torch.isnan(Ct_b[0]).any()
        Ht = torch.from_numpy(rs.rand(max(n, 1), k).astype(np.float32)).to(dev)    # n = 0: a real buffer, n passed apart
        P_a = torch.full((k, k + d), 3.0, device=dev)
        P_b = P_a.clone()
        _lib.surrogate_fused_tc(Ht, pool, idx, n, d, P_a, ws)
        _lib.surrogate_fused_tc_patches(Ht, pm, P_b, ws)
        assert_bits_equal(P_a, P_b, "surrogate %s" % name)
        # fused blend (single GPU form): A, B <- (1-w) A, B + w P
        A_a = torch.from_numpy(rs.rand(k, k).astype(np.float32)).to(dev); B_a = torch.from_numpy(rs.rand(k, d).astype(np.float32)).to(dev)
        A_b, B_b = A_a.clone(), B_a.clone()
        _lib.surrogate_fused_tc(Ht, pool, idx, n, d, None, ws, blend=(0.3, A_a, B_a))
        _lib.surrogate_fused_tc_patches(Ht, pm, None, ws, blend=(0.3, A_b, B_b))
        assert_bits_equal(A_a, A_b, "blend A %s" % name); assert_bits_equal(B_a, B_b, "blend B %s" % name)
    if kind == "u8":
        # against the uint8 pool itself (what step_pool reads on the fused path), clean indices
        pool8 = u8_pool_of(src.img, co[:N - 1], p)
        idx = torch.from_numpy(idx_clean).to(dev)
        Ct_a = torch.empty(300, k, device=dev); Ct_b = torch.empty(300, k, device=dev)
        _lib.cov_fused_tc(pool8, idx, 300, Whi, Wlo, Ct_a, scale=SCALE)
        _lib.cov_fused_tc_patches(src.minibatch(idx), Whi, Wlo, Ct_b)
        assert_bits_equal(Ct_a, Ct_b, "cov vs u8 pool")
    torch.cuda.synchronize()


@gpu
def test_fused_patches_reject_fp64_image():
    img = torch.zeros(20, 20, 1, dtype=torch.float64, device="cuda")
    src = ImagePatches(img, 8, np.zeros((4, 2), dtype=np.int32), precision="fp64")
    W = torch.zeros(64, 32, device="cuda")
    with pytest.raises(_lib.OnmfKernelError, match="ONMF_F32 or ONMF_STORE_U8"):
        _lib.cov_fused_tc_patches(src.minibatch(None), W, W, torch.empty(4, 32, device="cuda"))


@gpu
@pytest.mark.parametrize("kind", ["f32", "f64", "u8"])
@pytest.mark.parametrize("p,C", [(7, 1), (7, 3), (8, 1), (4, 3)])
def test_index_gather_equals_pool_rows(p, C, kind):
    rs = np.random.RandomState(p * 10 + C)
    H, W = 41, 53
    u8, img = make_image(rs, H, W, C, kind)
    N = 400
    co = corners(rs, H, W, p, N)
    co[3] = (0, W - p + 1)                              # patch leaves the image
    co[4] = (-1, 0)
    src = ImagePatches(img, p, co, precision="fp64" if kind == "f64" else "fp32")
    dt_ = src.engine_dtype
    pool = pool_of(img, src.coords, p, dt_)
    idx_np = rs.randint(5, N, size=333)
    idx_np[:4] = [3, 4, N, -2]                          # NaN rows: two bad corners, two bad indices
    idx_np[10:13] = idx_np[20]
    idx = torch.from_numpy(idx_np).to(img.device)
    ref = torch.empty(333, p * p * C, dtype=dt_, device=img.device)
    _lib.gather_rows(pool, idx, ref)
    got = src.gather(idx)
    assert_bits_equal(ref, got, "index gather")
    assert torch.isnan(got[:4]).all() and not torch.isnan(got[4:]).any()
    assert_bits_equal(pool, src.gather(), "gather of all columns")
    # pitched output rows
    wide = torch.full((333, p * p * C + 5), 2.0, dtype=dt_, device=img.device)
    _lib.gather_patches_mb(src.minibatch(idx), wide[:, :p * p * C])
    assert_bits_equal(ref, wide[:, :p * p * C], "pitched")
    assert (wide[:, p * p * C:] == 2.0).all()
    m = src.to_matrix()
    assert m.shape == (p * p * C, N) and m.dtype == np.float64


def _engine_pair(d, k, dtype, track_C, graph, use_tc=None):
    from onmf_ontf_ndl_b200 import OnmfEngine
    return [OnmfEngine(d, k, alpha=1.0, dtype=dtype, device=torch.device("cuda"), track_C=track_C, graph=graph, use_tc=use_tc)
            for _ in range(2)]


ENGINE_CASES = [
    # (p, C, k, kind, dtype, track_C, graph)
    (8, 1, 32, "f32", torch.float32, False, False),     # fused by reference, stream schedule
    (8, 1, 32, "f32", torch.float32, False, True),      # fused by reference, graph replay
    (6, 3, 36, "u8", torch.float32, False, True),       # fused, uint8 image vs uint8 pool
    (8, 1, 32, "f32", torch.float32, True, False),      # track_C: index gather + dense step
    (10, 1, 25, "f32", torch.float32, False, True),     # k = 25 (cfg1 / cfg3): SIMT products, index gather
    (10, 1, 25, "u8", torch.float32, False, False),     # k = 25, uint8 image vs the fp32 pool of its values
    (20, 1, 300, "f32", torch.float32, False, False),   # k > 256: pre-split tensor-core products
    (6, 3, 16, "f64", torch.float64, False, True),      # fp64 engine
]


@gpu
@pytest.mark.parametrize("p,C,k,kind,dtype,track_C,graph", ENGINE_CASES)
def test_engine_step_patches_equals_step_pool(p, C, k, kind, dtype, track_C, graph):
    rs = np.random.RandomState(k + p)
    H, W = 48, 40
    u8, img = make_image(rs, H, W, C, kind)
    N, n, d = 900, 256, p * p * C
    co = corners(rs, H, W, p, N)
    src = ImagePatches(img, p, co, precision="fp64" if dtype == torch.float64 else "fp32")
    e_ref, e_pat = _engine_pair(d, k, dtype, track_C, graph)
    fused = e_pat.fused_tc and not track_C
    if kind == "u8" and fused:
        pool, scale = u8_pool_of(src.img, co, p), SCALE
    else:
        pool, scale = pool_of(img, src.coords, p, dtype), 1.0
    W0 = rs.rand(d, k)                                  # raw initial dictionary: the FP64 first minibatch runs
    for e in (e_ref, e_pat):
        e.set_state(W0)
    # two index tensors in turn: a graph key (index pointer, dictionary slot) repeats, so the graph engines capture and replay
    idx_all = torch.from_numpy(rs.randint(0, N, size=(2, n))).cuda()
    for t in range(1, 9):
        H_ref = e_ref.step_pool(pool, idx_all[(t - 1) % 2], float(t), scale=scale)
        H_pat = e_pat.step_patches(src, idx_all[(t - 1) % 2], float(t))
        assert_bits_equal(H_ref, H_pat, "codes step %d" % t)
    for a, b, nm in zip(e_ref.state(), e_pat.state(), "WABC"):
        if a is not None:
            assert_bits_equal(a, b, nm)
    if graph and e_pat.graph:
        assert e_pat._plan.graph_steps() > 0
    torch.cuda.synchronize()


@gpu
def test_engine_step_patches_all_columns_and_multi_rank_form():
    """idx = None (every column) and the launch / all-reduce / finish form a multi-GPU engine takes"""
    rs = np.random.RandomState(3)
    u8, img = make_image(rs, 30, 30, 1, "f32")
    co = corners(rs, 30, 30, 8, 200)
    src = ImagePatches(img, 8, co)
    e_ref, e_pat = _engine_pair(64, 32, torch.float32, False, False)
    pool = pool_of(img, src.coords, 8, torch.float32)
    W0 = rs.rand(64, 32)
    for e in (e_ref, e_pat):
        e.set_state(W0)
    for t in (1, 2, 3):
        e_ref.step_pool(pool, None, float(t))
        e_pat.step_patches(src, None, float(t))
    # the two-phase form (what a rank of a process group runs), with an all-reduce over a group of one left out
    e_ref.world = e_pat.world = 2
    e_ref.pg = e_pat.pg = None
    e_ref._sb = e_pat._sb = None
    import torch.distributed as dist
    orig = dist.all_reduce
    dist.all_reduce = lambda *a, **kw: None
    try:
        idx = torch.from_numpy(rs.randint(0, 200, size=100)).cuda()
        for t in (4, 5):
            e_ref.step_pool(pool, idx, float(t))
            e_pat.step_patches(src, idx, float(t))
    finally:
        dist.all_reduce = orig
    for a, b, nm in zip(e_ref.state(), e_pat.state(), "WABC"):
        if a is not None:
            assert_bits_equal(a, b, nm)


@gpu
def test_graph_key_covers_image_and_corners():
    """Graph replays keyed on the image AND the corners: three patch sources (two images sharing one corner tensor, one
    image with two corner tensors) cycle through the graph path with the same index tensor; every step equals the same
    step on the stream schedule."""
    rs = np.random.RandomState(9)
    p, k, n, N = 8, 32, 256, 500
    _, img1 = make_image(rs, 40, 40, 1, "f32")
    _, img2 = make_image(rs, 40, 40, 1, "f32")
    co1, co3 = corners(rs, 40, 40, p, N), corners(rs, 40, 40, p, N)
    P1 = ImagePatches(img1, p, co1)
    P2 = ImagePatches(img2, p, co1)
    P2.coords = P1.coords                               # same corner tensor, different image
    P3 = ImagePatches(img1, p, co3)
    P3.img = P1.img                                     # same image tensor, different corners
    e_s, e_g = _engine_pair(p * p, k, torch.float32, False, False)
    e_g.graph = True
    W0 = rs.rand(p * p, k) / np.sqrt(p * p)             # normalised-size dictionary: every step takes the graph path
    for e in (e_s, e_g):
        e.set_state(W0)
    idx = torch.from_numpy(rs.randint(0, N, size=n)).cuda()
    seq = [P1, P1, P2, P2, P3, P3] * 3
    for t, src in enumerate(seq, 1):
        e_s.step_patches(src, idx, float(t))
        e_g.step_patches(src, idx, float(t))
        for a, b, nm in zip(e_s.state()[:3], e_g.state()[:3], "WAB"):
            assert_bits_equal(a, b, "%s after step %d" % (nm, t))
    assert e_g._plan.graph_steps() >= 6


def _driver_run(img, p, N, k, kw, by_reference, keep_code=True):
    """what a driver does under np.random.seed(21): draw N random patch corners, then train -- on the materialised X
    (extract_random_patches) or on the patches by reference (ImagePatches of sample_patch_coords).  Returns the training
    result and the next draw of the global RNG (both forms must consume it identically)."""
    from onmf_ontf_ndl_b200 import Online_NMF, patches
    np.random.seed(21)
    prec = kw.get("precision")
    if by_reference:
        X = ImagePatches(img, p, patches.sample_patch_coords(img.shape, p, N), precision=prec)
    elif img.dtype == np.uint8:                          # the fp32 values float(u8) * float(1/255) a uint8 image stands for
        vals = (img.astype(np.float32) * np.float32(SCALE)).astype(np.float64)
        X = patches.gather_patches(vals, patches.sample_patch_coords(img.shape, p, N), p)
    else:
        X = patches.extract_random_patches(img, p, N, precision=prec)
        X = X.reshape(-1, N) if X.ndim == 3 else X
    out = Online_NMF(X, n_components=k, keep_code=keep_code, **kw).train_dict()
    return out, np.random.rand()


@gpu
@pytest.mark.parametrize("case", ["cfg1_like", "fused", "fused_u8", "all_columns_fp64"])
def test_online_nmf_image_patches_equals_materialised(case):
    rs = np.random.RandomState(1)
    if case == "cfg1_like":                              # p = 10, k = 25, default track_C: index gather + SIMT products
        img, p, k, kw = rs.rand(64, 64), 10, 25, dict(iterations=6, batch_size=100, subsample=True)
    elif case == "fused":
        img, p, k, kw = rs.rand(48, 48), 8, 32, dict(iterations=6, batch_size=300, subsample=True, track_C=False)
    elif case == "fused_u8":
        img, p, k, kw = rs.randint(0, 256, size=(40, 40, 3)).astype(np.uint8), 4, 32, \
            dict(iterations=5, batch_size=200, subsample=True, track_C=False)
    else:
        img, p, k, kw = rs.rand(30, 30), 6, 12, dict(iterations=4, batch_size=50, subsample=False, precision="fp64")
    a, next_a = _driver_run(img, p, 600, k, kw, by_reference=False)
    b, next_b = _driver_run(img, p, 600, k, kw, by_reference=True)
    assert next_a == next_b
    for x, y, nm in zip(a, b, ("W", "A", "B", "C", "code")):
        if x is None:
            assert y is None, nm
        else:
            assert np.array_equal(x, y), nm
    c, _ = _driver_run(img, p, 600, k, kw, by_reference=True, keep_code=False)
    assert c[4] is None
    for x, y, nm in zip(a[:4], c[:4], "WABC"):
        if x is not None:
            assert np.array_equal(x, y), nm


def _gloo_worker(rank, world, port, out):
    import torch.distributed as dist
    from onmf_ontf_ndl_b200 import Online_NMF
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.cuda.set_device(0)
    res = {}
    rs = np.random.RandomState(4)
    img = rs.rand(50, 50)
    for name, p, k, kw in (("gather", 10, 25, dict(subsample=True)), ("fused", 8, 32, dict(subsample=True, track_C=False)),
                           ("all_columns", 8, 32, dict(subsample=False, track_C=False))):
        co = corners(rs, 50, 50, p, 501)
        src = ImagePatches(img, p, co)
        got = []
        for X in (src, src.to_matrix()):
            np.random.seed(3 if rank == 0 else 100 + rank)      # rank 0's draws are broadcast
            W, A, B, C, code = Online_NMF(X, n_components=k, iterations=5, batch_size=200, **kw).train_dict()
            got.append((W, A, B, C, code))
        same_as_matrix = all(x is None and y is None or np.array_equal(x, y) for x, y in zip(got[0], got[1]))
        Wt = torch.from_numpy(got[0][0]).cuda()
        gathered = [torch.empty_like(Wt) for _ in range(world)]
        dist.all_gather(gathered, Wt)
        same_ranks = all(torch.equal(gathered[0], t) for t in gathered)
        res[name] = dict(ok=bool(same_as_matrix and same_ranks), same_as_matrix=same_as_matrix, same_ranks=same_ranks)
    out[rank] = res
    dist.destroy_process_group()


@gpu
def test_online_nmf_image_patches_two_ranks_gloo_one_device():
    import torch.multiprocessing as mp
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_gloo_worker, args=(2, port, out), nprocs=2, join=True)
    for r in (0, 1):
        assert all(v["ok"] for v in out[r].values()), dict(out)


@gpu
def test_capacity_every_patch_of_a_2048_image():
    """All 4,068,289 positions of 32 x 32 patches in a 2048 x 2048 uint8 image (the materialised fp32 pool would be 16.7 GB):
    training by reference stays under 1 GB of device memory above the baseline."""
    from onmf_ontf_ndl_b200 import Online_NMF, patches
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    rs = np.random.RandomState(0)
    img = rs.randint(0, 256, size=(2048, 2048)).astype(np.uint8)
    co = patches.all_patch_coords(img.shape, 32)
    assert co.shape[0] == 2017 ** 2 == 4068289
    src = ImagePatches(img, 32, co)
    np.random.seed(0)
    m = Online_NMF(src, n_components=256, iterations=5, batch_size=4096, subsample=True, keep_code=False, track_C=False)
    W, A, B, C, code = m.train_dict()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    assert code is None and C is None
    assert np.isfinite(W).all() and np.abs(W).sum() > 0
    assert peak < 1 << 30, "peak %.1f MB" % (peak / 2 ** 20)
