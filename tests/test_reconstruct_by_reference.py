"""Banded reconstruction by reference (reconstruct.reconstruct_image, onmf_patch_grid_accumulate): the grid is coded and
averaged in bands of patches read out of the resident image, and must give the bits of the one-pass materialised
reconstruction (`_materialised_reconstruct`, the previous body of reconstruct_image) -- canvas, counts and codes."""
import zlib

import numpy as np
import pytest
import torch

from onmf_ontf_ndl_b200 import _host, _lib, patches
from onmf_ontf_ndl_b200 import reconstruct as rec
from onmf_ontf_ndl_b200.engine import OnmfEngine
from onmf_ontf_ndl_b200.patches import ImagePatches

gpu = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------------------------- reference
def _materialised_reconstruct(A, W, patch_size, recons_resolution=1, alpha=1, sub_iter=10, stopping_diff=0.01, coder="pgd",
                              H0=None, precision=None, return_code=False, include_last=False):
    """reconstruct_image as it was before banding: the whole patch matrix, its codes and reconstructions at once (verbatim,
    plus the corner grid of include_last)"""
    grid_shape = rec.grid_shape
    dev = _host.device()
    dtype = _host.torch_dtype(precision)
    A = np.asarray(A, dtype=np.float64)
    squeeze = A.ndim == 2
    A3 = A[:, :, None] if squeeze else A
    Hh, Ww, C = A3.shape
    k = int(patch_size)
    W = np.asarray(W, dtype=np.float64)
    d, r = W.shape
    if d != k * k * C:
        raise ValueError("dictionary has %d rows, expected patch_size^2 * channels = %d" % (d, k * k * C))
    ny, nx = grid_shape(Hh, Ww, k, recons_resolution)
    if include_last:
        ny, nx = len(range(0, Hh - k + 1, recons_resolution)), len(range(0, Ww - k + 1, recons_resolution))
    n = ny * nx
    canvas = torch.zeros(Hh, Ww, C, dtype=dtype, device=dev)
    count = torch.zeros(Hh, Ww, dtype=dtype, device=dev)
    if n == 0:
        out = canvas.cpu().numpy().astype(np.float64)
        return (out[:, :, 0] if squeeze else out), count.cpu().numpy().astype(np.float64)
    gy, gx = np.meshgrid(np.arange(ny) * recons_resolution, np.arange(nx) * recons_resolution, indexing="ij")
    coords = torch.from_numpy(np.stack([gy.reshape(-1), gx.reshape(-1)], 1).astype(np.int32)).to(dev)
    img = _host.to_device(A3, dtype, dev)
    Xt = torch.empty(n, d, dtype=dtype, device=dev)
    _lib.gather_patches(img, coords, k, Xt)                                  # K1
    Wd = _host.to_device(W, dtype, dev)
    if coder == "lasso_lars":
        eng = OnmfEngine(d, r, alpha=alpha, dtype=dtype, device=dev)
        Ht = eng.sparse_code(Xt, Wd, alpha=alpha).clone()                    # K2 + K3
    elif coder == "pgd":
        if H0 is None:
            # same stream as n calls of np.random.rand(r, 1); already sample-major
            Ht = _host.to_device(np.random.rand(n, r), dtype, dev)
        else:
            H0 = np.asarray(H0, dtype=np.float64)
            if H0.shape != (r, n):
                raise ValueError("H0 must have shape (r, n_patches) = (%d, %d)" % (r, n))
            Ht = _host.to_sample_major(H0, dtype, dev)                        # uploaded as it is, transposed on the device
        G = torch.empty(r, r, dtype=dtype, device=dev)
        Ct = torch.empty(n, r, dtype=dtype, device=dev)
        _lib.gram(Wd, G)
        _lib.cov(Xt, Wd, Ct)
        _lib.pgd_code_columns(G, Ct, alpha, sub_iter, stopping_diff, Ht)
    else:
        raise ValueError("coder must be 'pgd' or 'lasso_lars'")
    Wt = torch.empty(r, d, dtype=dtype, device=dev)
    _lib.transpose(Wd, Wt)
    R = torch.empty(n, d, dtype=dtype, device=dev)
    _lib.cov(Ht, Wt, R)                                                      # patch reconstructions (n x d) = Ht W^T
    _lib.patch_grid_mean(R, ny, nx, k, recons_resolution, C, Hh, Ww, canvas, count)
    out = canvas.cpu().numpy().astype(np.float64)
    res = (out[:, :, 0] if squeeze else out, count.cpu().numpy().astype(np.float64))
    if return_code:
        res = res + (_host.from_sample_major(Ht),)
    return res


def _np_mean_single(R, ny, nx, p, s, C, H, W):
    """one pass: every pixel sums its covering patches in ascending j, then divides by their number"""
    acc = np.zeros((H, W, C), dtype=R.dtype)
    cnt = np.zeros((H, W), dtype=R.dtype)
    for j in range(ny * nx):
        y, x = (j // nx) * s, (j % nx) * s
        acc[y:y + p, x:x + p] += R[j].reshape(p, p, C)
        cnt[y:y + p, x:x + p] += 1
    out = np.zeros_like(acc)
    np.divide(acc, cnt[:, :, None], out=out, where=cnt[:, :, None] > 0)
    return out, cnt


def _np_pixel_plan(ny, nx, p, s, H, W):
    """per pixel: first and last covering patch (first > last: none) and the owner own = min(y/s, ny-1)*nx + min(x/s, nx-1)"""
    y = np.arange(H)[:, None]
    x = np.arange(W)[None, :]
    gy_hi, gx_hi = np.minimum(y // s, ny - 1), np.minimum(x // s, nx - 1)
    gy_lo = np.where(y - p + 1 <= 0, 0, (y - p + s) // s)
    gx_lo = np.where(x - p + 1 <= 0, 0, (x - p + s) // s)
    covered = (gy_lo <= gy_hi) & (gx_lo <= gx_hi)
    cnt = np.where(covered, (gy_hi - gy_lo + 1) * (gx_hi - gx_lo + 1), 0)
    return gy_lo * nx + gx_lo, gy_hi * nx + gx_hi, covered, cnt


def _np_accumulate(canvas, count, Rb, j0, j1, ny, nx, p, s, C, H, W, plan):
    """numpy restatement of one onmf_patch_grid_accumulate call (include/onmf_b200.h)"""
    first, own, covered, cnt = plan
    start = covered & (first >= j0) & (first < j1)
    canvas[start] = 0
    for j in range(j0, j1):
        y, x = (j // nx) * s, (j % nx) * s
        canvas[y:y + p, x:x + p] += Rb[j - j0].reshape(p, p, C)
    fin = (own >= j0) & (own < j1)
    t = canvas.dtype.type
    canvas[fin & ~covered] = 0
    m = fin & covered
    canvas[m] = canvas[m] / cnt[m][:, None].astype(t)
    count[fin] = cnt[fin].astype(t)


def _random_splits(rs, n, nx):
    """cut points of [0, n): random bands, one-patch bands, and bands ending in the middle and at the end of a grid row"""
    cuts = set(rs.randint(1, n, size=min(n - 1, 6)).tolist()) if n > 1 else set()
    if n > 3:
        cuts |= {1, 2, n - 1}
    if nx > 2 and n > nx + 1:
        cuts |= {nx, nx + nx // 2}
    edges = [0] + sorted(c for c in cuts if 0 < c < n) + [n]
    return list(zip(edges[:-1], edges[1:]))


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.int64 if a.dtype == np.float64 else np.int32)


# ---------------------------------------------------------------------------------------------------------------- CPU tests
def test_band_plan_invariants():
    for n in list(range(0, 40)) + [99, 100, 101, 7105, 7106, 14209, 14210, 14211, 262144, 262145, 4068289]:
        for floor in (1, 3, 7, 64, 7105):
            for max_band in (0, 1, 2, 5, 64, 100, 7105, 14209, 65536, 262144):
                bands = rec._band_plan(n, max_band, floor)
                if n == 0:
                    assert bands == []
                    continue
                assert bands[0][0] == 0 and bands[-1][1] == n
                assert all(a[1] == b[0] for a, b in zip(bands, bands[1:]))
                sizes = [j1 - j0 for j0, j1 in bands]
                assert max(sizes) - min(sizes) <= 1, (n, max_band, floor, sizes)
                if n < floor:
                    assert len(bands) == 1
                else:
                    assert min(sizes) >= floor, (n, max_band, floor, sizes)
                # the floor takes precedence; bands stay within max_band whenever that leaves room for it
                assert max(sizes) <= max(max_band, 2 * floor - 1, n if n < floor else 0), (n, max_band, floor, sizes)
                if max_band >= 2 * floor - 1:
                    assert max(sizes) <= max_band, (n, max_band, floor, sizes)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("p,s,C", [(4, 1, 1), (4, 2, 3), (4, 4, 1), (3, 5, 3), (5, 3, 1)])
def test_accumulate_contract_in_numpy_equals_single_pass(p, s, C, dtype):
    rs = np.random.RandomState(p * 100 + s * 10 + C)
    for H, W, last in ((17, 23, False), (19, 16, True)):
        ny, nx = (len(range(0, H - p + (1 if last else 0), s)), len(range(0, W - p + (1 if last else 0), s)))
        n = ny * nx
        R = (rs.rand(n, p * p * C) - 0.3).astype(dtype)
        ref, ref_cnt = _np_mean_single(R, ny, nx, p, s, C, H, W)
        plan = _np_pixel_plan(ny, nx, p, s, H, W)
        for trial in range(4):
            bands = _random_splits(rs, n, nx) if trial else [(j, j + 1) for j in range(n)]
            canvas = np.full((H, W, C), np.nan, dtype=dtype)          # no memset: every pixel is written by its owner
            count = np.full((H, W), np.nan, dtype=dtype)
            for j0, j1 in bands:
                _np_accumulate(canvas, count, R[j0:j1], j0, j1, ny, nx, p, s, C, H, W, plan)
            assert np.array_equal(_bits(canvas), _bits(ref)), (H, W, bands)
            assert np.array_equal(_bits(count), _bits(ref_cnt)), (H, W, bands)


@pytest.mark.parametrize("case", ["patch_size", "precision", "precision_u8"])
def test_image_patches_mismatch_raises_before_device_use(case, monkeypatch):
    def no_device():
        raise AssertionError("device touched before validation")
    monkeypatch.setattr(_host, "device", no_device)
    src = ImagePatches.__new__(ImagePatches)          # patch size, geometry and precision are all that is checked first
    src.patch_size, src.H, src.W, src.C, src.d = 4, 20, 30, 1, 16
    src.precision, src.dtype = "fp32", torch.float32
    W = np.random.rand(16, 5)
    with pytest.raises(ValueError):
        if case == "patch_size":
            rec.reconstruct_image(src, np.random.rand(25, 5), 5, coder="lasso_lars")
        elif case == "precision":
            rec.reconstruct_image(src, W, 4, coder="lasso_lars", precision="fp64")
        else:
            src.dtype = torch.uint8
            rec.reconstruct_image(src, W, 4, coder="pgd", precision="fp64")


# ---------------------------------------------------------------------------------------------------------------- GPU tests
@gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("p,s,C,H,W", [(4, 1, 1, 33, 41), (5, 2, 3, 30, 27), (4, 4, 1, 26, 35), (3, 5, 3, 29, 31),
                                       (8, 3, 1, 64, 70)])
def test_accumulate_kernel_equals_single_pass(p, s, C, H, W, dtype):
    rs = np.random.RandomState(p + 7 * s + 13 * C)
    dev = torch.device("cuda")
    ny, nx = len(range(0, H - p + 1, s)), len(range(0, W - p + 1, s))
    n = ny * nx
    Rn = (rs.rand(n, p * p * C) - 0.3)
    R = torch.from_numpy(Rn).to(dev, dtype)
    ref = torch.empty(H, W, C, dtype=dtype, device=dev)
    ref_cnt = torch.empty(H, W, dtype=dtype, device=dev)
    _lib.patch_grid_mean(R, ny, nx, p, s, C, H, W, ref, ref_cnt)
    npd = np.float32 if dtype == torch.float32 else np.float64
    np_ref, np_cnt = _np_mean_single(R.cpu().numpy().astype(npd), ny, nx, p, s, C, H, W)
    assert np.array_equal(_bits(ref.cpu().numpy()), _bits(np_ref))
    assert np.array_equal(_bits(ref_cnt.cpu().numpy()), _bits(np_cnt))
    for trial in range(4):
        bands = _random_splits(rs, n, nx) if trial else [(j, j + 1) for j in range(n)]
        canvas = torch.full((H, W, C), float("nan"), dtype=dtype, device=dev)
        count = torch.full((H, W), float("nan"), dtype=dtype, device=dev)
        for j0, j1 in bands:
            _lib.patch_grid_accumulate(R[j0:j1], j0, j1, ny, nx, p, s, C, H, W, canvas, count)
        assert torch.equal(canvas.view(torch.int64 if dtype == torch.float64 else torch.int32),
                           ref.view(torch.int64 if dtype == torch.float64 else torch.int32)), bands
        assert torch.equal(count, ref_cnt), bands


def _dictionary(rs, d, r, raw=False):
    W = rs.rand(d, r)
    return W if raw else W / np.linalg.norm(W, axis=0)


def _assert_same(a, b, what):
    assert len(a) == len(b), what
    for x, y, nm in zip(a, b, ("canvas", "count", "code")):
        assert x.shape == y.shape, (what, nm)
        assert np.array_equal(_bits(x), _bits(y)), "%s: %s differs (max |diff| %.3g)" % (what, nm, np.max(np.abs(x - y)))


# (image shape, p, k, raw W): the fused tensor-core shape, the gather shape, a k > 256 shape, a raw dictionary (FP64 coder)
SHAPES = {"fused": ((36, 40), 8, 64, False), "gather": ((34, 31), 10, 25, False), "wide_k": ((30, 30), 8, 300, False),
          "raw_W": ((36, 40), 8, 64, True)}


@gpu
@pytest.mark.parametrize("shape", sorted(SHAPES))
@pytest.mark.parametrize("coder", ["lasso_lars", "pgd"])
@pytest.mark.parametrize("precision", ["fp32", "fp64"])
@pytest.mark.parametrize("C", [1, 3])
def test_banded_equals_materialised(shape, coder, precision, C, monkeypatch):
    # every grid here is below the coders' variant thresholds, so bands far below the production floor take the same
    # kernel variants as the whole grid: a floor of 1 lets a small max_band split them into many bands
    monkeypatch.setattr(_lib, "coder_band_floor", lambda device=None: 1)
    (H, Wd), p, k, raw = SHAPES[shape]
    if C == 3:
        p = max(p // 2, 3)
    rs = np.random.RandomState(zlib.crc32(repr((shape, coder, precision, C)).encode()))
    img = rs.rand(H, Wd, C) if C == 3 else rs.rand(H, Wd)
    W = _dictionary(rs, p * p * C, k, raw)
    for s in (1, 2, 3):
        for last in (False, True):
            kw = dict(coder=coder, precision=precision, return_code=True, include_last=last, alpha=0.5)
            np.random.seed(11)
            a = _materialised_reconstruct(img, W, p, s, **kw)
            n = a[2].shape[1]
            for max_band in (max(n // 7, 1), 53, 262144):
                np.random.seed(11)
                b = rec.reconstruct_image(img, W, p, s, max_band=max_band, **kw)
                _assert_same(a, b, (shape, coder, precision, C, s, last, max_band))


@gpu
@pytest.mark.parametrize("coder,k", [("lasso_lars", 25), ("lasso_lars", 49), ("pgd", 25)])
def test_bands_stay_on_the_whole_grid_variant(coder, k):
    # about 15,000 patches: above every coder threshold (LARS fast tier n <= 24 / 48 x SMs, PGD thread per sample n >= 16 x SMs).
    # max_band = 1000 asks for bands far below them; the floor keeps every band on the whole grid's side, bit for bit.
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    rs = np.random.RandomState(k)
    p = 5 if k == 25 else 7
    side = int(np.ceil(np.sqrt(max(15000, 2 * (48 * sms + 1) + 100)))) + p
    img = rs.rand(side, side)
    W = _dictionary(rs, p * p, k)
    np.random.seed(5)
    a = _materialised_reconstruct(img, W, p, 1, coder=coder, return_code=True, alpha=0.5)
    np.random.seed(5)
    b = rec.reconstruct_image(img, W, p, 1, coder=coder, return_code=True, alpha=0.5, max_band=1000)
    n = a[2].shape[1]
    assert len(rec._band_plan(n, 1000, _lib.coder_band_floor())) >= 2
    _assert_same(a, b, (coder, k, n))


@gpu
@pytest.mark.parametrize("coder", ["lasso_lars", "pgd"])
def test_image_patches_input(coder):
    rs = np.random.RandomState(3)
    u8 = rs.randint(0, 256, size=(40, 44)).astype(np.uint8)
    wide = u8.astype(np.float32) * np.float32(1.0 / 255.0)               # the values the kernels widen uint8 to
    p, k = 8, 64
    W = _dictionary(rs, p * p, k)
    src = ImagePatches(u8, p, np.zeros((0, 2), dtype=np.int32), scale=1.0 / 255.0)
    for s in (1, 3):
        np.random.seed(2)
        a = _materialised_reconstruct(wide, W, p, s, coder=coder, return_code=True)
        np.random.seed(2)
        b = rec.reconstruct_image(src, W, p, s, coder=coder, return_code=True)
        _assert_same(a, b, ("u8", coder, s))


@gpu
def test_trained_image_patches_feed_reconstruction():
    from onmf_ontf_ndl_b200 import Online_NMF
    rs = np.random.RandomState(4)
    img = rs.rand(48, 48).astype(np.float32)
    p, k = 8, 32
    src = ImagePatches(img, p, patches.all_patch_coords(img.shape, p))
    np.random.seed(0)
    W = Online_NMF(src, n_components=k, iterations=4, batch_size=300, subsample=True, keep_code=False,
                   track_C=False).train_dict()[0]
    a = _materialised_reconstruct(img, W, p, 1, coder="lasso_lars", return_code=True, include_last=True)
    b = rec.reconstruct_image(src, W, p, 1, coder="lasso_lars", return_code=True, include_last=True)
    _assert_same(a, b, "trained")
    assert np.all(np.isfinite(b[0])) and b[1].min() >= 1


@gpu
def test_include_last_is_the_drivers_one_shot_reconstruction():
    from onmf_ontf_ndl_b200 import Online_NMF
    rs = np.random.RandomState(6)
    img = rs.rand(30, 34)
    p, k, alpha = 6, 20, 0.5
    W = _dictionary(rs, p * p, k)
    X = patches.extract_patches_2d(img, p, precision="fp64")
    code = Online_NMF(X, n_components=k, alpha=alpha, precision="fp64").sparse_code(X, W)
    ref = rec.reconstruct_from_patches_2d(W, img.shape, code=code, precision="fp64")
    got, cnt = rec.reconstruct_image(img, W, p, 1, alpha=alpha, coder="lasso_lars", precision="fp64", include_last=True)
    assert cnt.min() >= 1
    assert np.max(np.abs(got - ref)) <= 1e-13


@gpu
def test_every_position_of_a_2048_image_in_bounded_memory():
    rs = np.random.RandomState(8)
    H = 2048
    yy, xx = np.meshgrid(np.linspace(0, 12, H), np.linspace(0, 9, H), indexing="ij")
    img = (0.5 + 0.25 * np.sin(yy) * np.cos(xx) + 0.1 * rs.rand(H, H)).astype(np.float32)
    p, k = 32, 256
    co = patches.all_patch_coords(img.shape, p)[rs.choice((H - p + 1) ** 2, k, replace=False)]
    W = np.stack([img[a:a + p, b:b + p].reshape(-1) for a, b in co], 1).astype(np.float64)
    W /= np.linalg.norm(W, axis=0)
    src = ImagePatches(img, p, np.zeros((0, 2), dtype=np.int32))
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    canvas, count = rec.reconstruct_image(src, W, p, 1, coder="lasso_lars", include_last=True, max_band=65536)
    peak = torch.cuda.max_memory_allocated() - base
    assert peak < 2 * 2 ** 30, peak                                         # the materialised path needs about 42 GB
    assert np.all(np.isfinite(canvas)) and count.min() >= 1
    # an interior window of a crop sees the same patches, codes and summation order as the full image
    y0, x0, c = 900, 1300, 320
    crop = img[y0:y0 + c, x0:x0 + c]
    a, a_cnt = _materialised_reconstruct(crop, W, p, 1, coder="lasso_lars", include_last=True)
    m = p - 1
    win = (slice(y0 + m, y0 + c - m), slice(x0 + m, x0 + c - m))
    assert np.array_equal(_bits(canvas[win]), _bits(a[m:c - m, m:c - m]))
    assert np.array_equal(count[win], a_cnt[m:c - m, m:c - m])
