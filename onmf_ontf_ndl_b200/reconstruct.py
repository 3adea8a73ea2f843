"""Batched patch reconstruction (SURVEY.md §8f.1).

The reference reconstructs an image by looping over a stride grid of patches in Python, coding ONE patch per call
and painting a running-mean canvas pixel by pixel (image_reconstruction.py:358-406: `update_code_within_radius(patch,
W, H0=None, r=None, alpha=1, sub_iter=10, stopping_diff=0.01)` at :384, running mean at :389-392).  Here the grid
is processed in bands of patches, each one K1 gather (or a read by reference), one Gram/covariance product, one batched
coder launch (the same projected-gradient iteration with the reference's per-patch stopping test, or the positive
LARS-lasso coder), one product Ht W^T and one range of the overlap-mean kernel.  Results equal the reference loop's (same
H0 stream) up to summation order, and do not depend on the band size.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _host, _lib, patches
from .engine import OnmfEngine


def grid_shape(H, W, patch_size, recons_resolution):
    """number of grid rows / columns of `for i in range(0, H - k, res)` (image_reconstruction.py:375-376)."""
    k, s = patch_size, recons_resolution
    return len(range(0, H - k, s)), len(range(0, W - k, s))


def _band_plan(n, max_band, floor):
    """Consecutive bands [(j0, j1), ...] of near-equal size covering [0, n).  Every band holds at least `floor` columns (a
    grid of fewer is one band): that keeps each coder call on the kernel variant the whole grid would take (see
    _lib.coder_band_floor).  A max_band below the floor is raised to it; the floor takes precedence, so a band holds at most
    max(max_band, 2 * floor - 1) columns."""
    n, floor = int(n), max(int(floor), 1)
    if n <= 0:
        return []
    mb = max(int(max_band), floor)
    nb = max(1, min(-(-n // mb), n // floor))
    base, rem = divmod(n, nb)
    bands, j = [], 0
    for b in range(nb):
        m = base + (1 if b < rem else 0)
        bands.append((j, j + m))
        j += m
    return bands


def reconstruct_image(A, W, patch_size, recons_resolution=1, alpha=1, sub_iter=10, stopping_diff=0.01, coder="pgd",
                      H0=None, precision=None, return_code=False, include_last=False, max_band=262144):
    """A: image (H x W) or (H x W x C), or an ImagePatches (patches.py) whose resident image is used as stored (fp32, fp64,
    or uint8 read as stored * scale; its corners are ignored, a one-channel image counts as grey); W: dictionary
    (patch_size^2 * C, r).  Returns (A_recons, overlap_count[, code (r x n_patches)]) as numpy float64.
    coder="pgd": the reference's projected-gradient coder, one independent run per patch; H0 (r x n_patches) defaults to
    np.random.rand(r, 1) per patch in loop order, like the reference.  coder="lasso_lars": the positive lasso (the
    commented-out alternative at image_reconstruction.py:380-383).
    The patch grid is `range(0, H - k, stride)` per axis, the reference loop's; include_last=True takes every offset
    0..H-k, sklearn's extract_patches_2d grid (with stride 1 and the lasso coder: the drivers' one-shot reconstruction).
    The grid is processed in bands of at most max_band patches (gathered or read by reference, coded, multiplied by W^T and
    added to the overlap mean band by band), so device memory is bounded by the band, not the image; the results are the
    bits of one pass over the whole grid."""
    if coder not in ("pgd", "lasso_lars"):
        raise ValueError("coder must be 'pgd' or 'lasso_lars'")
    k, s = int(patch_size), int(recons_resolution)
    src = A if isinstance(A, patches.ImagePatches) else None
    if src is not None:
        if k != src.patch_size:
            raise ValueError("patch_size %d differs from the ImagePatches' %d" % (k, src.patch_size))
        if precision is not None and _host.torch_dtype(precision) != src.engine_dtype:
            raise ValueError("precision %r differs from the ImagePatches' %s" % (precision, src.precision))
        dtype = src.engine_dtype
        Hh, Ww, C = src.H, src.W, src.C
        squeeze = C == 1
    else:
        dtype = _host.torch_dtype(precision)
        A = np.asarray(A, dtype=np.float64)
        squeeze = A.ndim == 2
        A3 = A[:, :, None] if squeeze else A
        Hh, Ww, C = A3.shape
    W = np.asarray(W, dtype=np.float64)
    d, r = W.shape
    if d != k * k * C:
        raise ValueError("dictionary has %d rows, expected patch_size^2 * channels = %d" % (d, k * k * C))
    ys = np.arange(0, Hh - k + (1 if include_last else 0), s)
    xs = np.arange(0, Ww - k + (1 if include_last else 0), s)
    ny, nx = len(ys), len(xs)
    n = ny * nx
    if coder == "pgd" and H0 is not None:
        H0 = np.asarray(H0, dtype=np.float64)
        if H0.shape != (r, n):
            raise ValueError("H0 must have shape (r, n_patches) = (%d, %d)" % (r, n))
    dev = _host.device()
    if n == 0:
        out = np.zeros((Hh, Ww, C))
        return (out[:, :, 0] if squeeze else out), np.zeros((Hh, Ww))
    canvas = torch.empty(Hh, Ww, C, dtype=dtype, device=dev)      # every pixel is written once by its owning band
    count = torch.empty(Hh, Ww, dtype=dtype, device=dev)
    img, scale = (src.img, src.scale) if src is not None else (_host.to_device(A3, dtype, dev), 1.0)
    Wd = _host.to_device(W, dtype, dev)
    Wt = torch.empty(r, d, dtype=dtype, device=dev)
    _lib.transpose(Wd, Wt)
    bands = _band_plan(n, max_band, _lib.coder_band_floor(dev))
    mmax = max(j1 - j0 for j0, j1 in bands)
    if coder == "lasso_lars":
        eng = OnmfEngine(d, r, alpha=alpha, dtype=dtype, device=dev)
        f = eng.derive_foreign(Wd)                                           # Gram (+ TF32 split) once for all bands
    else:
        G = torch.empty(r, r, dtype=dtype, device=dev)
        _lib.gram(Wd, G)
        Xt = torch.empty(mmax, d, dtype=dtype, device=dev)
        Ct = torch.empty(mmax, r, dtype=dtype, device=dev)
    R = torch.empty(mmax, d, dtype=dtype, device=dev)
    code = np.empty((r, n)) if return_code else None
    for j0, j1 in bands:
        m = j1 - j0
        jj = np.arange(j0, j1)
        corners = torch.from_numpy(np.stack([ys[jj // nx], xs[jj % nx]], 1).astype(np.int32)).to(dev)
        pm = _lib.make_patch_minibatch(img, k, corners, None, m, scale)
        if coder == "lasso_lars":
            # first tier 0 in every band: the tier hint an earlier band leaves in the workspace must not steer this one
            Ht = eng.sparse_code_patches(pm, f, alpha=alpha, first_tier=0)  # K1 (or by reference) + K2 + K3
        else:
            if H0 is None:
                # rand(m, r) band after band is the stream of n calls of np.random.rand(r, 1); already sample-major
                Ht = _host.to_device(np.random.rand(m, r), dtype, dev)
            else:
                Ht = _host.to_sample_major(H0[:, j0:j1], dtype, dev)
            _lib.gather_patches_mb(pm, Xt[:m])                               # K1
            _lib.cov(Xt[:m], Wd, Ct[:m])
            _lib.pgd_code_columns(G, Ct[:m], alpha, sub_iter, stopping_diff, Ht)
        _lib.cov(Ht, Wt, R[:m])                                              # patch reconstructions (m x d) = Ht W^T
        _lib.patch_grid_accumulate(R[:m], j0, j1, ny, nx, k, s, C, Hh, Ww, canvas, count)
        if return_code:
            code[:, j0:j1] = _host.from_sample_major(Ht)
    out = canvas.cpu().numpy().astype(np.float64)
    res = (out[:, :, 0] if squeeze else out, count.cpu().numpy().astype(np.float64))
    if return_code:
        res = res + (code,)
    return res


def reconstruct_from_patches_2d(patches_or_W, image_size, code=None, precision=None):
    """Overlap-averaged image from ALL its patches in sklearn's order -- the last two lines of the drivers' one-shot
    reconstruction (image_reconstruction.py:351-354, image_reconstruction_tensor.py:280-283, ising_reconstruction.py:196-199):

        patches_recons = np.dot(W, code).T.reshape(N, k, k);  img = reconstruct_from_patches_2d(patches_recons, dims)

    Two call forms: `reconstruct_from_patches_2d(patches (N, k, k[, C]), (H, W))` -- sklearn's signature, the patches are
    uploaded -- or `reconstruct_from_patches_2d(W (k*k*C, r), (H, W), code=code (r, N))`, which forms W code on the device
    (K2-style product) and never materialises the N x k x k array on the host.  Both end in the deterministic gather-form
    mean kernel onmf_patch_grid_mean.  Returns numpy float64 (H, W[, C])."""
    dev = _host.device()
    dtype = _host.torch_dtype(precision)
    Hh, Ww = int(image_size[0]), int(image_size[1])
    if code is None:
        P = np.asarray(patches_or_W, dtype=np.float64)
        if P.ndim not in (3, 4) or P.shape[1] != P.shape[2]:
            raise ValueError("patches must have shape (N, k, k) or (N, k, k, C)")
        n, k = P.shape[0], P.shape[1]
        C = 1 if P.ndim == 3 else P.shape[3]
        R = _host.to_device(P.reshape(n, -1), dtype, dev)
    else:
        W = np.asarray(patches_or_W, dtype=np.float64)
        d, r = W.shape
        C = int(image_size[2]) if len(image_size) > 2 else 1
        k = int(round(np.sqrt(d // C)))
        if k * k * C != d:
            raise ValueError("dictionary rows %d are not patch_size^2 * channels (channels = %d)" % (d, C))
        Ht = _host.to_sample_major(np.asarray(code, dtype=np.float64), dtype, dev)
        n = Ht.shape[0]
        if Ht.shape[1] != r:
            raise ValueError("code must have shape (r, N) = (%d, N)" % r)
        Wt = torch.empty(r, d, dtype=dtype, device=dev)
        _lib.transpose(_host.to_device(W, dtype, dev), Wt)
        R = torch.empty(n, d, dtype=dtype, device=dev)
        if n:
            _lib.cov(Ht, Wt, R)
    ny, nx = Hh - k + 1, Ww - k + 1
    if n != ny * nx:
        raise ValueError("expected (H-k+1)*(W-k+1) = %d patches, got %d" % (ny * nx, n))
    canvas = torch.empty(Hh, Ww, C, dtype=dtype, device=dev)
    _lib.patch_grid_mean(R, ny, nx, k, 1, C, Hh, Ww, canvas)
    out = canvas.cpu().numpy().astype(np.float64)
    return out[:, :, 0] if (C == 1 and len(image_size) == 2) else out


def reconstruct_network(G, W, embs, alpha=0, precision=None):
    """Batched form of Network_Reconstructor.reconstruct_network (network_reconstruction_nx.py:444-511).

    The reference walks the motif MCMC and, per step, builds ONE k x k adjacency patch (`get_single_patch_glauber`,
    :331-340), codes it with `SparseCoder(transform_alpha=0, 'lasso_lars', positive_code=True)` (:466-473), forms
    patch_recons = W code (:474-475) and folds every entry into a running-mean weight of the directed edge
    (emb[q], emb[r]) (:477-491).  The walk is the caller's (or patches.MotifChains on the device); given its states `embs`
    (recons_iter x k node labels, the embedding AFTER each update, i.e. what get_single_patch_glauber returns), this
    runs all steps at once: K1 motif patches -> K2 Gram/covariances -> K3 positive LARS at alpha -> Ht W^T -> one
    scatter kernel accumulating sum / count per directed pair.

    G: networkx graph (or scipy sparse adjacency, node labels = indices); W: (k*k, r) dictionary.  embs may also be an
    (n x k) int32 CUDA tensor of node positions (indices into G.nodes), e.g. from patches.MotifChains.sample; the patches,
    codes and reconstructions are those of the same states given as labels, and so are the pairs and counts (the sums are
    accumulated with FP64 atomics, whose order sets their last bits in either form).
    Returns (pairs (E x 2 node labels), weight (E,), count (E,)) sorted by (a, b) position in G.nodes -- the content
    of the reference's G_recons / G_overlap_count DiGraphs."""
    dev = _host.device()
    dtype = _host.torch_dtype(precision)
    W = np.asarray(W, dtype=np.float64)
    d, r = W.shape
    positions = isinstance(embs, torch.Tensor)
    if positions:
        if not embs.is_cuda or embs.dtype != torch.int32 or embs.dim() != 2:
            raise ValueError("embs as a tensor must be an (n x k) int32 CUDA tensor of node positions")
    else:
        embs = np.asarray(embs)
    n, kk = embs.shape
    if kk * kk != d:
        raise ValueError("dictionary has %d rows, expected k^2 = %d" % (d, kk * kk))
    if n == 0:
        return np.empty((0, 2), dtype=object), np.empty(0), np.empty(0, dtype=np.int64)
    rowptr, colidx, nodes = patches.graph_to_csr(G)
    if positions:
        # node positions (indices into G.nodes), e.g. MotifChains.sample: no per-entry label mapping on the host
        e = embs.to(dev).contiguous()
        if int(e.min()) < 0 or int(e.max()) >= len(nodes):
            raise ValueError("embs holds a node position outside [0, %d)" % len(nodes))
    else:
        pos = {u: i for i, u in enumerate(nodes)}
        emb_i = np.asarray([[pos[u] for u in row] for row in embs.tolist()], dtype=np.int32).reshape(n, kk)
        e = torch.from_numpy(emb_i).to(dev)
    Xt = torch.empty(n, d, dtype=dtype, device=dev)
    if n:
        _lib.motif_patches(torch.from_numpy(np.asarray(rowptr, dtype=np.int64)).to(dev),
                           torch.from_numpy(np.asarray(colidx, dtype=np.int32)).to(dev), e, Xt)      # K1
    Wd = _host.to_device(W, dtype, dev)
    eng = OnmfEngine(d, r, alpha=alpha, dtype=dtype, device=dev)
    Ht = eng.sparse_code(Xt, Wd, alpha=alpha)                                                        # K2 + K3
    Wt = torch.empty(r, d, dtype=dtype, device=dev)
    _lib.transpose(Wd, Wt)
    R = torch.empty(n, d, dtype=dtype, device=dev)
    if n:
        _lib.cov(Ht, Wt, R)                                                                          # patch_recons rows
    # Table size: a table of 2 * n * k^2 slots always suffices (every entry a distinct pair), but consecutive states of the
    # Glauber walk differ in one node, so a trajectory visits about n * (2k - 1) distinct directed pairs: start there (20 bytes
    # per slot -- the worst-case table of a 10^6-state trajectory at k = 21 would be 20 GB) and grow on the kernel's
    # "table full" report.  The rows of MotifChains.sample are time slices of independent chains, not one walk: each chain adds
    # up to k^2 pairs for its first state, so few samples per chain can need up to the worst case.  The start is not restated
    # for that ordering; the x4 growth below reaches the needed size in a few retries (log4 of k^2 / 8k, one retry at k = 21).
    worst = 2 * max(n * d, 1) + 2
    cap = 1024
    while cap < min(worst, 2 * n * 4 * kk + 2):
        cap *= 2
    while True:
        keys = torch.full((cap,), -1, dtype=torch.int64, device=dev)
        sums = torch.zeros(cap, dtype=torch.float64, device=dev)
        cnts = torch.zeros(cap, dtype=torch.int32, device=dev)
        failed = torch.zeros(1, dtype=torch.int32, device=dev)
        _lib.edge_scatter_add(R, e, keys, sums, cnts, failed)
        nf = int(failed.item())
        if nf == 0:
            break
        if cap >= worst:
            raise _lib.OnmfKernelError("edge_scatter_add could not place %d entries" % nf)
        del keys, sums, cnts
        cap *= 4
    return _table_result(keys, sums, cnts, nodes)


def _table_result(keys, sums, cnts, nodes):
    """(pairs, weight, count) of the occupied slots of an edge table, sorted by (a, b) position in nodes"""
    used = torch.nonzero(cnts > 0).flatten()
    kz = keys[used].cpu().numpy().astype(np.uint64)
    sm = sums[used].cpu().numpy()
    ct = cnts[used].cpu().numpy().astype(np.int64)
    order = np.argsort(kz, kind="stable")
    kz, sm, ct = kz[order], sm[order], ct[order]
    a, b = (kz >> np.uint64(32)).astype(np.int64), (kz & np.uint64(0xffffffff)).astype(np.int64)
    lab = np.asarray(nodes, dtype=object)
    pairs = np.stack([lab[a], lab[b]], axis=1) if len(kz) else np.empty((0, 2), dtype=object)
    return pairs, sm / np.maximum(ct, 1), ct


# First capacity of the streamed pair table (20 bytes per slot: 20 MB); it grows by doubling as pairs arrive.
_TABLE_START = 1 << 20
# Entries per scatter of the streamed form.  Before a scatter the table is grown to twice the slots in use plus the entries
# about to be added, so this sets the table's headroom (at most 2^24 slots, 320 MB: less than one full band's Xt at
# k = 21); it is large enough that the one host read of the slot count per scatter is a small part of the scatter.
_SCATTER_ENTRIES = 1 << 23


def _empty_table(cap, dev):
    return (torch.full((cap,), -1, dtype=torch.int64, device=dev), torch.zeros(cap, dtype=torch.float64, device=dev),
            torch.zeros(cap, dtype=torch.int32, device=dev))


def reconstruct_network_chains(chains, W, n_samples, steps_per_sample=1, alpha=0, precision=None, max_band=262144):
    """reconstruct_network(G, W, chains.sample(n_samples, steps_per_sample), alpha, precision) in device memory bounded by
    a band of states and the pair table, not by the trajectory: the streamed form of the drivers' reconstruct_network(
    recons_iter, is_glauber_recons) for long runs of patches.MotifChains.

    The n_chains x n_samples states are taken in bands: a chain range [c0, c1) times a run of consecutive samples, each at
    least _lib.coder_band_floor() states (unless the whole run is smaller) and at most about max_band, by _band_plan's rule.
    A band advances chains c0 .. c1-1 only (a trajectory depends on (seed, chain, step), so these are the states of one
    sample() call), forms its motif patches, codes them (first tier 0 in every band: an earlier band's tier hint must not
    steer this one), forms R = Ht W^T and adds R to one pair table with onmf_edge_table_add.  The table starts small and is
    moved into a larger one (onmf_edge_table_grow) whenever the next scatter could take its load above 1/2; no entry is
    ever rescattered.  Its final size is set by the distinct directed pairs visited, 20 bytes per slot at load <= 1/2.

    Returns (pairs, weight, count) as reconstruct_network: the same pairs and counts, the same codes and reconstructions,
    weights equal up to the order of the FP64 atomic sums.  chains.state and chains.step end where that sample() call
    leaves them.  A chain state that is not a homomorphism raises (OnmfKernelError) when its chain range is reached."""
    if not isinstance(chains, patches.MotifChains):
        raise ValueError("chains must be a patches.MotifChains")
    W = np.asarray(W, dtype=np.float64)
    if W.ndim != 2:
        raise ValueError("W must be a (k^2 x r) dictionary")
    d, r = W.shape
    kk = chains.kk
    if d != kk * kk:
        raise ValueError("dictionary has %d rows, expected k^2 = %d" % (d, kk * kk))
    n_samples, sps = int(n_samples), int(steps_per_sample)
    if n_samples < 0:
        raise ValueError("n_samples must be >= 0")
    if sps < 1:
        raise ValueError("steps_per_sample must be >= 1")
    dtype = _host.torch_dtype(precision)
    N = chains.n_chains
    if n_samples == 0 or N == 0:
        return np.empty((0, 2), dtype=object), np.empty(0), np.empty(0, dtype=np.int64)
    dev = chains.state.device
    floor = _lib.coder_band_floor(dev)
    plan = [(c0, c1, _band_plan(n_samples, max(max_band // (c1 - c0), 1), -(-floor // (c1 - c0))))
            for c0, c1 in _band_plan(N, max_band, floor)]
    mmax = max((c1 - c0) * (s1 - s0) for c0, c1, sb in plan for s0, s1 in sb)
    run = patches._MOTIF_STEPS[chains.mcmc]
    Wd = _host.to_device(W, dtype, dev)
    eng = OnmfEngine(d, r, alpha=alpha, dtype=dtype, device=dev)
    f = eng.derive_foreign(Wd)
    Wt = torch.empty(r, d, dtype=dtype, device=dev)
    _lib.transpose(Wd, Wt)
    emb = torch.empty(mmax, kk, dtype=torch.int32, device=dev)
    Xt = torch.empty(mmax, d, dtype=dtype, device=dev)
    R = torch.empty(mmax, d, dtype=dtype, device=dev)
    keys, sums, cnts = _empty_table(_TABLE_START, dev)
    claimed = torch.zeros(1, dtype=torch.int64, device=dev)
    failed = torch.zeros(1, dtype=torch.int32, device=dev)
    chunk = max(1, _SCATTER_ENTRIES // d)
    for c0, c1, sbands in plan:
        state = chains.state[c0:c1]
        for s0, s1 in sbands:
            m = (c1 - c0) * (s1 - s0)
            e = emb[:m]
            run(chains.rowptr, chains.colidx, state, c0, chains.seed, chains.step + s0 * sps, sps, e)
            _lib.motif_patches(chains.rowptr, chains.colidx, e, Xt[:m])                             # K1
            Ht = eng.sparse_code(Xt[:m], f, alpha=alpha, first_tier=0)                               # K2 + K3
            _lib.cov(Ht, Wt, R[:m])                                                                  # patch_recons rows
            for j0 in range(0, m, chunk):
                j1 = min(m, j0 + chunk)
                need = 2 * (int(claimed.item()) + (j1 - j0) * d)
                if need > keys.numel():
                    cap = keys.numel()
                    while cap < need:
                        cap *= 2
                    grown = _empty_table(cap, dev)
                    _lib.edge_table_grow(keys, sums, cnts, *grown, failed)
                    keys, sums, cnts = grown
                _lib.edge_table_add(R[j0:j1], e[j0:j1], keys, sums, cnts, claimed, failed)
    chains.step += n_samples * sps
    nf = int(failed.item())
    if nf:
        raise _lib.OnmfKernelError("edge_table_add / edge_table_grow could not place %d entries" % nf)
    return _table_result(keys, sums, cnts, chains.nodes)


def simple_graph_edges(pairs, weight):
    """The reference's final rounding (network_reconstruction_nx.py:499-507): undirected edge {a, b} when the mean
    weight of the directed pair rounds to a positive integer.  Returns a set of frozensets."""
    out = set()
    for (a, b), w in zip(pairs.tolist(), np.asarray(weight).tolist()):
        if np.round(w) > 0:
            out.add(frozenset((a, b)))
    return out
