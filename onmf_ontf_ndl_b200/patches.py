"""On-device patch pipelines (SURVEY.md §8f.2, §8f.4): the drivers build their d x N data matrices with O(N^2)
`np.append` loops; here the image / lattice / graph lives on the GPU, patch positions are drawn on the host in the
reference's RNG order, and one K1 kernel gathers every patch.  Outputs are numpy float64 in the reference's shapes
(or device tensors in the sample-major layout with device=True)."""
from __future__ import annotations

import numpy as np
import torch

from . import _host, _lib


def sample_patch_coords(shape, patch_size, num_patches):
    """Top-left corners in the reference's draw order: a = np.random.choice(H - k), b = np.random.choice(W - k),
    interleaved per patch (image_reconstruction.py:184-186, image_reconstruction_tensor.py:103-104,
    ising_reconstruction.py:57-58).  The last valid offset is excluded, like the reference."""
    k = patch_size
    out = np.empty((num_patches, 2), dtype=np.int32)
    for i in range(num_patches):
        out[i, 0] = np.random.choice(shape[0] - k)
        out[i, 1] = np.random.choice(shape[1] - k)
    return out


def gather_patches(img, coords, patch_size, precision=None, device=False):
    """img (H x W) or (H x W x C), coords (N x 2) -> data matrix X (k*k*C, N), feature f = (row*k + col)*C + ch.
    For a gray image this is `extract_random_patches` of image_reconstruction.py:173-206; for a colour image it is the
    mode-2 joint unfolding of the (k*k, 3, N) tensor of image_reconstruction_tensor.py:87-124 (see patches_to_tensor)."""
    dev = _host.device()
    dtype = _host.torch_dtype(precision)
    A = np.asarray(img, dtype=np.float64)
    A3 = A[:, :, None] if A.ndim == 2 else A
    C = A3.shape[2]
    co = torch.from_numpy(np.ascontiguousarray(np.asarray(coords, dtype=np.int32))).to(dev)
    n = co.shape[0]
    out = torch.empty(n, patch_size * patch_size * C, dtype=dtype, device=dev)
    if n:
        _lib.gather_patches(_host.to_device(A3, dtype, dev), co, patch_size, out)
    return out if device else _host.from_sample_major(out)


def extract_patches_2d(img, patch_size, precision=None, device=False):
    """ALL patches of an image in sklearn's order -- the data matrix the drivers build for reconstruction with
    `extract_patches_2d(data, (k, k)).reshape(N, -1).T` (image_reconstruction.py:163-166, ising_reconstruction.py:185-186):
    corners (i, j), i in 0..H-k, j in 0..W-k (the last offset INCLUDED, unlike the random sampler), row-major.
    Returns X (k*k*C, N) numpy float64, or the sample-major device tensor (N x k*k*C) with device=True."""
    A = np.asarray(img)
    return gather_patches(A, all_patch_coords(A.shape, patch_size), int(patch_size), precision, device)


def all_patch_coords(shape, patch_size, stride=1, include_last=True):
    """Top-left corners of a patch grid, row-major, as an (N x 2) int32 array.  include_last=True: every offset 0..H-k
    (sklearn's extract_patches_2d order); False: `range(0, H - k, stride)` -- the grid of the drivers' reconstruction loop
    (image_reconstruction.py:375-376), which leaves the last offset out."""
    k, s = int(patch_size), int(stride)
    if k > shape[0] or k > shape[1]:
        raise ValueError("patch_size %d larger than the image %s" % (k, tuple(shape[:2])))
    ys = np.arange(0, shape[0] - k + (1 if include_last else 0), s)
    xs = np.arange(0, shape[1] - k + (1 if include_last else 0), s)
    gy, gx = np.meshgrid(ys, xs, indexing="ij")
    return np.stack([gy.reshape(-1), gx.reshape(-1)], 1).astype(np.int32)


def extract_random_patches(img, patch_size, num_patches, precision=None):
    """Drop-in for the drivers' extract_random_patches: gray -> (k*k, N); colour -> tensor (k*k, C, N)."""
    A = np.asarray(img)
    co = sample_patch_coords(A.shape, patch_size, num_patches)
    X = gather_patches(A, co, patch_size, precision)
    return X if A.ndim == 2 else patches_to_tensor(X, A.shape[2])


class ImagePatches:
    """The data matrix X (d x N), d = p*p*C, of the p x p patches of ONE image at the corners `coords`, kept by reference:
    the image and the corners live on the device and no patch is ever written out.  X[(r*p + c)*C + ch, j] =
    img[y_j + r, x_j + c, ch] -- the feature order of gather_patches.  Pass it as `X` to Online_NMF, or to
    OnmfEngine.step_patches with minibatch indices into [0, N).

    img: (H x W) or (H x W x C) array or tensor.  uint8 keeps uint8 storage on the device (value = float32(stored) *
    float32(scale), scale defaulting to 1/255, the drivers' `data / 255`; fp32 engine only); any other dtype is stored in
    `precision` ("fp32" default, or "fp64").  A corner whose patch leaves the image stands for a NaN column."""

    def __init__(self, img, patch_size, coords, scale=None, precision=None):
        a = img.detach() if isinstance(img, torch.Tensor) else np.asarray(img)
        if a.ndim not in (2, 3):
            raise ValueError("img must be (H x W) or (H x W x C), got shape %s" % (tuple(a.shape),))
        co = coords.detach().cpu().numpy() if isinstance(coords, torch.Tensor) else np.asarray(coords)
        if co.ndim != 2 or co.shape[1] != 2:
            raise ValueError("coords must be an (N x 2) array of top-left corners, got shape %s" % (tuple(co.shape),))
        if co.size and not np.issubdtype(co.dtype, np.integer):
            raise ValueError("coords must be integers, got %s" % co.dtype)
        p = int(patch_size)
        H, W = int(a.shape[0]), int(a.shape[1])
        C = int(a.shape[2]) if a.ndim == 3 else 1
        if p <= 0 or p > H or p > W or C <= 0:
            raise ValueError("patch_size %d does not fit the image %s" % (p, (H, W)))
        u8 = (a.dtype == torch.uint8) if isinstance(a, torch.Tensor) else (a.dtype == np.uint8)
        if u8:
            if precision is not None and _host.torch_dtype(precision) != torch.float32:
                raise ValueError("a uint8 image is read by the fp32 engine only (precision must be fp32)")
            self.dtype = torch.uint8
            self.precision = "fp32"
            self.scale = 1.0 / 255.0 if scale is None else float(scale)
        else:
            if scale is not None:
                raise ValueError("scale applies to uint8 images only")
            self.dtype = _host.torch_dtype(precision)
            self.precision = "fp64" if self.dtype == torch.float64 else "fp32"
            self.scale = 1.0
        self.patch_size, self.H, self.W, self.C = p, H, W, C
        self.d, self.N = p * p * C, int(co.shape[0])
        dev = _host.device()
        if isinstance(a, torch.Tensor):
            t = a.to(dev, self.dtype if not u8 else torch.uint8)
        else:
            t = torch.from_numpy(np.ascontiguousarray(a if u8 else np.asarray(a, dtype=np.float64))).to(dev, self.dtype)
        self.img = t.reshape(H, W, C).contiguous()
        self.coords = torch.from_numpy(np.ascontiguousarray(co, dtype=np.int32).reshape(-1, 2)).to(dev)

    @property
    def shape(self):
        return (self.d, self.N)

    @property
    def engine_dtype(self):
        """dtype of the engine that reads these patches"""
        return torch.float64 if self.dtype == torch.float64 else torch.float32

    def minibatch(self, idx, n=None):
        """the C descriptor (onmf_patch_minibatch) of columns idx (int64 device tensor) or, idx None, columns 0..n-1"""
        n = int(idx.shape[0]) if idx is not None else (self.N if n is None else int(n))
        return _lib.make_patch_minibatch(self.img, self.patch_size, self.coords, idx, n, self.scale)

    def gather(self, idx=None, out=None, stream=None):
        """sample-major device tensor (n x d) of columns idx (None: all N), in the engine's dtype"""
        pm = self.minibatch(idx)
        if out is None:
            out = torch.empty(pm.n, self.d, dtype=self.engine_dtype, device=self.img.device)
        if pm.n:
            _lib.gather_patches_mb(pm, out, stream=stream)
        return out

    def to_matrix(self):
        """the (d x N) numpy float64 data matrix these patches stand for (small cases and tests)"""
        return _host.from_sample_major(self.gather())


def patches_to_tensor(X, channels):
    """(k*k*C, N) HWC data matrix -> the reference's (k*k, C, N) patch tensor (a view, no arithmetic)."""
    d, n = X.shape
    return X.reshape(d // channels, channels, n)


def graph_to_csr(G):
    """networkx Graph (or anything with .nodes / .neighbors) or a scipy sparse matrix -> (rowptr int64, colidx int32,
    node list); neighbour lists sorted, both directions present for undirected graphs."""
    if hasattr(G, "tocsr"):
        M = G.tocsr()
        M.sort_indices()
        return M.indptr.astype(np.int64), M.indices.astype(np.int32), list(range(M.shape[0]))
    nodes = list(G.nodes())
    pos = {u: i for i, u in enumerate(nodes)}
    rowptr = np.zeros(len(nodes) + 1, dtype=np.int64)
    cols = []
    for i, u in enumerate(nodes):
        nb = sorted(pos[v] for v in G.neighbors(u))
        cols.extend(nb)
        rowptr[i + 1] = len(cols)
    return rowptr, np.asarray(cols, dtype=np.int32), nodes


class SamplePool:
    """The data matrix X (d x N) held on the device in the sample-major layout: `Xt` (N x d, float32 or float64) is X^T.
    Pass it as `X` to Online_NMF to train on device-resident columns (for instance MotifChains.patches) without a host copy;
    the results are those of the same call on the host matrix X."""

    def __init__(self, Xt):
        if not isinstance(Xt, torch.Tensor) or not Xt.is_cuda or Xt.dim() != 2 or Xt.dtype not in (torch.float32, torch.float64):
            raise ValueError("Xt must be an (N x d) float32 / float64 CUDA tensor")
        self.Xt = Xt.contiguous()
        self.precision = "fp64" if Xt.dtype == torch.float64 else "fp32"

    @property
    def shape(self):
        return (self.Xt.shape[1], self.Xt.shape[0])


def _symmetric_csr(G):
    """graph_to_csr of a networkx graph or scipy adjacency, or a (rowptr, colidx[, nodes]) tuple; ValueError unless rows are
    ascending, in range and the adjacency is symmetric (M = M^T)."""
    if isinstance(G, tuple):
        rowptr, colidx = np.asarray(G[0], dtype=np.int64), np.asarray(G[1], dtype=np.int32)
        nodes = list(G[2]) if len(G) > 2 else list(range(len(rowptr) - 1))
    else:
        if hasattr(G, "is_directed") and G.is_directed():
            raise ValueError("motif chains need an undirected graph (got a directed one)")
        rowptr, colidx, nodes = graph_to_csr(G)
    n = len(rowptr) - 1
    if n <= 0 or len(nodes) != n or rowptr[0] != 0 or rowptr[-1] != len(colidx) or np.any(np.diff(rowptr) < 0):
        raise ValueError("malformed CSR")
    if n > np.iinfo(np.int32).max:
        raise ValueError("more than 2^31 - 1 nodes")
    rows = np.repeat(np.arange(n, dtype=np.int64), np.diff(rowptr))
    c64 = colidx.astype(np.int64)
    if len(c64) and (c64.min() < 0 or c64.max() >= n):
        raise ValueError("a neighbour index is outside the graph")
    if len(c64) > 1 and np.any((np.diff(c64) <= 0) & (rows[1:] == rows[:-1])):
        raise ValueError("CSR rows must be strictly ascending")
    if not np.array_equal(np.sort(rows * n + c64), np.sort(c64 * n + rows)):
        raise ValueError("the adjacency is not symmetric (directed graphs are not supported)")
    return rowptr, colidx, nodes


class MotifChains:
    """n_chains independent Glauber chains of homomorphisms of the path 0 - 1 - ... - kk-1 into an undirected graph, kept on the
    device: the motif MCMC of the NDL drivers (network_reconstruction_nx.py tree_sample / get_single_patch_glauber) without a
    host walk.  Every chain samples the same law; chain c's trajectory depends on (seed, c, step) only (include/onmf_b200.h,
    onmf_motif_chain), so two sample() calls give the bits of one longer call.

    G_or_csr: networkx graph, scipy sparse adjacency or a graph_to_csr tuple; it must be symmetric (ValueError otherwise).
    state: optional (n_chains x kk) initial states in node labels; by default each chain starts from a tree sample (a root
    uniform over the nodes with a neighbour, then uniform neighbours).  2 <= kk <= 32."""

    def __init__(self, G_or_csr, kk, n_chains, seed, state=None):
        rowptr, colidx, nodes = _symmetric_csr(G_or_csr)
        self.kk, self.n_chains = int(kk), int(n_chains)
        self.seed = int(seed)
        if not 0 <= self.seed < 2 ** 64:
            raise ValueError("seed must be in [0, 2^64)")
        self.nodes = nodes
        self.n_nodes = len(nodes)
        dev = _host.device()
        self.rowptr = torch.from_numpy(rowptr).to(dev)
        self.colidx = torch.from_numpy(np.ascontiguousarray(colidx)).to(dev)
        self.step = 0                                   # global Glauber steps run so far
        if state is None:
            self.state = torch.empty(self.n_chains, self.kk, dtype=torch.int32, device=dev)
            _lib.motif_chain_init(self.rowptr, self.colidx, self.state, 0, self.seed)
        else:
            pos = {u: i for i, u in enumerate(nodes)}
            st = np.asarray(state, dtype=object) if not isinstance(state, np.ndarray) else state
            if st.shape != (self.n_chains, self.kk):
                raise ValueError("state must have shape (n_chains, kk) = (%d, %d)" % (self.n_chains, self.kk))
            try:
                ix = np.asarray([[pos[u] for u in row] for row in st.tolist()], dtype=np.int32)
            except (KeyError, TypeError):
                raise ValueError("state names a node that is not in the graph")
            self.state = torch.from_numpy(ix.reshape(self.n_chains, self.kk)).to(dev)
        self._labels = None

    def sample(self, n_samples, steps_per_sample=1):
        """int32 device tensor (n_samples * n_chains x kk) of node positions: row s * n_chains + c is chain c after
        steps_per_sample * (s + 1) more steps.  Advances the chains and the step counter."""
        n_samples, sps = int(n_samples), int(steps_per_sample)
        out = torch.empty(n_samples * self.n_chains, self.kk, dtype=torch.int32, device=self.state.device)
        _lib.motif_chain(self.rowptr, self.colidx, self.state, 0, self.seed, self.step, sps, out)
        self.step += n_samples * sps
        return out

    def patches(self, n_samples, steps_per_sample=1, precision=None):
        """the sample-major (n_samples * n_chains x kk^2) motif-adjacency patches of sample(): row j, column q*kk + r =
        has_edge(x_j[q], x_j[r])"""
        emb = self.sample(n_samples, steps_per_sample)
        out = torch.empty(emb.shape[0], self.kk * self.kk, dtype=_host.torch_dtype(precision), device=emb.device)
        _lib.motif_patches(self.rowptr, self.colidx, emb, out)
        return out

    def labels(self, emb):
        """node labels (host object array, same shape) of node positions emb (device tensor or array)"""
        if self._labels is None:
            self._labels = np.empty(self.n_nodes, dtype=object)
            for i, u in enumerate(self.nodes):
                self._labels[i] = u
        e = emb.cpu().numpy() if isinstance(emb, torch.Tensor) else np.asarray(emb)
        return self._labels[e]


def frame_patch_coords(n_frames, shape, patch_size, num_patches):
    """Corners of num_patches patches in each of n_frames frames (H x W) stacked as one (n_frames * H x W) image: frame f, in
    order, draws sample_patch_coords(shape, patch_size, num_patches) and its rows are offset by f * H.  With one frame this
    is the drivers' draw.  ImagePatches(frames.reshape(n_frames * H, W), patch_size, coords) then stands for the patches of
    every frame by reference (no patch straddles two frames)."""
    H = int(shape[0])
    out = [sample_patch_coords(shape, patch_size, num_patches) for _ in range(int(n_frames))]
    for f, co in enumerate(out):
        co[:, 0] += f * H
    return np.concatenate(out) if out else np.empty((0, 2), dtype=np.int32)


class IsingChains:
    """n_chains independent checkerboard heat-bath chains of the Ising model (J = 1, no field) on an H x W torus, kept on the
    device: the lattice trajectory of the Ising driver (ising_simulator.ising_update / init_lattice) without a host loop.
    Every chain samples the Gibbs law P(sigma) ~ exp(beta sum_<ij> sigma_i sigma_j); chain c's trajectory depends on (seed, c,
    sweep) only (include/onmf_b200.h, onmf_ising_chain), so two sample() calls give the bits of one longer call.

    shape: (H, W), both even and >= 4.  state: optional (n_chains x H x W) +-1 initial lattices; by default each chain
    starts from independent uniform spins."""

    def __init__(self, shape, beta, n_chains, seed, state=None):
        if len(shape) != 2:
            raise ValueError("shape must be (H, W)")
        self.H, self.W = int(shape[0]), int(shape[1])
        if self.H < 4 or self.W < 4 or self.H % 2 or self.W % 2 or self.H * self.W >= 2 ** 31:
            raise ValueError("the lattice sides must be even and at least 4 (got %s)" % ((self.H, self.W),))
        self.beta = float(beta)
        if not np.isfinite(self.beta):
            raise ValueError("beta must be finite")
        self.n_chains = int(n_chains)
        if not 0 < self.n_chains <= 2 ** 32:
            raise ValueError("n_chains must be in [1, 2^32]")
        self.seed = int(seed)
        if not 0 <= self.seed < 2 ** 64:
            raise ValueError("seed must be in [0, 2^64)")
        self.sweep = 0                                  # global sweeps run so far
        if state is None:
            self.state = torch.empty(self.n_chains, self.H, self.W, dtype=torch.int8, device=_host.device())
            _lib.ising_chain_init(self.state, 0, self.seed)
        else:
            st = state.detach() if isinstance(state, torch.Tensor) else torch.from_numpy(np.asarray(state))
            if tuple(st.shape) != (self.n_chains, self.H, self.W):
                raise ValueError("state must have shape (n_chains, H, W) = %s" % ((self.n_chains, self.H, self.W),))
            if st.is_complex() or not bool(((st == 1) | (st == -1)).all()):
                raise ValueError("state must hold +-1 spins")
            self.state = st.to(_host.device(), torch.int8).contiguous()

    def sample(self, n_samples, sweeps_per_sample=1, precision=None):
        """device tensor (n_samples * n_chains x H x W) of +-1 in `precision` (fp32 default): row s * n_chains + c is chain c
        after sweeps_per_sample * (s + 1) more sweeps.  Advances the chains and the sweep counter."""
        n_samples, sps = int(n_samples), int(sweeps_per_sample)
        out = torch.empty(n_samples * self.n_chains, self.H, self.W, dtype=_host.torch_dtype(precision), device=self.state.device)
        _lib.ising_chain(self.state, 0, self.seed, self.beta, self.sweep, sps, out)
        self.sweep += n_samples * sps
        return out


def motif_patches(csr, emb, precision=None, device=False):
    """emb (N x kk) node positions (indices into the CSR) of N motif embeddings -> X (kk*kk, N) with
    X[q*kk + r, j] = has_edge(emb[j, q], emb[j, r])   (network_reconstruction_nx.py:302-305, 315-329)."""
    dev = _host.device()
    dtype = _host.torch_dtype(precision)
    rowptr, colidx = csr[0], csr[1]
    e = torch.from_numpy(np.ascontiguousarray(np.asarray(emb, dtype=np.int32))).to(dev)
    n, kk = e.shape
    out = torch.empty(n, kk * kk, dtype=dtype, device=dev)
    if n:
        _lib.motif_patches(torch.from_numpy(np.asarray(rowptr, dtype=np.int64)).to(dev),
                           torch.from_numpy(np.asarray(colidx, dtype=np.int32)).to(dev), e, out)
    return out if device else _host.from_sample_major(out)
