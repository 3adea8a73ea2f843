"""Streamed network reconstruction (reconstruct.reconstruct_network_chains, onmf_edge_table_add, onmf_edge_table_grow).

The streamed form takes the states of patches.MotifChains in bands and adds them to one growable pair table; it must give
what the one-pass reconstruct_network gives on the states of one sample() call of a twin chain object -- the same pairs and
counts, weights up to the order of the FP64 atomic sums -- and leave the chains where that call leaves them."""
import networkx as nx
import numpy as np
import pytest
import torch

from onmf_ontf_ndl_b200 import _lib, patches
from onmf_ontf_ndl_b200 import reconstruct as rec
from onmf_ontf_ndl_b200.patches import MotifChains

gpu = pytest.mark.gpu


def _graph(n_nodes=60, m_edges=200, seed=2):
    G = nx.gnm_random_graph(n_nodes, m_edges, seed=seed)
    G.add_edges_from((i, i + 1) for i in range(n_nodes - 1))
    return G


def _dictionary(kk, r, seed):
    W = np.random.default_rng(seed).random((kk * kk, r))
    return W / np.linalg.norm(W, axis=0)


def _twins(G, kk, n_chains, seed, mcmc, offset, sps):
    """two identical chain objects, both advanced by `offset` samples"""
    out = []
    for _ in range(2):
        ch = MotifChains(G, kk, n_chains, seed, mcmc=mcmc)
        if offset:
            ch.sample(offset, sps)
        out.append(ch)
    return out


def _assert_same(got, ref, ch, twin, what):
    (p, w, c), (p0, w0, c0) = got, ref
    assert np.array_equal(p.astype(np.int64), p0.astype(np.int64)), what
    assert np.array_equal(c, c0), what
    # the per-pair sums are accumulated with FP64 atomics, whose order sets their last bits
    assert np.allclose(w, w0, rtol=1e-12, atol=1e-14), what
    assert torch.equal(ch.state, twin.state) and ch.step == twin.step, what


def _streamed_vs_one_pass(G, W, kk, n_chains, n_samples, sps, seed, mcmc, precision, max_band, offset=2):
    ch, twin = _twins(G, kk, n_chains, seed, mcmc, offset, sps)
    ref = rec.reconstruct_network(G, W, twin.sample(n_samples, sps), alpha=0, precision=precision)
    got = rec.reconstruct_network_chains(ch, W, n_samples, sps, alpha=0, precision=precision, max_band=max_band)
    _assert_same(got, ref, ch, twin, (kk, n_chains, n_samples, sps, mcmc, precision, max_band))
    return got


def _count_calls(monkeypatch, module, name):
    calls = []
    fn = getattr(module, name)

    def counted(*a, **k):
        calls.append(1)
        return fn(*a, **k)
    monkeypatch.setattr(module, name, counted)
    return calls


# ------------------------------------------------------------------------------------------------------ 1. equal to one pass
@gpu
@pytest.mark.parametrize("mcmc", ["glauber", "pivot"])
@pytest.mark.parametrize("precision", ["fp32", "fp64"])
@pytest.mark.parametrize("kk", [2, 6, 21])
@pytest.mark.parametrize("sps", [1, 3])
def test_streamed_equals_one_pass(mcmc, precision, kk, sps, monkeypatch):
    # 24 chains x 10 samples = 240 states, far below the coder's variant thresholds, so bands far below the production floor
    # take the same kernel variants as the whole run: a floor of 1 lets a small max_band split it into many bands
    monkeypatch.setattr(_lib, "coder_band_floor", lambda device=None: 1)
    G = _graph()
    W = _dictionary(kk, 7 if kk > 2 else 3, kk)
    n_chains, n_samples = 24, 10
    for max_band, n_bands in ((262144, 1), (3 * n_chains, 4), (10, 3 * n_samples)):
        # one band; whole time slices, 3 or 2 per band; n_chains > max_band: chain ranges of 8, one sample each
        calls = []
        run = patches._MOTIF_STEPS[mcmc]
        monkeypatch.setitem(patches._MOTIF_STEPS, mcmc, lambda *a, **k: (calls.append(1), run(*a, **k))[1])
        for offset in (0, 2):                         # fresh chains, and chains an earlier sample() call has advanced
            calls.clear()
            _streamed_vs_one_pass(G, W, kk, n_chains, n_samples, sps, 5, mcmc, precision, max_band, offset)
            # the twins' offset calls, the twin's one sample() call and one chain call per band
            assert len(calls) == (2 if offset else 0) + 1 + n_bands
        monkeypatch.setitem(patches._MOTIF_STEPS, mcmc, run)


@gpu
def test_bands_above_the_coder_thresholds_keep_the_real_floor(monkeypatch):
    # 1000 chains x 16 samples = 16,000 states: above every LARS variant threshold (<= 48 x SMs).  max_band = 1000 asks for
    # bands far below them; the floor (48 x SMs + 1 states) keeps each band on the whole run's variant, so two bands of 8
    # time slices
    floor = _lib.coder_band_floor()
    n_chains = 1000
    n_samples = 2 * -(-floor // n_chains)
    calls = []
    run = patches._MOTIF_STEPS["pivot"]
    monkeypatch.setitem(patches._MOTIF_STEPS, "pivot", lambda *a, **k: (calls.append(1), run(*a, **k))[1])
    G = _graph(2000, 8000, 3)
    _streamed_vs_one_pass(G, _dictionary(6, 9, 1), 6, n_chains, n_samples, 1, 7, "pivot", "fp32", 1000, offset=0)
    assert len(calls) == 1 + 2                                       # the twin's sample() call and two bands


# ------------------------------------------------------------------------------------------------------------ 2. table growth
@gpu
@pytest.mark.parametrize("mcmc", ["glauber", "pivot"])
def test_table_grows_mid_run(mcmc, monkeypatch):
    monkeypatch.setattr(_lib, "coder_band_floor", lambda device=None: 1)
    monkeypatch.setattr(rec, "_TABLE_START", 1024)
    monkeypatch.setattr(rec, "_SCATTER_ENTRIES", 1024)            # scatters of 28 states at kk = 6
    grows = _count_calls(monkeypatch, _lib, "edge_table_grow")
    G = _graph(2000, 8000, 3)
    p, _, c = _streamed_vs_one_pass(G, _dictionary(6, 7, 2), 6, 64, 50, 1, 9, mcmc, "fp64", 640)
    assert len(grows) >= 3
    assert len(p) > 1024 and c.sum() == 64 * 50 * 36


def _mix64(x):
    x = np.asarray(x, dtype=np.uint64)
    with np.errstate(over="ignore"):
        x = x ^ (x >> np.uint64(30)); x = x * np.uint64(0xbf58476d1ce4e5b9)
        x = x ^ (x >> np.uint64(27)); x = x * np.uint64(0x94d049bb133111eb)
        x = x ^ (x >> np.uint64(31))
    return x


def _table(cap, dev):
    return rec._empty_table(cap, dev)


def _host_table(t):
    keys, sums, cnts = (x.cpu().numpy() for x in t)
    return keys.view(np.uint64), sums.view(np.uint64), cnts.view(np.uint32)


def _check_open_addressing(keys, sums, cnts):
    """every occupied slot lies on its key's probe sequence with no free slot before it (what a lookup relies on); free
    slots hold zero sums and counts"""
    cap = len(keys)
    empty = keys == np.uint64(0xFFFFFFFFFFFFFFFF)
    assert not np.any(sums[empty]) and not np.any(cnts[empty])
    occ = np.nonzero(~empty)[0]
    home = (_mix64(keys[occ]) & np.uint64(cap - 1)).astype(np.int64)
    for pos, h in zip(occ.tolist(), home.tolist()):
        span = np.arange(h, h + ((pos - h) % cap)) % cap
        assert not np.any(empty[span])


def _triples(keys, sums, cnts):
    occ = keys != np.uint64(0xFFFFFFFFFFFFFFFF)
    return sorted(zip(keys[occ].tolist(), sums[occ].tolist(), cnts[occ].tolist()))


def _filled_table(cap, n, kk, n_nodes, dtype, seed, dev):
    rng = np.random.default_rng(seed)
    emb = torch.from_numpy(rng.integers(0, n_nodes, size=(n, kk)).astype(np.int32)).to(dev)
    R = torch.from_numpy(rng.standard_normal((n, kk * kk))).to(dev, dtype)
    t = _table(cap, dev)
    claimed = torch.zeros(1, dtype=torch.int64, device=dev)
    failed = torch.zeros(1, dtype=torch.int32, device=dev)
    _lib.edge_table_add(R, emb, *t, claimed, failed)
    assert int(failed.item()) == 0
    return t, R, emb, claimed, failed


@gpu
def test_edge_table_grow_moves_every_triple():
    dev = torch.device("cuda", 0)
    t, R, emb, claimed, failed = _filled_table(1024, 50, 3, 20, torch.float64, 1, dev)   # <= 400 pairs: load <= 1/2
    old = _host_table(t)
    _check_open_addressing(*old)
    ref = _triples(*old)
    assert len(ref) == int(claimed.item()) > 100
    for cap in (2048, 1 << 16):
        g = _table(cap, dev)
        _lib.edge_table_grow(*t, *g, failed)
        new = _host_table(g)
        assert int(failed.item()) == 0
        assert _triples(*new) == ref                                  # bit-exact keys, sums and counts; none lost or doubled
        _check_open_addressing(*new)
        assert all(np.array_equal(a, b) for a, b in zip(_host_table(t), old))            # the old table is only read
        # the grown table is a table: adding the same entries again claims no slot and doubles every count
        c2 = torch.zeros(1, dtype=torch.int64, device=dev)
        _lib.edge_table_add(R, emb, *g, c2, failed)
        assert int(c2.item()) == 0 and int(failed.item()) == 0
        k3, _, n3 = _host_table(g)
        assert sorted(zip(k3[k3 != ~np.uint64(0)].tolist(), n3[k3 != ~np.uint64(0)].tolist())) == \
            sorted((k, 2 * c) for k, _, c in ref)


@gpu
def test_edge_table_grow_refusals_touch_nothing():
    dev = torch.device("cuda", 0)
    t, _, _, _, failed = _filled_table(1024, 50, 3, 20, torch.float64, 2, dev)
    old = _host_table(t)
    for cap in (1024, 512, 3000):                  # not larger; smaller; not a power of two
        g = _table(cap, dev)
        before = _host_table(g)
        with pytest.raises(_lib.OnmfKernelError):
            _lib.edge_table_grow(*t, *g, failed)
        assert all(np.array_equal(a, b) for a, b in zip(_host_table(g), before))
        assert all(np.array_equal(a, b) for a, b in zip(_host_table(t), old))
    g = _table(2048, dev)
    before = _host_table(g)
    lib = _lib.load()
    # an old capacity that is not a power of two, and a NULL pointer
    assert lib.onmf_edge_table_grow(t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), 1000, g[0].data_ptr(), g[1].data_ptr(),
                                    g[2].data_ptr(), 2048, failed.data_ptr(), None) == -1
    assert lib.onmf_edge_table_grow(t[0].data_ptr(), None, t[2].data_ptr(), 1024, g[0].data_ptr(), g[1].data_ptr(),
                                    g[2].data_ptr(), 2048, failed.data_ptr(), None) == -1
    torch.cuda.synchronize()
    assert all(np.array_equal(a, b) for a, b in zip(_host_table(g), before))
    assert all(np.array_equal(a, b) for a, b in zip(_host_table(t), old))
    assert int(failed.item()) == 0


# ---------------------------------------------------------------------------------------------------- 3. onmf_edge_table_add
@gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_edge_table_add_counts_new_pairs_and_equals_scatter_add(dtype):
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(3)
    kk, cap = 5, 1 << 14
    t = _table(cap, dev)
    ref = _table(cap, dev)
    claimed = torch.zeros(1, dtype=torch.int64, device=dev)
    failed = torch.zeros(1, dtype=torch.int32, device=dev)
    seen = set()
    for n, n_nodes in ((40, 30), (200, 60), (1, 60)):                # batches with repeats within and across calls
        e = rng.integers(0, n_nodes, size=(n, kk)).astype(np.int32)
        emb = torch.from_numpy(e).to(dev)
        R = torch.from_numpy(rng.standard_normal((n, kk * kk))).to(dev, dtype)
        before = int(claimed.item())
        _lib.edge_table_add(R, emb, *t, claimed, failed)
        _lib.edge_scatter_add(R, emb, *ref, failed)
        new = {(int(a), int(b)) for row in e for a in row for b in row} - seen
        seen |= new
        assert int(claimed.item()) - before == len(new)
    assert int(failed.item()) == 0
    nodes = list(range(60))
    p, w, c = rec._table_result(*t, nodes)
    p0, w0, c0 = rec._table_result(*ref, nodes)
    assert len(p) == len(seen)
    assert np.array_equal(p.astype(np.int64), p0.astype(np.int64)) and np.array_equal(c, c0)
    assert np.allclose(w, w0, rtol=1e-12, atol=1e-14)
    with pytest.raises(_lib.OnmfKernelError):                          # the slot counter is required
        rc = _lib.load().onmf_edge_table_add(_lib.dt(R), R.data_ptr(), kk * kk, emb.data_ptr(), 1, kk, t[0].data_ptr(),
                                             t[1].data_ptr(), t[2].data_ptr(), cap, None, failed.data_ptr(), None)
        _lib._check(rc, "onmf_edge_table_add")


# ---------------------------------------------------------------------------------------------------------- 4. bounded memory
def _torus(side):
    G = nx.Graph()
    G.add_nodes_from(range(side * side))
    for i in range(side):
        for j in range(side):
            G.add_edge(i * side + j, ((i + 1) % side) * side + j)
            G.add_edge(i * side + j, i * side + (j + 1) % side)
    return G


def _one_pass_bytes(n, kk, r, esize):
    """device bytes of reconstruct_network on n states, from its shapes: Xt and R (n x kk^2), the engine's Ct and Ht (n x r),
    the states (n x kk int32) and the first pair table (20 bytes per slot)"""
    d = kk * kk
    worst = 2 * max(n * d, 1) + 2
    cap = 1024
    while cap < min(worst, 2 * n * 4 * kk + 2):
        cap *= 2
    return 2 * n * d * esize + 2 * n * r * esize + 4 * n * kk + 20 * cap


@gpu
def test_streamed_memory_is_bounded_by_band_and_table():
    # a 200 x 200 torus has small balls, so few distinct pairs; 5 * 10^6 states at kk = 21 need more than 30 GB in one pass
    side, kk, r, n_chains, n_samples = 200, 21, 25, 50000, 100
    n, d = n_chains * n_samples, kk * kk
    assert _one_pass_bytes(n, kk, r, 4) > 30e9
    G = _torus(side)
    W = _dictionary(kk, r, 4)
    ch = MotifChains(G, kk, n_chains, 11, mcmc="pivot")
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    p, w, c = rec.reconstruct_network_chains(ch, W, n_samples, alpha=0, precision="fp32")
    peak = torch.cuda.max_memory_allocated() - base
    assert ch.step == n_samples and c.sum() == n * d and np.all(c > 0)
    # bound: the band buffers (states, Xt, R, codes, covariances, coder workspace), the table at its largest while it is
    # moved (at most 2x its final capacity, which is the power of two above 2 (distinct pairs + one scatter)), and 256 MB
    mmax = max(262144, 2 * _lib.coder_band_floor())
    band = mmax * (4 * kk + 2 * d * 4 + 2 * r * 4) + _lib.lasso_lars_workspace(torch.float32, r, mmax)
    cap = 1
    while cap < 2 * (len(p) + (rec._SCATTER_ENTRIES // d) * d):
        cap *= 2
    bound = band + 2 * 20 * cap + (256 << 20)
    assert bound < 8e9, bound
    assert peak <= bound, (peak, bound)
    # every pair is two positions of one path of kk nodes: within torus distance kk - 1
    a, b = p[:, 0].astype(np.int64), p[:, 1].astype(np.int64)
    di, dj = np.abs(a // side - b // side), np.abs(a % side - b % side)
    dist = np.minimum(di, side - di) + np.minimum(dj, side - dj)
    assert dist.max() <= kk - 1
    assert np.all(np.isfinite(w))


# --------------------------------------------------------------------------------------------------------------- 5. refusals
@gpu
def test_refusals_before_any_device_work(monkeypatch):
    G = _graph()
    ch = MotifChains(G, 6, 8, 1)
    state, step = ch.state.clone(), ch.step
    W = _dictionary(6, 7, 0)

    def no_kernels():
        raise AssertionError("a kernel was called")
    monkeypatch.setattr(_lib, "load", no_kernels)
    for args, kw in (((ch, W[:35], 4), {}), ((ch, W, -1), {}), ((ch, W, 4), {"steps_per_sample": 0}),
                     ((patches.graph_to_csr(G), W, 4), {}), ((ch, W[:, 0], 4), {})):
        with pytest.raises(ValueError):
            rec.reconstruct_network_chains(*args, **kw)
    assert torch.equal(ch.state, state) and ch.step == step
