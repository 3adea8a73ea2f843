"""NDL motif embeddings on the device (csrc/motif_chain.cu, patches.MotifChains, ndl.train_dict).

The kernels are held to oracle/motif_chain.py bit for bit (Philox4x32-10 and both chains restated in numpy); the oracle is
held to the chain's exact law on a small graph (every homomorphism enumerated, exact initial law and transition matrix) by
a chi-square test that three mutants with one plausible kernel bug each fail; and both are held, with the reference's own
trajectory, to the invariants of a Glauber chain of homomorphisms."""
import itertools

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.stats as ss

from oracle import motif_chain as mc

gpu = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------------------------ fixtures
def _csr(n, edges):
    """symmetric CSR (rowptr int64, colidx int32) and dense adjacency of an undirected edge list"""
    A = np.zeros((n, n), dtype=bool)
    for a, b in edges:
        A[a, b] = A[b, a] = True
    M = sp.csr_matrix(A.astype(np.int8))
    M.sort_indices()
    return M.indptr.astype(np.int64), M.indices.astype(np.int32), A


def _test_graph():
    """130 nodes: two hubs (0, 1) sharing 80 neighbours (an intersection of three warp strides), a sparse random remainder,
    a self-loop at node 5 and an isolated node 129"""
    rng = np.random.default_rng(11)
    edges = [(0, v) for v in range(2, 82)] + [(1, v) for v in range(2, 82)] + [(5, 5)]
    edges += [(int(a), int(b)) for a, b in rng.integers(2, 129, size=(260, 2)) if a != b]
    edges += [(v, v + 1) for v in range(2, 128)]
    return _csr(130, edges)


def _law_graph():
    """8 nodes, connected, with triangles (not bipartite)"""
    return _csr(8, [(i, (i + 1) % 8) for i in range(8)] + [(0, 2), (3, 6), (1, 5)])


LAW_KK, LAW_N, LAW_SEED, LAW_T = 4, 1 << 17, 2024, (0, 1, 5, 200)
# p-values of the oracle at (T = 0, 1, 5, 200) with this seed: 0.553, 0.324, 0.426, 0.820.  Mutants at T = 200: no last site
# 2.3e-58, union and rank-off 0 (states that are not homomorphisms).
P_MIN = 1e-3


class _ExactLaw:
    """Hom(P_kk, G) enumerated, the exact initial law p0 (root uniform, then uniform neighbours) and the exact Glauber matrix"""

    def __init__(self, A, kk):
        n = A.shape[0]
        self.n, self.kk = n, kk
        self.homs = [h for h in itertools.product(range(n), repeat=kk) if all(A[h[q], h[q + 1]] for q in range(kk - 1))]
        ix = {h: i for i, h in enumerate(self.homs)}
        H = len(self.homs)
        deg = A.sum(1)
        nz = int((deg > 0).sum())
        self.p0 = np.array([np.prod([1.0 / deg[h[q]] for q in range(kk - 1)]) / nz for h in self.homs])
        P = np.zeros((H, H))
        for h in self.homs:
            for i in range(kk):
                a = h[1] if i == 0 else h[i - 1]
                b = h[kk - 2] if i == kk - 1 else h[i + 1]
                S = np.nonzero(A[a] & A[b])[0]
                for v in S:
                    y = list(h)
                    y[i] = int(v)
                    P[ix[h], ix[tuple(y)]] += 1.0 / (kk * len(S))
        self.P = P
        self.code = {sum(h[q] * n ** (kk - 1 - q) for q in range(kk)): i for i, h in enumerate(self.homs)}

    def irreducible(self):
        H = len(self.homs)
        R = (self.P > 0).astype(np.float64) + np.eye(H)
        reach = np.eye(H)
        for _ in range(int(np.ceil(np.log2(H))) + 1):
            reach = np.minimum(reach @ R + reach, 1.0)
            R = np.minimum(R @ R, 1.0)
        return bool((reach > 0).all())

    def pvalue(self, x, T):
        """chi-square p-value of the empirical law of the states x against p0 P^T (0 when a state is not a homomorphism)"""
        pt = self.p0 @ np.linalg.matrix_power(self.P, T)
        keys = np.asarray(x, dtype=np.int64) @ (self.n ** np.arange(self.kk)[::-1])
        idx = np.array([self.code.get(int(k), -1) for k in keys])
        if (idx < 0).any():
            return 0.0
        obs = np.bincount(idx, minlength=len(self.homs))
        exp = pt * len(x)
        return float(ss.chi2.sf(((obs - exp) ** 2 / exp).sum(), len(self.homs) - 1))


@pytest.fixture(scope="module")
def law():
    rp, ci, A = _law_graph()
    L = _ExactLaw(A, LAW_KK)
    x0 = mc.chain_init(rp, ci, LAW_KK, LAW_N, 0, LAW_SEED)
    return L, A, x0


def _oracle_slices(A, x0, mutant=None):
    """{T: states after T steps} for T in LAW_T, continuing one run (the steps are numbered globally)"""
    out, x, t = {0: x0}, x0, 0
    for T in LAW_T[1:]:
        x = mc.run_dense(A, x, 0, LAW_SEED, t, T - t, mutant)
        out[T], t = x, T
    return out


# -------------------------------------------------------------------------------------------------------------- 1. Philox
def test_philox_known_answers():
    f = lambda w: " ".join("%08x" % int(v) for v in w)
    assert f(mc.philox4x32_10([0, 0, 0, 0], [0, 0])) == "6627e8d5 e169c58d bc57ac4c 9b00dbd8"
    assert f(mc.philox4x32_10([0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2)) == "408f276d 41c83b0e a20bc7c6 6d5451fd"
    assert f(mc.philox4x32_10([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0])) == \
        "d16cfe09 94fdcceb 5001e420 24126ea1"


def test_dense_oracle_is_the_csr_oracle():
    rp, ci, A = _test_graph()
    for kk in (2, 3, 7):
        x0 = mc.chain_init(rp, ci, kk, 40, 5, 99)
        _, fin = mc.run_chain(rp, ci, x0, 5, 99, 17, 3, 4)
        assert np.array_equal(mc.run_dense(A, x0, 5, 99, 17, 12), fin)


# ------------------------------------------------------------------------------------------------ 3./4. the law, exactly (CPU)
def test_oracle_chain_has_the_exact_law(law):
    L, A, x0 = law
    assert L.irreducible()
    xs = _oracle_slices(A, x0)
    for T in LAW_T:
        assert L.pvalue(xs[T], T) > P_MIN, T


@pytest.mark.parametrize("mutant", ["no_last_site", "union", "rank_off"])
def test_law_test_rejects_mutants(law, mutant):
    L, A, x0 = law
    xs = _oracle_slices(A, x0, mutant)
    assert min(L.pvalue(xs[T], T) for T in LAW_T[1:]) < P_MIN


# --------------------------------------------------------------------------------------- 5. invariants and the reference walk
def _step_changes(traj):
    """traj (steps x chains x kk) -> number of positions each consecutive pair of states differs in"""
    return (traj[1:] != traj[:-1]).sum(-1)


def test_reference_trajectory_invariants(golden_dir):
    g = np.load(golden_dir + "/network_recons.npz")
    e = g["graph_edges"]
    rp, ci, _ = _csr(int(g["n_nodes"]), e.tolist())
    embs = g["embs"]
    assert mc.is_homomorphism(rp, ci, embs).all()
    ch = _step_changes(embs[:, None, :])[:, 0]
    assert ch.max() <= 1 and int((ch == 0).sum()) == 132 and int((ch == 1).sum()) == 167


def test_oracle_trajectory_invariants():
    rp, ci, _ = _test_graph()
    x0 = mc.chain_init(rp, ci, 6, 8, 0, 3)
    out, _ = mc.run_chain(rp, ci, x0, 0, 3, 0, 60)
    assert mc.is_homomorphism(rp, ci, out).all()
    assert _step_changes(np.concatenate([x0[None], out])).max() <= 1


# ---------------------------------------------------------------------------------------------------------- 6. errors (CPU)
def test_directed_and_non_symmetric_graphs_are_refused():
    import networkx as nx
    from onmf_ontf_ndl_b200.patches import MotifChains
    with pytest.raises(ValueError):
        MotifChains(nx.DiGraph([(0, 1), (1, 2)]), 3, 4, 0)
    with pytest.raises(ValueError):
        MotifChains(sp.csr_matrix(np.array([[0, 1], [0, 0]])), 2, 4, 0)
    with pytest.raises(ValueError):
        MotifChains((np.array([0, 1, 1]), np.array([1], dtype=np.int32)), 2, 4, 0)


# ================================================================================================================== GPU
def _dev(*arrs):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrs]


@gpu
@pytest.mark.parametrize("kk", [2, 3, 21, 32])
def test_kernels_equal_the_oracle(kk):
    import torch
    from onmf_ontf_ndl_b200 import _lib
    rp, ci, _ = _test_graph()
    drp, dci = _dev(rp, ci)
    for seed, chain0, step0 in ((0, 0, 0), (0xDEADBEEF12345678, 77, 2 ** 32 - 5), (5, 3, 1000)):
        n_chains, n_samples, sps = 37, 9, 4
        ref0 = mc.chain_init(rp, ci, kk, n_chains, chain0, seed)
        st = torch.empty(n_chains, kk, dtype=torch.int32, device="cuda")
        _lib.motif_chain_init(drp, dci, st, chain0, seed)
        assert np.array_equal(st.cpu().numpy(), ref0), (kk, seed)
        out = torch.full((n_samples, n_chains, kk), -7, dtype=torch.int32, device="cuda")
        _lib.motif_chain(drp, dci, st, chain0, seed, step0, sps, out)
        ref_out, ref_fin = mc.run_chain(rp, ci, ref0, chain0, seed, step0, n_samples, sps)
        assert np.array_equal(out.cpu().numpy(), ref_out), (kk, seed)
        assert np.array_equal(st.cpu().numpy(), ref_fin), (kk, seed)


@gpu
def test_trajectory_does_not_depend_on_launch_or_split():
    import torch
    from onmf_ontf_ndl_b200 import _lib
    from onmf_ontf_ndl_b200.patches import MotifChains
    rp, ci, _ = _test_graph()
    drp, dci = _dev(rp, ci)
    kk, seed = 21, 42
    big = torch.empty(4096, kk, dtype=torch.int32, device="cuda")
    _lib.motif_chain_init(drp, dci, big, 0, seed)
    out_big = torch.empty(30, 4096, kk, dtype=torch.int32, device="cuda")
    _lib.motif_chain(drp, dci, big, 0, seed, 0, 1, out_big)
    for c in (0, 1, 31, 32, 1000, 4095 - 6):
        small = torch.empty(7, kk, dtype=torch.int32, device="cuda")
        _lib.motif_chain_init(drp, dci, small, c, seed)
        out_small = torch.empty(30, 7, kk, dtype=torch.int32, device="cuda")
        _lib.motif_chain(drp, dci, small, c, seed, 0, 1, out_small)
        assert torch.equal(out_small, out_big[:, c:c + 7]), c
        assert torch.equal(small, big[c:c + 7]), c
    # two calls = one longer call; steps_per_sample = 3 = every third row of steps_per_sample = 1
    a = MotifChains((rp, ci), kk, 64, seed)
    b = MotifChains((rp, ci), kk, 64, seed)
    s1 = torch.cat([a.sample(50), a.sample(50)])
    s2 = b.sample(100)
    assert torch.equal(s1, s2) and torch.equal(a.state, b.state) and a.step == b.step == 100
    c3 = MotifChains((rp, ci), kk, 64, seed)
    one = MotifChains((rp, ci), kk, 64, seed).sample(60).view(60, 64, kk)
    assert torch.equal(c3.sample(20, steps_per_sample=3).view(20, 64, kk), one[2::3])


@gpu
def test_device_law_and_invariants(law):
    import torch
    from onmf_ontf_ndl_b200.patches import MotifChains
    L, A, x0 = law
    rp, ci, _ = _law_graph()
    for T in LAW_T:
        ch = MotifChains((rp, ci), LAW_KK, LAW_N, LAW_SEED)
        if T == 0:
            x = ch.state.cpu().numpy()
            assert np.array_equal(x, x0)
        else:
            x = ch.sample(1, steps_per_sample=T).cpu().numpy()
        assert L.pvalue(x, T) > P_MIN, T
    # invariants on the test graph: every state a homomorphism, consecutive states differ in at most one position
    rp, ci, _ = _test_graph()
    ch = MotifChains((rp, ci), 21, 256, 9)
    x0 = ch.state.cpu().numpy()
    traj = ch.sample(40).view(40, 256, 21).cpu().numpy()
    assert mc.is_homomorphism(rp, ci, traj).all()
    assert _step_changes(np.concatenate([x0[None], traj])).max() <= 1


@gpu
def test_errors_touch_nothing():
    import networkx as nx
    import torch
    from onmf_ontf_ndl_b200 import _lib
    from onmf_ontf_ndl_b200.patches import MotifChains
    rp, ci, _ = _test_graph()
    drp, dci = _dev(rp, ci)
    # an initial state that is not a homomorphism (129 is isolated), and node positions outside the graph
    for bad in ([[2, 3, 129]], [[2, 3, 130]], [[-1, 2, 3]]):
        st = torch.tensor(bad, dtype=torch.int32, device="cuda")
        out = torch.full((4, 1, 3), -7, dtype=torch.int32, device="cuda")
        with pytest.raises(_lib.OnmfKernelError):
            _lib.motif_chain(drp, dci, st, 0, 1, 0, 1, out)
        assert (out == -7).all() and st.tolist() == bad
    G = nx.path_graph(5)
    with pytest.raises(_lib.OnmfKernelError):
        MotifChains(G, 3, 2, 0, state=[[0, 1, 2], [0, 2, 1]]).sample(1)
    with pytest.raises(ValueError):
        MotifChains(G, 3, 1, 0, state=[[0, 1, 99]])
    with pytest.raises(_lib.OnmfKernelError):
        MotifChains(G, 33, 4, 0)
    with pytest.raises(_lib.OnmfKernelError):
        MotifChains(nx.empty_graph(4), 3, 4, 0)
    with pytest.raises(ValueError):
        MotifChains(nx.DiGraph([(0, 1), (1, 0)]), 2, 4, 0)
    # the chains still run after the refusals
    ch = MotifChains(G, 3, 8, 0)
    assert mc.is_homomorphism(*_csr(5, list(G.edges()))[:2], ch.sample(5).cpu().numpy()).all()


@gpu
def test_labels_and_patches():
    import networkx as nx
    import torch
    from onmf_ontf_ndl_b200 import patches
    G = nx.relabel_nodes(nx.petersen_graph(), {i: "v%d" % i for i in range(10)})
    ch = patches.MotifChains(G, 5, 16, 1, state=[["v0", "v1", "v2", "v3", "v4"]] * 16)
    twin = patches.MotifChains(G, 5, 16, 1, state=[["v0", "v1", "v2", "v3", "v4"]] * 16)
    X = ch.patches(3, precision="fp64")
    emb = twin.sample(3)
    lab = twin.labels(emb)
    assert lab.shape == (48, 5) and all(G.has_edge(a, b) for row in lab for a, b in zip(row[:-1], row[1:]))
    ref = patches.motif_patches(patches.graph_to_csr(G), emb.cpu().numpy(), precision="fp64", device=True)
    assert X.dtype == torch.float64 and torch.equal(X, ref)


# ------------------------------------------------------------------------------------------------------------ 7. consumers
@gpu
def test_reconstruct_network_from_device_positions():
    import networkx as nx
    from onmf_ontf_ndl_b200 import reconstruct_network
    from onmf_ontf_ndl_b200.patches import MotifChains
    rng = np.random.default_rng(4)
    # one trajectory-like run (20 chains x 30 steps) and one of 256 independent first states that outgrows the pair table
    for n_nodes, m_edges, kk, n_chains, n_samples in ((60, 200, 6, 20, 30), (20000, 200000, 21, 256, 1)):
        G = nx.gnm_random_graph(n_nodes, m_edges, seed=2)
        G.add_edges_from((i, i + 1) for i in range(n_nodes - 1))
        W = rng.random((kk * kk, 7))
        W /= np.linalg.norm(W, axis=0)
        ch = MotifChains(G, kk, n_chains, 5)
        emb = ch.sample(n_samples)
        for prec in ("fp64", "fp32"):
            p_dev, w_dev, c_dev = reconstruct_network(G, W, emb, alpha=0, precision=prec)
            p_lab, w_lab, c_lab = reconstruct_network(G, W, ch.labels(emb), alpha=0, precision=prec)
            # same pairs and counts; the per-pair sums are accumulated by onmf_edge_scatter_add with FP64 atomics, whose order
            # (and so the last bits of a sum) differs between any two calls, label form included
            assert np.array_equal(p_dev.astype(np.int64), p_lab.astype(np.int64)) and np.array_equal(c_dev, c_lab)
            assert np.allclose(w_dev, w_lab, rtol=1e-12, atol=1e-14)
        if n_samples == 1:
            start = 1024
            while start < 2 * len(emb) * 4 * kk + 2:
                start *= 2
            assert len(p_dev) > start                       # the table grew


@gpu
@pytest.mark.parametrize("precision", ["fp32", "fp64"])
@pytest.mark.parametrize("subsample", [False, True])
def test_ndl_train_dict_equals_epochwise_online_nmf(precision, subsample):
    import networkx as nx
    from onmf_ontf_ndl_b200 import Online_NMF, _host, ndl
    from onmf_ontf_ndl_b200.patches import MotifChains
    G = nx.gnm_random_graph(80, 300, seed=7)
    G.add_edges_from((i, i + 1) for i in range(79))
    kk, r, sample_size, n_chains, seed = 6, 9, 200, 20, 13
    kw = dict(iterations=5, batch_size=50, alpha=None, subsample=subsample, precision=precision)
    for epochs in (1, 2):
        np.random.seed(31)
        got = ndl.train_dict(G, kk, r, epochs, kw["iterations"], sample_size, kw["batch_size"], n_chains=n_chains, seed=seed,
                             subsample=subsample, precision=precision)
        np.random.seed(31)
        ch = MotifChains(G, kk, n_chains, seed)
        res, nmf = None, None
        for _ in range(epochs):
            X = _host.from_sample_major(ch.patches(sample_size // n_chains, precision=precision))
            extra = {}
            if res is not None:
                extra = dict(ini_dict=res[0], ini_A=res[1], ini_B=res[2], ini_C=res[3], history=nmf.history)
            nmf = Online_NMF(X, r, **kw, **extra)
            res = nmf.train_dict()
        for a, b in zip(got, res):
            assert np.array_equal(np.asarray(a), np.asarray(b)), (precision, subsample, epochs)
