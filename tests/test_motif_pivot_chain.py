"""The NDL pivot chain on the device (csrc/motif_chain.cu onmf_motif_pivot_chain, patches.MotifChains(mcmc="pivot"),
ndl.train_dict(mcmc="pivot")).

The kernel is held to oracle/motif_pivot_chain.py bit for bit; the oracle's rule is held to the uniform law on Hom(P_kk, G)
exactly (the transition matrix of the rule on a small graph is built from every homomorphism: it is doubly stochastic,
reversible and irreducible); and oracle and device are held to that law by a chi-square test that three mutants of the
acceptance rule fail."""
import itertools

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.stats as ss

from oracle import motif_chain as mc
from oracle import motif_pivot_chain as mp

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
    """130 nodes: two hubs (0, 1) sharing 80 neighbours, a sparse random remainder, a self-loop at node 5 and an isolated
    node 129"""
    rng = np.random.default_rng(11)
    edges = [(0, v) for v in range(2, 82)] + [(1, v) for v in range(2, 82)] + [(5, 5)]
    edges += [(int(a), int(b)) for a, b in rng.integers(2, 129, size=(260, 2)) if a != b]
    edges += [(v, v + 1) for v in range(2, 128)]
    return _csr(130, edges)


def _law_graph():
    """8 nodes, connected, with triangles (not bipartite)"""
    return _csr(8, [(i, (i + 1) % 8) for i in range(8)] + [(0, 2), (3, 6), (1, 5)])


def _chord_cycle():
    """a 14-node cycle with 4 chords: sparse, so interior Glauber sites rarely move"""
    return _csr(14, [(i, (i + 1) % 14) for i in range(14)] + [(0, 7), (3, 10), (5, 12), (2, 4)])


LAW_KK, LAW_N, LAW_SEED, LAW_T = 4, 1 << 17, 2024, (0, 1, 2, 5, 50)
P_MIN = 1e-3


class _ExactPivotLaw:
    """Hom(P_kk, G) enumerated, the exact initial law p0 of chain_init (root uniform over the nodes with a neighbour, then
    uniform neighbours), the exact pivot matrix (proposal times min(1, num / den)) and, for comparison, the Glauber matrix"""

    def __init__(self, A, kk):
        n = A.shape[0]
        self.n, self.kk = n, kk
        self.homs = [h for h in itertools.product(range(n), repeat=kk) if all(A[h[q], h[q + 1]] for q in range(kk - 1))]
        ix = {h: i for i, h in enumerate(self.homs)}
        H = len(self.homs)
        deg = A.sum(1).astype(np.float64)
        nz = int((deg > 0).sum())
        self.p0 = np.array([np.prod([1.0 / deg[h[q]] for q in range(kk - 1)]) / nz for h in self.homs])
        P = np.zeros((H, H))
        for h in self.homs:
            for y in self.homs:
                if A[h[0], y[0]]:
                    prop = 1.0 / deg[h[0]] * np.prod([1.0 / deg[y[q]] for q in range(kk - 1)])
                    ratio = np.prod([deg[y[q]] / deg[h[q]] for q in range(1, kk - 1)])
                    P[ix[h], ix[y]] += prop * min(1.0, ratio)
            P[ix[h], ix[h]] += 1.0 - P[ix[h]].sum()
        self.P = P
        G = np.zeros((H, H))
        for h in self.homs:
            for i in range(kk):
                a = h[1] if i == 0 else h[i - 1]
                b = h[kk - 2] if i == kk - 1 else h[i + 1]
                S = np.nonzero(A[a] & A[b])[0]
                for v in S:
                    y = list(h)
                    y[i] = int(v)
                    G[ix[h], ix[tuple(y)]] += 1.0 / (kk * len(S))
        self.G = G
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


def _gap(P):
    ev = np.sort(np.abs(np.linalg.eigvals(P)))[::-1]
    return 1.0 - ev[1]


@pytest.fixture(scope="module")
def law():
    rp, ci, A = _law_graph()
    L = _ExactPivotLaw(A, LAW_KK)
    x0 = mc.chain_init(rp, ci, LAW_KK, LAW_N, 0, LAW_SEED)
    return L, A, x0


def _oracle_slices(A, x0, mutant=None):
    """{T: states after T pivot steps} for T in LAW_T, continuing one run (the steps are numbered globally)"""
    out, x, t = {0: x0}, x0, 0
    for T in LAW_T[1:]:
        x = mp.run_pivot_dense(A, x, 0, LAW_SEED, t, T - t, mutant)
        out[T], t = x, T
    return out


# ---------------------------------------------------------------------------------------------------------- the rule (CPU)
def test_pivot_matrix_is_exact_for_the_uniform_law(law):
    L = law[0]
    H = len(L.homs)
    assert H == 174
    assert (L.P >= 0).all() and np.allclose(L.P.sum(1), 1.0, rtol=0, atol=1e-15)
    pi = np.full(H, 1.0 / H)
    assert np.abs(pi @ L.P - pi).max() < 1e-15                  # stationary
    assert np.abs(L.P - L.P.T).max() < 1e-15                    # detailed balance for a uniform law
    assert L.irreducible()


def test_pivot_mixes_faster_than_glauber():
    """the spectral gaps quoted in DESIGN §7: exact matrices, kk = 4"""
    L = _ExactPivotLaw(_law_graph()[2], 4)
    assert round(_gap(L.G), 4) == 0.0097 and round(_gap(L.P), 2) == 0.31
    L = _ExactPivotLaw(_chord_cycle()[2], 4)
    assert len(L.homs) == 254
    assert round(_gap(L.G), 4) == 0.0031 and round(_gap(L.P), 2) == 0.20


def test_dense_oracle_is_the_csr_oracle():
    rp, ci, A = _test_graph()
    for kk in (2, 3, 7):
        x0 = mc.chain_init(rp, ci, kk, 40, 5, 99)
        _, fin = mp.run_pivot_chain(rp, ci, x0, 5, 99, 17, 3, 4)
        assert np.array_equal(mp.run_pivot_dense(A, x0, 5, 99, 17, 12), fin), kk


def test_oracle_chain_has_the_exact_law(law):
    L, A, x0 = law
    xs = _oracle_slices(A, x0)
    for T in LAW_T:
        assert L.pvalue(xs[T], T) > P_MIN, T


@pytest.mark.parametrize("mutant", ["no_mh", "pivot_degree", "inverted"])
def test_law_test_rejects_mutants(law, mutant):
    L, A, x0 = law
    xs = _oracle_slices(A, x0, mutant)
    assert min(L.pvalue(xs[T], T) for T in LAW_T[1:]) < P_MIN


def test_oracle_trajectory_invariants():
    rp, ci, _ = _test_graph()
    x0 = mc.chain_init(rp, ci, 6, 8, 0, 3)
    out, _ = mp.run_pivot_chain(rp, ci, x0, 0, 3, 0, 60)
    _assert_pivot_trajectory(rp, ci, np.concatenate([x0[None], out]))


def _assert_pivot_trajectory(rp, ci, traj):
    """every state a homomorphism; a step leaves the state unchanged or moves x[0] to a neighbour; and the chain moves"""
    assert mc.is_homomorphism(rp, ci, traj).all()
    moved = (traj[1:] != traj[:-1]).any(-1)
    a, b = traj[:-1, :, 0][moved], traj[1:, :, 0][moved]
    assert all(b_ in ci[rp[a_]:rp[a_ + 1]] for a_, b_ in zip(a.tolist(), b.tolist()))
    assert moved.mean() > 0.1


def test_unknown_mcmc_is_refused_before_the_device():
    from onmf_ontf_ndl_b200 import ndl
    from onmf_ontf_ndl_b200.patches import MotifChains
    rp, ci, _ = _law_graph()
    with pytest.raises(ValueError, match="mcmc"):
        MotifChains((rp, ci), 3, 4, 0, mcmc="metropolis")
    with pytest.raises(ValueError, match="mcmc"):
        ndl.train_dict((rp, ci), 3, 2, 1, 1, 4, 4, n_chains=4, mcmc="random_walk")


# ================================================================================================================== GPU
def _dev(*arrs):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrs]


@gpu
@pytest.mark.parametrize("kk", [2, 3, 21, 32])
def test_kernel_equals_the_oracle(kk):
    import torch
    from onmf_ontf_ndl_b200 import _lib
    rp, ci, _ = _test_graph()
    drp, dci = _dev(rp, ci)
    # 300 chains: two full blocks of 128 and a partial one
    for seed, chain0, step0, n_chains, n_samples, sps in ((0, 0, 0, 37, 9, 1), (0xDEADBEEF12345678, 77, 2 ** 32 - 5, 300, 4, 3),
                                                          (5, 3, 1000, 130, 6, 4)):
        st = torch.empty(n_chains, kk, dtype=torch.int32, device="cuda")
        _lib.motif_chain_init(drp, dci, st, chain0, seed)
        ref0 = st.cpu().numpy()
        out = torch.full((n_samples, n_chains, kk), -7, dtype=torch.int32, device="cuda")
        _lib.motif_pivot_chain(drp, dci, st, chain0, seed, step0, sps, out)
        ref_out, ref_fin = mp.run_pivot_chain(rp, ci, ref0, chain0, seed, step0, n_samples, sps)
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
    _lib.motif_pivot_chain(drp, dci, big, 0, seed, 0, 1, out_big)
    for c in (0, 1, 127, 128, 1000, 4095 - 6):
        small = torch.empty(7, kk, dtype=torch.int32, device="cuda")
        _lib.motif_chain_init(drp, dci, small, c, seed)
        out_small = torch.empty(30, 7, kk, dtype=torch.int32, device="cuda")
        _lib.motif_pivot_chain(drp, dci, small, c, seed, 0, 1, out_small)
        assert torch.equal(out_small, out_big[:, c:c + 7]), c
        assert torch.equal(small, big[c:c + 7]), c
    # two calls = one longer call; steps_per_sample = 3 = every third row of steps_per_sample = 1
    a = MotifChains((rp, ci), kk, 200, seed, mcmc="pivot")
    b = MotifChains((rp, ci), kk, 200, seed, mcmc="pivot")
    s1 = torch.cat([a.sample(50), a.sample(50)])
    s2 = b.sample(100)
    assert torch.equal(s1, s2) and torch.equal(a.state, b.state) and a.step == b.step == 100
    c3 = MotifChains((rp, ci), kk, 200, seed, mcmc="pivot")
    one = MotifChains((rp, ci), kk, 200, seed, mcmc="pivot").sample(60).view(60, 200, kk)
    assert torch.equal(c3.sample(20, steps_per_sample=3).view(20, 200, kk), one[2::3])
    # the Glauber chain of the same seed is another trajectory
    g = MotifChains((rp, ci), kk, 200, seed)
    assert not torch.equal(g.sample(100), s2)


@gpu
def test_device_law_and_invariants(law):
    from onmf_ontf_ndl_b200.patches import MotifChains
    L, A, x0 = law
    rp, ci, _ = _law_graph()
    for T in LAW_T:
        ch = MotifChains((rp, ci), LAW_KK, LAW_N, LAW_SEED, mcmc="pivot")
        if T == 0:
            x = ch.state.cpu().numpy()
            assert np.array_equal(x, x0)
        else:
            x = ch.sample(1, steps_per_sample=T).cpu().numpy()
        assert L.pvalue(x, T) > P_MIN, T
    rp, ci, _ = _test_graph()
    ch = MotifChains((rp, ci), 21, 256, 9, mcmc="pivot")
    x0 = ch.state.cpu().numpy()
    traj = ch.sample(40).view(40, 256, 21).cpu().numpy()
    _assert_pivot_trajectory(rp, ci, np.concatenate([x0[None], traj]))


@gpu
def test_errors_touch_nothing():
    import networkx as nx
    import torch
    from onmf_ontf_ndl_b200 import _lib
    from onmf_ontf_ndl_b200.patches import MotifChains
    rp, ci, _ = _test_graph()
    drp, dci = _dev(rp, ci)
    # states that are not homomorphisms (129 is isolated; 130 and -1 are outside the graph), kk = 1 and kk = 33
    good = mc.chain_init(rp, ci, 33, 2, 0, 1)
    for bad in ([[2, 3, 129]], [[2, 3, 130]], [[-1, 2, 3]], [[2], [3]], good.tolist()):
        st = torch.tensor(bad, dtype=torch.int32, device="cuda")
        out = torch.full((4,) + tuple(st.shape), -7, dtype=torch.int32, device="cuda")
        with pytest.raises(_lib.OnmfKernelError):
            _lib.motif_pivot_chain(drp, dci, st, 0, 1, 0, 1, out)
        assert (out == -7).all() and st.tolist() == bad
    G = nx.path_graph(5)
    with pytest.raises(_lib.OnmfKernelError):
        MotifChains(G, 3, 2, 0, state=[[0, 1, 2], [0, 2, 1]], mcmc="pivot").sample(1)
    ch = MotifChains(G, 3, 8, 0, mcmc="pivot")
    assert mc.is_homomorphism(*_csr(5, list(G.edges()))[:2], ch.sample(5).cpu().numpy()).all()


# ------------------------------------------------------------------------------------------------------------ consumers
@gpu
def test_reconstruct_network_from_device_pivot_positions():
    import networkx as nx
    from onmf_ontf_ndl_b200 import reconstruct_network
    from onmf_ontf_ndl_b200.patches import MotifChains
    rng = np.random.default_rng(4)
    G = nx.gnm_random_graph(60, 200, seed=2)
    G.add_edges_from((i, i + 1) for i in range(59))
    kk = 6
    W = rng.random((kk * kk, 7))
    W /= np.linalg.norm(W, axis=0)
    ch = MotifChains(G, kk, 20, 5, mcmc="pivot")
    emb = ch.sample(30)
    for prec in ("fp64", "fp32"):
        p_dev, w_dev, c_dev = reconstruct_network(G, W, emb, alpha=0, precision=prec)
        p_lab, w_lab, c_lab = reconstruct_network(G, W, ch.labels(emb), alpha=0, precision=prec)
        # the per-pair sums are FP64 atomics, whose order (and so the last bits) differs between any two calls
        assert np.array_equal(p_dev.astype(np.int64), p_lab.astype(np.int64)) and np.array_equal(c_dev, c_lab)
        assert np.allclose(w_dev, w_lab, rtol=1e-12, atol=1e-14)


@gpu
@pytest.mark.parametrize("precision", ["fp32", "fp64"])
@pytest.mark.parametrize("subsample", [False, True])
def test_ndl_train_dict_pivot_equals_epochwise_online_nmf(precision, subsample):
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
                             subsample=subsample, precision=precision, mcmc="pivot")
        np.random.seed(31)
        ch = MotifChains(G, kk, n_chains, seed, mcmc="pivot")
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
