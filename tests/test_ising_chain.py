"""Ising lattices on the device (csrc/ising_chain.cu, patches.IsingChains, ising.train_dict).

The kernels are held to oracle/ising_chain.py bit for bit (Philox4x32-10 words and the checkerboard heat-bath sweep restated
in numpy); the oracle and the device are held to the exact Gibbs law of a 4 x 4 torus (all 2^16 states enumerated) by
chi-square tests that four mutants with one plausible bug each fail, checkerboard Metropolis among them."""
import ctypes
import math

import numpy as np
import pytest
import scipy.stats as ss

from oracle import ising_chain as ic
from oracle import onmf_oracle as O

gpu = pytest.mark.gpu

LAW_BETAS = (0.05, 0.2, 0.44, 0.8)
LAW_SWEEPS, LAW_SEED = 60, 2024
LAW_N_CPU = 1 << 16            # chains of the oracle's (E, M) test
LAW_N_GPU = 1 << 20            # chains of the device's full-state test
P_MIN = 1e-3                   # the rule passes every case above this
P_MUTANT = 1e-6                # a mutant fails some case below this


# ------------------------------------------------------------------------------------------------------------------ fixtures
class _ExactLaw:
    """P(sigma) ~ exp(beta sum_<ij> sigma_i sigma_j) on the 4 x 4 torus, every state enumerated"""

    def __init__(self, beta, H=4, W=4):
        n = H * W
        self.H, self.W, self.n = H, W, n
        codes = np.arange(1 << n, dtype=np.int64)
        x = (((codes[:, None] >> np.arange(n)) & 1) * 2 - 1).reshape(-1, H, W)
        E, M = ic.energy_magnetisation(x)
        w = np.exp(-beta * (E - E.min()))
        self.p_state = w / w.sum()
        self.em_keys, inv = np.unique(self._em_key(E, M), return_inverse=True)
        self.p_em = np.bincount(inv, weights=self.p_state)

    def _em_key(self, E, M):
        return (np.asarray(E) + 2 * self.n) * (2 * self.n + 1) + (np.asarray(M) + self.n)

    @staticmethod
    def _chi2(obs, p):
        """chi-square p-value of counts obs against probabilities p, bins expecting fewer than 5 pooled into one"""
        exp = p * obs.sum()
        small = exp < 5
        o, e = obs[~small], exp[~small]
        if small.any():
            o, e = np.append(o, obs[small].sum()), np.append(e, exp[small].sum())
        return float(ss.chi2.sf(((o - e) ** 2 / e).sum(), len(o) - 1))

    def pvalue_em(self, x):
        """the (energy, magnetisation) histogram of states x (N x H x W)"""
        E, M = ic.energy_magnetisation(x)
        idx = np.searchsorted(self.em_keys, self._em_key(E, M))
        return self._chi2(np.bincount(idx, minlength=len(self.em_keys)).astype(np.float64), self.p_em)

    def pvalue_state(self, x):
        """the full-state histogram (2^16 bins) of states x (N x H x W)"""
        bits = (np.asarray(x).reshape(len(x), -1) > 0).astype(np.int64)
        code = bits @ (1 << np.arange(self.n, dtype=np.int64))
        return self._chi2(np.bincount(code, minlength=1 << self.n).astype(np.float64), self.p_state)


@pytest.fixture(scope="module")
def laws():
    return {b: _ExactLaw(b) for b in LAW_BETAS}


def _oracle_law_states(betas, mutant=None):
    """final states (len(betas) x LAW_N_CPU x 4 x 4) of the oracle chains after LAW_SWEEPS sweeps, one ensemble per beta"""
    x0 = ic.chain_init(4, 4, LAW_N_CPU, 0, LAW_SEED)
    thr = np.stack([ic.thresholds(b) for b in betas])
    _, fin = ic.run_chain(np.broadcast_to(x0, (len(betas),) + x0.shape), thr, 0, LAW_SEED, 0, 1, LAW_SWEEPS, mutant=mutant)
    return fin


# ------------------------------------------------------------------------------------------------------- thresholds (CPU)
def test_thresholds_match_python_and_refuse_non_finite_beta():
    from onmf_ontf_ndl_b200 import _lib
    for beta in (0.0, 0.05, 0.2, 0.44, 0.8, 1.5, 4.0, 30.0, -0.3, -30.0, 1e-300):
        got = _lib.ising_thresholds(beta)
        ref = [min(math.floor(2.0 ** 32 / (1.0 + math.exp(-2.0 * beta * (2 * j - 4)))), 2 ** 32 - 1) for j in range(5)]
        assert all(abs(a - b) <= 1 for a, b in zip(got, ref)), (beta, got, ref)
        assert got[2] == 2 ** 31, beta
        assert got == sorted(got) if beta >= 0 else got == sorted(got, reverse=True)
    assert _lib.ising_thresholds(30.0)[4] == 2 ** 32 - 1 and _lib.ising_thresholds(30.0)[0] == 0
    lib = _lib.load()
    for bad in (math.nan, math.inf, -math.inf):
        with pytest.raises(_lib.OnmfKernelError):
            _lib.ising_thresholds(bad)
        # refused before any launch, so the (never dereferenced) buffers need no device
        fake = ctypes.c_void_p(256)
        assert lib.onmf_ising_chain(4, 4, 1, 0, 0, bad, 0, 1, 1, fake, fake, 0, None) == -1
        assert b"beta" in lib.onmf_last_error()


# --------------------------------------------------------------------------------------------------------- the plan (CPU)
PINNED = {(4, 4): "smem", (6, 10): "smem", (200, 200): "smem", (10, 64): "smem", (480, 484): "smem",
          (482, 484): "global", (512, 512): "global", (1024, 1024): "global"}


def test_plan_invariants_and_pinned_forms():
    from onmf_ontf_ndl_b200 import _lib
    sides = list(range(4, 80, 2)) + [200, 256, 474, 476, 480, 482, 484, 512, 1024, 4096]
    for H in sides:
        for W in sides:
            p = _lib.ising_chain_plan(H, W)
            if H * W <= 227 * 1024:
                assert p["form"] == "smem" and p["smem"] == H * W <= 227 * 1024, (H, W, p)
                assert 32 <= p["threads"] <= 1024 and p["threads"] % 32 == 0, (H, W, p)
            else:
                assert p["form"] == "global" and p["smem"] == 0 and p["threads"] > 0, (H, W, p)
    for shape, form in PINNED.items():
        assert _lib.ising_chain_plan(*shape)["form"] == form, shape
    for H, W in ((3, 4), (4, 3), (2, 4), (4, 2), (0, 4), (5, 6), (-4, 4), (65536, 32768)):
        with pytest.raises(_lib.OnmfKernelError):
            _lib.ising_chain_plan(H, W)


# ----------------------------------------------------------------------------------------------------- the law (CPU, oracle)
def test_oracle_samples_the_exact_law(laws):
    fin = _oracle_law_states(LAW_BETAS)
    for b, x in zip(LAW_BETAS, fin):
        assert laws[b].pvalue_em(x) > P_MIN, b


@pytest.mark.parametrize("mutant,betas", [("metropolis", (0.44, 0.8)), ("simultaneous", (0.44,)), ("sign", (0.44,)),
                                          ("index_off", (0.44,))])
def test_law_test_rejects_mutants(laws, mutant, betas):
    fin = _oracle_law_states(betas, mutant)
    assert min(laws[b].pvalue_em(x) for b, x in zip(betas, fin)) < P_MUTANT, mutant


def test_oracle_init_and_words():
    x = ic.chain_init(6, 10, 5, 3, 9)
    assert x.dtype == np.int8 and set(np.unique(x)) == {-1, 1}
    # a chain's words depend on its global index only
    assert np.array_equal(ic.words(6, 10, 5, 3, 9, 7, 1)[2:], ic.words(6, 10, 3, 5, 9, 7, 1))
    # thinning and splitting
    thr = ic.thresholds(0.3)
    out, fin = ic.run_chain(x, thr, 3, 9, 0, 6)
    out3, fin3 = ic.run_chain(x, thr, 3, 9, 0, 2, 3)
    a, fa = ic.run_chain(x, thr, 3, 9, 0, 4)
    b, fb = ic.run_chain(fa, thr, 3, 9, 4, 2)
    assert np.array_equal(out[2::3], out3) and np.array_equal(fin, fin3)
    assert np.array_equal(np.concatenate([a, b]), out) and np.array_equal(fb, fin)


# -------------------------------------------------------------------------------------------------- patches, refusals (CPU)
def test_frame_patch_coords():
    from onmf_ontf_ndl_b200.patches import frame_patch_coords, sample_patch_coords
    np.random.seed(3)
    one = frame_patch_coords(1, (20, 30), 6, 50)
    np.random.seed(3)
    assert np.array_equal(one, sample_patch_coords((20, 30), 6, 50))
    np.random.seed(3)
    three = frame_patch_coords(3, (20, 30), 6, 50)
    np.random.seed(3)
    ref = [sample_patch_coords((20, 30), 6, 50) for _ in range(3)]
    for f in range(3):
        assert np.array_equal(three[50 * f:50 * (f + 1)], ref[f] + [20 * f, 0])
    assert three[:, 0].max() < 3 * 20 - 6 + 1


def test_python_refusals():
    from onmf_ontf_ndl_b200.patches import IsingChains
    for shape in ((5, 4), (4, 5), (2, 4), (4, 2), (0, 0), (4,)):
        with pytest.raises(ValueError):
            IsingChains(shape, 0.4, 2, 0)
    for beta in (math.nan, math.inf, -math.inf):
        with pytest.raises(ValueError):
            IsingChains((4, 4), beta, 2, 0)
    for state in (np.zeros((2, 4, 4)), np.full((2, 4, 4), 2), np.ones((1, 4, 4)), np.ones((2, 4, 6)), np.ones((2, 16))):
        with pytest.raises(ValueError):
            IsingChains((4, 4), 0.4, 2, 0, state=state)
    with pytest.raises(ValueError):
        IsingChains((4, 4), 0.4, 0, 0)


# ================================================================================================================== GPU
def _oracle_run(x0, beta, chain0, seed, sweep0, n_samples, sps):
    out, fin = ic.run_chain(x0, np.array(_lib_thr(beta), dtype=np.uint64), chain0, seed, sweep0, n_samples, sps)
    return out, fin


def _lib_thr(beta):
    from onmf_ontf_ndl_b200 import _lib
    return _lib.ising_thresholds(beta)


@gpu
@pytest.mark.parametrize("shape,n_chains,n_samples,sps", [((4, 4), 37, 5, 3), ((6, 10), 37, 5, 3), ((10, 64), 9, 4, 2),
                                                          ((200, 200), 3, 3, 2), ((512, 512), 2, 2, 2)])
def test_kernels_equal_the_oracle(shape, n_chains, n_samples, sps):
    import torch
    from onmf_ontf_ndl_b200 import _lib
    H, W = shape
    assert _lib.ising_chain_plan(H, W)["form"] == PINNED[shape]
    for seed, chain0, sweep0, beta in ((0, 0, 0, 0.44), (0xDEADBEEF12345678, 77, 2 ** 32 - 2, 0.8), (5, 3, 1000, -0.3)):
        ref0 = ic.chain_init(H, W, n_chains, chain0, seed)
        st = torch.empty(n_chains, H, W, dtype=torch.int8, device="cuda")
        _lib.ising_chain_init(st, chain0, seed)
        assert np.array_equal(st.cpu().numpy(), ref0), (shape, seed)
        ref_out, ref_fin = _oracle_run(ref0, beta, chain0, seed, sweep0, n_samples, sps)
        for dtype in (torch.float32, torch.float64):
            s2 = st.clone()
            out = torch.full((n_samples, n_chains, H, W), 7, dtype=dtype, device="cuda")
            _lib.ising_chain(s2, chain0, seed, beta, sweep0, sps, out)
            assert np.array_equal(out.cpu().numpy(), ref_out.astype(np.float64)), (shape, seed, dtype)
            assert np.array_equal(s2.cpu().numpy(), ref_fin), (shape, seed, dtype)


@gpu
@pytest.mark.parametrize("shape", [(6, 10), (512, 512)])
def test_trajectory_does_not_depend_on_launch_or_split(shape):
    import torch
    from onmf_ontf_ndl_b200 import _lib
    from onmf_ontf_ndl_b200.patches import IsingChains
    H, W = shape
    seed, beta = 42, 0.44
    n_big = 300 if shape == (6, 10) else 8
    big = torch.empty(n_big, H, W, dtype=torch.int8, device="cuda")
    _lib.ising_chain_init(big, 0, seed)
    out_big = torch.empty(6, n_big, H, W, device="cuda")
    _lib.ising_chain(big, 0, seed, beta, 0, 1, out_big)
    for c in ((0, 1, 31, 200, n_big - 3) if shape == (6, 10) else (0, 1, 5)):
        small = torch.empty(3, H, W, dtype=torch.int8, device="cuda")
        _lib.ising_chain_init(small, c, seed)
        out_small = torch.empty(6, 3, H, W, device="cuda")
        _lib.ising_chain(small, c, seed, beta, 0, 1, out_small)
        assert torch.equal(out_small, out_big[:, c:c + 3]), c
        assert torch.equal(small, big[c:c + 3]), c
    # two calls = one longer call; sweeps_per_sample = 3 = every third frame of sweeps_per_sample = 1
    n = 16 if shape == (6, 10) else 2
    a, b = IsingChains(shape, beta, n, seed), IsingChains(shape, beta, n, seed)
    s1 = torch.cat([a.sample(4), a.sample(5)])
    s2 = b.sample(9)
    assert torch.equal(s1, s2) and torch.equal(a.state, b.state) and a.sweep == b.sweep == 9
    c3 = IsingChains(shape, beta, n, seed)
    one = IsingChains(shape, beta, n, seed).sample(9, precision="fp64").view(9, n, H, W)
    assert torch.equal(c3.sample(3, sweeps_per_sample=3, precision="fp64").view(3, n, H, W), one[2::3])
    # a given initial state
    st = np.where(np.random.default_rng(1).random((n, H, W)) < 0.5, 1, -1)
    d = IsingChains(shape, beta, n, seed, state=st)
    ref_out, ref_fin = _oracle_run(st, beta, 0, seed, 0, 2, 1)
    assert np.array_equal(d.sample(2).cpu().numpy(), ref_out.reshape(2 * n, H, W).astype(np.float32))
    assert np.array_equal(d.state.cpu().numpy(), ref_fin)


@gpu
def test_device_samples_the_exact_law(laws):
    from onmf_ontf_ndl_b200.patches import IsingChains
    for b in LAW_BETAS:
        ch = IsingChains((4, 4), b, LAW_N_GPU, LAW_SEED + 1)
        x = ch.sample(1, sweeps_per_sample=LAW_SWEEPS).cpu().numpy()
        assert set(np.unique(x)) == {-1.0, 1.0}
        assert laws[b].pvalue_state(x) > P_MIN, b
        assert laws[b].pvalue_em(x) > P_MIN, b


@gpu
def test_errors_touch_nothing():
    import torch
    from onmf_ontf_ndl_b200 import _lib
    lib = _lib.load()
    st = torch.ones(3, 6, 10, dtype=torch.int8, device="cuda")
    before = st.clone()
    out = torch.full((2, 3, 6, 10), 7.0, device="cuda")
    p_st, p_out = _lib._ptr(st), _lib._ptr(out)
    cases = [dict(H=5), dict(W=2), dict(n_chains=0), dict(chain0=-1), dict(chain0=2 ** 32 - 2), dict(beta=math.nan),
             dict(n_samples=0), dict(sps=0), dict(out_dtype=7), dict(sweep0=2 ** 64 - 2), dict(state=None), dict(out=None)]
    for bad in cases:
        a = dict(H=6, W=10, n_chains=3, chain0=0, beta=0.4, sweep0=0, n_samples=2, sps=1, out_dtype=0, state=p_st, out=p_out)
        a.update(bad)
        rc = lib.onmf_ising_chain(a["H"], a["W"], a["n_chains"], a["chain0"], 1, a["beta"], a["sweep0"], a["n_samples"],
                                  a["sps"], a["state"], a["out"], a["out_dtype"], _lib._stream())
        assert rc == -1, bad
        torch.cuda.synchronize()
        assert torch.equal(st, before) and (out == 7.0).all(), bad
    for bad in (dict(H=5), dict(n_chains=0), dict(chain0=2 ** 32)):
        a = dict(H=6, W=10, n_chains=3, chain0=0)
        a.update(bad)
        assert lib.onmf_ising_chain_init(a["H"], a["W"], a["n_chains"], a["chain0"], 1, p_st, _lib._stream()) == -1, bad
        torch.cuda.synchronize()
        assert torch.equal(st, before), bad
    # the chains still run after the refusals
    _lib.ising_chain(st, 0, 1, 0.4, 0, 1, out)
    assert set(torch.unique(out).tolist()) <= {-1.0, 1.0}


@gpu
@pytest.mark.parametrize("precision", ["fp32", "fp64"])
@pytest.mark.parametrize("subsample", [False, True])
def test_ising_train_dict_equals_epochwise_online_nmf(precision, subsample):
    from onmf_ontf_ndl_b200 import Online_NMF, ising
    from onmf_ontf_ndl_b200.patches import ImagePatches, IsingChains, frame_patch_coords
    shape, beta, p, r, n_chains, sweeps, num_patches, seed = (20, 24), 0.44, 6, 12, 3, 4, 40, 13
    kw = dict(iterations=5, batch_size=30, alpha=None, subsample=subsample, precision=precision)
    for epochs in (1, 2):
        np.random.seed(31)
        got = ising.train_dict(shape, beta, p, r, epochs, kw["iterations"], num_patches, kw["batch_size"], n_chains=n_chains,
                               sweeps_per_epoch=sweeps, seed=seed, subsample=subsample, precision=precision)
        np.random.seed(31)
        ch = IsingChains(shape, beta, n_chains, seed)
        res, nmf = None, None
        for _ in range(epochs):
            frames = ch.sample(1, sweeps, precision=precision)
            co = frame_patch_coords(n_chains, shape, p, num_patches)
            X = ImagePatches(frames.reshape(n_chains * shape[0], shape[1]), p, co, precision=precision).to_matrix()
            extra = {}
            if res is not None:
                extra = dict(ini_dict=res[0], ini_A=res[1], ini_B=res[2], ini_C=res[3], history=nmf.history)
            nmf = Online_NMF(X, r, **kw, **extra)
            res = nmf.train_dict()
        for a, b in zip(got, res):
            assert np.array_equal(np.asarray(a), np.asarray(b)), (precision, subsample, epochs)


@gpu
def test_surrogate_error_of_the_trained_state():
    from onmf_ontf_ndl_b200 import ising
    np.random.seed(8)
    errors = []
    W, A, B, C, _ = ising.train_dict((24, 24), 0.44, 6, 12, 3, 6, 50, 40, n_chains=2, sweeps_per_epoch=5, seed=3,
                                     subsample=True, precision="fp64", errors=errors)
    assert len(errors) == 3 and C is not None
    ref = O.surrogate_error(W, A, B, C)
    assert abs(errors[-1] - ref) <= 1e-12 * (abs(np.trace(C)) + abs(ref)), (errors[-1], ref)
