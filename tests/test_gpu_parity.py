"""Parity of the CUDA path (through the C ABI / the reference-facing classes) against the oracle and the
reference's golden fixtures.  Tolerances (BASELINE.json north_star):
  fp64 mode : per-minibatch codes within 1e-4 relative L2 of the reference lasso_lars codes
              (measured ~1e-11; asserted at 1e-8 to catch regressions)
  fp32 mode : final dictionary per atom within 1e-3; reconstruction error within 0.5 %.
"""
import math
import os
import warnings

import numpy as np
import pytest
import torch

from onmf_ontf_ndl_b200 import Online_NMF, Online_NTF, OnmfEngine, _lib, update_code_within_radius
from oracle import c_oracle
from oracle import onmf_oracle as O

pytestmark = pytest.mark.gpu
warnings.filterwarnings("ignore")

CASES = ["cfg1_renoir_gray", "cfg1_alpha0", "cfg2_renoir_color_tensor", "cfg3_binary_motif", "cfg4_ising_pm1"]
CODE_TOL_FP64 = 1e-8       # north_star bar: 1e-4
CODE_TOL_FP32 = 2e-3       # per-minibatch fp32 codes (not a north_star bar; W / recon bars below are)
ATOM_TOL_FP32 = 1e-3       # north_star


def c_oracle_lars_single(G, c, alpha, d):
    return O.lars_lasso_positive(G, c, alpha, d)

RECON_TOL = 5e-3           # north_star: reconstruction error within 0.5 %


def dev():
    return torch.device("cuda", 0)


def rel(a, b):
    return float(np.linalg.norm(np.asarray(a, dtype=np.float64) - b) / max(np.linalg.norm(b), 1e-300))


def per_atom(W, Wref):
    return float(np.max(np.linalg.norm(W - Wref, axis=0) / np.maximum(np.linalg.norm(Wref, axis=0), 1e-30)))


def tt(x, dt):
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev(), dt)


def load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name + ".npz"))


def test_extension_is_the_native_library():
    lib = _lib.load()
    assert lib.onmf_built_arch() == 100
    assert torch.cuda.get_device_capability(0)[0] == 10


# ---------------------------------------------------------------------------------------------- K2 / K4
@pytest.mark.parametrize("dt,tol", [(torch.float64, 1e-13), (torch.float32, 2e-6)])
@pytest.mark.parametrize("n,d,k", [(300, 100, 25), (257, 300, 49), (1000, 441, 25), (513, 400, 100), (640, 1024, 256), (1, 7, 3)])
def test_gram_cov_surrogate(dt, tol, n, d, k):
    rng = np.random.default_rng(n + d + k)
    X, W = rng.random((n, d)), rng.random((d, k))
    H = rng.random((n, k)) * (rng.random((n, k)) < 0.2)
    Xt, Wd, Ht = tt(X, dt), tt(W, dt), tt(H, dt)
    G = torch.empty(k, k, dtype=dt, device=dev())
    Ct = torch.empty(n, k, dtype=dt, device=dev())
    P = torch.empty(k, k + d, dtype=dt, device=dev())
    ws = torch.empty(_lib.surrogate_workspace(dt, n, k, d), dtype=torch.uint8, device=dev())
    _lib.gram(Wd, G); _lib.cov(Xt, Wd, Ct); _lib.surrogate_partial(Ht, Xt, P, ws)
    Pn = P.cpu().numpy()
    assert rel(G.cpu().numpy(), W.T @ W) < tol and rel(Ct.cpu().numpy(), X @ W) < tol
    assert rel(Pn[:, :k], H.T @ H) < tol and rel(Pn[:, k:], H.T @ X) < tol
    A, B = rng.random((k, k)), rng.random((k, d))
    Ad, Bd = tt(A, dt), tt(B, dt)
    _lib.surrogate_blend(P, 0.25, Ad, Bd)
    Aref, Bref = O.aggregate(A, B, H.T, X.T, 4.0)
    assert rel(Ad.cpu().numpy(), Aref) < tol and rel(Bd.cpu().numpy(), Bref) < tol


def test_surrogate_is_deterministic_and_symmetric():
    rng = np.random.default_rng(0)
    n, d, k = 5000, 100, 25
    Ht = tt(rng.random((n, k)), torch.float32); Xt = tt(rng.random((n, d)), torch.float32)
    ws = torch.empty(_lib.surrogate_workspace(torch.float32, n, k, d), dtype=torch.uint8, device=dev())
    P1 = torch.empty(k, k + d, dtype=torch.float32, device=dev()); P2 = torch.empty_like(P1)
    _lib.surrogate_partial(Ht, Xt, P1, ws); _lib.surrogate_partial(Ht, Xt, P2, ws)
    assert torch.equal(P1, P2)                               # fixed-order split-K reduction
    assert torch.equal(P1[:, :k], P1[:, :k].T.contiguous())  # HtH bitwise symmetric


# ---------------------------------------------------------------------------------------------- K5
# fp32 tolerance: the sweep subtracts two O(100) numbers (W A[:,j] and B[j,:]) to get an O(0.01) update, so
# fp32 rounding is amplified ~1e4x on these synthetic magnitudes (measured 2e-4 at d=2700); fp64 pins the logic.
@pytest.mark.parametrize("dt,tol", [(torch.float64, 1e-12), (torch.float32, 1e-3)])
@pytest.mark.parametrize("d,k", [(100, 25), (300, 49), (441, 25), (400, 100), (1024, 256), (2700, 25), (77, 3), (5, 1)])
def test_update_dict(dt, tol, d, k):
    rng = np.random.default_rng(d * k)
    W = rng.random((d, k)); H = rng.random((k, 200))
    A, B = H @ H.T / 7, H @ rng.random((200, d)) / 7
    Wd, out = tt(W, dt), torch.empty(d, k, dtype=dt, device=dev())
    _lib.update_dict(Wd, tt(A, dt), tt(B, dt), out)
    ref = O.update_dict(W, A, B)
    got = out.cpu().numpy().astype(np.float64)
    assert per_atom(got, ref) < tol
    assert got.min() >= 0 and np.all(np.linalg.norm(got, axis=0) <= 1 + 1e-6)
    _lib.update_dict(Wd, tt(A, dt), tt(B, dt), Wd)                     # in place
    assert torch.equal(Wd, out)
    # zero aggregates: clamp + shrink only (first step of every run, SURVEY §A.1)
    z = torch.empty_like(out)
    _lib.update_dict(tt(W, dt), torch.zeros(k, k, dtype=dt, device=dev()), torch.zeros(k, d, dtype=dt, device=dev()), z)
    assert rel(z.cpu().numpy(), W / np.maximum(1.0, np.linalg.norm(W, axis=0))) < tol


# ---------------------------------------------------------------------------------------------- K3
@pytest.mark.parametrize("name", CASES)
def test_codes_vs_reference_golden_every_step(golden_dir, name):
    g = load(golden_dir, name)
    alpha = float(g["alpha"])
    for i in range(int(g["n_steps"])):
        W = g["W0"] if i == 0 else g["W_%d" % (i - 1)]
        Xb = g["X"][:, g["idx"][i]]
        Href = g["H_%d" % i]
        eng = OnmfEngine(W.shape[0], W.shape[1], alpha=alpha, dtype=torch.float64, device=dev(), collect_stats=True)
        H = eng.sparse_code(tt(Xb.T, torch.float64), tt(W, torch.float64)).cpu().numpy().T
        assert rel(H, Href) < CODE_TOL_FP64, (name, i)
        st = eng.read_stats()
        assert st["columns"] == Xb.shape[1] and st["flagged"] == 0
        if not (alpha == 0.0 and i > 0):          # alpha=0 on an ill-conditioned learned dictionary: NNLS is fp32-sensitive
            eng32 = OnmfEngine(W.shape[0], W.shape[1], alpha=alpha, dtype=torch.float32, device=dev())
            H32 = eng32.sparse_code(tt(Xb.T, torch.float32), tt(W, torch.float32)).cpu().numpy().T
            assert rel(H32, Href) < CODE_TOL_FP32, (name, i)


def test_codes_cfg5_and_overflow_path(golden_dir):
    """d=1024, k=256 on the raw U[0,1) W0: active sets exceed the 64-slot fast path -> exercises the large path."""
    g = load(golden_dir, "cfg5_synthetic")
    X = np.random.RandomState(int(g["x_seed"])).rand(1024, 160)
    W0 = np.random.RandomState(int(g["w0_seed"])).rand(1024, 256)
    Xb = X[:, g["idx"][0]]
    for dt, tol in ((torch.float64, CODE_TOL_FP64), (torch.float32, CODE_TOL_FP32)):
        eng = OnmfEngine(1024, 256, alpha=1.0, dtype=dt, device=dev(), collect_stats=True)
        H = eng.sparse_code(tt(Xb.T, dt), tt(W0, dt)).cpu().numpy().T
        assert rel(H, g["H_0"]) < tol
        st = eng.read_stats()
        assert st["overflow"] > 0 and st["max_active"] > 64 and st["columns"] == Xb.shape[1]


@pytest.mark.parametrize("d,k,n,alpha", [(64, 20, 333, 1.0), (64, 20, 64, 0.0), (50, 33, 100, 0.3), (120, 70, 90, 1.0),
                                          (200, 130, 60, 0.5), (30, 7, 1, 1.0), (16, 3, 5, 2.0)])
def test_codes_vs_c_oracle_fresh_inputs(d, k, n, alpha):
    rng = np.random.default_rng(d + k + n)
    W = rng.random((d, k)); W /= np.linalg.norm(W, axis=0)
    X = rng.random((d, n))
    if n > 3:
        X[:, 2] = 0.0                       # empty sample
        X[:, 3] = -X[:, 3]                  # all covariances negative -> never activates
    Href = c_oracle.sparse_code(X, W, alpha)
    eng = OnmfEngine(d, k, alpha=alpha, dtype=torch.float64, device=dev())
    H = eng.sparse_code(tt(X.T, torch.float64), tt(W, torch.float64)).cpu().numpy().T
    assert rel(H, Href) < CODE_TOL_FP64
    if n > 3:
        assert np.all(H[:, 2] == 0) and np.all(H[:, 3] == 0)
    assert H.min() >= -1e-12


def test_codes_satisfy_kkt_at_scale():
    """size-independent property at a bench-like shape: nonnegativity and lasso KKT conditions
    (G h - c + alpha >= 0 off the support up to the LARS last-segment shift, |.| small on the support)."""
    d, k, n, alpha = 1024, 256, 8192, 1.0
    g = torch.Generator(device=dev()); g.manual_seed(0)
    Xt = torch.rand(n, d, dtype=torch.float32, device=dev(), generator=g)
    W = torch.rand(d, k, dtype=torch.float32, device=dev(), generator=g)
    W = W / W.norm(dim=0, keepdim=True)
    eng = OnmfEngine(d, k, alpha=alpha, dtype=torch.float32, device=dev(), collect_stats=True)
    Ht = eng.sparse_code(Xt, W).clone()
    assert float(Ht.min()) >= 0.0
    G = (W.double().T @ W.double()); C = Xt.double() @ W.double()
    grad = Ht.double() @ G - C + alpha                          # n x k
    on = Ht > 0
    assert float(grad[on].abs().max()) < 0.05                    # alpha_eff in [0.9993, 1.0202]*alpha (SURVEY §B.2)
    assert float(grad[~on].min()) > -0.05
    st = eng.read_stats()
    assert st["columns"] == n and st["flagged"] <= n // 1000


# ---------------------------------------------------------------------------------------------- whole path
@pytest.mark.parametrize("name", ["cfg1_renoir_gray", "cfg3_binary_motif", "cfg4_ising_pm1", "cfg2_renoir_color_tensor"])
@pytest.mark.parametrize("precision", ["fp64", "fp32"])
def test_online_ntf_train_matches_reference(golden_dir, name, precision):
    """Online_NTF.train_dict_single under the reference's seed: same W0 / minibatch order (host RNG replay)."""
    g = load(golden_dir, name)
    seeds = {"cfg1_renoir_gray": 11, "cfg2_renoir_color_tensor": 21, "cfg3_binary_motif": 31, "cfg4_ising_pm1": 41}
    ns = int(g["n_steps"])
    k = g["W0"].shape[1]
    batch = g["idx"].shape[1]
    if name == "cfg2_renoir_color_tensor":
        X3, mode, joint = g["T"], 2, True
    else:
        X3, mode, joint = g["X"][:, :, None], 0, False
    np.random.seed(seeds[name])
    m = Online_NTF(X3, n_components=k, iterations=ns + 1, batch_size=batch, alpha=float(g["alpha"]), mode=mode,
                   learn_joint_dict=joint, precision=precision)
    W, A, B, code = m.train_dict_single()
    assert W.dtype == np.float64 and W.shape == g["W_final"].shape and code.shape == (X3.shape[1], k)
    assert float(m.history) == float(g["history_out"])
    if precision == "fp64":
        assert per_atom(W, g["W_final"]) < 1e-8 and rel(A, g["A_final"]) < 1e-8 and rel(B, g["B_final"]) < 1e-8
    else:
        assert per_atom(W, g["W_final"]) < ATOM_TOL_FP32
        assert rel(A, g["A_final"]) < 5e-3 and rel(B, g["B_final"]) < 5e-3
        # reconstruction error with reference codes for both dictionaries (SURVEY §8d)
        Xe = g["X"][:, :80]
        e_ref = np.linalg.norm(Xe - g["W_final"] @ O.sparse_code_sklearn(Xe, g["W_final"], float(g["alpha"]))) / np.linalg.norm(Xe)
        e_got = np.linalg.norm(Xe - W @ O.sparse_code_sklearn(Xe, W, float(g["alpha"]))) / np.linalg.norm(Xe)
        assert abs(e_got - e_ref) <= RECON_TOL * e_ref


def test_chained_epochs_alphaNone_beta(golden_dir):
    g2 = load(golden_dir, "cfg1_renoir_gray_epoch2")
    np.random.seed(12)
    m = Online_NTF(g2["X"][:, :, None], n_components=25, iterations=int(g2["n_steps"]) + 1, batch_size=g2["idx"].shape[1],
                   ini_dict=g2["W0"], ini_A=g2["A0"], ini_B=g2["B0"], history=float(g2["history_in"]), alpha=1,
                   precision="fp64")
    W, A, B, _ = m.train_dict_single()
    assert per_atom(W, g2["W_final"]) < 1e-8 and rel(A, g2["A_final"]) < 1e-8
    assert float(m.history) == float(g2["history_out"])
    g3 = load(golden_dir, "cfg1_alphaNone_beta_full")       # alpha=None -> 2, beta=0.75, subsample=False
    np.random.seed(13)
    m = Online_NTF(g3["X"][:, :, None], n_components=25, iterations=int(g3["n_steps"]) + 1, batch_size=200, alpha=None,
                   beta=0.75, subsample=False, precision="fp64")
    W, A, B, _ = m.train_dict_single()
    assert per_atom(W, g3["W_final"]) < 1e-8 and rel(A, g3["A_final"]) < 1e-8 and rel(B, g3["B_final"]) < 1e-8


def test_step_and_coder_methods(golden_dir):
    g = load(golden_dir, "cfg4_ising_pm1")
    i = 2
    W, A, B = g["W_%d" % (i - 1)], g["A_%d" % (i - 1)], g["B_%d" % (i - 1)]
    Xb = g["X"][:, g["idx"][i]]
    m = Online_NTF(g["X"][:, :, None], n_components=100, alpha=1, precision="fp64")
    H1, A1, B1, W1 = m.step(Xb, A, B, W, np.float64(i + 1))
    assert H1.shape == (Xb.shape[1], 100)                            # n x r like the reference
    assert rel(H1.T, g["H_%d" % i]) < 1e-8 and rel(A1, g["A_%d" % i]) < 1e-8 and rel(B1, g["B_%d" % i]) < 1e-8
    assert per_atom(W1, g["W_%d" % i]) < 1e-8 and float(m.history) == i + 2
    assert rel(m.joint_sparse_code_tensor(Xb, W).T, g["H_%d" % i]) < 1e-8
    assert per_atom(m.update_dict(W, A, B), g["W_%d" % i]) < 1e-8
    # Online_NMF: same arithmetic, r x n codes, driver-style 5-tuple
    nm = Online_NMF(g["X"], n_components=100, alpha=1, precision="fp64")
    assert rel(nm.sparse_code(Xb, W), g["H_%d" % i]) < 1e-8
    H2, agg, W2 = nm.step(Xb, [A, B], W, np.float64(i + 1))
    assert rel(H2, g["H_%d" % i]) < 1e-8 and rel(agg[0], g["A_%d" % i]) < 1e-8 and per_atom(W2, g["W_%d" % i]) < 1e-8


def test_online_nmf_train_dict_driver_style(golden_dir):
    """Online_NMF.train_dict (lasso coder, accumulating aggregates, subsample=True) == oracle loop; 5-tuple with Ct."""
    g = load(golden_dir, "cfg1_renoir_gray")
    X = g["X"][:, :400]
    np.random.seed(5)
    m = Online_NMF(X, n_components=25, iterations=4, batch_size=100, alpha=1, subsample=True, precision="fp64")
    W, At, Bt, Ct, H = m.train_dict()
    rs = np.random.RandomState(5)
    W0 = rs.rand(100, 25)
    idx = [rs.randint(400, size=100) for _ in range(3)]
    Wr, Ar, Br = W0, np.zeros((25, 25)), np.zeros((25, 100))
    Cr = np.zeros((100, 100)); code = np.zeros((25, 400))
    for i, ii in enumerate(idx, start=1):
        Hh, A1, B1, W1 = c_oracle.step(X[:, ii], Ar, Br, Wr, float(i), 1.0)
        Cr = (1 - 1.0 / i) * Cr + (1.0 / i) * X[:, ii] @ X[:, ii].T
        code[:, ii] += Hh
        Wr, Ar, Br = W1, A1, B1
    assert per_atom(W, Wr) < 1e-8 and rel(At, Ar) < 1e-8 and rel(Bt, Br) < 1e-8 and rel(Ct, Cr) < 1e-10
    assert rel(H, code) < 1e-8 and float(m.history) == 4.0
    err = O.surrogate_error(W, At, Bt, Ct)                      # ising_reconstruction.py:133 readout works
    assert np.isfinite(err)


def test_pgd_coder_and_shipped_compat(golden_dir):
    g = load(golden_dir, "pgd_coder")
    H = update_code_within_radius(g["X"], g["W"], H0=g["H0"], r=None, alpha=1, sub_iter=10, stopping_diff=0.01,
                                  precision="fp64")
    assert rel(H, g["H"]) < 1e-9
    H1 = update_code_within_radius(g["X"][:, :1], g["W"], H0=g["H0"][:, :1], r=None, alpha=1, sub_iter=10,
                                   stopping_diff=0.01, precision="fp64")
    assert rel(H1, g["H_single"]) < 1e-9
    # radius mode (src/onmf.py:260-263 incl. the H0 = H1 aliasing): the reference's own output
    Hr = update_code_within_radius(g["X"], g["W"], H0=g["H0"], r=0.5, alpha=0.3, sub_iter=3, stopping_diff=0.01,
                                   precision="fp64")
    assert rel(Hr, g["H_radius"]) < 1e-9
    Hr32 = update_code_within_radius(g["X"], g["W"], H0=g["H0"], r=0.5, alpha=0.3, sub_iter=3, stopping_diff=0.01)
    assert rel(Hr32, g["H_radius"]) < 1e-4
    with pytest.raises(ValueError):
        update_code_within_radius(g["X"], g["W"], H0=g["H0"], r=0.0)
    s = load(golden_dir, "shipped_onmf")                     # literal shipped src/onmf.py run, seed 71
    np.random.seed(int(s["seed"]))
    m = Online_NMF(s["X"], n_components=25, iterations=4, batch_size=60, alpha=1, subsample=True, compat="shipped_onmf",
                   precision="fp64")
    W, agg, code = m.train_dict()
    assert per_atom(W, s["W"]) < 1e-8 and rel(agg[0], s["A"]) < 1e-8 and rel(agg[1], s["B"]) < 1e-8
    assert rel(code, s["code"]) < 1e-8 and float(m.history) == float(s["history_out"])


# ---------------------------------------------------------------------------------------------- K1
def test_gathers(golden_dir):
    g = load(golden_dir, "cfg1_renoir_gray")
    for dt in (torch.float64, torch.float32):
        img = tt(g["img"], dt); co = torch.from_numpy(g["coords"].astype(np.int32)).to(dev())
        out = torch.empty(co.shape[0], 100, dtype=dt, device=dev())
        _lib.gather_patches(img, co, 10, out)
        assert np.array_equal(out.cpu().numpy().T, g["X"].astype(out.cpu().numpy().dtype))
    g2 = load(golden_dir, "cfg2_renoir_color_tensor")
    img = tt(g2["img"], torch.float64); co = torch.from_numpy(g2["coords"].astype(np.int32)).to(dev())
    out = torch.empty(co.shape[0], 300, dtype=torch.float64, device=dev())
    _lib.gather_patches(img, co, 10, out)
    assert np.array_equal(out.cpu().numpy().T, g2["X"])              # HWC feature order == mode-2 joint unfolding
    g4 = load(golden_dir, "cfg4_ising_pm1")
    img = tt(g4["img"], torch.float32); co = torch.from_numpy(g4["coords"].astype(np.int32)).to(dev())
    out = torch.empty(co.shape[0], 400, dtype=torch.float32, device=dev())
    _lib.gather_patches(img, co, 20, out)
    assert np.array_equal(out.cpu().numpy().T.astype(np.float64), g4["X"])
    pool = tt(g["X"].T, torch.float64); idx = torch.from_numpy(g["idx"][0].astype(np.int64)).to(dev())
    xb = torch.empty(len(idx), 100, dtype=torch.float64, device=dev())
    _lib.gather_rows(pool, idx, xb)
    assert np.array_equal(xb.cpu().numpy().T, g["X"][:, g["idx"][0]])
    src = tt(np.arange(35 * 77, dtype=np.float64).reshape(35, 77), torch.float64)
    dst = torch.empty(77, 35, dtype=torch.float32, device=dev())
    _lib.transpose(src, dst)
    assert torch.equal(dst, src.T.to(torch.float32))
    # empty inputs are no-ops
    _lib.gather_rows(pool, idx[:0], xb[:0])


def test_empty_minibatch_and_loud_failures():
    eng = OnmfEngine(20, 5, alpha=1.0, dtype=torch.float32, device=dev())
    W0 = torch.rand(20, 5, device=dev())
    eng.set_state(W0.cpu().numpy())
    eng.step(torch.empty(0, 20, device=dev()), 1.0)                 # a rank may own zero columns
    W, A, B, _ = eng.state()
    assert float(A.abs().max()) == 0.0
    with pytest.raises(_lib.OnmfKernelError):
        eng.step(None, 2.0)
    before = [x.clone() for x in eng.state()[:3]]
    with pytest.raises(_lib.OnmfKernelError):
        eng._plan.step(eng._sb, None, None, 5, 0.5, eng._cur)       # n > 0 with no minibatch: refused before any launch
    torch.cuda.synchronize()
    assert all(torch.equal(x, y) for x, y in zip(eng.state()[:3], before))
    with pytest.raises(_lib.OnmfKernelError):
        _lib.gram(torch.rand(4, 3), torch.empty(3, 3))               # CPU tensors are refused, not silently handled
    with pytest.raises(_lib.OnmfKernelError):
        OnmfEngine(10, 600, device=dev()).sparse_code(torch.rand(4, 10, device=dev()))   # k > 512 unsupported


# ---------------------------------------------------------------------------------------------- tensor-core path
@pytest.mark.parametrize("n,d,k", [(256, 64, 64), (300, 128, 96), (1000, 400, 100), (4096, 1024, 256), (513, 300, 52), (33, 32, 32)])
def test_tensor_core_gemms_vs_fp64(n, d, k):
    """tcgen05 3xTF32 products against float64; tolerance 2e-5 = the round-toward-zero accumulation bias of the
    tensor core over the capped 32-K-block chain (DESIGN.md), far below the 1.5e-3 of plain TF32."""
    g = torch.Generator(device=dev()); g.manual_seed(n + d + k)
    X = torch.rand(n, d, device=dev(), generator=g); W = torch.rand(d, k, device=dev(), generator=g)
    H = torch.rand(n, k, device=dev(), generator=g) * (torch.rand(n, k, device=dev(), generator=g) < 0.2)
    assert _lib.tc_supported(k, d)
    def split(x):
        hi, lo = torch.empty_like(x), torch.empty_like(x)
        _lib.split_tf32(x, hi, lo)
        return hi, lo
    Xh, Xl = split(X); Wh, Wl = split(W); Hh, Hl = split(H)
    assert torch.equal(Xh + Xl, X)                                   # the split is exact
    assert torch.equal(Xh.view(torch.int32) & 0x1FFF, torch.zeros_like(Xh, dtype=torch.int32))   # hi is a TF32 number
    Ct = torch.full((n, k), float("nan"), device=dev())
    _lib.cov_tc(Xh, Xl, Wh, Wl, Ct)
    P = torch.full((k, k + d), float("nan"), device=dev())
    ws = torch.empty(_lib.surrogate_tc_workspace(n, k, d), dtype=torch.uint8, device=dev())
    _lib.surrogate_partial_tc(Hh, Hl, Xh, Xl, P, ws)
    P2 = torch.empty_like(P); _lib.surrogate_partial_tc(Hh, Hl, Xh, Xl, P2, ws)
    assert torch.equal(P, P2)                                        # deterministic split-K
    Xd, Wd, Hd = X.double(), W.double(), H.double()
    relt = lambda a, b: float((a.double() - b).norm() / b.norm())
    assert relt(Ct, Xd @ Wd) < 2e-5 and relt(P[:, :k], Hd.T @ Hd) < 2e-5 and relt(P[:, k:], Hd.T @ Xd) < 2e-5


def test_tensor_core_and_cuda_core_paths_agree_end_to_end(golden_dir):
    """same online run with and without the tensor-core GEMMs: dictionaries agree far inside the fp32 bar."""
    g = load(golden_dir, "cfg4_ising_pm1")
    X, W0 = g["X"], g["W0"]
    outs = []
    for use_tc in (True, False):
        eng = OnmfEngine(400, 100, alpha=1.0, dtype=torch.float32, device=dev(), use_tc=use_tc)
        assert eng.use_tc == use_tc
        eng.set_state(W0)
        pool = tt(X.T, torch.float32)
        for i in range(int(g["n_steps"])):
            idx = torch.from_numpy(g["idx"][i].astype(np.int64)).to(dev())
            Xb = torch.empty(len(idx), 400, dtype=torch.float32, device=dev())
            _lib.gather_rows(pool, idx, Xb)
            eng.step(Xb, float(i + 1))
        W, A, B, _ = eng.state()
        torch.cuda.synchronize()
        outs.append(W.cpu().numpy().astype(np.float64))
        assert per_atom(outs[-1], g["W_final"]) < ATOM_TOL_FP32
    assert per_atom(outs[0], outs[1]) < 5e-4      # both are fp32 paths with different summation orders


# ---------------------------------------------------------------------------------------------- batched reconstruction (§8f.1)
def test_batched_reconstruction_matches_reference_loop(golden_dir):
    from onmf_ontf_ndl_b200 import reconstruct_image
    g = load(golden_dir, "reconstruct_color")
    rec, cnt, code = reconstruct_image(g["img"], g["W"], int(g["patch"]), int(g["stride"]), alpha=1, sub_iter=10,
                                       stopping_diff=0.01, coder="pgd", H0=g["H0"], precision="fp64", return_code=True)
    assert rel(code, g["codes"]) < 1e-10 and rel(rec, g["recons"]) < 1e-10 and np.array_equal(cnt, g["count"])
    rec32, _ = reconstruct_image(g["img"], g["W"], int(g["patch"]), int(g["stride"]), alpha=1, coder="pgd", H0=g["H0"],
                                 precision="fp32")
    assert rel(rec32, g["recons"]) < 1e-4
    # default H0 = the reference's RNG stream (one np.random.rand(r, 1) per patch, loop order)
    np.random.seed(7)
    recd, _ = reconstruct_image(g["img"], g["W"], 5, 2, precision="fp64")
    np.random.seed(7)
    ny, nx = len(range(0, 36 - 5, 2)), len(range(0, 40 - 5, 2))
    H0 = np.stack([np.random.rand(25, 1)[:, 0] for _ in range(ny * nx)], 1)
    ref, _, _ = O.reconstruct_image_loop(g["img"], g["W"], 5, 2, 1, 10, 0.01, H0)
    assert rel(recd, ref) < 1e-10
    # lasso_lars coder variant (image_reconstruction.py:380-383) on a gray image, stride 3
    gray = g["img"][:, :, 0]
    Wg = np.abs(g["W"][:25, :12]); Wg /= np.linalg.norm(Wg, axis=0)
    recl, cntl = reconstruct_image(gray, Wg, 5, 3, alpha=0.1, coder="lasso_lars", precision="fp64")
    refl, cntr, _ = O.reconstruct_image_loop(gray, Wg, 5, 3, 0.1, 0, 0, np.zeros((12, 200)),
                                             coder=lambda patch, h0: c_oracle.sparse_code(patch, Wg, 0.1))
    assert rel(recl, refl) < 1e-9 and np.array_equal(cntl, cntr) and recl.shape == gray.shape


def test_patch_grid_mean_equals_sklearn_overlap_average():
    from sklearn.feature_extraction.image import extract_patches_2d, reconstruct_from_patches_2d
    rng = np.random.default_rng(0)
    img = rng.random((17, 23))
    P = extract_patches_2d(img, (4, 4)) + rng.random((14 * 20, 4, 4))          # ising_reconstruction.py:185,199 use these
    ref = reconstruct_from_patches_2d(P, (17, 23))
    R = tt(P.reshape(len(P), -1), torch.float64)
    canvas = torch.empty(17, 23, 1, dtype=torch.float64, device=dev())
    _lib.patch_grid_mean(R, 14, 20, 4, 1, 1, 17, 23, canvas)
    assert rel(canvas.cpu().numpy()[:, :, 0], ref) < 1e-14


# ---------------------------------------------------------------------------------------------- full-length runs, fp32 bars
@pytest.mark.parametrize("name", ["full_cfg1", "full_cfg2", "full_cfg3", "full_cfg4"])
def test_full_length_run_fp32_bars(golden_dir, name):
    """BASELINE.json configs at full minibatch size for 100 / 100 / 25 / 25 iterations in the fp32 production mode:
    final dictionary per atom within 1e-3 of the reference's, reconstruction error within 0.5 %."""
    g = load(golden_dir, name)
    scale = 255.0 if name in ("full_cfg1", "full_cfg2") else 1.0
    X = g["pool_u8"].astype(np.float64) / scale
    ntr, k, iters, batch, alpha = int(g["n_train"]), int(g["k"]), int(g["iters"]), int(g["batch"]), float(g["alpha"])
    np.random.seed(int(g["seed"]))
    m = Online_NTF(X[:, :ntr, None], n_components=k, iterations=iters + 1, batch_size=batch, alpha=alpha, mode=0,
                   learn_joint_dict=False, precision="fp32")
    W, A, B, _ = m.train_dict_single()
    assert float(m.history) == float(g["history"])
    assert per_atom(W, g["W"]) < ATOM_TOL_FP32, per_atom(W, g["W"])
    assert rel(A, g["A"]) < 2e-3 and rel(B, g["B"]) < 2e-3
    Xe = X[:, ntr:ntr + 400]                       # the 400 held-out columns oracle/make_golden_full.py used
    e_got = np.linalg.norm(Xe - W @ O.sparse_code_sklearn(Xe, W, alpha)) / np.linalg.norm(Xe)
    assert abs(e_got - float(g["recon"])) <= RECON_TOL * float(g["recon"])
    assert m.lars_stats["flagged"] <= m.lars_stats["columns"] // 1000


# ---------------------------------------------------------------------------------------------- on-device patch pipelines (§8f.2, §8f.4)
def test_patch_pipeline_helpers(golden_dir):
    from onmf_ontf_ndl_b200 import patches
    g = load(golden_dir, "cfg1_renoir_gray")
    np.random.seed(3)
    X = patches.extract_random_patches(g["img"], 10, 50, precision="fp64")
    np.random.seed(3)
    co = np.array([[np.random.choice(g["img"].shape[0] - 10), np.random.choice(g["img"].shape[1] - 10)] for _ in range(50)])
    assert np.array_equal(X, O.gather_patches_gray(g["img"], co, 10))            # same RNG order, exact copy
    g2 = load(golden_dir, "cfg2_renoir_color_tensor")
    T = patches.patches_to_tensor(patches.gather_patches(g2["img"], g2["coords"], 10, precision="fp64"), 3)
    assert np.array_equal(T, g2["T"])                                           # the reference's (k*k, 3, N) tensor
    # motif patches on a random graph with a self-loop and an isolated node
    import networkx as nx
    G = nx.gnp_random_graph(60, 0.1, seed=1)
    G.add_edge(5, 5)
    csr = patches.graph_to_csr(G)
    rng = np.random.default_rng(2)
    emb = rng.integers(0, 60, size=(300, 7))
    Xm = patches.motif_patches(csr, emb, precision="fp32")
    ref = O.motif_patches({u: set(G.neighbors(u)) for u in G.nodes()}, emb)
    assert np.array_equal(Xm, ref) and Xm.shape == (49, 300) and Xm[0, np.where(emb[:, 0] == 5)[0]].all()
    for j in range(3):                                                          # equals networkx's own has_edge
        for q in range(7):
            for r in range(7):
                assert Xm[q * 7 + r, j] == float(G.has_edge(emb[j, q], emb[j, r]))
    # tiled kernel (k*k <= 1024 entries per patch) and flat kernel (k = 33), fp64, node indices outside the graph -> 0
    adj = {u: set(G.neighbors(u)) for u in G.nodes()}
    for kk, nn in ((21, 97), (33, 41), (1, 5), (32, 33)):
        emb = rng.integers(0, 60, size=(nn, kk))
        for prec in ("fp64", "fp32"):
            assert np.array_equal(patches.motif_patches(csr, emb, precision=prec), O.motif_patches(adj, emb))
    e = torch.tensor([[0, -1, 60, 5, 5]], dtype=torch.int32, device=dev())
    out = torch.full((1, 25), 7.0, device=dev())
    _lib.motif_patches(torch.from_numpy(csr[0]).to(dev()), torch.from_numpy(csr[1]).to(dev()), e, out)
    want = np.zeros((5, 5)); want[3, 3] = want[3, 4] = want[4, 3] = want[4, 4] = 1.0      # the self-loop at node 5
    for a_, b_ in ((0, 3), (0, 4)):
        want[a_, b_] = want[b_, a_] = float(G.has_edge(0, 5))
    want[0, 0] = float(G.has_edge(0, 0))
    assert np.array_equal(out.cpu().numpy().reshape(5, 5), want)


def test_codes_large_active_sets_all_tiers():
    """alpha = 0 (NNLS end of the path) on d=1024, k=256: active sets far beyond 128 atoms -> every tier of the coder
    including the global-memory one; plus the k <= 512 class."""
    rng = np.random.default_rng(5)
    d, k, n = 1024, 256, 6
    W = rng.random((d, k)); W /= np.linalg.norm(W, axis=0)
    Htrue = rng.random((k, n)) * (rng.random((k, n)) < 0.8)        # X is an exact nonnegative combination of ~200 atoms
    X = W @ Htrue
    Href = c_oracle.sparse_code(X, W, 0.0)
    eng = OnmfEngine(d, k, alpha=0.0, dtype=torch.float64, device=dev(), collect_stats=True)
    H = eng.sparse_code(tt(X.T, torch.float64), tt(W, torch.float64)).cpu().numpy().T
    st = eng.read_stats()
    assert st["max_active"] > 128 and st["columns"] == n, st
    assert rel(H, Href) < 1e-6 and rel(H, Htrue) < 1e-6          # (the path ends in a long near-degenerate tail: looser bar)
    d, k, n = 96, 300, 40                                       # k-class 4 (<= 512 atoms), more atoms than features
    W = rng.random((d, k)); W /= np.linalg.norm(W, axis=0)
    X = rng.random((d, n))
    Href = c_oracle.sparse_code(X, W, 0.2)
    H = OnmfEngine(d, k, alpha=0.2, dtype=torch.float64, device=dev()).sparse_code(tt(X.T, torch.float64), tt(W, torch.float64)).cpu().numpy().T
    assert rel(H, Href) < CODE_TOL_FP64
    H32 = OnmfEngine(d, k, alpha=0.2, dtype=torch.float32, device=dev()).sparse_code(tt(X.T, torch.float32), tt(W, torch.float32)).cpu().numpy().T
    assert rel(H32, Href) < 5e-3


# ---------------------------------------------------------------------------------------------- fp32 robustness regressions
def test_fp32_near_tie_column_and_fp64_gram(golden_dir):
    """A column (found in the two-rank test problem) where two atoms tie within one fp32 ulp at a knot: sklearn's
    strictly-positive step rule then steps past the second atom if the tie rounds to an exact one, which changed the fp32
    code by 22 %.  The fp32 coder takes the zero-length step instead and must agree with the fp64 coder (and the oracle)
    with either Gram precision; the FP64-accumulated Gram must be the correctly rounded product."""
    z = load(golden_dir, "fp32_tie_column")
    d, k = 64, 32
    G64 = tt(z["G64"], torch.float64)
    Href = c_oracle_lars_single(z["G64"], z["c32"].astype(np.float64), 0.5, d)
    assert set(np.nonzero(Href)[0]) == {7, 10, 20, 22, 29}
    for G in (G64, G64.float().contiguous()):
        for reps in (1, 5):
            Ct = tt(np.tile(z["c32"][None, :], (reps, 1)), torch.float32)
            Ht = torch.zeros(reps, k, device=dev())
            ws = torch.zeros(_lib.lasso_lars_workspace(torch.float32, k, reps), dtype=torch.uint8, device=dev())
            _lib.lasso_lars(G, Ct, d, 0.5, Ht, ws)
            torch.cuda.synchronize()
            for r in range(reps):
                assert rel(Ht[r].cpu().numpy().astype(np.float64), Href) < 1e-4
    # onmf_gram_f64: fp32 dictionary, FP64 accumulation, bitwise symmetric, odd shapes
    rng = np.random.default_rng(11)
    for (dd, kk) in ((64, 32), (300, 49), (441, 25), (1024, 256), (70, 130)):
        W = rng.random((dd, kk)).astype(np.float32)
        Wd = tt(W, torch.float32)
        G = torch.empty(kk, kk, dtype=torch.float64, device=dev())
        G32 = torch.empty(kk, kk, dtype=torch.float32, device=dev())
        ws = torch.empty(_lib.gram_f64_workspace(dd, kk), dtype=torch.uint8, device=dev())
        _lib.gram_f64(Wd, G, ws, G32=G32)
        torch.cuda.synchronize()
        ref = W.astype(np.float64).T @ W.astype(np.float64)
        assert np.abs(G.cpu().numpy() - ref).max() <= 1e-13 * np.abs(ref).max()
        assert torch.equal(G, G.T.contiguous())
        assert np.array_equal(G32.cpu().numpy(), G.cpu().numpy().astype(np.float32))


def test_surrogate_error_readout(golden_dir):
    """tr(W A W^T) - 2 tr(W B) + tr(C) (ising_reconstruction.py:133,164) from the engine's resident state vs the oracle."""
    g = load(golden_dir, "cfg4_ising_pm1")
    X = g["X"]
    d = X.shape[0]
    k = int(g["W0"].shape[1]) if "W0" in g else 12
    rng = np.random.default_rng(3)
    W0 = g["W0"] if "W0" in g else rng.random((d, k))
    for dt_, tol in ((torch.float64, 1e-10), (torch.float32, 1e-4)):
        eng = OnmfEngine(d, k, alpha=1.0, dtype=dt_, device=dev(), track_C=True, use_tc=False)
        eng.set_state(W0)
        Xt = tt(X.T, dt_)
        A, B, C, W = np.zeros((k, k)), np.zeros((k, d)), np.zeros((d, d)), W0
        for t in (1, 2, 3):
            eng.step(Xt, float(t))
            H, A1, B1, W1 = c_oracle.step(X, A, B, W, float(t), 1.0)
            C = (1 - 1.0 / t) * C + (1.0 / t) * (X @ X.T)
            A, B, W = A1, B1, W1
        ref = O.surrogate_error(W, A, B, C)
        got = eng.surrogate_error()
        scale = abs(np.trace(C)) + abs(ref)
        assert abs(got - ref) <= tol * scale, (got, ref)


def test_fused_step_equals_python_composed_schedule(monkeypatch):
    """OnmfEngine(fused=True) (one onmf_step call per minibatch) and fused=False (the same kernels composed from Python
    with torch events) must give bitwise identical state, in both precisions and with external codes / track_C.
    (Both on the pre-split tensor-core kernels: the Python-composed schedule does not use the minibatch-by-reference ones.)"""
    monkeypatch.setenv("ONMF_B200_FUSED_TC", "0")
    rng = np.random.default_rng(7)
    d, k, n = 64, 32, 777
    X = rng.random((n, d)); W0 = rng.random((d, k))
    for dt_ in (torch.float32, torch.float64):
        for kw in ({}, {"track_C": True, "use_tc": False}):
            res = []
            for fused in (True, False):
                l0 = _lib.launch_count()
                eng = OnmfEngine(d, k, alpha=0.7, dtype=dt_, device=dev(), fused=fused, **kw)
                eng.set_state(W0)
                Xt = tt(X, dt_)
                H = None
                for t in (1, 2, 3, 4):
                    H = eng.step(Xt, float(t)).clone()
                eng.step(Xt, 5.0, codes=H)                          # aggregate externally supplied codes
                eng.step(Xt[:0], 6.0)                                # empty shard
                W, A, B, C = eng.state()
                torch.cuda.synchronize()
                res.append((H, W.clone(), A.clone(), B.clone(), None if C is None else C.clone(), eng.launches - l0))
            for a, b in zip(res[0][:5], res[1][:5]):
                assert (a is None and b is None) or torch.equal(a, b)
            assert res[0][5] == res[1][5]                            # same launch accounting


# ---------------------------------------------------------------------------------------------- the benchmarked config (cfg5)
def _cfg5_inputs(g):
    ntr = int(g["n_train"])
    X = np.random.RandomState(int(g["x_seed"])).rand(1024, ntr + int(g["n_holdout"]))
    W0 = np.random.RandomState(int(g["seed"])).rand(1024, int(g["k"]))
    assert abs(W0.sum() - float(g["W0_checksum"])) < 1e-9
    return X, W0, ntr


def test_cfg5_per_step_codes_on_learned_dictionaries(golden_dir):
    """d=1024, k=256 (the shape bench.py times), 10 steps of the reference at minibatch 2048 (fixture full_cfg5).

    fp64 engine: per-step codes against the reference's lasso_lars codes at EVERY step (<= 1e-8), final W / A / B.
    fp32 production path (tensor-core products, fused onmf_step, hybrid 64-slot first tier): at every step >= 2 the fp32
    engine is put on the trajectory's state (W, A, B from the fp64 engine, which equals the reference's to ~1e-9) and
    codes the same minibatch through OnmfEngine.step; codes within 2e-3, no column may leave the first tier
    (overflow == 0) -- this is the regime the benchmark runs in (unit-norm learned dictionary, mean active set ~16)."""
    g = load(golden_dir, "full_cfg5")
    X, W0, ntr = _cfg5_inputs(g)
    k, iters = int(g["k"]), int(g["iters"])
    pool64 = tt(X[:, :ntr].T, torch.float64)
    pool32 = pool64.float().contiguous()
    e64 = OnmfEngine(1024, k, alpha=1.0, dtype=torch.float64, device=dev(), collect_stats=True)
    e32 = OnmfEngine(1024, k, alpha=1.0, dtype=torch.float32, device=dev(), collect_stats=True, use_tc=True, fused=True)
    assert e32.use_tc and e32.fused
    e64.set_state(W0)
    nb = g["idx"].shape[1]
    xb64 = torch.empty(nb, 1024, dtype=torch.float64, device=dev())
    xb32 = torch.empty(nb, 1024, dtype=torch.float32, device=dev())
    worst32 = 0.0
    for i in range(iters):
        idx = torch.from_numpy(g["idx"][i].astype(np.int64)).to(dev())
        Href = g["H_%d" % i]                                   # (n x r)
        if i >= 2:
            Wc, Ac, Bc, _ = e64.state()
            e32.set_state(Wc, Ac, Bc)
            e32.stats.zero_()
            _lib.gather_rows(pool32, idx, xb32)
            H32 = e32.step(xb32, float(i + 1)).cpu().numpy().astype(np.float64)
            st = e32.read_stats()
            assert st["overflow"] == 0 and st["columns"] == nb and st["flagged"] == 0, (i, st)
            assert st["max_active"] <= 64
            worst32 = max(worst32, rel(H32, Href))
            assert rel(H32, Href) < CODE_TOL_FP32, (i, rel(H32, Href))
        _lib.gather_rows(pool64, idx, xb64)
        H64 = e64.step(xb64, float(i + 1)).cpu().numpy()
        assert rel(H64, Href) < CODE_TOL_FP64, (i, rel(H64, Href))
    W, A, B, _ = e64.state()
    torch.cuda.synchronize()
    assert per_atom(W.cpu().numpy(), g["W"]) < 1e-8 and rel(A.cpu().numpy(), g["A"]) < 1e-8 and rel(B.cpu().numpy(), g["B"]) < 1e-8
    assert e64.read_stats()["flagged"] == 0


def test_cfg5_full_run_fp32_bars(golden_dir):
    """the same 10-step run end to end in the fp32 production mode through the reference-facing class: final dictionary per
    atom within 1e-3, A / B within 2e-3, held-out reconstruction error within 0.5 % (north_star bars at the benchmarked
    shape)."""
    g = load(golden_dir, "full_cfg5")
    X, W0, ntr = _cfg5_inputs(g)
    np.random.seed(int(g["seed"]))
    m = Online_NTF(X[:, :ntr, None], n_components=int(g["k"]), iterations=int(g["iters"]) + 1, batch_size=int(g["batch"]),
                   alpha=1.0, mode=0, learn_joint_dict=False, precision="fp32")
    W, A, B, _ = m.train_dict_single()
    assert float(m.history) == float(g["history"])
    assert per_atom(W, g["W"]) < ATOM_TOL_FP32, per_atom(W, g["W"])
    assert rel(A, g["A"]) < 2e-3 and rel(B, g["B"]) < 2e-3
    Xe = X[:, ntr:]
    e_got = np.linalg.norm(Xe - W @ O.sparse_code_sklearn(Xe, W, 1.0)) / np.linalg.norm(Xe)
    assert abs(e_got - float(g["recon"])) <= RECON_TOL * float(g["recon"])
    assert m.lars_stats["flagged"] <= m.lars_stats["columns"] // 1000


# ---------------------------------------------------------------------------------------------- shipped re-binding + lasso coder
def test_shipped_rebinding_with_lasso_coder(golden_dir):
    """compat='shipped_onmf' (src/onmf.py:217: every step starts from the INITIAL aggregates) combined with the lasso coder:
    the dictionary update runs on the side stream and must see the re-copied A, B (OnmfEngine.reset_aggregates orders the
    copies and re-marks the state) -- compared with the same recursion on the oracle."""
    g = load(golden_dir, "cfg1_renoir_gray")
    X = g["X"][:, :500]
    W0, A0, B0 = g["W_3"], g["A_3"], g["B_3"]
    for prec, tol in (("fp64", 1e-8), ("fp32", 1e-3)):
        np.random.seed(17)
        m = Online_NMF(X, n_components=25, iterations=6, batch_size=120, ini_dict=W0, ini_agg=[A0, B0], history=4, alpha=1,
                       subsample=True, compat="shipped_onmf", coder="lasso_lars", precision=prec)
        W, agg, code = m.train_dict()
        rs = np.random.RandomState(17)
        Wr, A1, B1 = W0, A0, B0
        for i in range(1, 6):
            ii = rs.randint(500, size=120)
            H = c_oracle.sparse_code(X[:, ii], Wr, 1.0)
            A1, B1 = O.aggregate(A0, B0, H, X[:, ii], float(4 + i))       # blend from the INITIAL aggregates
            Wr = O.update_dict(Wr, A0, B0)                                # update with the INITIAL aggregates
        assert per_atom(W, Wr) < tol and rel(agg[0], A1) < tol and rel(agg[1], B1) < tol, prec
        assert float(m.history) == 10.0


def test_online_nmf_alpha_none_follows_the_coder():
    X = np.random.rand(12, 30)
    assert Online_NMF(X)._alpha() == 2                                    # lasso_lars: src/ontf.py:79-81
    assert Online_NMF(X, coder="pgd")._alpha() == 0 and Online_NMF(X, compat="shipped_onmf")._alpha() == 0   # src/onmf.py:82-84
    assert Online_NMF(X, alpha=0.5)._alpha() == 0.5


# ---------------------------------------------------------------------------------------------- batched network reconstruction (§8f.1)
def test_batched_network_reconstruction_matches_reference(golden_dir):
    """all MCMC states of a trajectory at once (motif patches -> alpha=0 LARS -> W h -> scatter-mean) against the weights
    and overlap counts of the UNMODIFIED Network_Reconstructor.reconstruct_network (network_reconstruction_nx.py:444-511)."""
    import networkx as nx
    from onmf_ontf_ndl_b200 import reconstruct_network
    from onmf_ontf_ndl_b200.reconstruct import simple_graph_edges
    g = load(golden_dir, "network_recons")
    G = nx.Graph()
    G.add_nodes_from(range(int(g["n_nodes"])))
    G.add_edges_from(g["graph_edges"].tolist())
    # (fp32: alpha = 0 on binary patches is the NNLS end of the path -- ties and ill-conditioning; measured 6e-3)
    for prec, tol in (("fp64", 1e-9), ("fp32", 1e-2)):
        pairs, weight, count = reconstruct_network(G, g["W"], g["embs"], alpha=0, precision=prec)
        assert np.array_equal(np.asarray(pairs.tolist()), g["pairs"]) and np.array_equal(count, g["count"])
        assert np.max(np.abs(weight - g["weight"])) < tol * max(1.0, np.abs(g["weight"]).max()), prec
    assert simple_graph_edges(pairs, weight) == {frozenset(e) for e in g["simple_edges"].tolist()}
    # empty trajectory
    p0, w0, c0 = reconstruct_network(G, g["W"], np.empty((0, 6), dtype=np.int64))
    assert len(p0) == 0 and len(w0) == 0
    # unrelated states (every directed pair distinct): the pair table starts at the size a Glauber walk needs and grows
    rng = np.random.default_rng(3)
    G2 = nx.gnm_random_graph(500, 6000, seed=1)
    kk, r, n = 21, 5, 100
    embs = rng.integers(0, 500, size=(n, kk))
    W2 = rng.random((kk * kk, r)); W2 /= np.linalg.norm(W2, axis=0)
    pairs2, weight2, count2 = reconstruct_network(G2, W2, embs, alpha=0, precision="fp64")
    adj = {u: set(G2.neighbors(u)) for u in G2.nodes()}
    wref, cref = O.reconstruct_network_loop(adj, W2, embs, alpha=0.0)
    assert len(pairs2) == len(wref) > 2 * n * 4 * kk
    got = {(int(a), int(b)): (w, c) for (a, b), w, c in zip(pairs2.tolist(), weight2.tolist(), count2.tolist())}
    assert all(got[key][1] == cref[key] and abs(got[key][0] - wref[key]) < 1e-9 for key in wref)


# ---------------------------------------------------------------------------------------------- robustness of the gathers / large shapes
def test_gather_index_checks_and_large_dictionary_fallbacks():
    pool = torch.rand(10, 8, device=dev())
    idx = torch.tensor([0, 9, 10, -1, 3], dtype=torch.int64, device=dev())
    out = torch.zeros(5, 8, device=dev())
    _lib.gather_rows(pool, idx, out)
    assert torch.equal(out[0], pool[0]) and torch.equal(out[1], pool[9]) and torch.equal(out[4], pool[3])
    assert torch.isnan(out[2]).all() and torch.isnan(out[3]).all()                 # bad indices: NaN rows, no wild reads
    img = torch.rand(12, 9, device=dev())
    co = torch.tensor([[0, 0], [8, 5], [9, 0], [0, 6], [-1, 2]], dtype=torch.int32, device=dev())
    P = torch.zeros(5, 16, device=dev())
    _lib.gather_patches(img, co, 4, P)
    assert torch.equal(P[1], img[8:12, 5:9].reshape(-1)) and torch.isnan(P[2]).all() and torch.isnan(P[3]).all() and torch.isnan(P[4]).all()
    # dictionary update beyond one cluster's shared memory: cooperative-grid fallback == oracle
    rng = np.random.default_rng(4)
    d, k = 20000, 64
    assert _lib.update_dict_workspace(torch.float64, d, k) > 0 and _lib.update_dict_workspace(torch.float32, 1024, 256) == 0
    W = rng.random((d, k)); H = rng.random((k, 50))
    A, B = H @ H.T / 7, H @ rng.random((50, d)) / 7
    for dt_, tol in ((torch.float64, 1e-12), (torch.float32, 1e-3)):
        out = torch.empty(d, k, dtype=dt_, device=dev())
        _lib.update_dict(tt(W, dt_), tt(A, dt_), tt(B, dt_), out)
        assert per_atom(out.cpu().numpy().astype(np.float64), O.update_dict(W, A, B)) < tol
    # projected-gradient coder with a Gram beyond shared memory (k = 300 > 238): read through L1/L2
    d, k, n = 64, 300, 40
    Wp = rng.random((d, k)); Xp = rng.random((d, n)); H0 = rng.random((k, n))
    H = update_code_within_radius(Xp, Wp, H0=H0, r=None, alpha=0.5, sub_iter=3, stopping_diff=0.0, precision="fp64")
    assert rel(H, O.update_code_within_radius(Xp, Wp, H0.copy(), r=None, alpha=0.5, sub_iter=3, stopping_diff=0.0)) < 1e-10


# ---------------------------------------------------------------------------------------------- CUDA-graph step, narrow storage
def test_graph_replayed_step_is_bitwise_the_stream_schedule():
    """OnmfEngine(graph=True): from the third step on the whole step is one CUDA graph launch (onmf_step_graph); state and
    codes must be bit-identical to the two-stream schedule, in both precisions, on the SIMT and the tensor-core path."""
    rng = np.random.default_rng(9)
    for (d, k, n) in ((100, 25, 700), (64, 32, 515)):
        X = rng.random((n, d)); W0 = rng.random((d, k))
        for dt_ in (torch.float32, torch.float64):
            res = []
            for graph in (True, False):
                l0 = _lib.launch_count()
                eng = OnmfEngine(d, k, alpha=0.7, dtype=dt_, device=dev(), graph=graph)
                assert eng.graph == graph
                eng.set_state(W0)
                Xt = tt(X, dt_)
                H = None
                for t in range(1, 10):
                    H = eng.step(Xt, float(t)).clone()
                    if t == 5:
                        eng.step(Xt[:0], 5.5)                    # another key in between (empty shard): falls back / new graph
                W, A, B, _ = eng.state()
                torch.cuda.synchronize()
                res.append((H, W.clone(), A.clone(), B.clone(), eng._plan.graph_steps(), eng.launches - l0))
            for a, b in zip(res[0][:4], res[1][:4]):
                assert torch.equal(a, b)
            assert res[0][4] >= 5 and res[1][4] == 0                 # replays really happened
            assert res[0][5] == res[1][5]                            # same kernels per step either way


def test_narrow_storage_step_host_matches_fp32_stream():
    """uint8 / float16 host minibatches through OnmfEngine.step_host: widened on the device (x/255 for uint8), results equal
    the fp32 stream of the same values bit for bit."""
    rng = np.random.default_rng(10)
    d, k, n = 64, 32, 1000
    X8 = rng.integers(0, 256, size=(n, d), dtype=np.uint8)
    W0 = rng.random((d, k))
    Xf = torch.from_numpy(X8.astype(np.float32)) * np.float32(1.0 / 255.0)
    outs = []
    for host in (torch.from_numpy(X8).pin_memory(), Xf.pin_memory()):
        eng = OnmfEngine(d, k, alpha=0.5, dtype=torch.float32, device=dev())
        eng.set_state(W0)
        for t in (1, 2, 3, 4):
            H = eng.step_host(host, float(t)).clone()
        W, A, B, _ = eng.state()
        torch.cuda.synchronize()
        outs.append((H, W.clone(), A.clone()))
    for a, b in zip(*outs):
        assert torch.equal(a, b)
    x16 = torch.from_numpy(rng.random((n, d)).astype(np.float16))
    hi, lo = torch.empty(n, d, device=dev()), torch.empty(n, d, device=dev())
    _lib.widen(x16.to(dev()), 1.0, hi, lo)
    assert torch.equal(hi + lo, x16.to(dev()).float())
    wide = torch.empty(n, d, device=dev())
    _lib.widen(torch.from_numpy(X8).to(dev()), 1.0 / 255.0, wide)
    assert torch.equal(wide.cpu(), Xf)


# ---------------------------------------------------------------------------------------------- fused tensor-core products
@pytest.mark.parametrize("n,d,k,n_pool", [(256, 64, 64, 300), (300, 128, 96, 300), (1000, 400, 100, 1500), (4096, 1024, 256, 5000),
                                           (513, 300, 52, 700), (33, 32, 32, 40), (20000, 256, 128, 20000)])
def test_fused_tensor_core_products_vs_fp64(n, d, k, n_pool):
    """onmf_cov_fused_tc / onmf_surrogate_fused_tc (minibatch gathered by index and split to TF32 hi/lo inside the kernels)
    against float64, same 2e-5 bar as the pre-split kernels; the narrow storage formats; the fused blend; determinism."""
    g = torch.Generator(device=dev()); g.manual_seed(n + d + k)
    pool = torch.rand(n_pool, d, device=dev(), generator=g)
    idx = torch.randint(0, n_pool, (n,), device=dev(), generator=g)
    W = torch.rand(d, k, device=dev(), generator=g)
    H = torch.rand(n, k, device=dev(), generator=g) * (torch.rand(n, k, device=dev(), generator=g) < 0.2)
    assert _lib.fused_tc_supported(k, d)
    Wh, Wl = torch.empty_like(W), torch.empty_like(W)
    _lib.split_tf32(W, Wh, Wl)
    relt = lambda a, b: float((a.double() - b).norm() / b.norm())
    ws = torch.empty(_lib.surrogate_fused_tc_workspace(n, k, d), dtype=torch.uint8, device=dev())
    for use_idx in (True, False):
        ii = idx if use_idx else None
        nn = n if use_idx else min(n, n_pool)
        Xd = (pool[idx] if use_idx else pool[:nn]).double()
        Hn = H[:nn].contiguous()
        Ct = torch.full((nn, k), float("nan"), device=dev())
        _lib.cov_fused_tc(pool, ii, nn, Wh, Wl, Ct)
        assert relt(Ct, Xd @ W.double()) < 2e-5, (use_idx, relt(Ct, Xd @ W.double()))
        P = torch.full((k, k + d), float("nan"), device=dev())
        _lib.surrogate_fused_tc(Hn, pool, ii, nn, d, P, ws)
        Hd = Hn.double()
        assert relt(P[:, :k], Hd.T @ Hd) < 2e-5 and relt(P[:, k:], Hd.T @ Xd) < 2e-5
        P2 = torch.empty_like(P)
        _lib.surrogate_fused_tc(Hn, pool, ii, nn, d, P2, ws)
        assert torch.equal(P, P2)                                    # deterministic
        A = torch.rand(k, k, device=dev(), generator=g); B = torch.rand(k, d, device=dev(), generator=g)
        A2, B2 = A.clone(), B.clone()
        _lib.surrogate_fused_tc(Hn, pool, ii, nn, d, None, ws, blend=(0.25, A2, B2))
        assert torch.allclose(A2, 0.75 * A + 0.25 * P[:, :k], rtol=1e-6, atol=1e-6) and torch.allclose(B2, 0.75 * B + 0.25 * P[:, k:], rtol=1e-6, atol=1e-6)
    # narrow storage: uint8 (x / 255) and float16 pools give exactly what the widened fp32 pool gives
    p8 = torch.randint(0, 256, (n_pool, d), dtype=torch.uint8, device=dev(), generator=g)
    pf = p8.float() * np.float32(1.0 / 255.0)
    C8, Cf = torch.empty(n, k, device=dev()), torch.empty(n, k, device=dev())
    _lib.cov_fused_tc(p8, idx, n, Wh, Wl, C8, scale=1.0 / 255.0); _lib.cov_fused_tc(pf, idx, n, Wh, Wl, Cf)
    assert torch.equal(C8, Cf)
    P8, Pf = torch.empty(k, k + d, device=dev()), torch.empty(k, k + d, device=dev())
    _lib.surrogate_fused_tc(H, p8, idx, n, d, P8, ws, scale=1.0 / 255.0); _lib.surrogate_fused_tc(H, pf, idx, n, d, Pf, ws)
    assert torch.equal(P8, Pf)
    p16 = torch.rand(n_pool, d, device=dev(), generator=g).half()
    _lib.cov_fused_tc(p16, idx, n, Wh, Wl, C8); _lib.cov_fused_tc(p16.float(), idx, n, Wh, Wl, Cf)
    assert torch.equal(C8, Cf)
    # an index outside the pool poisons its row (like the K1 gather), never reads out of bounds
    bad = idx.clone(); bad[0] = n_pool + 5
    _lib.cov_fused_tc(pool, bad, n, Wh, Wl, Cf)
    assert torch.isnan(Cf[0]).all() and not torch.isnan(Cf[1:]).any()


def test_minibatch_by_reference_engine_matches_presplit_engine(monkeypatch, golden_dir):
    """The production fp32 step with the minibatch passed by reference (gemm_fused.cu: gather + TF32 split inside the
    tensor-core kernels, blend fused into the reduction) against the pre-split tensor-core kernels and the golden run."""
    g = load(golden_dir, "cfg4_ising_pm1")
    X, W0 = g["X"], g["W0"]
    pool = tt(X.T, torch.float32)
    outs = []
    for fused_tc in ("1", "0"):
        monkeypatch.setenv("ONMF_B200_FUSED_TC", fused_tc)
        eng = OnmfEngine(400, 100, alpha=1.0, dtype=torch.float32, device=dev(), collect_stats=True)
        assert eng.use_tc and eng.fused_tc == (fused_tc == "1")
        eng.set_state(W0)
        for i in range(int(g["n_steps"])):
            idx = torch.from_numpy(g["idx"][i].astype(np.int64)).to(dev())
            H = eng.step_pool(pool, idx, float(i + 1))
            if i > 0:
                assert rel(H.cpu().numpy().T, g["H_%d" % i]) < CODE_TOL_FP32
        W, A, B, _ = eng.state()
        torch.cuda.synchronize()
        outs.append((W.cpu().numpy().astype(np.float64), A.cpu().numpy().astype(np.float64)))
        assert per_atom(outs[-1][0], g["W_final"]) < ATOM_TOL_FP32
        if fused_tc == "1":
            assert eng.Xhi is None and eng.Hhi is None          # no hi/lo copies of the minibatch or the codes exist
    assert per_atom(outs[0][0], outs[1][0]) < 5e-4 and rel(outs[0][1], outs[1][1]) < 1e-4


def test_fast_tier_matches_general_kernel():
    """csrc/lars_fast.cuh (the warp-uniform first tier of the fp32 coder for k > 64) against the general kernel on the same
    covariances: learned unit-norm dictionaries (clean paths, <= 64 active atoms), a raw U[0,1) dictionary (most columns
    outgrow the 64 slots and are handed on), alpha = 0 (long paths, degenerate tails), k < 256 (padded lanes) and the
    k <= 512 class."""
    rng = np.random.default_rng(21)
    def run(G64, Ct, d, alpha, fast):
        n, k = Ct.shape
        Ht = torch.full((n, k), float("nan"), device=dev())
        ws = torch.zeros(_lib.lasso_lars_workspace(torch.float32, k, n), dtype=torch.uint8, device=dev())
        stats = torch.zeros(8, dtype=torch.int64, device=dev())
        saved = _lib.get_option(_lib.OPT_LARS_FAST_TIER)
        _lib.set_option(_lib.OPT_LARS_FAST_TIER, fast)
        try:
            _lib.lasso_lars(G64, Ct, d, alpha, Ht, ws, stats=stats)
            torch.cuda.synchronize()
        finally:
            _lib.set_option(_lib.OPT_LARS_FAST_TIER, saved)
        return Ht, stats.cpu().numpy()
    assert _lib.get_option(_lib.OPT_LARS_FAST_TIER) == 1                 # the default
    for (d, k, n, alpha, unit) in [(1024, 256, 3000, 1.0, True), (1024, 256, 300, 1.0, False), (256, 200, 500, 0.0, True),
                                   (512, 160, 700, 0.3, True), (300, 384, 400, 0.5, True),
                                   # 64 < k <= 128: the shared-memory-Gram form of the fast tier (32 slots)
                                   (400, 100, 3000, 1.0, True), (200, 128, 500, 0.2, True), (300, 70, 300, 0.0, True),
                                   (400, 100, 200, 1.0, False)]:
        W = rng.random((d, k))
        if unit:
            W /= np.linalg.norm(W, axis=0)
        X = rng.random((n, d))
        Wt = tt(W, torch.float32)
        G64 = (Wt.double().T @ Wt.double()).contiguous()
        G64 = ((G64 + G64.T) / 2).contiguous()
        Ct = (tt(X, torch.float32) @ Wt).contiguous()
        H1, s1 = run(G64, Ct, d, alpha, 1)
        H0, s0 = run(G64, Ct, d, alpha, 0)
        assert not torch.isnan(H1).any() and not torch.isnan(H0).any()   # every column written by some tier
        assert s1[0] == n and s0[0] == n, (s1, s0)                       # columns finished
        assert torch.equal(H1, H0), (d, k, n, alpha, float((H1 - H0).abs().max()), int((H1 != H0).any(1).sum()))


def test_fast_tier_edge_columns():
    """Columns that leave the clean path or stop at once, through the fast tier and through the general kernel: an all-zero
    and an all-negative covariance row (empty code), alpha above every covariance, exact ties from a duplicated atom
    (degenerate pivot: handed to the general tier), max_iter = 1 and 3 (every column handed on), a tiny alpha.  Same bits,
    every column finished, no hang."""
    rng = np.random.default_rng(33)
    for (d, k) in ((256, 200), (160, 100)):
        n = 64
        W = rng.random((d, k)); W /= np.linalg.norm(W, axis=0)
        W[:, 7] = W[:, 3]                                             # two identical atoms
        X = rng.random((n, d))
        X[0] = 0.0
        Wt = tt(W, torch.float32)
        G64 = (Wt.double().T @ Wt.double()).contiguous()
        G64 = ((G64 + G64.T) / 2).contiguous()
        Ct = (tt(X, torch.float32) @ Wt).contiguous()
        Ct[1] = -Ct[1]                                                # nothing is positively correlated
        Ct[2] = 0.0
        for alpha, max_iter in ((1.0, 1000), (1e4, 1000), (1e-3, 1000), (0.5, 1), (0.5, 3)):
            outs = []
            for fast in (1, 0):
                Ht = torch.full((n, k), float("nan"), device=dev())
                ws = torch.zeros(_lib.lasso_lars_workspace(torch.float32, k, n), dtype=torch.uint8, device=dev())
                stats = torch.zeros(8, dtype=torch.int64, device=dev())
                saved = _lib.get_option(_lib.OPT_LARS_FAST_TIER)
                _lib.set_option(_lib.OPT_LARS_FAST_TIER, fast)
                try:
                    _lib.lasso_lars(G64, Ct, d, alpha, Ht, ws, max_iter=max_iter, stats=stats)
                    torch.cuda.synchronize()
                finally:
                    _lib.set_option(_lib.OPT_LARS_FAST_TIER, saved)
                assert not torch.isnan(Ht).any() and int(stats[0]) == n
                outs.append(Ht)
            assert torch.equal(outs[0], outs[1]), (d, k, alpha, max_iter)
            assert float(outs[0][0].abs().max()) == 0.0 and float(outs[0][1].abs().max()) == 0.0 and float(outs[0][2].abs().max()) == 0.0
            if alpha == 1e4:
                assert float(outs[0].abs().max()) == 0.0
            assert float(outs[0].min()) >= 0.0


def test_fast_tier_small_dictionaries():
    """k <= 64 on small minibatches: one column per warp in the fast kernel (2 atoms per lane) against the general kernel
    (4 / 2 columns per warp).  The slots sit on different lanes, so the FP64 sums of a join are taken in a different order:
    agreement to rounding, not bit for bit; plus the C oracle on the same covariances."""
    rng = np.random.default_rng(44)
    for (d, k, n, alpha) in [(100, 25, 1000, 1.0), (300, 49, 3000, 1.0), (441, 25, 500, 0.5), (64, 20, 300, 0.0), (50, 33, 100, 0.3),
                             (120, 64, 700, 1.0), (40, 32, 200, 0.0), (30, 7, 64, 0.1)]:
        W = rng.random((d, k)); W /= np.linalg.norm(W, axis=0)
        X = rng.random((n, d))
        if n > 2:
            X[1] = 0.0
        Wt = tt(W, torch.float32)
        G64 = (Wt.double().T @ Wt.double()).contiguous()
        G64 = ((G64 + G64.T) / 2).contiguous()
        Ct = (tt(X, torch.float32) @ Wt).contiguous()
        outs = []
        for fast in (1, 0):
            Ht = torch.full((n, k), float("nan"), device=dev())
            ws = torch.zeros(_lib.lasso_lars_workspace(torch.float32, k, n), dtype=torch.uint8, device=dev())
            stats = torch.zeros(8, dtype=torch.int64, device=dev())
            saved = _lib.get_option(_lib.OPT_LARS_FAST_TIER)
            _lib.set_option(_lib.OPT_LARS_FAST_TIER, fast)
            try:
                _lib.lasso_lars(G64, Ct, d, alpha, Ht, ws, stats=stats)
                torch.cuda.synchronize()
            finally:
                _lib.set_option(_lib.OPT_LARS_FAST_TIER, saved)
            assert not torch.isnan(Ht).any() and int(stats[0]) == n, (d, k, n, alpha, fast, stats.cpu().numpy())
            outs.append(Ht.cpu().numpy().astype(np.float64))
        assert rel(outs[0], outs[1]) < 2e-5, (d, k, n, alpha, rel(outs[0], outs[1]))
        assert (outs[0] >= 0).all()
        # the oracle on the SAME fp32 covariances and the FP64 Gram
        cs = Ct.cpu().numpy().astype(np.float64)
        Gn = G64.cpu().numpy()
        Href = np.stack([c_oracle_lars_single(Gn, cs[i], alpha, d) for i in range(min(n, 60))])
        assert rel(outs[0][:Href.shape[0]], Href) < 2e-3, (d, k, n, alpha)


def test_spectral_norm_kernel():
    """onmf_spectral_norm (FP64 Gram + largest eigenvalue by repeated squaring) against numpy's SVD: generic, rank-one,
    repeated and nearly repeated top singular values, a zero matrix, one column; fp32 and fp64 inputs; and n in {1024, 1040,
    5000, 1e5} x k in {1, 2, 64, 65, 256, 512}, where the FP64 Gram takes its 16-way split over n with a partial last chunk.
    Every case within the header's 1e-5 of the norm of the dtype-rounded matrix."""
    rng = np.random.default_rng(55)
    cases = []
    cases.append(rng.random((700, 25)))
    cases.append(rng.standard_normal((64, 100)))
    cases.append(np.outer(rng.random(300), rng.random(49)))                       # rank one
    Q, _ = np.linalg.qr(rng.standard_normal((200, 30)))
    cases.append(Q @ np.diag([3.0, 3.0, 3.0] + [1.0] * 27))                       # triple top singular value
    cases.append(Q @ np.diag([2.0, 2.0 * (1 - 1e-4), 2.0 * (1 - 1e-5)] + list(np.linspace(1.9, 0.1, 27))))   # near-degenerate
    cases.append(np.zeros((50, 7)))
    cases.append(rng.random((1000, 1)))
    cases.append(rng.random((3, 238)) * 1e-3)
    shapes = [(n, k) for n in (1024, 1040, 5000, 100000) for k in (1, 2, 64, 65, 256, 512)]
    for M in cases + shapes:
        for dt_ in (torch.float64, torch.float32):
            if isinstance(M, tuple):
                n, k = M
                Mr = rng.random((n, k)) - 0.3 * (k > 1) * rng.random(k)                 # tilted: a dominant but not lone top
            else:
                n, k = M.shape
                Mr = M
            Mr = Mr.astype(np.float32 if dt_ == torch.float32 else np.float64).astype(np.float64)
            ref = math.sqrt(max(np.linalg.eigvalsh(Mr.T @ Mr)[-1], 0.0)) if n > 4 * k else np.linalg.norm(Mr, 2)
            out = torch.full((1,), float("nan"), dtype=torch.float64, device=dev())
            ws = torch.empty(_lib.spectral_norm_workspace(n, k), dtype=torch.uint8, device=dev())
            _lib.spectral_norm(tt(Mr, dt_), out, ws)
            got = float(out[0])
            assert abs(got - ref) <= 1e-5 * ref or got == ref == 0.0, (n, k, dt_, got, ref)


# ---------------------------------------------------------------------------------------------- K1 vector forms, batched PGD
def test_vector_gathers_equal_scalar_forms():
    """The 16-byte forms of the patch gather / transpose (taken whenever shapes and alignment allow) move the same bytes
    as the scalar kernels: bit-equal to plain indexing, for fp32 and fp64, gray and colour, incl. poisoned patches."""
    g = torch.Generator(device=dev()); g.manual_seed(5)
    for dt in (torch.float32, torch.float64):
        # (the last two shapes have more than 1024 sixteen-byte pieces per patch: the flat vector kernel instead of the tiled one)
        for (H, Wd, C, p) in ((40, 37, 1, 10), (33, 41, 3, 10), (64, 64, 1, 20), (19, 23, 3, 3), (50, 50, 2, 7), (16, 16, 1, 16),
                              (40, 40, 1, 32), (70, 70, 1, 46), (80, 80, 1, 66)):
            img = torch.rand(H, Wd, C, dtype=dt, device=dev(), generator=g)
            n = 777
            co = torch.stack([torch.randint(0, H - p + 1, (n,), device=dev(), generator=g),
                              torch.randint(0, Wd - p + 1, (n,), device=dev(), generator=g)], 1).to(torch.int32)
            co[5] = torch.tensor([H - p + 1, 0]); co[6] = torch.tensor([-1, 0]); co[7] = torch.tensor([0, Wd - p + 1])
            co = co.contiguous()
            d = p * p * C
            for ld in (d, d + 4, d + 1):                       # pitch d + 1 breaks the 16-byte pitch -> scalar kernel
                buf = torch.zeros(n, ld, dtype=dt, device=dev())
                out = buf[:, :d]
                _lib.gather_patches(img, co, p, out)
                ok = torch.ones(n, dtype=torch.bool, device=dev()); ok[5:8] = False
                ii = torch.nonzero(ok).flatten()
                a, b = co[ii, 0].long(), co[ii, 1].long()
                rr = torch.arange(p, device=dev())
                ref = img[(a[:, None, None] + rr[None, :, None]), (b[:, None, None] + rr[None, None, :])].reshape(len(ii), d)
                assert torch.equal(out[ii], ref), (dt, H, Wd, C, p, ld)
                assert torch.isnan(out[5:8]).all()
                if ld > d:
                    assert float(buf[:, d:].abs().max()) == 0.0   # nothing written beyond a patch's d features
    for (r, c) in ((64, 128), (68, 132), (4, 4), (1024, 300), (300, 1024), (35, 77), (36, 77), (200, 8)):
        for ti in (torch.float32, torch.float64):
            for to in (torch.float32, torch.float64):
                src = torch.rand(r, c, dtype=ti, device=dev(), generator=g)
                dst = torch.empty(c, r, dtype=to, device=dev())
                _lib.transpose(src, dst)
                assert torch.equal(dst, src.T.to(to)), (r, c, ti, to)


@pytest.mark.parametrize("k", [5, 12, 25, 32])
def test_thread_per_sample_pgd_equals_warp_per_sample(k):
    """pgd_code_columns takes one thread per sample for k <= 32 on large batches; same iteration and stopping test as the
    warp-per-sample kernel (and the oracle's update_code_within_radius per column), sums in index order."""
    rng = np.random.default_rng(k)
    d, n = 40, 16 * 160 + 37                                    # above the 16 * SMs switch on a 148-SM part
    W = rng.random((d, k)); W /= np.maximum(1.0, np.linalg.norm(W, axis=0))
    X = rng.random((d, n)); H0 = rng.random((k, n))
    H0[:, 3] = 0.0                                              # zero start: dist = x / 0 on the first sweep
    for dt, tol in ((torch.float64, 1e-12), (torch.float32, 2e-5)):
        Wd = tt(W, dt); Xt = tt(X.T, dt)
        G = torch.empty(k, k, dtype=dt, device=dev()); Ct = torch.empty(n, k, dtype=dt, device=dev())
        _lib.gram(Wd, G); _lib.cov(Xt, Wd, Ct)
        for sub_iter, stop in ((10, 0.01), (3, 0.0), (25, 0.05)):
            big = tt(H0.T, dt)
            _lib.pgd_code_columns(G, Ct, 0.7, sub_iter, stop, big)                 # thread per sample
            small = tt(H0.T, dt)
            for lo in range(0, n, 500):                                            # chunks below the switch: warp per sample
                _lib.pgd_code_columns(G, Ct[lo:lo + 500], 0.7, sub_iter, stop, small[lo:lo + 500])
            a, b = big.cpu().numpy().astype(np.float64), small.cpu().numpy().astype(np.float64)
            fin = np.isfinite(b).all(axis=1)
            assert np.array_equal(fin, np.isfinite(a).all(axis=1))
            # a column whose stopping test sits within rounding of the threshold may take one sweep more or less
            bad = np.linalg.norm(a[fin] - b[fin], axis=1) > tol * np.maximum(np.linalg.norm(b[fin], axis=1), 1e-30)
            assert bad.sum() <= (0 if dt == torch.float64 else 2), (k, dt, sub_iter, int(bad.sum()))
        if dt == torch.float64:
            ref = np.stack([O.update_code_within_radius(X[:, j:j + 1], W, H0[:, j:j + 1].copy(), None, 0.7, 25, 0.05)[:, 0]
                            for j in range(0, 64) if j != 3], 0)
            got = np.delete(a[:64], 3, axis=0)
            assert rel(got, ref) < 1e-10


def test_sklearn_order_patch_helpers_one_shot_reconstruction():
    """the drivers' one-shot reconstruction (image_reconstruction.py:335-357, ising_reconstruction.py:179-201):
    extract_patches_2d(data, (k, k)) -> sparse_code -> np.dot(W, code).T -> reconstruct_from_patches_2d, against sklearn's
    own two functions and numpy on the same code."""
    from sklearn.feature_extraction.image import extract_patches_2d, reconstruct_from_patches_2d
    from onmf_ontf_ndl_b200 import patches, reconstruct_from_patches_2d as recon_b200
    rng = np.random.default_rng(11)
    for shape, k in (((23, 31), 5), ((18, 20, 3), 4)):
        img = rng.random(shape)
        ref = extract_patches_2d(img, (k, k))
        X = patches.extract_patches_2d(img, k, precision="fp64")
        assert np.array_equal(X, ref.reshape(len(ref), -1).T)
        r = 7
        W = rng.random((X.shape[0], r)); W /= np.linalg.norm(W, axis=0)
        code = Online_NMF(X, n_components=r, iterations=1, batch_size=10, alpha=0.1, precision="fp64").sparse_code(X, W)
        assert rel(code, c_oracle.sparse_code(X, W, 0.1)) < 1e-9
        pr = np.dot(W, code).T.reshape((len(ref),) + ref.shape[1:])
        want = reconstruct_from_patches_2d(pr, shape)
        assert rel(recon_b200(pr, shape[:2], precision="fp64"), want) < 1e-13
        assert rel(recon_b200(W, shape, code=code, precision="fp64"), want) < 1e-13
        assert rel(recon_b200(W, shape, code=code), want) < 1e-5
    with pytest.raises(ValueError):
        recon_b200(pr[:-1], shape[:2])
