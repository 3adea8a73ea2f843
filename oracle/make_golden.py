"""Generate tests/golden/*.npz by running the UNMODIFIED reference.

TEST INFRASTRUCTURE ONLY.  Needs a checkout of the reference, named by ONMF_REFERENCE_ROOT:

    ONMF_REFERENCE_ROOT=<reference checkout> python oracle/make_golden.py

Every fixture holds the inputs (X or the patch tensor, W0, the minibatch index sequence,
alpha, history...) and the per-step outputs (H, A, B, W) of the reference's own
`Online_NTF.step` (src/ontf.py:117-154) / `Online_NMF.step` (src/onmf.py:119-167), recorded
through a subclass that only wraps `step` -- no reference arithmetic is re-implemented here.
The numpy global RNG is seeded before each run; the same stream is replayed with a private
RandomState to recover W0 (src/ontf.py:213) and the per-step `randint` draws (src/ontf.py:230).

Configs are cut-down versions of BASELINE.json's cfg1..cfg5 (same d, k, data kind; smaller
minibatch / fewer steps so the fixtures stay small and the CPU suite fast).
"""
import os
import sys
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from oracle.ref_loader import load_reference, REFERENCE_ROOT  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")
warnings.filterwarnings("ignore")


def _renoir(gray):
    from PIL import Image
    img = Image.open(os.path.join(REFERENCE_ROOT, "Data", "renoir", "0.jpg"))
    if gray:
        img = img.convert("L")   # image_reconstruction.py:85
    return np.asarray(img) / 255  # image_reconstruction.py:88


def _coords(rs, shape, k, n):
    # interleaved draws like image_reconstruction.py:184-186 (np.random.choice(x - k))
    out = np.empty((n, 2), dtype=np.int64)
    for i in range(n):
        out[i, 0] = rs.choice(shape[0] - k)
        out[i, 1] = rs.choice(shape[1] - k)
    return out


def run_ntf(ontf, X3, k, steps, batch, alpha, seed, mode=0, joint=False, beta=None,
            ini=None, history=0, subsample=True):
    """Runs reference Online_NTF.train_dict_single and records every step."""
    trace = []

    class Rec(ontf.Online_NTF):
        def step(self, X, A, B, W, t):
            out = super().step(X, A, B, W, t)
            trace.append(dict(X=np.array(X), H=out[0].T.copy(), A=out[1].copy(), B=out[2].copy(),
                              W=out[3].copy(), t=float(t)))
            return out

    kw = dict(n_components=k, iterations=steps + 1, batch_size=batch, alpha=alpha, mode=mode,
              learn_joint_dict=joint, beta=beta, history=history, subsample=subsample)
    if ini is not None:
        kw.update(ini_dict=ini[0], ini_A=ini[1], ini_B=ini[2])
    np.random.seed(seed)
    m = Rec(X3, **kw)
    W, A, B, code = m.train_dict_single()
    # replay RNG
    rs = np.random.RandomState(seed)
    U = np.reshape(np.moveaxis(X3, mode, 0), (X3.shape[mode], -1))
    Xm = U.T if joint else U
    d, n = Xm.shape
    W0 = rs.rand(d, k) if ini is None else np.array(ini[0])
    idx = []
    for i in range(steps):
        if subsample:
            ii = rs.randint(n, size=batch)
            assert np.array_equal(Xm[:, ii], trace[i]["X"]), "RNG replay mismatch"
        else:
            ii = np.arange(n)
        idx.append(ii)
    return dict(Xm=Xm, W0=W0, idx=np.array(idx), trace=trace, W=W, A=A, B=B,
                history_out=float(m.history))


def pack(res, **extra):
    d = dict(X=res["Xm"], W0=res["W0"], idx=res["idx"], W_final=res["W"], A_final=res["A"],
             B_final=res["B"], history_out=res["history_out"])
    for i, tr in enumerate(res["trace"]):
        for key in ("H", "A", "B", "W"):
            d["%s_%d" % (key, i)] = tr[key]
        d["t_%d" % i] = tr["t"]
    d["n_steps"] = len(res["trace"])
    d.update(extra)
    return d


def main(which=None, out_dir=None):
    """which: iterable of fixture names (file stems) to write, None = all.  The data draws of every section always run
    (they share one RandomState stream); only the selected sections run the reference."""
    global OUT
    onmf, ontf = load_reference()
    if out_dir is not None:
        OUT = out_dir
    os.makedirs(OUT, exist_ok=True)
    want = (lambda name: True) if which is None else (lambda name: name in set(which))
    rs = np.random.RandomState(1234)

    # ---- cfg1: Renoir gray 10x10 patches, d=100, k=25, alpha=1 ------------------------
    img = _renoir(gray=True)
    crop = img[100:260, 80:260].copy()                       # 160 x 180 crop kept as a gather fixture
    co = _coords(rs, crop.shape, 10, 1500)
    X = np.stack([crop[a:a + 10, b:b + 10].reshape(-1) for a, b in co], axis=1)
    if want("cfg1_renoir_gray") or want("cfg1_renoir_gray_epoch2"):
        r1 = run_ntf(ontf, X[:, :, None], 25, steps=8, batch=300, alpha=1, seed=11)
        if want("cfg1_renoir_gray"):
            np.savez_compressed(os.path.join(OUT, "cfg1_renoir_gray.npz"),
                                **pack(r1, alpha=1.0, img=crop, coords=co, patch=10))
    if want("cfg1_renoir_gray_epoch2"):
        # chained epoch: carry (W, A, B, history) like image_reconstruction.py:300-309
        r1b = run_ntf(ontf, X[:, :, None], 25, steps=4, batch=300, alpha=1, seed=12,
                      ini=(r1["W"], r1["A"], r1["B"]), history=r1["history_out"])
        np.savez_compressed(os.path.join(OUT, "cfg1_renoir_gray_epoch2.npz"),
                            **pack(r1b, alpha=1.0, A0=r1["A"], B0=r1["B"], history_in=r1["history_out"]))
    if want("cfg1_alphaNone_beta_full"):
        # alpha=None (=> 2, src/ontf.py:79-81), beta=0.75, all columns (subsample=False)
        r1c = run_ntf(ontf, X[:, :200, None], 25, steps=3, batch=200, alpha=None, seed=13, beta=0.75,
                      subsample=False)
        np.savez_compressed(os.path.join(OUT, "cfg1_alphaNone_beta_full.npz"),
                            **pack(r1c, alpha=2.0, beta=0.75))
    if want("cfg1_alpha0"):
        # alpha=0 (network_reconstruction_nx.py:468 regime; ~all columns on the final LARS segment)
        r1d = run_ntf(ontf, X[:, :, None], 25, steps=3, batch=200, alpha=0, seed=14)
        np.savez_compressed(os.path.join(OUT, "cfg1_alpha0.npz"), **pack(r1d, alpha=0.0))

    # ---- cfg2: Renoir colour, tensor (k*k, 3, N), mode=2 joint => d=300, k=49 ----------
    imgc = _renoir(gray=False)
    cropc = imgc[100:200, 80:200, :].copy()
    coc = _coords(rs, cropc.shape, 10, 600)
    T = np.stack([cropc[a:a + 10, b:b + 10, :].reshape(100, 3) for a, b in coc], axis=2)
    if want("cfg2_renoir_color_tensor"):
        r2 = run_ntf(ontf, T, 49, steps=5, batch=200, alpha=1, seed=21, mode=2, joint=True)
        np.savez_compressed(os.path.join(OUT, "cfg2_renoir_color_tensor.npz"),
                            **pack(r2, alpha=1.0, img=cropc, coords=coc, patch=10, T=T, mode=2, joint=1))

    # ---- cfg3: binary 21x21 motif-adjacency-like patches, d=441, k=25 -------------------
    n3 = 800
    P = np.zeros((21, 21, n3))
    for j in range(n3):
        # path motif (i,i+1 adjacent) + random extra symmetric edges, like
        # network_reconstruction_nx.py:302-305 patches of a sparse graph
        Aj = np.zeros((21, 21))
        ii = np.arange(20)
        Aj[ii, ii + 1] = 1
        Aj[ii + 1, ii] = 1
        extra = rs.rand(21, 21) < 0.04
        extra = np.triu(extra, 2)
        Aj = np.maximum(Aj, extra + extra.T)
        P[:, :, j] = Aj
    X3 = P.reshape(441, n3)
    X3[:, 5] = 0.0                                            # an all-zero column (empty patch)
    if want("cfg3_binary_motif"):
        r3 = run_ntf(ontf, X3[:, :, None], 25, steps=4, batch=300, alpha=1, seed=31)
        np.savez_compressed(os.path.join(OUT, "cfg3_binary_motif.npz"), **pack(r3, alpha=1.0))

    # ---- cfg4: +-1 Ising-like 20x20 spin patches, d=400, k=100 (X may be negative) -----
    lat = rs.choice([-1.0, 1.0], size=(60, 60))
    for _ in range(3):                                         # a few smoothing sweeps -> domains
        nb = np.roll(lat, 1, 0) + np.roll(lat, -1, 0) + np.roll(lat, 1, 1) + np.roll(lat, -1, 1)
        flip = rs.rand(60, 60) < 0.7
        lat = np.where(flip & (nb != 0), np.sign(nb), lat)
    co4 = _coords(rs, lat.shape, 20, 500)
    X4 = np.stack([lat[a:a + 20, b:b + 20].reshape(-1) for a, b in co4], axis=1)
    if want("cfg4_ising_pm1"):
        r4 = run_ntf(ontf, X4[:, :, None], 100, steps=4, batch=200, alpha=1, seed=41)
        np.savez_compressed(os.path.join(OUT, "cfg4_ising_pm1.npz"),
                            **pack(r4, alpha=1.0, img=lat, coords=co4, patch=20))

    # ---- cfg5: synthetic U[0,1), d=1024, k=256 ------------------------------------------
    # kept light: X and W0 are regenerated from seeds by the tests (RandomState(5).rand(1024,160),
    # RandomState(51).rand(1024,256)); per-step H in float64, final W/A/B in float32.
    if want("cfg5_synthetic"):
        X5 = np.random.RandomState(5).rand(1024, 160)
        r5 = run_ntf(ontf, X5[:, :, None], 256, steps=3, batch=48, alpha=1, seed=51)
        d5 = dict(x_seed=5, w0_seed=51, idx=r5["idx"], alpha=1.0, n_steps=3,
                  history_out=r5["history_out"], W_final=r5["W"].astype(np.float32),
                  A_final=r5["A"].astype(np.float32), B_final=r5["B"].astype(np.float32))
        for i, tr in enumerate(r5["trace"]):
            d5["H_%d" % i] = tr["H"]
            d5["t_%d" % i] = tr["t"]
        np.savez_compressed(os.path.join(OUT, "cfg5_synthetic.npz"), **d5)

    # ---- shipped src/onmf.py: PGD coder + step, RNG-replayed H0 --------------------------
    np.random.seed(61)
    Xs = X[:, :120]
    Ws = np.random.rand(100, 25)
    H0 = np.random.rand(25, 120)
    if want("pgd_coder"):
      Hp = onmf.update_code_within_radius(Xs, Ws, H0=H0.copy(), r=None, alpha=1, sub_iter=10,
                                        stopping_diff=0.01)
      Hp_r = onmf.update_code_within_radius(Xs, Ws, H0=H0.copy(), r=0.5, alpha=0.3, sub_iter=3,
                                            stopping_diff=0.01)
      Hp_1 = onmf.update_code_within_radius(Xs[:, :1], Ws, H0=H0[:, :1].copy(), r=None, alpha=1,
                                            sub_iter=10, stopping_diff=0.01)
      np.savez_compressed(os.path.join(OUT, "pgd_coder.npz"), X=Xs, W=Ws, H0=H0, H=Hp, H_radius=Hp_r,
                          H_single=Hp_1)

    # shipped Online_NMF.train_dict (gen-3): literal behaviour incl. the aggregate re-binding
    # (src/onmf.py:217) and the random-H0 coder; RNG replay: W0, then per step idx, H0.
    if want("shipped_onmf"):
        np.random.seed(71)
        m = onmf.Online_NMF(Xs, n_components=25, iterations=4, batch_size=60, alpha=1, subsample=True)
        Wn, aggn, coden = m.train_dict()
        np.savez_compressed(os.path.join(OUT, "shipped_onmf.npz"), X=Xs, seed=71, W=Wn, A=aggn[0],
                            B=aggn[1], code=coden, history_out=float(m.history))
    # ---- reconstruction loop (image_reconstruction.py:358-406): the reference's own coder per patch, painting restated
    from oracle import onmf_oracle as O
    if want("reconstruct_color"):
        imgr = _renoir(gray=False)[200:236, 150:190, :].copy()                 # 36 x 40 x 3 crop
        np.random.seed(81)
        Wr = np.random.rand(75, 25)
        Wr /= np.linalg.norm(Wr, axis=0)
        ny, nx = len(range(0, 36 - 5, 2)), len(range(0, 40 - 5, 2))
        H0r = np.random.rand(ny * nx, 25).T                                    # same stream as one rand(r, 1) per patch
        rec, cnt, codes = O.reconstruct_image_loop(
            imgr, Wr, 5, 2, 1, 10, 0.01, H0r,
            coder=lambda patch, h0: onmf.update_code_within_radius(patch, Wr, H0=h0.copy(), r=None, alpha=1, sub_iter=10,
                                                                   stopping_diff=0.01))
        np.savez_compressed(os.path.join(OUT, "reconstruct_color.npz"), img=imgr, W=Wr, H0=H0r, recons=rec, count=cnt,
                            codes=codes, patch=5, stride=2)

    # ---- network reconstruction (network_reconstruction_nx.py:444-511): the UNMODIFIED driver method on a generated graph.
    # The constructor reads a comma edge-list file; the instance is created without it and given the attributes the
    # method uses (G, W, k1, k2, is_glauber_recons).  The two DiGraphs the method builds (running-mean weights, overlap
    # counts) are local variables: they are captured by handing the driver module a networkx proxy that remembers the
    # DiGraph instances it creates; the MCMC states by wrapping get_single_patch_glauber.  No reference line is edited.
    if want("network_recons"):
        import networkx as nx
        from oracle.ref_loader import load_reference_driver
        nrx = load_reference_driver("network_reconstruction_nx")
        Gn = nx.gnp_random_graph(40, 0.15, seed=3)
        Gn.add_edges_from((i, (i + 1) % 40) for i in range(40))              # connected: every node has neighbours
        rec_ = object.__new__(nrx.Network_Reconstructor)
        rec_.G, rec_.k1, rec_.k2 = Gn, 0, 5
        rec_.is_glauber_recons, rec_.is_glauber_dict, rec_.sample_size = True, True, 200
        np.random.seed(91)
        Bm = rec_.path_adj(0, 5)
        emb0 = rec_.tree_sample(Bm, np.random.choice(np.asarray([i for i in Gn])))
        Xn, _ = rec_.get_patches_glauber(Bm, emb0)                            # (36 x 200) training patches (:315-329)
        Wn_, _, _, _ = ontf.Online_NTF(Xn[:, :, None], 9, iterations=7, batch_size=50, alpha=1).train_dict_single()
        rec_.W = Wn_
        states = []
        orig_single = rec_.get_single_patch_glauber

        def rec_single(B, emb):
            Xp, e2 = orig_single(B, emb)
            states.append(np.array(e2).copy())
            return Xp, e2
        rec_.get_single_patch_glauber = rec_single

        class NxProxy:
            def __init__(self, real):
                self._real, self.made = real, []

            def __getattr__(self, name):
                return getattr(self._real, name)

            def DiGraph(self, *a, **k):
                g_ = self._real.DiGraph(*a, **k)
                self.made.append(g_)
                return g_
        proxy = NxProxy(nrx.nx)
        nrx.nx = proxy
        np.random.seed(92)
        Gs = rec_.reconstruct_network(recons_iter=300)
        nrx.nx = proxy._real
        Gw, Gc = proxy.made[0], proxy.made[1]
        pairs = sorted(Gw.edges)
        np.savez_compressed(os.path.join(OUT, "network_recons.npz"), graph_edges=np.asarray(sorted(Gn.edges)), n_nodes=40,
                            W=Wn_, embs=np.asarray(states), pairs=np.asarray(pairs),
                            weight=np.asarray([Gw[a][b]["weight"] for a, b in pairs]),
                            count=np.asarray([Gc[a][b]["weight"] for a, b in pairs]),
                            simple_edges=np.asarray(sorted(tuple(sorted(e)) for e in Gs.edges)), alpha=0.0)

    # ---- a reference DRIVER end to end: Image_Reconstructor_tensor.train_dict (image_reconstruction_tensor.py:220-262,
    # patch sampling :87-124, epoch chaining through ini_dict / ini_A / ini_B / history) with the reference's own
    # Online_NTF, unmodified, on a crop of Data/renoir/0.jpg saved as a lossless PNG.
    if want("driver_tensor"):
        import tempfile
        from PIL import Image
        from oracle.ref_loader import load_reference_driver
        irt = load_reference_driver("image_reconstruction_tensor")
        crop8 = np.asarray(Image.open(os.path.join(REFERENCE_ROOT, "Data", "renoir", "0.jpg")).convert("RGB"))[120:200, 90:190, :].copy()
        cwd = os.getcwd()
        with tempfile.TemporaryDirectory() as tmp:
            os.makedirs(os.path.join(tmp, "Image_dictionary"))
            Image.fromarray(crop8).save(os.path.join(tmp, "crop.png"))
            os.chdir(tmp)
            try:
                np.random.seed(95)
                drv = irt.Image_Reconstructor_tensor(path="crop.png", n_components=16, iterations=3, sub_iterations=5,
                                                     batch_size=20, num_patches=60, patch_size=6, is_color=True)
                Wd_ = drv.train_dict(mode=2, learn_joint_dict=True)
                hist = float(drv.ntf.history)
            finally:
                os.chdir(cwd)
        np.savez_compressed(os.path.join(OUT, "driver_tensor.npz"), img_u8=crop8, seed=95, n_components=16, iterations=3,
                            sub_iterations=5, batch_size=20, num_patches=60, patch_size=6, mode=2, joint=1, W=Wd_,
                            history=hist)
    print("golden fixtures written to", OUT)
    for f in sorted(os.listdir(OUT)):
        print("  %-40s %8.1f KB" % (f, os.path.getsize(os.path.join(OUT, f)) / 1024))


if __name__ == "__main__":
    main(sys.argv[1:] or None)
