"""Full-length reference runs for the fp32 production-mode bars (final dictionary per atom <= 1e-3, reconstruction
error within 0.5 %).  TEST INFRASTRUCTURE ONLY; needs a reference checkout named by ONMF_REFERENCE_ROOT.  Takes ~15
CPU-minutes.

    python oracle/make_golden_full.py [cfg1 cfg2 cfg3 cfg4]

cfg1 is BASELINE.json configs[0] at full size (Renoir gray 10x10 patches, d=100, k=25, batch 1000, alpha=1,
100 iterations); cfg2..cfg4 keep d, k and the full minibatch size at 100 / 25 / 25 iterations (the reference needs
2-3 ms per column on one core: 15 / 9 / 22 CPU-minutes).  Only seeds, the integer-valued data pool and the final
(W, A, B) + a held-out reconstruction error are stored.  cfg5 is the benchmarked shape (d=1024, k=256, synthetic
U[0,1) data regenerated from a seed by the test) at minibatch 2048 for 10 iterations, with the minibatch indices and
the reference's codes of EVERY step, so that the GPU tests can compare per-step codes on the learned (unit-norm)
dictionaries the benchmark actually runs on.  Every config draws from its own RandomState, so any subset can be
regenerated on its own (tests/test_oracle_vs_reference.py does that for cfg1).
"""
import os
import sys
import time
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from oracle.ref_loader import load_reference, REFERENCE_ROOT  # noqa: E402
from oracle import onmf_oracle as O  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")
warnings.filterwarnings("ignore")


def recon_error(W, Xe, alpha):
    H = O.sparse_code_sklearn(Xe, W, alpha)
    return float(np.linalg.norm(Xe - W @ H) / np.linalg.norm(Xe))


def run(ontf, X, k, iters, batch, alpha, seed):
    np.random.seed(seed)
    m = ontf.Online_NTF(X[:, :, None], n_components=k, iterations=iters + 1, batch_size=batch, alpha=alpha, mode=0,
                        learn_joint_dict=False)
    t = time.time()
    W, A, B, _ = m.train_dict_single()
    return W, A, B, float(m.history), time.time() - t


def main(which):
    onmf, ontf = load_reference()
    from PIL import Image
    if "cfg1" in which:
        rs = np.random.RandomState(2024)
        img = np.asarray(Image.open(os.path.join(REFERENCE_ROOT, "Data", "renoir", "0.jpg")).convert("L"))   # uint8
        co = np.stack([rs.randint(0, img.shape[0] - 10, 6000), rs.randint(0, img.shape[1] - 10, 6000)], 1)
        P8 = np.stack([img[a:a + 10, b:b + 10].reshape(-1) for a, b in co], axis=1).astype(np.uint8)      # 100 x 6000
        X = P8 / 255
        W, A, B, h, sec = run(ontf, X[:, :5000], 25, 100, 1000, 1, 101)
        np.savez_compressed(os.path.join(OUT, "full_cfg1.npz"), pool_u8=P8, n_train=5000, k=25, iters=100, batch=1000,
                            alpha=1.0, seed=101, W=W, A=A, B=B, history=h, recon=recon_error(W, X[:, 5000:5400], 1.0))
        print("cfg1 done in %.0f s" % sec, flush=True)
    if "cfg2" in which:
        rs = np.random.RandomState(2025)
        img = np.asarray(Image.open(os.path.join(REFERENCE_ROOT, "Data", "renoir", "0.jpg")))                # uint8 RGB
        co = np.stack([rs.randint(0, img.shape[0] - 10, 8400), rs.randint(0, img.shape[1] - 10, 8400)], 1)
        P8 = np.stack([img[a:a + 10, b:b + 10, :].reshape(-1) for a, b in co], axis=1).astype(np.uint8)   # 300 x 8400 (HWC)
        X = P8 / 255
        W, A, B, h, sec = run(ontf, X[:, :8000], 49, 100, 4000, 1, 102)
        np.savez_compressed(os.path.join(OUT, "full_cfg2.npz"), pool_u8=P8, n_train=8000, k=49, iters=100, batch=4000,
                            alpha=1.0, seed=102, W=W, A=A, B=B, history=h, recon=recon_error(W, X[:, 8000:8400], 1.0))
        print("cfg2 done in %.0f s" % sec, flush=True)
    if "cfg3" in which:
        rs = np.random.RandomState(2026)
        n3 = 12400
        P = np.zeros((21, 21, n3), dtype=np.uint8)
        ii = np.arange(20)
        P[ii, ii + 1, :] = 1
        P[ii + 1, ii, :] = 1
        extra = np.triu(rs.rand(21, 21, n3) < 0.04, 0)
        for j in range(n3):
            e = np.triu(extra[:, :, j], 2)
            P[:, :, j] = np.maximum(P[:, :, j], e + e.T)
        P8 = P.reshape(441, n3)
        X = P8.astype(np.float64)
        W, A, B, h, sec = run(ontf, X[:, :12000], 25, 25, 10000, 1, 103)
        np.savez_compressed(os.path.join(OUT, "full_cfg3.npz"), pool_u8=P8, n_train=12000, k=25, iters=25, batch=10000,
                            alpha=1.0, seed=103, W=W, A=A, B=B, history=h, recon=recon_error(W, X[:, 12000:12400], 1.0))
        print("cfg3 done in %.0f s" % sec, flush=True)
    if "cfg4" in which:
        rs = np.random.RandomState(2027)
        lat = rs.choice([-1.0, 1.0], size=(200, 200))
        for _ in range(4):
            nb = np.roll(lat, 1, 0) + np.roll(lat, -1, 0) + np.roll(lat, 1, 1) + np.roll(lat, -1, 1)
            flip = rs.rand(200, 200) < 0.7
            lat = np.where(flip & (nb != 0), np.sign(nb), lat)
        co = np.stack([rs.randint(0, 180, 17000), rs.randint(0, 180, 17000)], 1)
        P8 = np.stack([lat[a:a + 20, b:b + 20].reshape(-1) for a, b in co], axis=1).astype(np.int8)       # +-1 spins
        X = P8.astype(np.float64)
        W, A, B, h, sec = run(ontf, X[:, :16600], 100, 25, 16384, 1, 104)
        np.savez_compressed(os.path.join(OUT, "full_cfg4.npz"), pool_u8=P8, n_train=16600, k=100, iters=25, batch=16384,
                            alpha=1.0, seed=104, W=W, A=A, B=B, history=h, recon=recon_error(W, X[:, 16600:17000], 1.0))
        print("cfg4 done in %.0f s" % sec, flush=True)
    if "cfg5" in which:
        # the benchmarked shape.  X = RandomState(55).rand(1024, 8592) (8192 training + 400 held-out columns) is
        # regenerated by the test; W0 and the minibatch indices come from the reference's own global-RNG draws
        # (np.random.seed(105): rand(d, k) then one randint(n, size=batch) per step, src/ontf.py:213,230).
        n_tr, n_ho, k5, it5, b5 = 8192, 400, 256, 10, 2048
        X = np.random.RandomState(55).rand(1024, n_tr + n_ho)
        trace = []

        class Rec(ontf.Online_NTF):
            def step(self, Xb, A, B, W, t):
                out = super().step(Xb, A, B, W, t)
                trace.append(out[0].copy())          # H1 (n x r), src/ontf.py:136
                return out

        np.random.seed(105)
        m = Rec(X[:, :n_tr, None], n_components=k5, iterations=it5 + 1, batch_size=b5, alpha=1, mode=0,
                learn_joint_dict=False)
        t0 = time.time()
        W, A, B, _ = m.train_dict_single()
        sec = time.time() - t0
        rs = np.random.RandomState(105)              # replay of the global stream
        W0 = rs.rand(1024, k5)
        idx = np.stack([rs.randint(n_tr, size=b5) for _ in range(it5)])
        d5 = dict(x_seed=55, n_train=n_tr, n_holdout=n_ho, k=k5, iters=it5, batch=b5, alpha=1.0, seed=105, idx=idx,
                  W=W, A=A, B=B, history=float(m.history), recon=recon_error(W, X[:, n_tr:], 1.0),
                  W0_checksum=float(W0.sum()))
        for i, H in enumerate(trace):
            d5["H_%d" % i] = H                       # (batch x k) float64, ~11 % non-zero
        np.savez_compressed(os.path.join(OUT, "full_cfg5.npz"), **d5)
        print("cfg5 done in %.0f s" % sec, flush=True)


if __name__ == "__main__":
    main(sys.argv[1:] or ["cfg1", "cfg2", "cfg3", "cfg4", "cfg5"])
