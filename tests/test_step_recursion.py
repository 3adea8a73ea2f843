"""The online step as a whole (csrc/step.cu onmf_step*, engine.py) with the codes held fixed, against an fp64 restatement.

With codes supplied (OnmfEngine.step(..., codes=H)) the coder drops out and a step is linear algebra: the dictionary update
with the OLD aggregates, the partial sums P = [H^T H | H^T X] (and P2 = X X^T with track_C) and the blends
A <- (1-w) A + w P_A, B <- (1-w) B + w P_B, C <- (1-w) C + w P2, w = t^-beta.  Each GPU case runs twelve steps in one
schedule form, reads the device state after every step and compares it with oracle.onmf_oracle.step_given_codes applied to
the device's PREVIOUS state, so the bars do not compound:
  fp64                 : 1e-12 relative per entry of A / B / C, 1e-12 per atom of W, surrogate_error 1e-11 relative
  fp32 SIMT products   : 16x the error of a float32 emulation of the same step (split-K order of the kernels); C 4x
  fp32 tensor cores    : per entry w * 2e-5 * sum_s |H_si| |X_sj| (the 3xTF32 chain bound, DESIGN K2 / K4) plus the blend's
                         own fp32 rounding; W as in test_update_dict_variants
and the same sequence enqueued without any host synchronisation must end bit-identical (a cross-step ordering race).
test_mutants_are_far_above_the_bars shows that plausible bugs of the recursion land far above these bars."""
import os
import socket

import numpy as np
import pytest
import torch

import _bcd_worker as BW
from oracle import onmf_oracle as O

EPS32 = float(np.finfo(np.float32).eps)
B200_SMS = 148
UNUSED = 3                                    # atom no code ever uses: A_jj = 0, the update's step is 1 / (0 + 1)
# n per step, cycled twice: 0 and 1; the SIMT surrogate's ceil(n/64) cap (65: 2 splits; 9473: 148 = 2 x SMs / tiles);
# the tensor-core chain cap (1025 samples > 32 K-blocks); xxt's ceil(n/256) (300: 2 splits, 1025: 5, 9473: 38)
# (the largest first: the engine sizes its buffers once, so the second cycle replays the graphs of the first)
SLOTS = (9473, 0, 1025, 1, 300, 65)
SLOTS_D400 = (2000, 0, 1025, 1, 300, 65)
SLOTS_BIG_C = (40000, 0, 1025, 1, 300, 65)    # d = 100: 40000 > 16384 samples, where xxt fell back to one split
TB = [(1, 1.0), (37, 0.6), (1, 0.6), (37, 1.0)]
C_FACTOR = 4                                  # the C emulation sums in the kernel's own order: only FMA contraction differs


# ------------------------------------------------------------------------------------------------------------ inputs
def _unit(W):
    return W / np.linalg.norm(W, axis=0)


def codes(rng, n, k):
    """nonnegative, ~20 % dense; atom UNUSED never used; sample 0 all zero when n >= 2"""
    H = rng.random((n, k)) * (rng.random((n, k)) < 0.2)
    H[:, UNUSED] = 0.0
    if n >= 2:
        H[0] = 0.0
    return H


def start_state(rng, d, k):
    """unit nonnegative dictionary; A, B blended from one minibatch of codes that leave atom UNUSED out"""
    W0 = _unit(rng.random((d, k)) + 0.05)
    H, X = codes(rng, 64, k), rng.random((64, d))
    return W0, H.T @ H / 64, H.T @ X / 64


def steps_of(t0):
    return [float(t0 + i) for i in range(2 * 6)]


# ------------------------------------------------------------------------------------------------ fp32 emulation
def surrogate_splits(n, k, d, sms=B200_SMS):
    """onmf_surrogate_partial's split-K count (gemm_simt.cu pick_splits)"""
    tiles = -(-k // 128) * (-(-k // 128) + -(-d // 128))
    return int(max(1, min(-(-2 * sms // tiles), -(-n // 64), 256)))


def xxt_splits(n, d, ws_bytes, esz, sms=B200_SMS):
    """onmf_xxt_partial's split-K count: ceil(2 SMs / tiles), ceil(n / 256), and what the workspace holds"""
    tiles = (-(-d // 128)) ** 2
    s = max(1, min(-(-2 * sms // tiles), -(-n // 256)))
    return int(max(1, min(s, ws_bytes // (d * d * esz)))) if s > 1 else 1


def split_sum_f32(L, R, splits):
    """L^T R in float32 the way the split-K SIMT kernels form it: each split sums its chunk of samples in order (chunks of
    round_up(ceil(n / splits), 16)), the partials are added in split order"""
    L, R = np.asarray(L, np.float32), np.asarray(R, np.float32)
    n = L.shape[0]
    out = np.zeros((L.shape[1], R.shape[1]), np.float32)
    if n == 0:
        return out
    chunk = -(-(-(-n // splits)) // 16) * 16
    parts = np.zeros((splits,) + out.shape, np.float32)
    starts = np.arange(splits) * chunk
    for i in range(chunk):
        rows = starts + i
        ok = rows < n
        if not ok.any():
            break
        r = rows[ok]
        parts[ok] += L[r][:, :, None] * R[r][:, None, :]
    for s in range(splits):
        out += parts[s]
    return out


def blend_f32(P, w, Y):
    w32 = np.float32(w)
    return (np.float32(1.0) - w32) * np.asarray(Y, np.float32) + w32 * P


def emulate_step_f32(X, H, W, A, B, C, w, xxt_ws=0, sms=B200_SMS):
    """float32 emulation of one SIMT step: the dictionary half is _bcd_worker.emulate_fp32, the products sample-ordered in
    float32 with the kernels' split counts, the blends in float32.  Returns float64 (W1, A1, B1, C1)."""
    n, d = X.shape
    k = H.shape[1]
    s = surrogate_splits(n, k, d, sms)
    A1 = blend_f32(split_sum_f32(H, H, s), w, A)
    B1 = blend_f32(split_sum_f32(H, X, s), w, B)
    C1 = None
    if C is not None:
        C1 = blend_f32(split_sum_f32(X, X, xxt_splits(n, d, xxt_ws, 4, sms)), w, C).astype(np.float64)
    return BW.emulate_fp32(W, A, B), A1.astype(np.float64), B1.astype(np.float64), C1


# ------------------------------------------------------------------------------------------------------------ bars
def entry_ratio(got, ref, bar):
    return float(np.max(np.abs(got - ref) / (bar + 1e-300))) if ref.size else 0.0


def step_ratios(kind, prev, X, H, t, beta, got, xxt_ws=0, sms=B200_SMS):
    """error-to-bar ratio of each part of one step: prev / got = (W, A, B, C) of the device before / after the step
    (float64 copies of the stored values), X (n x d) and H (n x k) the minibatch and codes as the kernels read them"""
    W, A, B, C = prev
    Wr, Ar, Br, Cr = O.step_given_codes(X.T, H.T, W, A, B, C, t, beta)
    w = float(t) ** (-beta)
    r = {}
    if kind == "f64":
        r["W"] = BW.atom_err(got[0], Wr) / 1e-12
        for name, g, ref in (("A", got[1], Ar), ("B", got[2], Br), ("C", got[3], Cr)):
            if ref is not None:
                r[name] = entry_ratio(g, ref, 1e-12 * np.abs(ref))
        return r
    r["W"] = BW.atom_err(got[0], Wr) / min(max(16 * BW.atom_err(BW.emulate_fp32(W, A, B), Wr), 1e-6), 1e-5)
    _, Ae, Be, Ce = emulate_step_f32(X, H, W, A, B, C, w, xxt_ws, sms)
    if kind == "simt":
        for name, g, ref, e in (("A", got[1], Ar, Ae), ("B", got[2], Br, Be)):
            r[name] = np.max(np.abs(g - ref)) / max(16 * np.max(np.abs(e - ref)), EPS32 * np.max(np.abs(ref)), 1e-30)
    else:
        assert kind == "tc"
        for name, g, ref, prev_, S in (("A", got[1], Ar, A, H.T @ H), ("B", got[2], Br, B, H.T @ X)):
            # nonnegative H, X: sum_s |H_si| |X_sj| is the product itself
            bar = w * 2e-5 * S + 2 * EPS32 * ((1 - w) * np.abs(prev_) + w * S)
            r[name] = entry_ratio(g, ref, bar)
    if Cr is not None:
        r["C"] = np.max(np.abs(got[3] - Cr)) / max(C_FACTOR * np.max(np.abs(Ce - Cr)), EPS32 * np.max(np.abs(Cr)), 1e-30)
    return r


def surrogate_ratio(state, got):
    W, A, B, C = state
    t0, t1 = np.sum((W.T @ W) * A), np.trace(W @ B)
    t2 = np.trace(C) if C is not None else 0.0
    return abs(got - (t0 - 2 * t1 + t2)) / (1e-11 * (abs(t0) + 2 * abs(t1) + abs(t2)))


# ------------------------------------------------------------------------------------------------------------- CPU
def test_step_given_codes_reproduces_the_oracle_step(golden_dir):
    """step_given_codes with O.step's own codes is O.step"""
    g = np.load(os.path.join(golden_dir, "cfg1_renoir_gray.npz"))
    X = g["X"][:, g["idx"][0][:60]]
    rng = np.random.default_rng(1)
    W, A, B = g["W0"], rng.random((25, 25)), rng.random((25, 100))
    H, A1, B1, W1 = O.step(X, A, B, W, 3.0, 1.0, beta=0.6)
    W2, A2, B2, C2 = O.step_given_codes(X, H, W, A, B, None, 3.0, beta=0.6)
    assert C2 is None
    for a, b in ((W1, W2), (A1, A2), (B1, B2)):
        assert np.array_equal(a, b)
    C = rng.random((100, 100))
    _, _, _, C3 = O.step_given_codes(X, H, W, A, B, C, 3.0, beta=0.6)
    assert np.allclose(C3, (1 - 3.0 ** -0.6) * C + 3.0 ** -0.6 * X @ X.T, rtol=1e-14, atol=0)


def test_run_given_codes_reproduces_a_golden_run(golden_dir):
    """fed the recorded codes of the reference run cfg1_renoir_gray, run_given_codes lands on its A / B / W"""
    g = np.load(os.path.join(golden_dir, "cfg1_renoir_gray.npz"))
    n = int(g["idx"].shape[0])
    Xs = [g["X"][:, g["idx"][i]] for i in range(n)]
    Hs = [g["H_%d" % i] for i in range(n)]
    ts = [float(g["t_%d" % i]) for i in range(n)]
    k, d = g["W0"].shape[1], g["X"].shape[0]
    W, A, B, C = O.run_given_codes(Xs, Hs, g["W0"], np.zeros((k, k)), np.zeros((k, d)), ts)
    assert C is None
    for got, ref in ((W, g["W_final"]), (A, g["A_final"]), (B, g["B_final"])):
        assert np.max(np.abs(got - ref)) <= 1e-12 * np.max(np.abs(ref)), np.max(np.abs(got - ref))


def _mutant_run(d, k, slots, t0, beta, track_C, seed, xxt_ws=0):
    """the GPU tests' fp32 SIMT inputs stepped by the fp64 oracle (states rounded to float32 as the device stores them);
    per step, every mutant's error over its fp32 bar"""
    rng = np.random.default_rng(seed)
    W, A, B = (BW.rounded(x, "float32") for x in start_state(rng, d, k))
    C = np.zeros((d, d)) if track_C else None
    seq = [(BW.rounded(rng.random((n, d)), "float32"), BW.rounded(codes(rng, n, k), "float32")) for n in slots]
    worst = {}
    put = lambda m, v: worst.__setitem__(m, max(worst.get(m, 0.0), float(v)))
    prevX, prevH, prev_t, P2_prev = np.zeros((0, d)), np.zeros((0, k)), None, np.zeros((d, d))
    for i, t in enumerate(steps_of(t0)):
        X, H = seq[i % len(seq)]
        w = t ** -beta
        Wr, Ar, Br, Cr = O.step_given_codes(X.T, H.T, W, A, B, C, t, beta)
        _, Ae, Be, Ce = emulate_step_f32(X, H, W, A, B, C, w, xxt_ws)
        barW = min(max(16 * BW.atom_err(BW.emulate_fp32(W, A, B), Wr), 1e-6), 1e-5)
        barA = max(16 * np.max(np.abs(Ae - Ar)), EPS32 * np.max(np.abs(Ar)))
        barB = max(16 * np.max(np.abs(Be - Br)), EPS32 * np.max(np.abs(Br)))
        put("no_lag", BW.atom_err(O.update_dict(W, Ar, Br), Wr) / barW)
        ab = lambda w_, HX=(H, X): (np.max(np.abs((1 - w_) * A + w_ * HX[0].T @ HX[0] - Ar)) / barA,
                                    np.max(np.abs((1 - w_) * B + w_ * HX[0].T @ HX[1] - Br)) / barB)
        if prev_t is not None:
            put("stale_w", max(ab(prev_t ** -beta)))
        if beta != 1.0:
            put("w_1_over_t", max(ab(1.0 / t)))
        if i > 0:
            put("other_parity", max(ab(w, (prevH, prevX))))
        if track_C:
            barC = max(C_FACTOR * np.max(np.abs(Ce - Cr)), EPS32 * np.max(np.abs(Cr)))
            if X.shape[0] == 0:
                put("p2_not_zeroed", np.max(np.abs((1 - w) * C + w * P2_prev - Cr)) / barC)
            else:
                P2_prev = X.T @ X
        # the read-out after this step with the Gram of the dictionary before it
        st = (BW.rounded(Wr, "float32"), BW.rounded(Ar, "float32"), BW.rounded(Br, "float32"),
              None if Cr is None else BW.rounded(Cr, "float32"))
        G_old = W.T @ W
        wrong = np.sum(G_old * st[1]) - 2 * np.trace(st[0] @ st[2]) + (np.trace(st[3]) if track_C else 0.0)
        put("sur_prev_gram", surrogate_ratio(st, wrong))
        W, A, B, C = st
        prevX, prevH, prev_t = X, H, t
    return worst


@pytest.mark.parametrize("case", ["d64_t1_b1", "d64_t37_b06_C"])
def test_mutants_are_far_above_the_bars(case):
    """numpy restatements of the recursion with one bug each land >= 10x above the fp32 bars on the GPU tests' inputs:
    no one-step lag, the previous step's w (a stale w_dev), w = 1/t whatever beta, the other parity's partial sums P[cur^1],
    P2 not zeroed on an empty step, the read-out with the Gram of the previous dictionary"""
    if case == "d64_t1_b1":
        worst = _mutant_run(64, 32, SLOTS, 1, 1.0, False, 11)
        expect = ("no_lag", "stale_w", "other_parity", "sur_prev_gram")
    else:
        ws = 64 * 64 * 64 * 4 + 256
        worst = _mutant_run(64, 32, SLOTS, 37, 0.6, True, 12, ws)
        expect = ("no_lag", "stale_w", "w_1_over_t", "other_parity", "p2_not_zeroed", "sur_prev_gram")
    print(case, {m: "%.3g" % v for m, v in worst.items()})
    for m in expect:
        assert worst[m] >= 10, (m, worst[m])


def test_single_split_xxt_is_far_above_the_c_bar():
    """at d = 100, n = 40000 (k = 25: the engine's workspace holds 64 splits of the d x d product) the one-CTA sequential
    fp32 X X^T the workspace fallback used to take lands >= 5x above the C bar of the split form"""
    rng = np.random.default_rng(5)
    d, n = 100, 40000
    X = BW.rounded(rng.random((n, d)), "float32")
    ref = X.T @ X
    ws = max(surrogate_splits(n, 25, d) * 25 * 125 * 4, 64 * d * d * 4) + 256
    s = xxt_splits(n, d, ws, 4)
    assert s == 64
    bar = C_FACTOR * np.max(np.abs(split_sum_f32(X, X, s) - ref))
    seq = np.max(np.abs(split_sum_f32(X, X, 1) - ref))
    print("single-split / C bar = %.2f" % (seq / bar))
    assert seq >= 5 * bar, seq / bar


def test_split_rules_mirror_the_kernels():
    """the split counts the emulation uses, at the shapes of the GPU tests (a retuned kernel rule fails here first)"""
    assert [surrogate_splits(n, 32, 64) for n in SLOTS] == [148, 1, 17, 1, 5, 2]
    assert [xxt_splits(n, 64, 64 * 64 * 64 * 4 + 256, 4) for n in SLOTS] == [38, 1, 5, 1, 2, 1]
    assert xxt_splits(16385, 100, 64 * 100 * 100 * 4 + 256, 4) == 64
    assert xxt_splits(2000, 400, 64 * 400 * 400 * 4 + 256, 4) == 8


# ------------------------------------------------------------------------------------------------------------- GPU
def _dev():
    return torch.device("cuda", 0)


def _np(t):
    return None if t is None else t.detach().cpu().numpy().astype(np.float64)


# form -> (dtype, d, k, feed, engine keyword arguments, env, slots, ratio kind)
FORMS = {
    "f64_streams": ("float64", 64, 32, "dense", dict(graph=False), {}, SLOTS, "f64"),
    "f64_graph": ("float64", 64, 32, "dense", dict(graph=True), {}, SLOTS, "f64"),
    "f64_composed": ("float64", 64, 32, "dense", dict(fused=False), {}, SLOTS, "f64"),
    "f32_simt_streams": ("float32", 64, 32, "dense", dict(use_tc=False, graph=False), {}, SLOTS, "simt"),
    "f32_simt_graph": ("float32", 64, 32, "dense", dict(use_tc=False, graph=True), {}, SLOTS, "simt"),
    "f32_by_ref_streams": ("float32", 64, 32, "dense", dict(graph=False), {}, SLOTS, "tc"),
    "f32_by_ref_graph": ("float32", 64, 32, "dense", dict(graph=True), {}, SLOTS, "tc"),
    "f32_presplit_env": ("float32", 64, 32, "dense", dict(graph=False), {"ONMF_B200_FUSED_TC": "0"}, SLOTS, "tc"),
    "f32_presplit_k300": ("float32", 64, 300, "dense", dict(graph=True), {}, SLOTS, "tc"),
    "f32_pool_u8": ("float32", 64, 32, "pool_u8", dict(graph=True), {}, SLOTS, "tc"),
    "f32_pool_f16": ("float32", 64, 32, "pool_f16", dict(graph=False), {}, SLOTS, "tc"),
    "f32_patches_streams": ("float32", 64, 32, "patches", dict(graph=False), {}, SLOTS, "tc"),
    "f32_patches_graph": ("float32", 64, 32, "patches", dict(graph=True), {}, SLOTS, "tc"),
    "f32_host_f32": ("float32", 64, 32, "host_f32", dict(), {}, SLOTS, "tc"),
    "f32_host_u8": ("float32", 64, 32, "host_u8", dict(), {}, SLOTS, "tc"),
    "f32_C_d64": ("float32", 64, 32, "dense", dict(track_C=True), {}, SLOTS, "tc"),
    "f64_C_d100": ("float64", 100, 25, "dense", dict(track_C=True), {}, SLOTS_BIG_C, "f64"),
    "f32_C_d100": ("float32", 100, 25, "dense", dict(track_C=True), {}, SLOTS_BIG_C, "simt"),
    "f32_C_d400": ("float32", 400, 100, "dense", dict(track_C=True, graph=False), {}, SLOTS_D400, "tc"),
}


def assert_path(form, eng):
    """each form really reaches the entry point it stands for"""
    dt, d, k, feed, kw, env, _, kind = FORMS[form]
    assert eng.fused == (form != "f64_composed")
    assert eng.use_tc == (kind == "tc")
    # by reference (onmf_step_mb / onmf_step_patches): fp32 tensor cores at k <= 256 without track_C, unless switched off
    assert (eng.fused_tc and not eng.track_C) == (kind == "tc" and k <= 256 and not eng.track_C and not env)
    assert eng.graph == (eng.fused and kw.get("graph", True))
    # graph replays: the second cycle of the six resident minibatches; never with track_C (its d x d blend takes w from
    # the host)
    assert eng._plan is None or eng._plan.graph_steps() == (6 if eng.graph and not eng.track_C else 0), form


class Feeder:
    """resident minibatches of one form, their codes, and the X the kernels read (float64, n x d)"""

    def __init__(self, form, seed):
        dt, d, k, feed, kw, env, slots, kind = FORMS[form]
        self.feed, self.d, self.k = feed, d, k
        rng = np.random.default_rng(seed)
        tdt = getattr(torch, dt)
        self.state0 = start_state(rng, d, k)
        self.items = []
        if feed == "patches":
            from onmf_ontf_ndl_b200.patches import ImagePatches, all_patch_coords
            p = int(round(np.sqrt(d)))
            img = rng.random((60, 70)).astype(np.float32)
            co = all_patch_coords(img.shape, p)
            self.src = ImagePatches(img, p, co)
        if feed.startswith("pool"):
            n_pool = 5000
            if feed == "pool_u8":
                pool = rng.integers(0, 256, size=(n_pool, d), dtype=np.uint8)
                self.pool, self.scale = torch.from_numpy(pool).to(_dev()), 1.0 / 255.0
                pool_vals = pool.astype(np.float32) * np.float32(1.0 / 255.0)
            else:
                pool = rng.random((n_pool, d)).astype(np.float16)
                self.pool, self.scale = torch.from_numpy(pool).to(_dev()), 1.0
                pool_vals = pool.astype(np.float32)
        for n in slots:
            H = BW.rounded(codes(rng, n, k), dt)
            item = dict(n=n, H=H, Hd=torch.from_numpy(H).to(_dev(), tdt))
            if feed == "dense":
                X = BW.rounded(rng.random((n, d)), dt)
                item.update(X=X, Xd=torch.from_numpy(X).to(_dev(), tdt))
            elif feed.startswith("pool"):
                idx = rng.integers(0, n_pool, size=n)
                item.update(X=pool_vals[idx].astype(np.float64), idx=torch.from_numpy(idx).to(_dev()))
            elif feed == "patches":
                idx = rng.integers(0, self.src.N, size=n)
                c = self.src.coords.cpu().numpy()[idx]
                item.update(X=O.gather_patches_gray(img.astype(np.float64), c, p).T.reshape(n, d),
                            idx=torch.from_numpy(idx).to(_dev()))
            elif feed == "host_f32":
                X = BW.rounded(rng.random((n, d)), dt)
                item.update(X=X, host=torch.from_numpy(X.astype(np.float32)).pin_memory())
            else:
                X8 = rng.integers(0, 256, size=(n, d), dtype=np.uint8)
                item.update(X=(X8.astype(np.float32) * np.float32(1.0 / 255.0)).astype(np.float64),
                            host=torch.from_numpy(X8).pin_memory())
            self.items.append(item)

    def step(self, eng, i, t):
        """one step on item i; returns the codes the step aggregated (n x k, float64) when the device chose them"""
        it = self.items[i % len(self.items)]
        if self.feed == "dense":
            eng.step(it["Xd"], t, codes=it["Hd"])
        elif self.feed.startswith("pool"):
            eng.step_pool(self.pool, it["idx"], t, scale=self.scale, codes=it["Hd"])
        elif self.feed == "patches":
            eng.step_patches(self.src, it["idx"], t, codes=it["Hd"])
        else:
            return eng.step_host(it["host"], t).clone()       # step_host runs the coder: its codes are the given ones
        return None


def _run(form, seed, t0, beta, sync):
    from onmf_ontf_ndl_b200 import OnmfEngine
    dt, d, k, feed, kw, env, slots, kind = FORMS[form]
    fd = Feeder(form, seed)
    eng = OnmfEngine(d, k, alpha=0.5, beta=beta, dtype=getattr(torch, dt), device=_dev(), **kw)
    W0, A0, B0 = fd.state0
    eng.set_state(W0, A0, B0, np.zeros((d, d)) if eng.track_C else None)
    worst, host_codes = {}, []
    state = lambda: tuple(_np(x) for x in eng.state())
    prev = state() if sync else None
    for i, t in enumerate(steps_of(t0)):
        Hc = fd.step(eng, i, t)
        if Hc is not None:
            host_codes.append(Hc)
        if not sync:
            continue
        got = state()
        torch.cuda.synchronize()
        it = fd.items[i % len(fd.items)]
        H = _np(Hc) if Hc is not None else it["H"]
        ws = eng._ws_sur.numel() if eng._ws_sur is not None else 0
        r = step_ratios(kind, prev, it["X"], H, t, beta, got, ws, torch.cuda.get_device_properties(0).multi_processor_count)
        r["sur"] = surrogate_ratio(got, eng.surrogate_error())
        for key, v in r.items():
            worst[key] = max(worst.get(key, 0.0), float(v))
        prev = got
    final = [x.clone() for x in eng.state() if x is not None]
    torch.cuda.synchronize()
    return eng, worst, final, host_codes


@pytest.mark.gpu
@pytest.mark.parametrize("form", list(FORMS))
def test_step_form_against_fp64_restatement(form, monkeypatch):
    """twelve steps of one schedule form against step_given_codes on the device's previous state; then the same sequence
    enqueued without host synchronisation ends bit-identical"""
    dt, d, k, feed, kw, env, slots, kind = FORMS[form]
    for key, v in env.items():
        monkeypatch.setenv(key, v)
    i = list(FORMS).index(form)
    t0, beta = TB[i % len(TB)]
    eng, worst, final, codes_sync = _run(form, 100 + i, t0, beta, True)
    assert_path(form, eng)
    print("step %s (t0=%g beta=%g): largest error / bar %s" % (form, t0, beta, {key: "%.3g" % v for key, v in worst.items()}))
    for key, v in worst.items():
        assert v <= 1.0, (form, key, v)
    eng2, _, final2, codes_async = _run(form, 100 + i, t0, beta, False)
    for a, b in zip(final, final2):
        assert torch.equal(a, b), form
    for a, b in zip(codes_sync, codes_async):
        assert torch.equal(a, b), form


def _gloo_worker(rank, world, port, out):
    import torch.distributed as dist
    from onmf_ontf_ndl_b200 import OnmfEngine
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.cuda.set_device(0)
    res = {}
    for form, t0, beta in (("f64_streams", 37, 0.6), ("f32_by_ref_streams", 1, 1.0), ("f32_C_d64", 37, 1.0)):
        dt, d, k, feed, kw, env, slots, kind = FORMS[form]
        fd = Feeder(form, 7)
        eng = OnmfEngine(d, k, alpha=0.5, beta=beta, dtype=getattr(torch, dt), device=_dev(), process_group=dist.group.WORLD,
                         **kw)
        W0, A0, B0 = fd.state0
        eng.set_state(W0, A0, B0, np.zeros((d, d)) if eng.track_C else None)
        prev = tuple(_np(x) for x in eng.state())
        worst = {}
        for i, t in enumerate(steps_of(t0)):
            it = fd.items[i % len(fd.items)]
            lo, hi = (it["n"] * rank) // world, (it["n"] * (rank + 1)) // world      # this rank's columns
            eng.step(it["Xd"][lo:hi].contiguous(), t, codes=it["Hd"][lo:hi].contiguous())
            got = tuple(_np(x) for x in eng.state())
            torch.cuda.synchronize()
            ws = eng._ws_sur.numel()
            for key, v in step_ratios(kind, prev, it["X"], it["H"], t, beta, got, ws,
                                      torch.cuda.get_device_properties(0).multi_processor_count).items():
                worst[key] = max(worst.get(key, 0.0), float(v))
            prev = got
        Wt = eng.state()[0].contiguous()
        gathered = [torch.empty_like(Wt) for _ in range(world)]
        dist.all_gather(gathered, Wt)
        same = all(torch.equal(gathered[0], x) for x in gathered)
        res[form] = dict(ok=bool(same and max(worst.values()) <= 1.0 and eng.world == world and not eng.graph),
                         same_ranks=same, worst=worst)
    out[rank] = res
    dist.destroy_process_group()


@pytest.mark.gpu
def test_two_gloo_ranks_split_the_minibatch_by_columns():
    """onmf_step_launch[_mb] + all-reduce of P (and P2) + onmf_step_finish on two gloo ranks sharing cuda:0: every step
    matches the fp64 restatement of the whole minibatch at the single-GPU bars, and the ranks' dictionaries are identical"""
    import torch.multiprocessing as mp
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_gloo_worker, args=(2, port, out), nprocs=2, join=True)
    for r in (0, 1):
        print("rank", r, {f: {key: "%.3g" % v for key, v in x["worst"].items()} for f, x in out[r].items()})
        assert all(v["ok"] for v in out[r].values()), dict(out)


RING = 4096


@pytest.mark.gpu
def test_graph_weight_ring_over_three_wraps():
    """3 x 4096 + 17 graph-replayed steps enqueued without a host sync, two resident minibatches alternating with fixed
    codes from A = B = 0: then A_T = a_T P_0 + b_T P_1 with scalar recursions a, b, and likewise B.  A replay that read
    another step's weight from the pinned ring breaks this far beyond 1e-12."""
    from onmf_ontf_ndl_b200 import OnmfEngine
    d, k, n, beta = 32, 16, 40, 0.7
    rng = np.random.default_rng(21)
    X = [rng.random((n, d)) for _ in range(2)]
    H = [codes(rng, n, k) for _ in range(2)]
    eng = OnmfEngine(d, k, alpha=0.5, beta=beta, dtype=torch.float64, device=_dev(), graph=True)
    eng.set_state(_unit(rng.random((d, k)) + 0.05))
    Xd = [torch.from_numpy(x).to(_dev()) for x in X]
    Hd = [torch.from_numpy(h).to(_dev()) for h in H]
    T = 3 * RING + 17
    a = b = 0.0
    for t in range(1, T + 1):
        i = (t - 1) % 2
        eng.step(Xd[i], float(t), codes=Hd[i])
        w = float(t) ** -beta
        a, b = (1 - w) * a + w * (i == 0), (1 - w) * b + w * (i == 1)
    _, A, B, _ = eng.state()
    torch.cuda.synchronize()
    assert eng._plan.graph_steps() == T - 2
    for got, P in ((A, [h.T @ h for h in H]), (B, [h.T @ x for h, x in zip(H, X)])):
        ref = a * P[0] + b * P[1]
        err = np.max(np.abs(_np(got) - ref) / (np.abs(ref) + 1e-300))
        print("weight ring: %d replays, largest relative error %.2e" % (T - 2, err))
        assert err <= 1e-12, err


# ------------------------------------------------------------------------------------------------ direct kernel cases
def _gamma(m, eps):
    return m * eps / (1 - m * eps)


@pytest.mark.gpu
@pytest.mark.parametrize("d", [64, 100, 200])
def test_xxt_partial_at_split_edges(d):
    """onmf_xxt_partial at n = 256 s +- 1 over its split counts, fp64 within the summation bound of its split form; with a
    workspace that holds exactly the splits it wants, one that holds fewer (it then uses as many as fit) and none"""
    from onmf_ontf_ndl_b200 import _lib
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    tiles = (-(-d // 128)) ** 2
    want = -(-2 * sms // tiles)
    rng = np.random.default_rng(d)
    for s in sorted({1, 2, 5, 63, want}):
        for n in (256 * s - 1, 256 * s + 1):
            X = rng.random((n, d))
            ref = X.T @ X
            Xd = torch.from_numpy(X).to(_dev())
            s_full = xxt_splits(n, d, 1 << 40, 8, sms)
            outs = {}
            for ws_bytes in (2 * s_full * d * d * 8, s_full * d * d * 8, max(s_full // 3, 1) * d * d * 8 + 7, 0):
                ws = torch.empty(ws_bytes, dtype=torch.uint8, device=_dev()) if ws_bytes else None
                P2 = torch.full((d, d), float("nan"), dtype=torch.float64, device=_dev())
                _lib.xxt_partial(Xd, P2, ws)
                torch.cuda.synchronize()
                used = xxt_splits(n, d, ws_bytes, 8, sms)
                chunk = -(-(-(-n // used)) // 16) * 16
                err = np.max(np.abs(_np(P2) - ref) / ref)
                assert err <= _gamma(chunk + used + 1, 2.0 ** -53), (d, n, ws_bytes, used, err)
                outs[ws_bytes] = _np(P2)
            assert np.array_equal(outs[2 * s_full * d * d * 8], outs[s_full * d * d * 8]), (d, n)    # exact fit: same splits
    # fp32: the sample-ordered split form, as many splits as the workspace holds
    n = 40000
    X = BW.rounded(rng.random((n, d)), "float32")
    ref = X.T @ X
    Xd = torch.from_numpy(X).to(_dev(), torch.float32)
    for ws_bytes in (64 * d * d * 4 + 256, 16 * d * d * 4):
        used = xxt_splits(n, d, ws_bytes, 4, sms)
        P2 = torch.empty(d, d, device=_dev())
        _lib.xxt_partial(Xd, P2, torch.empty(ws_bytes, dtype=torch.uint8, device=_dev()))
        emu = np.max(np.abs(split_sum_f32(X, X, used) - ref))
        err = np.max(np.abs(_np(P2) - ref))
        print("xxt fp32 d=%d n=%d splits=%d: error %.3g, emulation %.3g" % (d, n, used, err, emu))
        assert err <= C_FACTOR * emu, (d, ws_bytes, used, err, emu)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", ["float32", "float64"])
def test_blend_and_axpby_leave_guards_untouched(dt):
    """onmf_surrogate_blend / onmf_surrogate_blend_dev / onmf_axpby at counts that are not multiples of 256: every entry
    within one rounding of each operation of the fp64 formula, the entries past the end untouched; blend_dev reads w from
    device memory"""
    from onmf_ontf_ndl_b200 import _lib
    tdt = getattr(torch, dt)
    eps = EPS32 if dt == "float32" else 2.0 ** -52
    rng = np.random.default_rng(3)
    for k, d in ((7, 13), (33, 100), (250, 513)):
        P = BW.rounded(rng.random((k, k + d)), dt)
        A0, B0 = BW.rounded(rng.random((k, k)), dt), BW.rounded(rng.random((k, d)), dt)
        w = 0.3 if dt == "float64" else float(np.float32(0.3))
        for dev_w in (False, True):
            Ag = torch.full((k * k + 300,), 7.0, dtype=tdt, device=_dev())
            Bg = torch.full((k * d + 300,), 7.0, dtype=tdt, device=_dev())
            Ag[:k * k] = torch.from_numpy(A0.ravel()).to(_dev(), tdt)
            Bg[:k * d] = torch.from_numpy(B0.ravel()).to(_dev(), tdt)
            Pd = torch.from_numpy(P).to(_dev(), tdt)
            A, B = Ag[:k * k].view(k, k), Bg[:k * d].view(k, d)
            if dev_w:
                wd = torch.tensor([0.3], dtype=torch.float64, device=_dev())
                _lib._check(_lib.load().onmf_surrogate_blend_dev(_lib.dt(Pd), _lib._ptr(Pd), k, d, _lib._ptr(wd), _lib._ptr(A),
                                                                 _lib._ptr(B), _lib._stream()), "onmf_surrogate_blend_dev")
            else:
                _lib.surrogate_blend(Pd, 0.3, A, B)
            torch.cuda.synchronize()
            for got, Y, Pp in ((A, A0, P[:, :k]), (B, B0, P[:, k:])):
                ref = (1 - w) * Y + w * Pp
                assert np.all(np.abs(_np(got) - ref) <= 3 * eps * ((1 - w) * Y + w * Pp)), (k, d, dev_w)
            assert torch.all(Ag[k * k:] == 7.0) and torch.all(Bg[k * d:] == 7.0)
    for count in (1, 255, 257, 1000003):
        x = BW.rounded(rng.random(count), dt)
        y = BW.rounded(rng.random(count), dt)
        yg = torch.full((count + 300,), 7.0, dtype=tdt, device=_dev())
        yg[:count] = torch.from_numpy(y).to(_dev(), tdt)
        a = 0.25 if dt == "float64" else float(np.float32(0.25))
        _lib.axpby(0.25, torch.from_numpy(x).to(_dev(), tdt), 0.75, yg[:count])
        torch.cuda.synchronize()
        ref = a * x + (1 - a) * y
        assert np.all(np.abs(_np(yg[:count]) - ref) <= 3 * eps * ref), count
        assert torch.all(yg[count:] == 7.0)


@pytest.mark.gpu
@pytest.mark.parametrize("d,k,withC", [(4096, 512, True), (100, 25, False), (77, 33, True), (1, 1, True)])
def test_surrogate_error_kernel(d, k, withC):
    """onmf_surrogate_error on fp64 inputs (k^2 > 1024 and a large d k included; C = None reads as tr C = 0) against
    O.surrogate_error at 1e-13 of the sum of the terms' magnitudes"""
    from onmf_ontf_ndl_b200 import _lib
    rng = np.random.default_rng(d + k)
    W = rng.random((d, k)) - 0.3
    A, B = rng.random((k, k)), rng.random((k, d)) - 0.5
    C = rng.random((d, d)) if withC else None
    t = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(_dev())
    G = t(W.T @ W)
    out = torch.empty(3, dtype=torch.float64, device=_dev())
    _lib.surrogate_error(t(W), G, t(A), t(B), t(C) if withC else None, out)
    o = _np(out)
    ref = O.surrogate_error(W, A, B, C if withC else np.zeros((d, d)))
    scale = np.sum((np.abs(W).T @ np.abs(W)) * A) + 2 * np.sum(np.abs(W) * np.abs(B.T)) + (np.trace(C) if withC else 0.0)
    assert abs(o[0] - 2 * o[1] + o[2] - ref) <= 1e-13 * scale
    if not withC:
        assert o[2] == 0.0


@pytest.mark.gpu
def test_convert_is_the_rounding_of_torch():
    """onmf_convert f64 -> f32 bit-equal to Tensor.float() on ties, overflow to +-inf, subnormals and NaN, past the
    16 x SMs x 256 grid-stride edge; f32 -> f64 exact"""
    from onmf_ontf_ndl_b200 import _lib
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    edge = 16 * sms * 256
    rng = np.random.default_rng(8)
    f32max = float(np.finfo(np.float32).max)
    special = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, f32max, -f32max, f32max * (1 + 2.0 ** -25), f32max * 1.0000001,
                        -f32max * 1.0000001, 1e39, -1e300, 1e-40, -1e-40, 1e-45, 7e-46, 1.4e-45, 1e-50, 2.0 ** -149,
                        2.0 ** -150, 3 * 2.0 ** -151, 1.0 + 2.0 ** -24, 1.0 + 3 * 2.0 ** -24, 1.0 + 2.0 ** -24 + 2.0 ** -60,
                        1.0 - 2.0 ** -25, 2.0 ** -126 * (1 - 2.0 ** -24)])
    for count in (len(special), edge - 1, edge + 1, 2 * edge + 5):
        x = np.concatenate([special, rng.standard_normal(max(count - len(special), 0)) * np.exp(rng.uniform(-120, 100, max(count - len(special), 0)))])[:count]
        src = torch.from_numpy(x).to(_dev())
        dst = torch.full((count + 64,), 5.0, dtype=torch.float32, device=_dev())
        _lib.convert(src, dst[:count])
        torch.cuda.synchronize()
        ref = src.float()
        assert torch.equal(dst[:count].view(torch.int32)[~torch.isnan(ref)], ref.view(torch.int32)[~torch.isnan(ref)]), count
        assert torch.equal(torch.isnan(dst[:count]), torch.isnan(ref)) and torch.all(dst[count:] == 5.0)
        back = torch.full((count + 64,), 5.0, dtype=torch.float64, device=_dev())
        _lib.convert(ref, back[:count])
        torch.cuda.synchronize()
        assert torch.equal(back[:count][~torch.isnan(ref)], ref.double()[~torch.isnan(ref)]) and torch.all(back[count:] == 5.0)
