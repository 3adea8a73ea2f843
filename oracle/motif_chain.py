"""numpy restatement of csrc/motif_chain.cu: Philox4x32-10 and the batched Glauber chain of path homomorphisms.

The device code is fixed bit for bit by this file (include/onmf_b200.h, onmf_motif_chain_init / onmf_motif_chain):

  * Philox4x32-10 (Salmon et al., SC'11; the Random123 constants): multipliers 0xD2511F53, 0xCD9E8D57, Weyl key increments
    0x9E3779B9, 0xBB67AE85, ten rounds.  Key = the 64-bit seed (lo, hi).
  * init, chain c (global index chain0 + c), draw q: counter (q, 0, c, 1).  Root x[0] = mulhi32(word0, n_nodes); while the
    root has no neighbour it is redrawn from counter (0, a, c, 1), a = 1, 2, ...  (uniform over the nodes with a
    neighbour).  x[q] = N(x[q-1])[mulhi32(word0, deg)] for q >= 1 (x[q-1] when it has no neighbour, which only a
    non-symmetric graph allows).
  * Glauber step t (t = step0 + 1, step0 + 2, ...) of chain c: counter (t_lo, t_hi, c, 0); site i = mulhi32(word0, kk);
    x[i] <- S[mulhi32(word1, |S|)] with S = N(x[i-1]) & N(x[i+1]) (interior), N(x[1]) (i = 0), N(x[kk-2]) (i = kk-1), in
    ascending node order.  |S| = 0 (possible only for a non-symmetric graph) leaves the state unchanged.

The package never imports this module; the tests compare the kernels against it.
"""
from __future__ import annotations

import numpy as np

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
_MASK = np.uint64(0xFFFFFFFF)
_S32 = np.uint64(32)


def philox4x32_10(ctr, key):
    """ctr (..., 4), key (..., 2) unsigned 32-bit words (broadcast) -> (..., 4) uint32"""
    c = np.asarray(ctr, dtype=np.uint64)
    k = np.asarray(key, dtype=np.uint64)
    c0, c1, c2, c3 = c[..., 0], c[..., 1], c[..., 2], c[..., 3]
    k0, k1 = k[..., 0], k[..., 1]
    for rnd in range(10):
        if rnd:
            k0 = (k0 + W0) & _MASK
            k1 = (k1 + W1) & _MASK
        p0 = M0 * c0
        p1 = M1 * c2
        c0, c1, c2, c3 = ((p1 >> _S32) ^ c1 ^ k0) & _MASK, p1 & _MASK, ((p0 >> _S32) ^ c3 ^ k1) & _MASK, p0 & _MASK
    return np.stack(np.broadcast_arrays(c0, c1, c2, c3), -1).astype(np.uint32)


def mulhi32(u, m):
    """floor(u * m / 2^32) for unsigned 32-bit u and 0 <= m < 2^32"""
    return ((np.asarray(u, dtype=np.uint64) * np.asarray(m, dtype=np.uint64)) >> _S32).astype(np.int64)


def _key(seed):
    s = int(seed) & 0xFFFFFFFFFFFFFFFF
    return np.array([s & 0xFFFFFFFF, s >> 32], dtype=np.uint64)


def chain_init(rowptr, colidx, kk, n_chains, chain0, seed):
    """-> (n_chains x kk) int32 initial states (tree_sample of a path)"""
    rowptr = np.asarray(rowptr, dtype=np.int64)
    colidx = np.asarray(colidx, dtype=np.int64)
    n_nodes = len(rowptr) - 1
    deg = np.diff(rowptr)
    if not deg.any():
        raise ValueError("the graph has no edge")
    key = _key(seed)
    cs = (int(chain0) + np.arange(n_chains, dtype=np.uint64)) & _MASK
    z = np.zeros_like(cs)
    x = np.empty((n_chains, kk), dtype=np.int64)
    x[:, 0] = mulhi32(philox4x32_10(np.stack([z, z, cs, z + 1], -1), key)[:, 0], n_nodes)
    a = 0
    while True:
        bad = deg[x[:, 0]] == 0
        if not bad.any():
            break
        a += 1
        w = philox4x32_10(np.stack([z[bad], z[bad] + a, cs[bad], z[bad] + 1], -1), key)[:, 0]
        x[bad, 0] = mulhi32(w, n_nodes)
    for q in range(1, kk):
        w = philox4x32_10(np.stack([z + q, z, cs, z + 1], -1), key)[:, 0]
        u = x[:, q - 1]
        x[:, q] = np.where(deg[u] > 0, colidx[np.minimum(rowptr[u] + mulhi32(w, deg[u]), len(colidx) - 1)], u)
    return x.astype(np.int32)


def candidate_set(rowptr, colidx, x, i):
    """S of site i for one state x (ascending)"""
    kk = len(x)
    if i == 0:
        return colidx[rowptr[x[1]]:rowptr[x[1] + 1]]
    if i == kk - 1:
        return colidx[rowptr[x[kk - 2]]:rowptr[x[kk - 2] + 1]]
    a = colidx[rowptr[x[i - 1]]:rowptr[x[i - 1] + 1]]
    b = colidx[rowptr[x[i + 1]]:rowptr[x[i + 1] + 1]]
    return np.intersect1d(a, b, assume_unique=True)


def glauber_step(rowptr, colidx, x, t, c, key):
    """one step of one chain in place (x: kk ints, t: global step, c: global chain index)"""
    kk = len(x)
    w = philox4x32_10(np.array([t & 0xFFFFFFFF, (t >> 32) & 0xFFFFFFFF, c & 0xFFFFFFFF, 0], dtype=np.uint64), key)
    i = int(mulhi32(w[0], kk))
    S = candidate_set(rowptr, colidx, x, i)
    x[i] = int(S[mulhi32(w[1], len(S))]) if len(S) else int(x[i])


def run_chain(rowptr, colidx, state, chain0, seed, step0, n_samples, steps_per_sample=1):
    """-> (out (n_samples x n_chains x kk) int32, final state); `state` (n_chains x kk) is not modified"""
    rowptr = np.asarray(rowptr, dtype=np.int64)
    colidx = np.asarray(colidx, dtype=np.int64)
    st = np.array(state, dtype=np.int64)
    n_chains, kk = st.shape
    key = _key(seed)
    out = np.empty((n_samples, n_chains, kk), dtype=np.int32)
    for c in range(n_chains):
        x = st[c]
        t = int(step0)
        for s in range(n_samples):
            for _ in range(steps_per_sample):
                t += 1
                glauber_step(rowptr, colidx, x, t, int(chain0) + c, key)
            out[s, c] = x
    return out, st.astype(np.int32)


def is_homomorphism(rowptr, colidx, x):
    """every consecutive pair of the path is an edge (x: (..., kk))"""
    rowptr = np.asarray(rowptr, dtype=np.int64)
    colidx = np.asarray(colidx, dtype=np.int64)
    x = np.asarray(x).reshape(-1, np.shape(x)[-1])
    n = len(rowptr) - 1
    ok = np.ones(len(x), dtype=bool)
    for j, row in enumerate(x):
        if row.min() < 0 or row.max() >= n:
            ok[j] = False
            continue
        for q in range(len(row) - 1):
            nb = colidx[rowptr[row[q]]:rowptr[row[q] + 1]]
            if not np.any(nb == row[q + 1]):
                ok[j] = False
                break
    return ok


def run_dense(adj, state, chain0, seed, step0, n_steps, mutant=None):
    """run_chain's final states for many chains at once on a dense boolean adjacency (small graphs): the same steps, vectorised
    over chains.  mutant (tests only) restates one plausible kernel bug: "no_last_site" (site drawn from [0, kk-1)), "union"
    (candidates from N(x[i-1]) | N(x[i+1])), "rank_off" (at an interior site, the element of the shorter row after the chosen
    hit, wrapping around the row)."""
    adj = np.asarray(adj, dtype=bool)
    x = np.array(state, dtype=np.int64)
    C, kk = x.shape
    key = _key(seed)
    cs = (int(chain0) + np.arange(C, dtype=np.uint64)) & _MASK
    z = np.zeros_like(cs)
    rows = np.arange(C)
    deg = adj.sum(1)
    for t in range(int(step0) + 1, int(step0) + int(n_steps) + 1):
        w = philox4x32_10(np.stack([z + (t & 0xFFFFFFFF), z + (t >> 32), cs, z], -1), key)
        i = mulhi32(w[:, 0], kk - 1 if mutant == "no_last_site" else kk)
        a = x[rows, np.where(i == 0, 1, i - 1)]
        b = x[rows, np.where(i == kk - 1, kk - 2, i + 1)]
        S = (adj[a] | adj[b]) if mutant == "union" else (adj[a] & adj[b])
        m = S.sum(1)
        r = mulhi32(w[:, 1], m)
        v = np.argmax(np.cumsum(S, 1) > r[:, None], 1)
        if mutant == "rank_off":
            short = np.where((deg[a] <= deg[b])[:, None], adj[a], adj[b])
            cum = np.cumsum(short, 1)
            nxt = cum[rows, v] % np.maximum(short.sum(1), 1)
            interior = (i > 0) & (i < kk - 1)
            v = np.where(interior, np.argmax(cum > nxt[:, None], 1), v)
        x[rows, i] = np.where(m > 0, v, x[rows, i])
    return x.astype(np.int32)
