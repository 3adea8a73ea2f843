"""numpy restatement of the pivot chain of csrc/motif_chain.cu (onmf_motif_pivot_chain), bit for bit.

The state x[0..kk-1] is a homomorphism of the path 0 - 1 - ... - kk-1, x[0] the pivot; deg(v) = rowptr[v+1] - rowptr[v].
Pivot step t (t = step0 + 1, step0 + 2, ...) of chain c takes word j (j = 0 ... kk) from word (j & 3) of Philox4x32-10
(oracle/motif_chain.py) at counter (t_lo, t_hi, c, 2 + (j >> 2)), key = the seed:

  * proposal: y[0] = N(x[0])[mulhi32(word 0, deg x[0])]; y[q] = N(y[q-1])[mulhi32(word q, deg y[q-1])], q = 1 ... kk-1;
  * acceptance: num = prod_{q=1}^{kk-2} deg(y[q]), den = prod_{q=1}^{kk-2} deg(x[q]) (fp64, in that order); x <- y iff
    word kk * 2^-32 * den < num.  A y[q], q <= kk-2, without a neighbour (only in a non-symmetric graph) refuses the proposal.

This is the Metropolis-Hastings rule for the uniform law on Hom(P_kk, G): the proposal has probability
deg(x[0])^-1 prod_{q=0}^{kk-2} deg(y[q])^-1, and the pivot's degrees cancel in q(y -> x) / q(x -> y) = num / den.  Initial states
are those of motif_chain.chain_init.  The package never imports this module; the tests compare the kernel against it.
"""
from __future__ import annotations

import numpy as np

from .motif_chain import _MASK, _key, mulhi32, philox4x32_10

_TWO_M32 = 2.0 ** -32


def _words(t, cs, kk, key):
    """(len(cs) x (kk + 1)) uint32 words of pivot step t for the global chain indices cs"""
    z = np.zeros_like(cs)
    blocks = [philox4x32_10(np.stack([z + (t & 0xFFFFFFFF), z + ((t >> 32) & 0xFFFFFFFF), cs, z + 2 + b], -1), key)
              for b in range((kk >> 2) + 1)]
    return np.concatenate(blocks, -1)[:, :kk + 1]


def pivot_step(rowptr, colidx, x, t, c, key):
    """one pivot step of one chain in place (x: kk ints, t: global step, c: global chain index)"""
    kk = len(x)
    w = _words(int(t), np.array([int(c) & 0xFFFFFFFF], dtype=np.uint64), kk, key)[0]
    deg = lambda v: int(rowptr[v + 1] - rowptr[v])
    y = np.empty(kk, dtype=np.int64)
    u, num = int(x[0]), 1.0
    for q in range(kk):
        y[q] = colidx[rowptr[u] + int(mulhi32(w[q], deg(u)))]
        u = int(y[q])
        if q == kk - 1:
            break
        if deg(u) == 0:
            return
        if q > 0:
            num *= float(deg(u))
    den = 1.0
    for q in range(1, kk - 1):
        den *= float(deg(int(x[q])))
    if float(w[kk]) * _TWO_M32 * den < num:
        x[:] = y


def run_pivot_chain(rowptr, colidx, state, chain0, seed, step0, n_samples, steps_per_sample=1):
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
                pivot_step(rowptr, colidx, x, t, int(chain0) + c, key)
            out[s, c] = x
    return out, st.astype(np.int32)


def run_pivot_dense(adj, state, chain0, seed, step0, n_steps, mutant=None):
    """run_pivot_chain's final states for many chains at once on a dense boolean adjacency (small graphs): the same steps,
    vectorised over chains.  mutant (tests only) restates one plausible bug of the acceptance rule: "no_mh" (every proposal
    accepted), "pivot_degree" (the pivot's degree ratio deg(y[0]) / deg(x[0]) kept in the ratio), "inverted" (den / num
    instead of num / den)."""
    adj = np.asarray(adj, dtype=bool)
    x = np.array(state, dtype=np.int64)
    C, kk = x.shape
    key = _key(seed)
    cs = (int(chain0) + np.arange(C, dtype=np.uint64)) & _MASK
    deg = adj.sum(1)
    cum = np.cumsum(adj, 1)
    for t in range(int(step0) + 1, int(step0) + int(n_steps) + 1):
        w = _words(t, cs, kk, key)
        y = np.empty_like(x)
        u = x[:, 0]
        ok = np.ones(C, dtype=bool)
        num = np.ones(C)
        for q in range(kk):
            r = mulhi32(w[:, q], deg[u])
            y[:, q] = np.argmax(cum[u] > r[:, None], 1)
            u = y[:, q]
            if q < kk - 1:
                ok &= deg[u] > 0
                if q > 0:
                    num = num * deg[u]
        den = np.ones(C)
        for q in range(1, kk - 1):
            den = den * deg[x[:, q]]
        if mutant == "pivot_degree":
            num, den = num * deg[y[:, 0]], den * deg[x[:, 0]]
        if mutant == "inverted":
            num, den = den, num
        acc = ok & (w[:, kk] * _TWO_M32 * den < num)
        if mutant == "no_mh":
            acc = ok
        x = np.where(acc[:, None], y, x)
    return x.astype(np.int32)
