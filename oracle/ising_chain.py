"""numpy restatement of csrc/ising_chain.cu: checkerboard heat-bath chains of the Ising model on an H x W torus.

The device code is fixed bit for bit by this file (include/onmf_b200.h, onmf_ising_chain_init / onmf_ising_chain):

  * Spins are int8 +-1, (n_chains x H x W) row-major; H and W even and >= 4.  colour(y, x) = (y + x) & 1.  The sites of one
    colour are numbered m = 0, 1, ... in row-major order.
  * Sweep t (t = 1, 2, ... counts sweeps globally) updates colour 0, then colour 1.  Site m of colour k of chain c (global
    index chain0 + c) takes word (m & 3) of Philox4x32-10 (oracle/motif_chain.py) at counter (t_lo, t_hi, c, 2 (m >> 2) + k)
    with key = the seed, and becomes +1 iff that word < thr[(s + 4) / 2], s the sum of its four torus neighbours.
  * thr[j] = min(floor(2^32 / (1 + exp(-2 beta (2j - 4)))), 2^32 - 1), the heat-bath law P(+1 | s) in 32 bits.  The table is
    an input here, so this file and the C library never have to agree on exp to the ulp (thresholds() is its restatement).
  * The initial state is sweep t = 0 with every threshold 2^31: independent uniform +-1.

The package never imports this module; the tests compare the kernels against it.
"""
from __future__ import annotations

import math

import numpy as np

from .motif_chain import _key, philox4x32_10

_MASK = 0xFFFFFFFF
HALF = 1 << 31


def thresholds(beta):
    """the heat-bath table thr[0..4] (uint64) for inverse temperature beta, s = 2j - 4"""
    return np.array([min(int(math.floor(2.0 ** 32 / (1.0 + math.exp(-2.0 * beta * (2 * j - 4))))), _MASK)
                     for j in range(5)], dtype=np.uint64)


def sites(H, W, colour):
    """flat indices y * W + x of the sites of one colour, in their order m"""
    y = np.repeat(np.arange(H), W // 2)
    x = 2 * np.tile(np.arange(W // 2), H) + ((y + colour) & 1)
    return y * W + x


def words(H, W, n_chains, chain0, seed, t, colour):
    """(n_chains x H*W/2) uint32: the word each site of `colour` draws at sweep t"""
    n = H * W // 2
    G = (n + 3) // 4
    cs = (int(chain0) + np.arange(n_chains, dtype=np.uint64)) & np.uint64(_MASK)
    ctr = np.empty((n_chains, G, 4), dtype=np.uint64)
    ctr[..., 0] = int(t) & _MASK
    ctr[..., 1] = (int(t) >> 32) & _MASK
    ctr[..., 2] = cs[:, None]
    ctr[..., 3] = 2 * np.arange(G, dtype=np.uint64) + colour
    return philox4x32_10(ctr, _key(seed)).reshape(n_chains, 4 * G)[:, :n]


def _update(x, own, w, thr, mutant):
    """new values of the sites `own` (flat indices) of x (..., C, H, W) from their words w (C x n)"""
    nbs = np.roll(x, 1, -2) + np.roll(x, -1, -2) + np.roll(x, 1, -1) + np.roll(x, -1, -1)     # int8, |s| <= 4
    s = nbs.reshape(x.shape[:-2] + (-1,))[..., own]
    if mutant == "sign":                                        # the sign of the neighbour sum flipped
        s = -s
    j = (s + 4) // 2
    if mutant == "index_off":                                   # the threshold one entry too far
        j = np.minimum(j + 1, 4)
    thr = np.asarray(thr, dtype=np.uint64)
    p = np.choose(j, [thr[..., i, None, None] for i in range(5)])
    if mutant == "metropolis":
        # flip with probability min(1, exp(-2 beta sigma s)) = min(1, P(-sigma | s) / P(sigma | s)): the reference's
        # acceptance, which forces a flip whenever sigma s <= 0
        sig = x.reshape(x.shape[:-2] + (-1,))[..., own]
        pp = p.astype(np.float64) / 2.0 ** 32
        acc = np.where(sig > 0, (1.0 - pp) / pp, pp / (1.0 - pp))
        flip = w < np.floor(np.minimum(acc, 1.0) * 2.0 ** 32)
        return np.where(flip, -sig, sig).astype(np.int8)
    return np.where(w < p, 1, -1).astype(np.int8)


def chain_init(H, W, n_chains, chain0, seed):
    """-> (n_chains x H x W) int8 initial states (sweep 0, every threshold 2^31)"""
    x = np.empty((n_chains, H * W), dtype=np.int8)
    for k in (0, 1):
        x[:, sites(H, W, k)] = np.where(words(H, W, n_chains, chain0, seed, 0, k) < HALF, 1, -1)
    return x.reshape(n_chains, H, W)


def run_chain(state, thr, chain0, seed, sweep0, n_samples, sweeps_per_sample=1, mutant=None):
    """-> (out (n_samples x ... x n_chains x H x W) int8, final state); `state` is not modified.

    state (..., n_chains, H, W) +-1, thr (..., 5): leading axes are ensembles that share the chains' words (one per table, for
    instance).  Sweeps sweep0 + 1 ... sweep0 + n_samples * sweeps_per_sample; out[s] is the state after sweep
    sweep0 + (s + 1) * sweeps_per_sample.  mutant (tests only) restates one plausible bug: "metropolis" (checkerboard
    Metropolis with the reference's acceptance), "simultaneous" (both colours updated from the state before the sweep),
    "sign" (s negated), "index_off" (thr[min(j + 1, 4)])."""
    x = np.array(state, dtype=np.int8)
    H, W = x.shape[-2:]
    C = x.shape[-3]
    flat = x.reshape(x.shape[:-2] + (H * W,))                  # a view of x
    own = [sites(H, W, k) for k in (0, 1)]
    out = np.empty((n_samples,) + x.shape, dtype=np.int8)
    t = int(sweep0)
    for s in range(n_samples):
        for _ in range(sweeps_per_sample):
            t += 1
            if mutant == "simultaneous":
                new = [_update(x, own[k], words(H, W, C, chain0, seed, t, k), thr, None) for k in (0, 1)]
                for k in (0, 1):
                    flat[..., own[k]] = new[k]
                continue
            for k in (0, 1):
                flat[..., own[k]] = _update(x, own[k], words(H, W, C, chain0, seed, t, k), thr, mutant)
        out[s] = x
    return out, x


def energy_magnetisation(x):
    """(E, M) of states x (..., H, W): E = -sum over the 2HW torus bonds of s_i s_j, M = sum of the spins"""
    x = np.asarray(x, dtype=np.int64)
    E = -(x * np.roll(x, 1, -1)).sum((-2, -1)) - (x * np.roll(x, 1, -2)).sum((-2, -1))
    return E, x.sum((-2, -1))
