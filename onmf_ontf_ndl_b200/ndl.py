"""Network dictionary learning (NDL) with the motif MCMC on the device.

The reference's Network_Reconstructor.train_dict (network_reconstruction_nx.py:342-391) walks ONE Glauber chain of path
embeddings on the host, turns `sample_size` consecutive states into k x k adjacency patches per epoch, and runs one
Online_NMF per epoch, carrying ini_dict / ini_A / ini_B / ini_C / history from epoch to epoch (SURVEY.md §3.4).  Here the
patches of an epoch come from patches.MotifChains -- n_chains independent chains on the device, continued across epochs --
and are trained on where they are (patches.SamplePool): no state or patch crosses to the host.
"""
from __future__ import annotations

from .onmf import Online_NMF
from .patches import MotifChains, SamplePool


def train_dict(G, kk, n_components, iterations, sub_iterations, sample_size, batch_size, alpha=None, n_chains=100, seed=0,
               subsample=False, precision=None, mcmc="glauber"):
    """`iterations` epochs of NDL on the graph G (networkx graph or symmetric scipy adjacency) with the path motif on kk nodes.

    Epoch e draws sample_size = n_chains * m motif patches, m consecutive states (one step apart) of every chain, in
    time-slice order (row s * n_chains + c is chain c after its s-th step of the epoch), and returns exactly what

        Online_NMF(X, n_components, iterations=sub_iterations, batch_size=batch_size, ini_dict=W, ini_A=At, ini_B=Bt,
                   ini_C=Ct, history=h, alpha=alpha, subsample=subsample, precision=precision).train_dict()

    returns on the host matrix X of the same patches (epoch 0 without the ini_* / history keywords), under the same global
    numpy RNG state.  mcmc: "glauber" or "pivot", the chain of patches.MotifChains (the drivers' is_glauber_dict = True /
    False).  Returns the last epoch's (W, At, Bt, Ct, H)."""
    if int(iterations) < 1:
        raise ValueError("iterations (epochs) must be at least 1")
    if int(sample_size) <= 0 or int(n_chains) <= 0 or int(sample_size) % int(n_chains):
        raise ValueError("sample_size (%d) must be a positive multiple of n_chains (%d)" % (sample_size, n_chains))
    chains = MotifChains(G, kk, n_chains, seed, mcmc=mcmc)
    m = int(sample_size) // int(n_chains)
    res = None
    nmf = None
    for _ in range(int(iterations)):
        X = SamplePool(chains.patches(m, precision=precision))
        kw = dict(iterations=sub_iterations, batch_size=batch_size, alpha=alpha, subsample=subsample, precision=precision)
        if res is not None:
            W, At, Bt, Ct, _ = res
            kw.update(ini_dict=W, ini_A=At, ini_B=Bt, ini_C=Ct, history=nmf.history)
        nmf = Online_NMF(X, n_components, **kw)
        res = nmf.train_dict()
    return res
