"""Dictionary learning along Ising lattice trajectories with the lattices sampled on the device.

The reference's Ising_Reconstructor (ising_reconstruction.py) trains Online_NMF on random patches of lattices from an Ising
MCMC trajectory that ising_simulator.ising_update produces one site at a time on the host, carrying ini_dict / ini_A / ini_B
/ ini_C / history from epoch to epoch and plotting the surrogate error tr(W A W^T) - 2 tr(W B) + tr(C).  Here the lattices
come from patches.IsingChains -- n_chains independent heat-bath chains on the device, continued across epochs -- and the
patches are read out of the frames where they are (patches.ImagePatches): no lattice or patch crosses to the host.
"""
from __future__ import annotations

from .onmf import Online_NMF
from .patches import ImagePatches, IsingChains, frame_patch_coords


def train_dict(shape, ising_beta, patch_size, n_components, iterations, sub_iterations, num_patches, batch_size, alpha=None,
               n_chains=1, sweeps_per_epoch=1, seed=0, subsample=False, precision=None, errors=None):
    """`iterations` epochs of ONMF on patch_size x patch_size patches of Ising lattices of `shape` at inverse temperature
    ising_beta (`beta` is Online_NMF's forgetting exponent).

    Epoch e advances the chains sweeps_per_epoch sweeps, takes one frame per chain (F = n_chains frames), draws
    coords = patches.frame_patch_coords(F, shape, patch_size, num_patches) (num_patches corners per frame, from the global
    numpy RNG) and returns exactly what

        Online_NMF(ImagePatches(frames.reshape(F * H, W), patch_size, coords).to_matrix(), n_components,
                   iterations=sub_iterations, batch_size=batch_size, ini_dict=W, ini_A=At, ini_B=Bt, ini_C=Ct, history=h,
                   alpha=alpha, subsample=subsample, precision=precision).train_dict()

    returns (epoch 0 without the ini_* / history keywords), under the same global numpy RNG state.  errors: an optional
    list; each epoch appends the surrogate error of its trained state, read on the device.  Returns the last epoch's
    (W, At, Bt, Ct, H)."""
    if int(iterations) < 1:
        raise ValueError("iterations (epochs) must be at least 1")
    if int(sweeps_per_epoch) < 1:
        raise ValueError("sweeps_per_epoch must be at least 1")
    chains = IsingChains(shape, ising_beta, n_chains, seed)
    H, W = chains.H, chains.W
    res = None
    nmf = None
    for _ in range(int(iterations)):
        frames = chains.sample(1, sweeps_per_epoch, precision=precision)
        coords = frame_patch_coords(chains.n_chains, (H, W), patch_size, num_patches)
        X = ImagePatches(frames.reshape(chains.n_chains * H, W), patch_size, coords, precision=precision)
        kw = dict(iterations=sub_iterations, batch_size=batch_size, alpha=alpha, subsample=subsample, precision=precision)
        if res is not None:
            W_, At, Bt, Ct, _ = res
            kw.update(ini_dict=W_, ini_A=At, ini_B=Bt, ini_C=Ct, history=nmf.history)
        nmf = Online_NMF(X, n_components, **kw)
        res = nmf.train_dict()
        if errors is not None:
            errors.append(nmf.surrogate_error())
    return res
