"""Device pivot chains (patches.MotifChains(mcmc="pivot"), onmf_motif_pivot_chain) beside the Glauber chain, on the graph of
prof_motif_chain.py (seeded, 10^6 nodes, mean degree about 20, 5 hubs of degree about 10^4).
    1. Rates, for both chains: kk = 21 and kk = 6, 10^4, 10^5 and 10^6 chains.  The timed call is
       MotifChains.sample(1, steps_per_sample=S) (validation kernel + S steps + one output slice), CUDA events around it, S
       chosen from a probe so that each run lasts about 2 s.  steps_per_s = chains x steps / time; site_updates_per_s counts
       kk per pivot step and 1 per Glauber step.
    2. Mixing, for both chains: the integrated autocorrelation time (IAT) of the number of edges in the kk x kk patch (half
       the patch's sum; the graph has no self-loop), 2,000 chains, 2,000 recorded samples after 1,000 discarded ones, one
       sample every pivot step and every kk Glauber steps.  The autocovariance is averaged over chains around the pivot
       chain's mean (both chains sample the same law; the Glauber chains' own means stay near their start), and the IAT
       is 1 + 2 sum_{tau <= W} rho(tau) with Sokal's window (the least W >= 5 IAT(W)).  When no W < 1,000 samples
       qualifies, the value at W = 1,000 is a lower bound (window_converged = false).  The IAT is given in steps and, at
       each measured chain count, in seconds (IAT steps / steps per second of one chain), with effective samples per
       second = steps_per_s / IAT steps.
One JSON line per measurement, each with the GPU name and power limit read in the same run.
    python profiles/tools/prof_pivot_chain.py"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from onmf_ontf_ndl_b200 import patches  # noqa: E402
from prof_motif_chain import gpu_info, make_graph, timed_sample  # noqa: E402

KKS, CHAINS = (21, 6), (10_000, 100_000, 1_000_000)
IAT_CHAINS, IAT_BURN, IAT_SAMPLES, IAT_CHUNK = 2_000, 1_000, 2_000, 250


def edge_counts(ch, n_samples, thin):
    """(n_samples x n_chains) float64: edges of the patch of every recorded state"""
    out = []
    for s0 in range(0, n_samples, IAT_CHUNK):
        X = ch.patches(min(IAT_CHUNK, n_samples - s0), steps_per_sample=thin)
        out.append(X.sum(1, dtype=torch.float64).view(-1, ch.n_chains) / 2)
    return torch.cat(out)


def iat(f, mu):
    """Sokal-windowed integrated autocorrelation time (in samples) of the columns of f around mu -> (iat, window, converged)"""
    R = f.shape[0]
    g = f - mu
    F = torch.fft.rfft(g, n=2 * R, dim=0)
    acov = torch.fft.irfft(F.real ** 2 + F.imag ** 2, n=2 * R, dim=0)[:R].sum(1)
    acov = acov / (torch.arange(R, 0, -1, dtype=acov.dtype, device=acov.device) * f.shape[1])
    rho = (acov / acov[0]).cpu().numpy()
    tau = 1 + 2 * np.cumsum(rho[1:R // 2])
    ok = np.nonzero(np.arange(1, R // 2) >= 5 * tau)[0]
    if len(ok):
        return float(tau[ok[0]]), int(ok[0] + 1), True
    return float(tau[-1]), R // 2 - 1, False


def main():
    name, power = gpu_info()
    rp, ci = make_graph()
    csr = (rp, ci)
    deg = np.diff(rp)
    base = dict(gpu=name, power_limit=power, nodes=len(rp) - 1, entries=int(rp[-1]), max_degree=int(deg.max()),
                mean_degree=round(float(deg.mean()), 2))
    print(json.dumps(dict(base, what="graph")), flush=True)

    rate = {}
    for mcmc in ("pivot", "glauber"):
        for kk in KKS:
            for n_chains in CHAINS:
                ch = patches.MotifChains(csr, kk, n_chains, seed=1, mcmc=mcmc)
                timed_sample(ch, 5)                                    # warm-up (module load, L2)
                probe = 20
                dt = timed_sample(ch, probe)
                steps = max(probe, int(probe * 2.0 / max(dt, 1e-6)))
                dt = timed_sample(ch, steps)
                sps = n_chains * steps / dt
                rate[mcmc, kk, n_chains] = sps
                print(json.dumps(dict(base, what="rate", mcmc=mcmc, kk=kk, chains=n_chains, steps=steps, seconds=round(dt, 3),
                                      steps_per_s=sps, site_updates_per_s=sps * (kk if mcmc == "pivot" else 1))), flush=True)
                del ch
                torch.cuda.empty_cache()

    for kk in KKS:
        f = {}
        for mcmc, thin in (("pivot", 1), ("glauber", kk)):
            ch = patches.MotifChains(csr, kk, IAT_CHAINS, seed=3, mcmc=mcmc)
            ch.sample(1, steps_per_sample=IAT_BURN * thin)
            f[mcmc] = edge_counts(ch, IAT_SAMPLES, thin)
        mu = float(f["pivot"].mean())
        for mcmc, thin in (("pivot", 1), ("glauber", kk)):
            tau, W, conv = iat(f[mcmc], mu)
            rec = dict(base, what="iat", mcmc=mcmc, kk=kk, chains=IAT_CHAINS, samples=IAT_SAMPLES, steps_per_sample=thin,
                       burn_in_steps=IAT_BURN * thin, observable="patch edges", pivot_mean=round(mu, 4),
                       chain_mean=round(float(f[mcmc].mean()), 4), variance=float(f[mcmc].var()), iat_steps=tau * thin,
                       window_samples=W, window_converged=conv)
            for n_chains in CHAINS:
                sps = rate[mcmc, kk, n_chains]
                rec["iat_seconds_at_%d_chains" % n_chains] = tau * thin * n_chains / sps
                rec["eff_samples_per_s_at_%d_chains" % n_chains] = sps / (tau * thin)
            print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
