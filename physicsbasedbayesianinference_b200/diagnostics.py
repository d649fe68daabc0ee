"""Convergence diagnostics of ensemble chains (build-defined: the reference has none).

Nested R-hat (Margossian, Hoffman, Sountsov, Riou-Durand, Vehtari, Gelman, "Nested R-hat: assessing the convergence
of Markov chain Monte Carlo when running many short chains", Bayesian Analysis, 2024) is the R-hat of many short
chains.  The chains are grouped into K superchains of M chains each (M = superchainSize: chains k M .. k M + M - 1 form
superchain k, and the chains of one superchain share their initial point, Ensemble.setPosition(qStd, superchainSize=M)).
With N draws per chain in the window, per dimension:

    f.mk  mean of chain m of superchain k;  s2_mk  its within-chain variance (N - 1 in the denominator)
    f..k  mean of superchain k;             f...   the grand mean
    B^    = 1/(K-1) sum_k (f..k - f...)^2
    B~_k  = 1/(M-1) sum_m (f.mk - f..k)^2        (0 when M = 1)
    W~_k  = 1/M sum_m s2_mk                      (0 when N = 1)
    W^    = 1/K sum_k (B~_k + W~_k)
    nR^   = sqrt(1 + B^ / W^)

K < 2, and M = 1 together with N = 1, are refused (ValueError).  With M = 1, nR^2 = R^2 + 1/N, where R^ is the classic
(non-split) Gelman-Rubin R-hat: nested R-hat is then the classic one up to that 1/N.  Both need only each chain's mean
and within-chain variance, which HMC.run(chainDiagnostics=True) accumulates on the GPU for every chain.

Effective sample size, estimator: for one coordinate, the chains are centred on the GRAND mean over chains and draws (they
are exchangeable: same target, independent particles -- centring every chain on its own mean would
hide exactly the slow component a poorly mixing chain has not traversed yet), the autocovariance is
computed by FFT per chain and AVERAGED over the traced chains, then
Geyer's initial-positive-sequence truncation gives the integrated autocorrelation time tau;
ESS = (number of draws) x (number of chains) / tau.  Runs on the tensors' device (torch.fft)."""
from __future__ import annotations

import math


def ess(trace):
    """trace: torch tensor (S, C) -- S draws of C chains of ONE coordinate.  Returns total ESS."""
    import torch

    x = trace.to(torch.float64)
    S, C = x.shape
    xc = x - x.mean()
    n = 1 << (2 * S - 1).bit_length()
    f = torch.fft.rfft(xc, n=n, dim=0)
    acov = torch.fft.irfft(f * f.conj(), n=n, dim=0)[:S] / S
    acov = acov.mean(dim=1).cpu()
    if float(acov[0]) <= 0:
        return float(S * C)
    rho = (acov / acov[0]).tolist()
    tau = -1.0
    t = 0
    while t + 1 < S:
        pair = rho[t] + rho[t + 1]
        if pair < 0:
            break
        tau += 2.0 * pair
        t += 2
    tau = max(tau, 1.0 / math.log10(max(S, 10)))
    return float(S * C / tau)


def ess_min_over_dims(trace, numParticlesTotal=None):
    """trace: (D, C, S) positions of C traced particles over S iterations.  Returns
    (min over dimensions of the ESS of the traced chains, the same scaled to the whole ensemble)."""
    D, C, S = trace.shape
    vals = [ess(trace[d].transpose(0, 1)) for d in range(D)]
    m = min(vals)
    scale = (numParticlesTotal / C) if numParticlesTotal else 1.0
    return m, m * scale


def _as_float64(x):
    import numpy as np
    import torch

    if isinstance(x, np.ndarray):
        x = torch.from_numpy(x)
    return x.to(torch.float64)


def _superchain_sums(chainMean, chainVar, numDraws, M):
    """This process's part of nested R-hat: (K, mean of the superchain means, their centred sum of squares,
    sum_k (B~_k + W~_k)), per dimension, float64."""
    import torch

    D, C = chainMean.shape
    K = C // M
    cm = chainMean.reshape(D, K, M)
    sm = cm.mean(dim=2)  # superchain means (D, K)
    if M > 1:
        btil = (cm - sm[:, :, None]).square().sum(dim=2) / (M - 1)
    else:
        btil = torch.zeros_like(sm)
    wtil = chainVar.reshape(D, K, M).mean(dim=2) if numDraws > 1 else torch.zeros_like(sm)
    if K > 0:
        mu = sm.mean(dim=1)
        ss = (sm - mu[:, None]).square().sum(dim=1)  # centred: two passes, never sum x^2 - (sum x)^2 / K
    else:
        mu = ss = torch.zeros(D, dtype=torch.float64, device=chainMean.device)
    return K, mu, ss, (btil + wtil).sum(dim=1)


def _gather_parts(K, mu, ss, s, group):
    """Every rank's (K, mu, ss, s), in rank order (one all_gather; gloo: CPU tensors, NCCL: device tensors)."""
    import torch
    import torch.distributed as dist

    world = dist.get_world_size(group)
    dev = mu.device if dist.get_backend(group) == "nccl" else torch.device("cpu")
    D = mu.shape[0]
    mine = torch.cat([torch.tensor([float(K)], dtype=torch.float64, device=mu.device), mu, ss, s]).to(dev)
    out = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(out, mine, group=group)
    return [(int(t[0].item()), t[1:1 + D].to(mu.device), t[1 + D:1 + 2 * D].to(mu.device),
             t[1 + 2 * D:].to(mu.device)) for t in out]


def nested_rhat_from_moments(chainMean, chainVar, numDraws, superchainSize=1, group=None):
    """Nested R-hat from per-chain moments (see the module docstring).

    chainMean, chainVar: (D, C) per-chain means and within-chain variances (N - 1 denominator) of numDraws draws each,
    torch tensors or NumPy arrays; chains k M .. k M + M - 1 form superchain k (M = superchainSize).  group: a
    torch.distributed process group whose ranks each hold a shard of whole superchains; their parts are combined in
    rank order (Chan et al.'s pairwise update of the superchain means), so every rank gets identical numbers.  None:
    this process's chains alone.

    Returns (rhat, between, within): per-dimension nR^, B^ and W^, float64 tensors on the device of chainMean."""
    M, N = int(superchainSize), int(numDraws)
    if M < 1 or N < 1:
        raise ValueError("superchainSize and numDraws must be >= 1")
    if M == 1 and N == 1:
        raise ValueError("nested R-hat needs superchainSize > 1 or more than one draw per chain")
    mean = _as_float64(chainMean)
    var = _as_float64(chainVar).to(mean.device)
    if mean.dim() != 2 or var.shape != mean.shape:
        raise ValueError("chainMean and chainVar must both be (D, C)")
    if mean.shape[1] % M:
        raise ValueError(f"superchainSize {M} does not divide the {mean.shape[1]} chains")
    parts = [_superchain_sums(mean, var, N, M)]
    if group is not None:
        parts = _gather_parts(*parts[0], group)
    K, mu, ss, s = parts[0]
    for Kb, mub, ssb, sb in parts[1:]:
        if Kb == 0:
            continue
        if K == 0:
            K, mu, ss, s = Kb, mub, ssb, sb
            continue
        delta = mub - mu
        tot = K + Kb
        mu = mu + delta * (Kb / tot)
        ss = ss + ssb + delta * delta * (K * Kb / tot)
        s = s + sb
        K = tot
    if K < 2:
        raise ValueError(f"nested R-hat needs at least 2 superchains, got {K}")
    between = ss / (K - 1)
    within = s / K
    return (1.0 + between / within).sqrt(), between, within


def nested_rhat(draws, superchainSize=1):
    """Nested R-hat of full chains: draws (D, C, S) -- S draws of C chains, the layout of HMC.getSamples and of
    HMC.run(...)["trace"] -- as a torch tensor or NumPy array.  Returns (rhat, between, within) as
    nested_rhat_from_moments, float64 on the device of draws."""
    x = _as_float64(draws)
    if x.dim() != 3:
        raise ValueError("draws must be (D, C, S)")
    N = x.shape[2]
    if N < 1:
        raise ValueError("draws must hold at least one draw per chain")
    mean = x.mean(dim=2)
    var = (x - mean[:, :, None]).square().sum(dim=2) / (N - 1) if N > 1 else mean.new_zeros(mean.shape)
    return nested_rhat_from_moments(mean, var, N, superchainSize)
