"""Float64 NumPy reference for the Gaussian-mixture family (EHMC_FAMILY_GAUSSIAN_MIXTURE) and for the tempered run
(ehmc_hmc_run_tempered, include/ehmc.h) -- TEST INFRASTRUCTURE ONLY, used by tests/test_tempering_cpu.py and
tests/test_tempering_gpu.py.  The potential follows the interface of oracle/hmc_oracle.py (energy / grad over q of
shape (D,) or (D, P)), and the tempered loop is driven by that module's Philox stream and leapfrog.

It lives beside the tests rather than in oracle/hmc_oracle.py: that module is the port of the reference's own code and
the fixture set its golden tests pin, and the reference has neither mixtures nor replica exchange.  swap_uniform is the
bit-level specification of the replica-exchange block of the RNG stream.
"""
from __future__ import annotations

import numpy as np

from oracle import hmc_oracle as O

PHILOX_SWAP_BLOCK = 0xFFFFFFFE


class GaussianMixture:
    """U = -log sum_k w_k prod_d N(q_d; mu_kd, sigma_kd^2), without (D/2) log 2 pi and log sum_k w_k, as a max-shifted
    log-sum-exp."""

    family = 8

    def __init__(self, weights, means, stds):
        self.w = np.asarray(weights, dtype=np.float64)
        self.mu = np.asarray(means, dtype=np.float64)
        self.sd = np.asarray(stds, dtype=np.float64)
        self.c = np.log(self.w) - np.sum(np.log(self.sd), axis=1)

    def _a(self, q):
        q2 = q.reshape(q.shape[0], -1)
        x = q2[None, :, :] - self.mu[:, :, None]                        # (K, D, P)
        a = self.c[:, None] - 0.5 * np.sum(x * x / (self.sd**2)[:, :, None], axis=1)  # (K, P)
        return a, x

    def energy(self, q):
        a, _ = self._a(q)
        amax = a.max(axis=0)
        U = -(amax + np.log(np.sum(np.exp(a - amax), axis=0)))
        return U[0] if q.ndim == 1 else U

    def grad(self, q):
        a, x = self._a(q)
        r = np.exp(a - a.max(axis=0))
        r /= r.sum(axis=0)
        g = np.sum(r[:, None, :] * x / (self.sd**2)[:, :, None], axis=0)
        return g.reshape(q.shape)


def swap_uniform(seed, iteration, particle_ids, dtype=np.float64):
    """The replica-exchange uniform of the pairs whose lower particles have the given global ids at Philox iteration
    `iteration`: block 0xFFFFFFFE of the stream (oracle.hmc_oracle.philox_stream's counter and key), float32
    (x >> 8) 2^-24, float64 ((x >> 6) << 27 | y >> 5) 2^-53."""
    pid = np.asarray(particle_ids, dtype=np.uint64)
    lo, hi = pid & np.uint64(0xFFFFFFFF), pid >> np.uint64(32)
    k0 = seed & 0xFFFFFFFF
    k1 = ((seed >> 32) ^ (iteration >> 32)) & 0xFFFFFFFF
    x, y, _, _ = O.philox4x32_10(lo, hi, PHILOX_SWAP_BLOCK, iteration & 0xFFFFFFFF, k0, k1)
    if np.dtype(dtype) == np.float32:
        return (x >> np.uint32(8)).astype(np.float64) * 2.0**-24
    u53 = ((x >> np.uint32(6)).astype(np.uint64) << np.uint64(27)) | (y >> np.uint32(5)).astype(np.uint64)
    return u53.astype(np.float64) * 2.0**-53


def tempered_run(q0, mass, pot, betas, num_iterations, temperature, step_size, n_steps, seed, iteration0=0,
                 particle_offset=0, boltzmann=O.BOLTZMANN):
    """ehmc_hmc_run_tempered of one float64 ensemble, restated iteration by iteration: particle i is slot i mod R of
    system i // R; slot r draws p = z (sqrt(m kB T) (1 / sqrt(beta_r))) from philox_stream, runs the reference's
    leapfrog and rejects iff u > min(1, exp(beta_r (oldH - newH))); then the pairs (r, r + 1) with
    r = iteration (mod 2) swap iff swap_uniform < min(1, exp((beta_r - beta_r+1)(U_r - U_r+1))) (U of the kept
    states; NaN rejects).  Returns dict(q, samples (D, P, S), accepted[P], swaps[P], roundtrips[P // R],
    accept (S, P) and swap (S, P) decisions: swap[k, i] for the lower particle i of each pair proposed at k)."""
    q = np.array(q0, dtype=np.float64, copy=True)
    mass = np.asarray(mass, dtype=np.float64)
    b = np.asarray(betas, dtype=np.float64)
    R = b.shape[0]
    D, P = q.shape
    S = int(num_iterations)
    ids = np.arange(P, dtype=np.uint64) + np.uint64(particle_offset)
    lvl = np.arange(P) % R
    beta = b[lvl]
    pstd = O.momentum_std(mass, temperature, boltzmann) * (1.0 / np.sqrt(beta))
    label = np.where(lvl == 0, 1, np.where(lvl == R - 1, 2, 0))
    out = dict(samples=np.empty((D, P, S)), accepted=np.zeros(P, dtype=np.int64), swaps=np.zeros(P, dtype=np.int64),
               roundtrips=np.zeros(P // R, dtype=np.int64), accept=np.zeros((S, P), dtype=bool),
               swap=np.zeros((S, P), dtype=bool))
    for k in range(S):
        it = iteration0 + k
        z, u = O.philox_stream(seed, it, ids, D, np.float64)
        p0 = z * pstd
        q1, p1 = O.leapfrog(q, p0, mass, step_size, n_steps, pot.grad)
        U0, U1 = pot.energy(q), pot.energy(q1)
        old_h = 0.5 * np.sum(p0 * p0, axis=0) / mass + U0
        new_h = 0.5 * np.sum(p1 * p1, axis=0) / mass + U1
        with np.errstate(over="ignore", invalid="ignore"):
            reject = u > np.minimum(1, np.exp(beta * (old_h - new_h)))
        q = np.where(reject[None, :], q, q1)
        Uk = np.where(reject, U0, U1)
        out["accept"][k] = ~reject
        out["accepted"] += ~reject
        if R > 1:
            lo = np.nonzero((lvl % 2 == it % 2) & (lvl + 1 < R))[0]
            hi = lo + 1
            us = swap_uniform(seed, it, ids[lo], np.float64)
            with np.errstate(over="ignore", invalid="ignore"):
                ex = np.exp((b[lvl[lo]] - b[lvl[hi]]) * (Uk[lo] - Uk[hi]))
                acc = ~np.isnan(ex) & (us < np.minimum(1.0, ex))
            out["swap"][k, lo] = acc
            out["swaps"][lo] += acc
            s_lo, s_hi = lo[acc], hi[acc]
            q[:, s_lo], q[:, s_hi] = q[:, s_hi].copy(), q[:, s_lo].copy()
            label[s_lo], label[s_hi] = label[s_hi].copy(), label[s_lo].copy()
            cold = lvl == 0
            out["roundtrips"] += (cold & (label == 2))[cold]
            label[cold] = 1
            label[lvl == R - 1] = 2
        out["samples"][:, :, k] = q
    out["q"] = q
    return out
