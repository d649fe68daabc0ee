"""CPU oracle for the ensemble-HMC leapfrog hot path -- TEST INFRASTRUCTURE ONLY.

This module is a vectorised NumPy float64 restatement of the reference's
algorithm.  It is imported ONLY by ``tests/``, ``__graft_entry__.smoke()`` and
``bench.py``'s ``cpu_baseline`` / ``--impl reference`` legs, and there only as
the checker / timed CPU baseline.  The product package
(``physicsbasedbayesianinference_b200``) never imports it.

Parity status
-------------
* PINNED against the reference itself: ``oracle/ref_runner.py`` executes the
  UNMODIFIED files under ``/root/reference/src`` (through the ``jax`` stand-in in
  ``oracle/jax_standin``; JAX cannot be installed in this image) and
  ``tests/golden/make_golden.py`` stores their outputs under ``tests/golden``.
  ``tests/test_oracle_golden.py`` checks every function below against those
  fixtures (bit-exact for element-wise families, <=1e-13 relative where the
  reference goes through a BLAS dot whose summation order is unspecified) and
  against the reference's own known answers KA1-KA3 (SURVEY.md section 8c).
* "parity unpinned" by the reference for the models it does not contain
  (dense 100-D Gaussian, Neal's funnel, logistic regression, ensemble N-body as
  an HMC potential): for those the *loop* (rows H, J, L of SURVEY.md section 8a)
  is the reference's, driven by a NumPy float64 closed-form gradient that is
  cross-checked by finite differences in the tests.

Reference lines each function follows are cited in the docstrings
(paths relative to ``/root/reference``).
"""
from __future__ import annotations

import numpy as np

# scipy.constants values (ensemble.py:13, HMC.py:13, potential.py:13); literal so
# that the oracle does not depend on the installed SciPy's CODATA release.
BOLTZMANN = 1.380649e-23
GRAV_CONST = 6.6743e-11


# --------------------------------------------------------------------------
# Potential families (vectorised over particles: q is (D, P))
# --------------------------------------------------------------------------
class DiagGaussian:
    """harmonicPotentialND: U = 0.5 * dot(k, q**2)   (src/potential.py:18-27)."""

    family = 1

    def __init__(self, k):
        self.k = np.asarray(k, dtype=np.float64)

    def energy(self, q):
        return 0.5 * np.dot(self.k, q**2)

    def grad(self, q):
        if q.ndim == 1:
            return self.k * q
        return self.k[:, None] * q


class DenseGaussian:
    """U = 0.5 (q-mu)^T Lambda (q-mu); grad = Lambda (q-mu).

    Model of src/tests/test_HMC.py:122-125 (2-D, mean (5,5), cov [[4,-3],[-3,4]])
    scaled to config 2 (100-D).  The additive log-normaliser cancels in
    oldH - newH (src/HMC.py:108-115) and is omitted.
    """

    family = 2

    def __init__(self, precision, mean=None):
        self.prec = np.asarray(precision, dtype=np.float64)
        d = self.prec.shape[0]
        self.mean = np.zeros(d) if mean is None else np.asarray(mean, dtype=np.float64)

    def _x(self, q):
        return q - (self.mean if q.ndim == 1 else self.mean[:, None])

    def energy(self, q):
        x = self._x(q)
        return 0.5 * np.sum(x * (self.prec @ x), axis=0)

    def grad(self, q):
        return self.prec @ self._x(q)


class Funnel:
    """Neal's funnel: v = q[0] ~ N(0, s^2), q[k] ~ N(0, e^v), k = 1..D-1.

    U = v^2/(2 s^2) + 0.5 e^{-v} sum_k q_k^2 + 0.5 (D-1) v   (build-defined; SURVEY 8d C5)
    scale_v, scale_x: the same potential in rescaled coordinates, v = scale_v q[0], x_k = scale_x q[k]
    (what the build's mass adaptation produces; both 1 = the plain funnel).
    """

    family = 3

    def __init__(self, num_dims, sigma_v=3.0, scale_v=1.0, scale_x=1.0):
        self.D = int(num_dims)
        self.s = float(sigma_v)
        self.a = float(scale_v)
        self.c = float(scale_x)

    def energy(self, q):
        v = self.a * q[0]
        s2 = np.sum((self.c * q[1:]) ** 2, axis=0)
        return v * v / (2.0 * self.s**2) + 0.5 * np.exp(-v) * s2 + 0.5 * (self.D - 1) * v

    def grad(self, q):
        v = self.a * q[0]
        ev = np.exp(-v)
        x = self.c * q[1:]
        s2 = np.sum(x**2, axis=0)
        g = np.empty_like(q)
        g[0] = self.a * (v / self.s**2 - 0.5 * ev * s2 + 0.5 * (self.D - 1))
        g[1:] = self.c * (ev * x)
        return g


class CoinToss:
    """Independent coin biases under a flat prior: the reference's NumPyro sample model
    (samples/NumpyroExamples/CoinToss/CoinToss.py:21-25, Uniform(0,1) priors and Bernoulli
    observations), whose potential is -log_density (CoinTossExample.py:75-90):

        U = -sum_d [ k_d ln q_d + (n_d - k_d) ln(1 - q_d) ]
        dU/dq_d = -k_d / q_d + (n_d - k_d) / (1 - q_d)   (references/NotesOnParticleBasedHMC.pdf eq. 22)
    """

    family = 6

    def __init__(self, successes, trials):
        self.k = np.asarray(successes, dtype=np.float64).reshape(-1)
        self.n = np.asarray(trials, dtype=np.float64).reshape(-1)
        self.D = self.k.shape[0]

    def energy(self, q):
        k = self.k.reshape((-1,) + (1,) * (q.ndim - 1))
        nk = (self.n - self.k).reshape(k.shape)
        with np.errstate(invalid="ignore", divide="ignore"):
            return -np.sum(k * np.log(q) + nk * np.log(1.0 - q), axis=0)

    def grad(self, q):
        k = self.k.reshape((-1,) + (1,) * (q.ndim - 1))
        nk = (self.n - self.k).reshape(k.shape)
        with np.errstate(invalid="ignore", divide="ignore"):
            return -k / q + nk / (1.0 - q)


class NBody:
    """Pairwise gravitational potential with every ensemble particle being a
    whole B-body system.  Coordinates are flattened component-major,
    d = c*B + b, the reference's own convention (src/potential.py:83-84
    ``q.reshape(shape)`` with shape (3, N)).

    U = -G sum_{i<j} m_i m_j / sqrt(|r_i - r_j|^2 + eps^2)
        (sign as in samples/NBody/MiscFunctions.py:163-169; the src/potential.py:56-69
        version has the opposite sign -- SURVEY row N1).
    -grad_i U / m_i = G sum_{j != i} m_j (r_j - r_i)/|r_j - r_i|^3 for eps = 0, which is
    exactly src/potential.py:40-53 (getAccelNBody).
    """

    family = 4

    def __init__(self, masses, G=GRAV_CONST, eps=0.0):
        self.m = np.asarray(masses, dtype=np.float64)
        self.B = self.m.shape[0]
        self.G = float(G)
        self.eps = float(eps)

    def _r(self, q):
        q = q.reshape(3, self.B, -1)  # (3, B, P)
        return q

    def energy(self, q):
        one = q.ndim == 1
        r = self._r(q)
        dr = r[:, :, None, :] - r[:, None, :, :]  # (3, B, B, P): r_i - r_j
        d2 = np.sum(dr * dr, axis=0) + self.eps**2
        iu = np.triu_indices(self.B, 1)
        mm = (self.m[:, None] * self.m[None, :])[iu]
        U = -self.G * np.sum(mm[:, None] / np.sqrt(d2[iu]), axis=0)
        return U[0] if one else U

    def grad(self, q):
        shape = q.shape
        r = self._r(q)
        dr = r[:, :, None, :] - r[:, None, :, :]  # r_i - r_j
        d2 = np.sum(dr * dr, axis=0) + self.eps**2
        idx = np.arange(self.B)
        d2[idx, idx, :] = 1.0
        inv3 = d2 ** (-1.5)
        inv3[idx, idx, :] = 0.0
        w = self.G * self.m[:, None, None] * self.m[None, :, None] * inv3  # (B,B,P)
        g = np.sum(w[None] * dr, axis=2)  # (3, B, P)
        return g.reshape(shape)


class Logistic:
    """Bayesian logistic regression (build-defined; SURVEY 8d C3).

    U(theta) = sum_n [softplus(x_n.theta) - y_n x_n.theta] + 0.5 |theta|^2 / s^2
    grad     = X^T (sigmoid(X theta) - y) + theta / s^2
    """

    family = 5

    def __init__(self, X, y, prior_scale=1.0):
        self.X = np.asarray(X, dtype=np.float64)
        self.y = np.asarray(y, dtype=np.float64)
        self.s = float(prior_scale)

    def energy(self, q):
        one = q.ndim == 1
        th = q.reshape(q.shape[0], -1)
        s = self.X @ th  # (N, P)
        U = np.sum(np.logaddexp(0.0, s) - self.y[:, None] * s, axis=0)
        U = U + 0.5 * np.sum(th * th, axis=0) / self.s**2
        return U[0] if one else U

    def grad(self, q):
        th = q.reshape(q.shape[0], -1)
        s = self.X @ th
        r = 1.0 / (1.0 + np.exp(-s)) - self.y[:, None]
        g = self.X.T @ r + th / self.s**2
        return g.reshape(q.shape)


def get_accel_nbody(q, mass, i, G=GRAV_CONST):
    """src/potential.py:30-53 restated: acceleration of body i, q is (3, N)."""
    r = np.delete(q, i, axis=1) - q[:, [i]]
    m = np.delete(mass, i)
    return np.sum(G * m * r / np.linalg.norm(r, axis=0) ** 3, axis=1)


# --------------------------------------------------------------------------
# Integrators (src/integrator.py)
# --------------------------------------------------------------------------
def num_steps(final_time, step_size):
    """src/integrator.py:51 -- float floor, e.g. int(0.3/0.1) == 2."""
    return int(final_time / step_size)


def leapfrog(q, p, mass, step_size, n_steps, grad):
    """Leapfrog.integrate, src/integrator.py:105-120, all particles at once.

    Same element-wise arithmetic and evaluation order as the reference's
    per-particle loop; returns new (q, p) (inputs are not modified).
    """
    h = step_size
    q = np.array(q, dtype=np.float64, copy=True)
    v = p / mass  # :106
    a = -grad(q) / mass  # :108 -> :73
    for _ in range(n_steps):  # :111
        q += v * h + 0.5 * a * h**2  # :112-115
        a2 = -grad(q) / mass  # :116
        v += 0.5 * (a + a2) * h  # :117
        a = a2  # :118
    return q, v * mass  # :120


def stormer_verlet(q, p, mass, step_size, n_steps, grad):
    """StormerVerlet.integrate, src/integrator.py:142-163 (L+1 position updates,
    backward-difference velocity)."""
    h = step_size
    q = np.array(q, dtype=np.float64, copy=True)
    v = p / mass  # :143
    q_past = q.copy()  # :145
    q = q + v * h + 0.5 * (-grad(q) / mass) * h**2  # :146-150
    for _ in range(n_steps):  # :153
        tmp = q.copy()
        q = 2 * q - q_past + (-grad(q) / mass) * h**2  # :155-159
        q_past = tmp
    v = (q - q_past) / h  # :162
    return q, v * mass  # :163


def leapfrog_nbody_reference_mode(q, p, mass, step_size, n_steps, G=GRAV_CONST):
    """Leapfrog.integrate in the reference's N-body mode (gradient falsy,
    src/integrator.py:57-59,75-85): the ensemble's particles ARE the bodies and
    body i completes all its steps before body i+1 starts while reading the
    shared q (the sequential-in-time quirk, SURVEY section 3c)."""
    h = step_size
    q = np.array(q, dtype=np.float64, copy=True)
    p = np.array(p, dtype=np.float64, copy=True)
    for i in range(q.shape[1]):
        v = p[:, i] / mass[i]
        a = get_accel_nbody(q, mass, i, G)
        for _ in range(n_steps):
            q[:, i] += v * h + 0.5 * a * h**2
            a2 = get_accel_nbody(q, mass, i, G)
            v = v + 0.5 * (a + a2) * h
            a = a2
        p[:, i] = v * mass[i]
    return q, p


# --------------------------------------------------------------------------
# HMC driver (src/HMC.py, src/ensemble.py)
# --------------------------------------------------------------------------
def momentum_std(mass, temperature, boltzmann=BOLTZMANN):
    """src/ensemble.py:88 -- sqrt((mass * kB) * T), left-to-right."""
    return np.sqrt(mass * boltzmann * temperature)


def hamiltonian(q, p, mass, pot):
    """src/HMC.py:109-114: 0.5 * dot(p, p) / m + U(q)."""
    return 0.5 * np.sum(p * p, axis=0) / mass + pot.energy(q)


def hmc_iter(q, z, u, mass, temperature, step_size, n_steps, pot,
             integrator="Leapfrog", boltzmann=BOLTZMANN, bug_compat=True):
    """One pass of the getSamples loop body, src/HMC.py:154-179.

    z: (D,P) standard normals, u: (P,) uniforms, exactly the draws the reference
    takes from NumPy's global MT19937 (SURVEY row L3).
    Returns (q_next, p_stored, accept[bool P], oldH, newH).
    """
    p0 = z * momentum_std(mass, temperature, boltzmann)  # ensemble.py:88-91
    integ = leapfrog if integrator == "Leapfrog" else stormer_verlet
    q1, p1 = integ(q, p0, mass, step_size, n_steps, pot.grad)  # HMC.py:161
    old_h = hamiltonian(q, p0, mass, pot)  # :108-110
    new_h = hamiltonian(q1, -p1, mass, pot)  # :164, :111-114
    with np.errstate(over="ignore", invalid="ignore"):
        ratio = np.exp(old_h - new_h)  # :115
    acc_prob = np.minimum(1, ratio)  # :168
    reject = u > acc_prob  # :173
    q_next = np.where(reject[None, :], q, q1)  # :175
    # :176 stores oldQ (sic) into p for rejected particles; :164 only rebinds a local,
    # so the stored momentum is the UN-flipped p (SURVEY rows L1, L2).
    p_store = np.where(reject[None, :], q if bug_compat else p0, p1)
    return q_next, p_store, ~reject, old_h, new_h


def hmc_iter_diag_mass(q, z, u, mass, mass_diag, temperature, step_size, n_steps, pot, boltzmann=BOLTZMANN):
    """One HMC iteration with the DIAGONAL mass matrix M[d, i] = mass[i] * mass_diag[d], written out in the original
    coordinates (build-defined: the reference's mass is one scalar per particle, src/ensemble.py:42; this is the
    independent statement of what HMC.run(adaptMass=True) computes through rescaled coordinates, where
    mass_diag = 1 / massScale**2).  Leapfrog in kick-drift-kick form; momentum p = sqrt(M kT) z.
    Returns (q_next, accept, oldH, newH)."""
    M = mass[None, :] * np.asarray(mass_diag, dtype=np.float64)[:, None]
    p = z * np.sqrt(M * boltzmann * temperature)
    old_h = 0.5 * np.sum(p * p / M, axis=0) + pot.energy(q)
    x = q.copy()
    g = pot.grad(x)
    for _ in range(int(n_steps)):
        p = p - 0.5 * step_size * g
        x = x + step_size * p / M
        g = pot.grad(x)
        p = p - 0.5 * step_size * g
    new_h = 0.5 * np.sum(p * p / M, axis=0) + pot.energy(x)
    with np.errstate(over="ignore", invalid="ignore"):
        acc_prob = np.minimum(1, np.exp(old_h - new_h))
    reject = u > acc_prob
    return np.where(reject[None, :], q, x), ~reject, old_h, new_h


def ensemble_stats(q_kept, accept, old_h, new_h):
    """The 2D+3 ensemble statistics of one iteration (build-defined; the reference has none): the vector
    ehmc_hmc_iter returns and parallel.unpack_stats reads (physicsbasedbayesianinference_b200/parallel.py,
    csrc/k_small.cuh WarpStats), as plain float64 sums over the particles:
        [0] n_accept, [1] sum min(1, exp(oldH - newH)) (src/HMC.py:168), [2] sum H of the kept state (newH where the
        proposal was accepted, oldH where it was not, src/HMC.py:173-176), [3 .. 3+D) sum q_d, [3+D .. 3+2D) sum q_d^2
        of the kept positions q_kept (D, P).
    Non-finite energies are not handled here (the kernels count a NaN ratio as acceptance probability 1)."""
    q_kept = np.asarray(q_kept, dtype=np.float64)
    accept = np.asarray(accept, dtype=bool)
    old_h = np.asarray(old_h, dtype=np.float64)
    new_h = np.asarray(new_h, dtype=np.float64)
    with np.errstate(over="ignore"):
        acc_prob = np.minimum(1.0, np.exp(old_h - new_h))
    kept_h = np.where(accept, new_h, old_h)
    return np.concatenate([[float(np.sum(accept)), np.sum(acc_prob), np.sum(kept_h)], np.sum(q_kept, axis=1),
                           np.sum(q_kept * q_kept, axis=1)])


def adaptive_run(q0, mass, pot, num_iterations, temperature, step_size, n_steps, seed, *, iteration0=0,
                 particle_offset=0, adapt_iterations=None, target=0.8, lag=1, gain0=1.5, kappa=0.5, min_step=1e-6,
                 max_step=1e3, max_move=0.7, bug_compat=False, boltzmann=BOLTZMANN):
    """HMC.run(adapt=True, keepNumSteps=True) of one float64 ensemble, replayed iteration by iteration
    (build-defined; the reference has no adaptation):
    * iteration k draws z, u from philox_stream(seed, iteration0 + k, particle ids, D, float64) and runs hmc_iter
      (src/HMC.py:154-179) with the step size of iteration k and a fixed number of leapfrog steps;
    * its statistics (ensemble_stats) give acceptRate = n_accept / P, meanAcceptProb, meanH;
    * the Robbins-Monro rule of parallel.StepSizeAdapter, restated: for k < adapt_iterations,
          j += 1;  log h += clip(gain0 / j^kappa * (meanAcceptProb - target), -max_move, max_move),
          log h clipped to [log min_step, log max_step],  h = exp(log h)
      and the lag schedule of HMC.run(adaptLag=lag): the statistics of iteration k set the step size of iteration
      k + 1 + lag (iterations 0 .. lag keep the incoming step size, later ones the newest update).
    Returns dict(stepSize[S], acceptRate[S], meanAcceptProb[S], meanH[S], q (D, P) after the run, trace (D, P, S),
    mean[D], var[D] (moments pooled over the iterations), finalStepSize: the newest step size, what HMC.run leaves in
    HMC.stepSize)."""
    q = np.array(q0, dtype=np.float64, copy=True)
    mass = np.asarray(mass, dtype=np.float64)
    D, P = q.shape
    S = int(num_iterations)
    n_adapt = S if adapt_iterations is None else min(S, int(adapt_iterations))
    ids = np.arange(P, dtype=np.uint64) + np.uint64(particle_offset)
    log_h = np.log(step_size)
    lo, hi = np.log(min_step), np.log(max_step)
    sched = [float(step_size)] * (S + 1 + lag)  # step size of every iteration
    h_new = float(step_size)
    j = 0
    out = dict(stepSize=[], acceptRate=[], meanAcceptProb=[], meanH=[])
    trace = np.empty((D, P, S))
    sums = np.zeros(2 * D)
    for k in range(S):
        h = sched[k]
        z, u = philox_stream(seed, iteration0 + k, ids, D, np.float64)
        q, _, acc, old_h, new_h = hmc_iter(q, z, u, mass, temperature, h, n_steps, pot, boltzmann=boltzmann,
                                           bug_compat=bug_compat)
        st = ensemble_stats(q, acc, old_h, new_h)
        out["stepSize"].append(h)
        out["acceptRate"].append(st[0] / P)
        out["meanAcceptProb"].append(st[1] / P)
        out["meanH"].append(st[2] / P)
        sums += st[3:]
        trace[:, :, k] = q
        if k < n_adapt:
            acc_prob = st[1] / P if np.isfinite(st[1]) else 0.0
            j += 1
            log_h = min(max(log_h + min(max(gain0 / j**kappa * (acc_prob - target), -max_move), max_move), lo), hi)
            h_new = float(np.exp(log_h))
            for t in range(k + 1 + lag, S + 1 + lag):
                sched[t] = h_new
    n = max(S, 1) * P
    mean = sums[:D] / n
    out.update(q=q, trace=trace, mean=mean, var=sums[D:] / n - mean * mean, finalStepSize=h_new)
    return out


def get_samples(num_dims, num_particles, mass, pot, num_samples, temperature, q_std,
                simul_time, step_size, integrator="Leapfrog", record=None):
    """HMC.getSamples, src/HMC.py:123-183, drawing from NumPy's GLOBAL legacy
    MT19937 stream in the reference's order (call np.random.seed(s) first):
    standard_normal((D,P))*qStd, then per iteration standard_normal((D,P)) and
    uniform(size=P)  (SURVEY row L3; verified bit-equal to scipy's norm.rvs)."""
    D, P = num_dims, num_particles
    L = num_steps(simul_time, step_size)
    samples = np.zeros((D, P, num_samples))
    momenta = np.zeros((D, P, num_samples))
    q = np.random.standard_normal((D, P)) * q_std  # ensemble.py:72-74
    for it in range(num_samples):
        z = np.random.standard_normal((D, P))  # ensemble.py:89-91
        # the reference draws u AFTER integrating (HMC.py:170) -- same stream position
        u = np.random.uniform(size=P)
        q, p, acc, oh, nh = hmc_iter(q, z, u, mass, temperature, step_size, L, pot, integrator)
        if record is not None:
            record.append(dict(z=z, u=u, accept=acc, oldH=oh, newH=nh))
        samples[:, :, it] = q
        momenta[:, :, it] = p
    return samples, momenta


# --------------------------------------------------------------------------
# Philox4x32-10 -- specification of the engine's device RNG stream
# (build-defined; the reference only has NumPy's MT19937, which is a host stream)
# --------------------------------------------------------------------------
_M0 = np.uint64(0xD2511F53)
_M1 = np.uint64(0xCD9E8D57)
_W0 = 0x9E3779B9
_W1 = 0xBB67AE85
_MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Vectorised Philox4x32-10 (Salmon et al. 2011).  Inputs broadcastable
    uint32 arrays / ints; returns four uint32 arrays."""
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint64) & _MASK for c in (c0, c1, c2, c3))
    c0, c1, c2, c3 = np.broadcast_arrays(c0, c1, c2, c3)
    k0 = int(k0) & 0xFFFFFFFF
    k1 = int(k1) & 0xFFFFFFFF
    for _ in range(10):
        p0 = _M0 * c0
        p1 = _M1 * c2
        hi0, lo0 = p0 >> np.uint64(32), p0 & _MASK
        hi1, lo1 = p1 >> np.uint64(32), p1 & _MASK
        c0, c1, c2, c3 = (hi1 ^ c1 ^ np.uint64(k0), lo1, hi0 ^ c3 ^ np.uint64(k1), lo0)
        k0 = (k0 + _W0) & 0xFFFFFFFF
        k1 = (k1 + _W1) & 0xFFFFFFFF
    return tuple(c.astype(np.uint32) for c in (c0, c1, c2, c3))


PHILOX_UNIFORM_BLOCK = 0xFFFFFFFF
PHILOX_STREAM_VERSION = 2  # == EHMC_RNG_STREAM_VERSION (include/ehmc.h)


def philox_stream(seed, iteration, particle_ids, num_dims, dtype=np.float32):
    """The engine's production RNG stream (include/ehmc.h, "RNG stream").

    counter = (particle id low 32, particle id high 32, block, iteration low 32)
    key     = (seed low 32, seed high 32 XOR iteration high 32)
    fp32: block b yields the normals of dimensions 4b..4b+3 through two
          Box-Muller pairs (x,y)->(z0,z1), (z,w)->(z2,z3);
          u1 = ((x>>8)+1) 2^-24 in (0,1], u2 = (y>>8) 2^-24 in [0,1).
    fp64: block b yields dimensions 2b, 2b+1 from one pair built out of 53-bit
          uniforms: u1 = (((x>>6)<<27 | (y>>5)) + 1) 2^-53,  u2 = ((z>>6)<<27 | (w>>5)) 2^-53.
    Metropolis uniform (stream version 2, PHILOX_STREAM_VERSION): fp32 with D mod 4 in {1, 2} -- the last normal
          block D // 4 leaves its words z, w unused -- (z>>8) 2^-24 of THAT block; otherwise block 0xFFFFFFFF:
          fp32 (x>>8) 2^-24, fp64 ((x>>6)<<27 | y>>5) 2^-53.  (Version 1 always used block 0xFFFFFFFF.)
    Returns (z[D,P], u[P]) in float64 evaluated from the exact integer stream.
    """
    pid = np.asarray(particle_ids, dtype=np.uint64)
    lo, hi = pid & _MASK, pid >> np.uint64(32)
    k0 = seed & 0xFFFFFFFF
    k1 = ((seed >> 32) ^ (iteration >> 32)) & 0xFFFFFFFF
    it = iteration & 0xFFFFFFFF
    D = num_dims
    z = np.zeros((D, pid.shape[0]))
    if np.dtype(dtype) == np.float32:
        for b in range((D + 3) // 4):
            x, y, zz, w = philox4x32_10(lo, hi, b, it, k0, k1)
            for j, (a, c) in enumerate(((x, y), (zz, w))):
                u1 = ((a >> np.uint32(8)).astype(np.float64) + 1.0) * 2.0**-24
                u2 = (c >> np.uint32(8)).astype(np.float64) * 2.0**-24
                r = np.sqrt(-2.0 * np.log(u1))
                for t, val in enumerate((r * np.cos(2 * np.pi * u2), r * np.sin(2 * np.pi * u2))):
                    d = 4 * b + 2 * j + t
                    if d < D:
                        z[d] = val
        if D % 4 in (1, 2):
            _, _, x, _ = philox4x32_10(lo, hi, D // 4, it, k0, k1)
        else:
            x, _, _, _ = philox4x32_10(lo, hi, PHILOX_UNIFORM_BLOCK, it, k0, k1)
        u = (x >> np.uint32(8)).astype(np.float64) * 2.0**-24
    else:
        def u53(a, c):
            return ((a >> np.uint32(6)).astype(np.uint64) << np.uint64(27)) | (c >> np.uint32(5)).astype(np.uint64)

        for b in range((D + 1) // 2):
            x, y, zz, w = philox4x32_10(lo, hi, b, it, k0, k1)
            u1 = (u53(x, y).astype(np.float64) + 1.0) * 2.0**-53
            u2 = u53(zz, w).astype(np.float64) * 2.0**-53
            r = np.sqrt(-2.0 * np.log(u1))
            z[2 * b] = r * np.cos(2 * np.pi * u2)
            if 2 * b + 1 < D:
                z[2 * b + 1] = r * np.sin(2 * np.pi * u2)
        x, y, _, _ = philox4x32_10(lo, hi, PHILOX_UNIFORM_BLOCK, it, k0, k1)
        u = u53(x, y).astype(np.float64) * 2.0**-53
    return z, u


# --------------------------------------------------------------------------
# Effective sample size (build-defined; the reference has no ESS)
# --------------------------------------------------------------------------
def ess_geyer(x):
    """ESS of chains x[S, C] (S draws, C independent chains of one coordinate):
    centred on the grand mean, FFT autocovariance averaged over chains, Geyer initial-positive-sequence
    truncation.  Returns total ESS over all chains."""
    x = np.asarray(x, dtype=np.float64)
    S, C = x.shape
    xc = x - x.mean()  # grand mean: the chains are exchangeable
    n = 1 << (2 * S - 1).bit_length()
    f = np.fft.rfft(xc, n=n, axis=0)
    acov = np.fft.irfft(f * np.conj(f), n=n, axis=0)[:S] / S
    acov = acov.mean(axis=1)
    if acov[0] <= 0:
        return float(S * C)
    rho = acov / acov[0]
    tau = -1.0
    t = 0
    while t + 1 < S:
        pair = rho[t] + rho[t + 1]
        if pair < 0:
            break
        tau += 2.0 * pair
        t += 2
    tau = max(tau, 1.0 / np.log10(max(S, 10)))
    return float(S * C / tau)
