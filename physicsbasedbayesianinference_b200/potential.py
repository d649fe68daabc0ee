"""Potentials -- host mirror of the reference's ``src/potential.py``.

The reference hands arbitrary Python callables (``potential(q[:, i])``,
``gradient(q[:, i])``) to the integrator (src/integrator.py:73, src/HMC.py:102).
A GPU engine cannot call Python per particle, so potentials are *family
descriptors*: objects that are callable like the reference's functions
(``pot(q)`` -> U, ``pot.gradient(q)`` -> grad U, for ``q`` of shape (D,) or (D, P))
AND carry the family id + parameters the fused CUDA kernels consume.  Every
evaluation runs on the GPU through ``ehmc_potential_eval``; there is no CPU path.

Reference names kept: harmonicPotentialND, getAccelNBody, gravitationalPotential,
nBodyPotential, noPotential (src/potential.py:18-142).  The finite-difference
helpers nBodyForce / getForceArray are numerical-differentiation fallbacks that the
HMC path never uses (SURVEY.md section 2, row 4): they raise NotImplementedError
and point to the analytic ``.gradient``.
"""
from __future__ import annotations

import numpy as np

from . import _lib

# scipy.constants.G as imported by the reference (src/potential.py:13)
gravConst = 6.6743e-11


class Potential:
    """Base class of the potential-family descriptors."""

    family = 0

    def __init__(self, numDimensions):
        self.numDimensions = int(numDimensions)
        self._handles = {}

    # -- parameters handed to ehmc_potential_create ---------------------------------
    def _params(self):
        return []

    def _scalars(self):
        return []

    def handle(self, bits, ctx=None):
        """Device-resident parameter pack for float32/float64 kernels (cached)."""
        ctx = ctx or _lib.Context.get()
        key = (id(ctx), int(bits))
        h = self._handles.get(key)
        if h is None:
            h = _lib.PotentialHandle(ctx, self.family, self._params(), self._scalars(), bits)
            self._handles[key] = h
        return h

    # -- evaluation (always on the GPU) ------------------------------------------------
    def _eval(self, q, want_energy, want_grad):
        # the context of the device the tensor LIVES on (not the current device): the kernel is launched there
        ctx = _lib.Context.get(q.device.index if getattr(q, "is_cuda", False) else None)
        if isinstance(q, np.ndarray) or not hasattr(q, "is_cuda"):
            qa = np.asarray(q)
            one = qa.ndim == 1
            dt = np.float32 if qa.dtype == np.float32 else np.float64
            q2 = np.ascontiguousarray(qa.reshape(qa.shape[0], -1), dtype=dt)
            e = np.empty(q2.shape[1], dtype=dt) if want_energy else None
            g = np.empty_like(q2) if want_grad else None
            _lib.potential_eval(ctx, self.handle(q2.dtype.itemsize * 8, ctx), q2, e, g)
            if one:
                return (e[0] if want_energy else None), (g[:, 0] if want_grad else None)
            return e, g
        import torch

        one = q.dim() == 1
        q2 = q.reshape(q.shape[0], -1).contiguous()
        e = torch.empty(q2.shape[1], dtype=q2.dtype, device=q2.device) if want_energy else None
        g = torch.empty_like(q2) if want_grad else None
        _lib.potential_eval(ctx, self.handle(q2.element_size() * 8, ctx), q2, e, g, _lib.current_stream_ptr(q2))
        if one:
            return (e[0] if want_energy else None), (g[:, 0] if want_grad else None)
        return e, g

    def __call__(self, q):
        return self._eval(q, True, False)[0]

    def gradient(self, q):
        return self._eval(q, False, True)[1]

    # -- mass adaptation (HMC.run(adaptMass=True)) --------------------------------------
    def rescaled(self, scales):
        """The same potential in the coordinates q' = q / scales, U'(q') = U(scales * q'), as a descriptor of the
        SAME family (so the kernels are untouched).  HMC on U' with the particle's scalar mass is HMC on U with
        the diagonal mass matrix M_d = mass / scales_d**2."""
        raise NotImplementedError(f"{type(self).__name__} has no rescaled form: mass adaptation is not available "
                                  "for this family")

    def projectScales(self, scales):
        """The per-dimension scales this family can absorb (identity unless dimensions are tied)."""
        return np.asarray(scales, dtype=np.float64)


class HarmonicPotential(Potential):
    """U = 0.5 * dot(k, q**2) -- harmonicPotentialND (src/potential.py:18-27)."""

    family = _lib.FAMILY_DIAG_GAUSSIAN

    def __init__(self, springConsts):
        self.springConsts = np.atleast_1d(np.asarray(springConsts, dtype=np.float64)).copy()
        super().__init__(self.springConsts.shape[0])

    def _params(self):
        return [self.springConsts]

    def rescaled(self, scales):
        return HarmonicPotential(self.springConsts * np.asarray(scales, dtype=np.float64) ** 2)


class GaussianPotential(Potential):
    """U = 0.5 (q - mean)^T precision (q - mean): minus the log of a multivariate
    normal density up to its constant, which cancels in oldH - newH (src/HMC.py:108-115).
    The targets of src/tests/test_HMC.py:46-49 and :122-125."""

    family = _lib.FAMILY_DENSE_GAUSSIAN

    def __init__(self, precision=None, mean=None, cov=None):
        if (precision is None) == (cov is None):
            raise ValueError("give exactly one of precision= or cov=")
        if precision is None:
            precision = np.linalg.inv(np.asarray(cov, dtype=np.float64))
        self.precision = np.ascontiguousarray(precision, dtype=np.float64)
        if self.precision.ndim != 2 or self.precision.shape[0] != self.precision.shape[1]:
            raise ValueError("precision must be a square matrix")
        d = self.precision.shape[0]
        self.mean = np.zeros(d) if mean is None else np.ascontiguousarray(mean, dtype=np.float64)
        if self.mean.shape != (d,):
            raise ValueError("mean must have one entry per dimension")
        super().__init__(d)

    def _params(self):
        return [self.precision, self.mean]

    def rescaled(self, scales):
        s = np.asarray(scales, dtype=np.float64)
        return GaussianPotential(precision=self.precision * s[:, None] * s[None, :], mean=self.mean / s)


class FunnelPotential(Potential):
    """Neal's funnel: v = q[0] ~ N(0, sigmaV^2), q[k] ~ N(0, e^v).

    scaleV, scaleX: the funnel in rescaled coordinates, v = scaleV * q[0], x_k = scaleX * q[k] (one scale for all x:
    they are exchangeable) -- what mass adaptation produces (Potential.rescaled)."""

    family = _lib.FAMILY_FUNNEL

    def __init__(self, numDimensions, sigmaV=3.0, scaleV=1.0, scaleX=1.0):
        self.sigmaV = float(sigmaV)
        self.scaleV = float(scaleV)
        self.scaleX = float(scaleX)
        if not (self.scaleV > 0 and self.scaleX > 0):
            raise ValueError("scaleV and scaleX must be > 0")
        super().__init__(numDimensions)

    def _scalars(self):
        if self.scaleV == 1.0 and self.scaleX == 1.0:
            return [self.numDimensions, self.sigmaV]
        return [self.numDimensions, self.sigmaV, self.scaleV, self.scaleX]

    def projectScales(self, scales):
        s = np.array(scales, dtype=np.float64)
        s[1:] = np.sqrt(np.mean(s[1:] ** 2))  # pooled variance of the exchangeable dimensions
        return s

    def rescaled(self, scales):
        s = np.asarray(scales, dtype=np.float64)
        if not np.allclose(s[1:], s[1], rtol=1e-12):
            raise ValueError("the funnel family ties the scales of q[1:] (use projectScales)")
        return FunnelPotential(self.numDimensions, self.sigmaV, self.scaleV * s[0], self.scaleX * s[1])


class CoinTossPotential(Potential):
    """Independent coin biases q_d in (0, 1) under a flat prior -- the model of the reference's
    NumPyro sample (samples/NumpyroExamples/CoinToss/CoinToss.py:6-25):

        U(q) = -sum_d [ k_d ln q_d + (n_d - k_d) ln(1 - q_d) ]

    successes k_d out of trials n_d per coin.  The gradient -k/q + (n-k)/(1-q) vanishes at
    q = k/n (references/NotesOnParticleBasedHMC.pdf eq. 22; CoinTossExample.py:102-109)."""

    family = _lib.FAMILY_COIN_TOSS

    def __init__(self, successes, trials):
        self.successes = np.atleast_1d(np.asarray(successes, dtype=np.float64)).copy()
        self.trials = np.atleast_1d(np.asarray(trials, dtype=np.float64)).copy()
        if self.successes.shape != self.trials.shape:
            raise ValueError("successes and trials must have the same length")
        super().__init__(self.successes.shape[0])

    @classmethod
    def fromObservations(cls, *coins):
        """One 0/1 outcome array per coin, as in CoinToss.data.json (c1, c2)."""
        return cls([float(np.sum(c)) for c in coins], [float(np.size(c)) for c in coins])

    def _params(self):
        return [self.successes, self.trials]


class HierarchicalNormalPotential(Potential):
    """The normal-normal hierarchical model (NumPyro's eight-schools example):

        mu ~ N(muLoc, muScale^2),  tau ~ HalfCauchy(tauScale),  theta_j ~ N(mu, tau^2),  y_j ~ N(theta_j, sigma_j^2)

    with J groups and known sigma_j, sampled in NumPyro's unconstrained coordinates (D = J + 2):
    q[0] = mu, q[1] = eta = ln tau, q[2 + j] = theta_j (centered=True) or thetaTilde_j with
    theta_j = mu + tau thetaTilde_j (centered=False, the non-centred form that has no funnel in (eta, theta)).
    U(q) is minus the log posterior density, Jacobian of eta included, additive constants dropped.

    scale: the same potential in rescaled coordinates, U'(q) = U(scale * q) -- what mass adaptation produces
    (Potential.rescaled)."""

    family = _lib.FAMILY_HIERARCHICAL_NORMAL

    EIGHT_SCHOOLS_Y = (28.0, 8.0, -3.0, 7.0, -1.0, 1.0, 18.0, 12.0)
    EIGHT_SCHOOLS_SIGMA = (15.0, 10.0, 16.0, 11.0, 9.0, 11.0, 10.0, 18.0)

    def __init__(self, y, sigma, muLoc=0.0, muScale=5.0, tauScale=5.0, centered=False, scale=None):
        self.y = np.atleast_1d(np.asarray(y, dtype=np.float64)).copy()
        self.sigma = np.atleast_1d(np.asarray(sigma, dtype=np.float64)).copy()
        if self.y.ndim != 1 or self.sigma.shape != self.y.shape:
            raise ValueError("y and sigma must be 1-D with one entry per group")
        J = self.y.shape[0]
        if not 1 <= J <= 30:
            raise ValueError(f"the hierarchical normal kernels take 1 <= J <= 30 groups (got {J})")
        if not np.all(np.isfinite(self.y)):
            raise ValueError("y must be finite")
        if not np.all((self.sigma > 0) & np.isfinite(self.sigma)):
            raise ValueError("sigma must be > 0")
        self.muLoc, self.muScale, self.tauScale = float(muLoc), float(muScale), float(tauScale)
        if not np.isfinite(self.muLoc):
            raise ValueError("muLoc must be finite")
        if not (self.muScale > 0 and np.isfinite(self.muScale) and self.tauScale > 0 and np.isfinite(self.tauScale)):
            raise ValueError("muScale and tauScale must be > 0")
        if centered not in (True, False, 0, 1):
            raise ValueError("centered must be True or False")
        self.centered = bool(centered)
        self.scale = None if scale is None else np.asarray(scale, dtype=np.float64).copy()
        if self.scale is not None and (self.scale.shape != (J + 2,) or not np.all((self.scale > 0) & np.isfinite(self.scale))):
            raise ValueError("scale must hold J + 2 entries > 0")
        super().__init__(J + 2)

    @classmethod
    def eightSchools(cls, centered=False):
        """The eight-schools data and priors of NumPyro's example (muLoc 0, muScale 5, tauScale 5)."""
        return cls(cls.EIGHT_SCHOOLS_Y, cls.EIGHT_SCHOOLS_SIGMA, 0.0, 5.0, 5.0, centered)

    def _params(self):
        return [self.y, self.sigma] + ([] if self.scale is None else [self.scale])

    def _scalars(self):
        return [self.muLoc, self.muScale, self.tauScale, 1.0 if self.centered else 0.0]

    def rescaled(self, scales):
        s = np.asarray(scales, dtype=np.float64)
        base = np.ones(self.numDimensions) if self.scale is None else self.scale
        return HierarchicalNormalPotential(self.y, self.sigma, self.muLoc, self.muScale, self.tauScale, self.centered,
                                           scale=base * s)

    def modelParameters(self, q):
        """dict(mu, tau, theta) of positions q in this descriptor's coordinates: q is a NumPy array or a torch
        tensor of shape (D,), (D, P) or (D, P, S); mu and tau have q's shape without the first axis, theta has
        (J,) + that shape."""
        s = np.ones(self.numDimensions) if self.scale is None else self.scale
        if hasattr(q, "is_cuda"):  # torch
            import torch

            exp = torch.exp
            sv = torch.as_tensor(s, dtype=q.dtype, device=q.device)
        else:
            q = np.asarray(q, dtype=np.float64)
            exp = np.exp
            sv = s
        if q.shape[0] != self.numDimensions:
            raise ValueError(f"q must have {self.numDimensions} rows (mu, eta, J group effects)")
        st = sv[2:].reshape((-1,) + (1,) * (q.ndim - 1))
        mu = sv[0] * q[0]
        tau = exp(sv[1] * q[1])
        x = st * q[2:]
        theta = x if self.centered else mu + tau * x
        return dict(mu=mu, tau=tau, theta=theta)


class NBodyPotential(Potential):
    """Every ensemble particle is a whole B-body system; coordinates are flattened
    component-major, d = c*B + b (the reference's own convention, src/potential.py:83-84).

    U = -G sum_{i<j} m_i m_j / sqrt(|r_i - r_j|^2 + eps^2)
    (sign of samples/NBody/MiscFunctions.py:163-169; for eps = 0, -grad_i U / m_i is
    getAccelNBody, src/potential.py:30-53)."""

    family = _lib.FAMILY_NBODY

    def __init__(self, masses, G=gravConst, eps=0.0):
        self.masses = np.atleast_1d(np.asarray(masses, dtype=np.float64)).copy()
        self.G = float(G)
        self.eps = float(eps)
        super().__init__(3 * self.masses.shape[0])

    def _params(self):
        return [self.masses]

    def _scalars(self):
        return [self.G, self.eps]


class LogisticPotential(Potential):
    """Bayesian logistic regression with a N(0, priorScale^2) prior:
    U(theta) = sum_n [softplus(x_n.theta) - y_n x_n.theta] + 0.5 |theta|^2 / priorScale^2."""

    family = _lib.FAMILY_LOGISTIC

    PRECISIONS = {"fp32": 0.0, "bf16": 1.0, "fp16x3": 2.0, "auto": 3.0}

    def __init__(self, X, y, priorScale=1.0, precision="auto"):
        """precision selects the gradient kernel of float32 ensembles (float64 always runs the exact one):
        "auto" (default): the tcgen05 tensor-core GEMM chain at float32 accuracy ("fp16x3") unless the fp16
        split cannot represent X, then "fp32";  "fp16x3": force it -- every operand a 2-term fp16 split,
        3 MMA passes per GEMM, trajectories within 1e-5 of the float64 oracle (BASELINE config 3);
        "fp32": exact CUDA-core gradient;  "bf16": single-pass bf16 tensor-core chain, 2.7x faster than
        "fp16x3" but 5e-3 gradient accuracy -- outside the tolerance, opt-in only."""
        if precision not in self.PRECISIONS:
            raise ValueError("precision must be one of " + ", ".join(sorted(self.PRECISIONS)))
        self.precision = precision
        self.X = np.ascontiguousarray(X, dtype=np.float64)
        self.y = np.ascontiguousarray(y, dtype=np.float64)
        if self.X.ndim != 2 or self.y.shape != (self.X.shape[0],):
            raise ValueError("X must be (N, D) and y (N,)")
        self.priorScale = float(priorScale)
        super().__init__(self.X.shape[1])

    def _params(self):
        return [self.X, self.y]

    def _scalars(self):
        return [self.priorScale, self.PRECISIONS[self.precision]]


def _descriptor(potential):
    """Resolve what a user passed as potential=/gradient= to a descriptor."""
    if isinstance(potential, Potential):
        return potential
    owner = getattr(potential, "__self__", None)  # bound .gradient / .__call__
    if isinstance(owner, Potential):
        return owner
    raise TypeError(
        "potential/gradient must be a potential-family descriptor from "
        "physicsbasedbayesianinference_b200.potential (HarmonicPotential, GaussianPotential, "
        "FunnelPotential, ...) or its .gradient; arbitrary Python callables cannot run inside the "
        "fused CUDA trajectory kernels and this engine has no CPU fallback")


# ---------------------------------------------------------------------------
# reference-named functions (src/potential.py)
# ---------------------------------------------------------------------------
def harmonicPotentialND(q, springConsts):
    """src/potential.py:18-27 -- q is (D,) or (D, P); evaluated on the GPU."""
    return HarmonicPotential(springConsts)(q)


def getAccelNBody(q, mass, i):
    """Acceleration of the i-th body of an N-body system, q is (numDimensions=3, N)
    (src/potential.py:30-53): a_i = G sum_{j != i} m_j (r_j - r_i) / |r_j - r_i|^3, evaluated on
    the GPU as -grad_i U / m_i of the NBodyPotential family (one ensemble particle = the system)."""
    q = np.asarray(q, dtype=np.float64)
    mass = np.asarray(mass, dtype=np.float64)
    if q.shape[0] != 3:
        raise ValueError("getAccelNBody on the GPU supports 3-D positions")
    g = NBodyPotential(mass, gravConst, 0.0).gradient(np.ascontiguousarray(q).reshape(-1))
    return -g.reshape(3, -1)[:, i] / mass[i]


def gravitationalPotential(r1, r2, mass1, mass2):
    """Potential between two masses with the reference's sign, +G m1 m2 / |r1 - r2|
    (src/potential.py:56-69; note SURVEY row N1: the physical sign is the opposite)."""
    q = np.stack([np.asarray(r1, dtype=np.float64), np.asarray(r2, dtype=np.float64)], axis=1)
    return -NBodyPotential([mass1, mass2], gravConst, 0.0)(np.ascontiguousarray(q).reshape(-1))


def nBodyPotential(q, mass, shape=None):
    """src/potential.py:72-101 (reference sign: + sum_{i<j} G m_i m_j / r_ij)."""
    q = np.asarray(q, dtype=np.float64)
    if shape is not None:
        q = q.reshape(shape)
    return -NBodyPotential(mass, gravConst, 0.0)(np.ascontiguousarray(q).reshape(-1))


def noPotential(q):
    """src/potential.py:141-142."""
    return 0


def nBodyForce(q, mass):
    raise NotImplementedError(
        "nBodyForce is the reference's finite-difference fallback (src/potential.py:104-119), never used by "
        "the HMC path; use NBodyPotential(mass).gradient(q) (analytic, on the GPU)")


def getForceArray(q, potentialFunc, dq):
    """src/potential.py:122-138 computed -approx_fprime per particle; here: the analytic
    gradient of a descriptor, evaluated on the GPU."""
    return -_descriptor(potentialFunc).gradient(q)
