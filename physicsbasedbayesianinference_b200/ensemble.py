"""Ensemble -- host mirror of the reference's ``src/ensemble.py`` (the particle container).

State layout is the reference's: ``q``, ``p`` are ``(numDimensions, numParticles)``
arrays with the particle index contiguous (already structure-of-arrays),
``mass`` and ``weights`` are ``(numParticles,)``.

Two backings:
 * host (default): NumPy float64 arrays exactly like the reference; the engine
   stages them through the C-ABI's host path.  ``setPosition`` / ``setMomentum``
   draw from NumPy's global MT19937 through ``scipy.stats.norm.rvs`` like
   src/ensemble.py:72-74,88-91, so a script seeded with ``np.random.seed`` sees the
   reference's numbers.
 * device (``device="cuda"``): torch CUDA tensors (float32 by default) that the
   kernels use in place; initialisation draws from the engine's Philox stream
   (ehmc_set_position / ehmc_set_momentum).
"""
from __future__ import annotations

import numpy as np

from . import _lib

# scipy.constants.k as imported by the reference (src/ensemble.py:13)
boltzmannConst = 1.380649e-23


class Ensemble:
    """Data structure holding positions, momenta, masses and probabilistic weights
    of every particle (src/ensemble.py:17-43)."""

    def __init__(self, numDimensions, numParticles, dtype=None, device=None, seed=0, particleOffset=0):
        self.numParticles = int(numParticles)
        self.numDimensions = int(numDimensions)
        self.seed = int(seed)
        self.particleOffset = int(particleOffset)  # global index of particle 0 (multi-GPU shards)
        self._drawCount = 0
        self._posCount = 0
        if device is None:
            self.device = None
            dt = np.dtype(np.float64 if dtype is None else dtype)
            if dt not in (np.dtype(np.float32), np.dtype(np.float64)):
                raise TypeError("dtype must be float32 or float64")
            self.dtype = dt
            self.q = np.zeros((numDimensions, numParticles), dtype=dt)  # ensemble.py:40
            self.p = np.zeros((numDimensions, numParticles), dtype=dt)  # :41
            self.mass = np.ones(numParticles, dtype=dt)  # :42
            self.weights = np.zeros(numParticles, dtype=dt)  # :43
        else:
            import torch

            self.device = torch.device(device)
            if self.device.type != "cuda":
                raise ValueError("device backing must be a CUDA device (host backing: device=None)")
            tdt = {None: torch.float32, np.float32: torch.float32, np.float64: torch.float64,
                   "float32": torch.float32, "float64": torch.float64}.get(dtype, dtype)
            if tdt not in (torch.float32, torch.float64):
                raise TypeError("dtype must be float32 or float64")
            self.dtype = tdt
            self.q = torch.zeros((numDimensions, numParticles), dtype=tdt, device=self.device)
            self.p = torch.zeros((numDimensions, numParticles), dtype=tdt, device=self.device)
            self.mass = torch.ones(numParticles, dtype=tdt, device=self.device)
            self.weights = torch.zeros(numParticles, dtype=tdt, device=self.device)

    def __iter__(self):
        """Unpacking helper.  The reference's version (src/ensemble.py:45-50) returns a
        tuple naming a non-existent ``self.potential`` and raises AttributeError; this
        one yields the four arrays that exist."""
        return iter((self.q, self.p, self.mass, self.weights))

    @property
    def onDevice(self):
        return self.device is not None

    def _ctx(self):
        return _lib.Context.get(self.device.index if self.onDevice and self.device.index is not None else None)

    def setPosition(self, qStd, superchainSize=1):
        """Distribute positions with a normal distribution of standard deviation qStd
        (src/ensemble.py:63-76).  Rebinds and returns ``self.q``.

        superchainSize M > 1 starts superchains for nested R-hat (diagnostics.py): every particle takes the draw of
        the first particle of its superchain, global particle id // M.  M must divide numParticles and
        particleOffset, so that no superchain straddles two shards.  M = 1 draws exactly as before."""
        M = int(superchainSize)
        if M < 1 or self.numParticles % M or self.particleOffset % M:
            raise ValueError(f"superchainSize {superchainSize} must be >= 1 and divide numParticles "
                             f"({self.numParticles}) and particleOffset ({self.particleOffset})")
        D, P = self.numDimensions, self.numParticles
        if not self.onDevice:
            from scipy.stats import norm

            if M == 1:
                self.q = norm.rvs(scale=qStd, size=(D, P)).astype(self.dtype, copy=False)
            else:
                self.q = np.repeat(norm.rvs(scale=qStd, size=(D, P // M)), M, axis=1).astype(self.dtype, copy=False)
            return self.q
        import torch

        self.q = torch.empty((D, P), dtype=self.dtype, device=self.device)
        # fresh positions on every call, like the reference's norm.rvs: call k > 0 draws from the Philox key
        # seed XOR k * 0x9E3779B97F4A7C15 (call 0: the seed itself, the stream documented in ehmc.h)
        seed = (self.seed ^ ((self._posCount * 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF)) & 0xFFFFFFFFFFFFFFFF
        self._posCount += 1
        _lib.set_position(self._ctx(), self.q, qStd, seed, self.particleOffset,
                          _lib.current_stream_ptr(self.q))
        if M > 1:
            # the first chain's draw of every superchain (whose global id, a multiple of M, does not depend on sharding)
            self.q.copy_(self.q.view(D, P // M, M)[:, :, :1].expand(D, P // M, M).reshape(D, P))
        return self.q

    def setMomentum(self, temperature):
        """Distribute momenta thermally: p = z * sqrt(mass * kB * T) (src/ensemble.py:78-93).
        Rebinds and returns ``self.p``."""
        if not self.onDevice:
            from scipy.stats import norm

            pStd = np.sqrt(np.asarray(self.mass, dtype=np.float64) * boltzmannConst * temperature)
            self.p = norm.rvs(scale=pStd, size=(self.numDimensions, self.numParticles)).astype(self.dtype, copy=False)
            return self.p
        import torch

        self.p = torch.empty((self.numDimensions, self.numParticles), dtype=self.dtype, device=self.device)
        self._drawCount += 1
        _lib.set_momentum(self._ctx(), self.p, self.mass, boltzmannConst, temperature, self.seed,
                          (1 << 63) + self._drawCount, self.particleOffset, _lib.current_stream_ptr(self.p))
        return self.p

    def particle(self, particleNum):
        """Information about the particleNum-th particle (src/ensemble.py:95-114)."""
        if not 0 <= particleNum < self.numParticles:
            raise IndexError(f"Index {particleNum} out of bounds. " f"numParticles={self.numParticles}")
        return (
            self.q[:, particleNum],
            self.p[:, particleNum],
            self.mass[particleNum],
            self.weights[particleNum],
        )
