"""HMC driver -- host mirror of the reference's ``src/HMC.py``.

``HMC.getSamples`` keeps the reference's signature and return value
(``samples[D, P, S]``, ``momenta[D, P, S]``) but every iteration of its loop body
(src/HMC.py:154-179: momentum refresh, old Hamiltonian, trajectory, new
Hamiltonian, Metropolis test, restore) is ONE fused CUDA kernel launched through
``ehmc_hmc_iter``.

RNG.  ``rng="numpy"`` (default for host ensembles) draws the momentum normals
and the Metropolis uniforms from NumPy's global MT19937 in the reference's order
(SURVEY.md row L3) and feeds them to the kernel, so ``np.random.seed(s)`` followed
by ``getSamples`` reproduces the reference's chain.  ``rng="philox"`` (default for
device ensembles) draws inside the kernel from the counter-based Philox stream.

Reference quirks kept (SURVEY.md section 8a, rows L1/L2), both visible only in the
returned momenta: the stored momentum is the un-flipped integrated ``p``
(src/HMC.py:164 rebinds a local), and rejected particles get their OLD POSITION
written into ``p`` (src/HMC.py:176 ``= oldQ[:, mask]``, sic).  ``bugCompat=False``
stores the old momentum instead.
"""
from __future__ import annotations

from types import SimpleNamespace

import numpy as np

from . import _lib
from .ensemble import boltzmannConst
from .integrator import Leapfrog, StormerVerlet
from .potential import Potential, _descriptor


class HMC:
    """Class with getSamples method (src/HMC.py:20-71)."""

    def __init__(self, ensemble, simulTime, stepSize, density, potential=None, gradient=None, method="Leapfrog",
                 rng=None, seed=None, bugCompat=True, rejectNonFinite=None):
        """
        ensemble (Ensemble)
        simulTime (float): duration of the Hamiltonian simulation
        stepSize (float)
        density: kept for signature compatibility; a potential-family descriptor (or an
                 object with a ``.potential`` descriptor) is accepted here too
        potential: potential-family descriptor equal to -ln(density)
        gradient: optional, the descriptor's ``.gradient`` (or the descriptor)
        method (str): "Leapfrog" or "Stormer-Verlet"
        """
        self.ensemble = ensemble
        self.simulTime = simulTime
        self.stepSize = stepSize
        self.density = density

        desc = None
        for cand in (potential, gradient, density, getattr(density, "potential", None)):
            if cand is None:
                continue
            try:
                desc = _descriptor(cand)
                break
            except TypeError:
                continue
        if desc is None:
            _descriptor(potential if potential is not None else (gradient if gradient is not None else density))
        self.potential = desc
        self.gradient = desc.gradient

        if method == "Leapfrog":
            self.integrator = Leapfrog(ensemble, stepSize, simulTime, self.gradient)
        elif method == "Stormer-Verlet":
            self.integrator = StormerVerlet(ensemble, stepSize, simulTime, self.gradient)
        else:
            raise ValueError("Invalid integration method selected.")
        self.method = method

        if rng is None:
            rng = "philox" if ensemble.onDevice else "numpy"
        if rng not in ("numpy", "philox"):
            raise ValueError("rng must be 'numpy' or 'philox'")
        self.rng = rng
        self.seed = ensemble.seed if seed is None else int(seed)
        self.bugCompat = bool(bugCompat)
        # None: the reference's rule (a NaN ratio is ACCEPTED, src/HMC.py:168-173) for getSamples() / step(), rejection
        # for run() -- an adaptive ensemble run must survive the divergent trajectories its own step-size search causes
        # (funnel neck: inf - inf energies), one accepted NaN particle poisons the all-reduced moments for good
        self.rejectNonFinite = None if rejectNonFinite is None else bool(rejectNonFinite)
        self._inRun = False
        self.iteration = 0  # Philox iteration counter (persists across getSamples calls)
        self.massScale = None  # per-dimension coordinate scales of run(adaptMass=True): M_d = mass / massScale_d^2
        self.lastAccept = None

    # U(x) = -log(p(x))
    def potentialFunc(self, q):
        """Potential at position q (src/HMC.py:75-84), evaluated on the GPU."""
        return self.potential(q)

    def _kinetic(self, p):
        m = self.ensemble.mass
        return 0.5 * (p * p).sum(0) / m

    def getWeights(self, q, p):
        """exp(-H) of every particle (src/HMC.py:86-104)."""
        h = self._kinetic(p) + self.potential(q)
        return np.exp(-h) if isinstance(h, np.ndarray) else h.neg().exp()

    def getWeightsRatio(self, newQ, newP, oldQ, oldP):
        """exp(oldH - newH) of every particle (src/HMC.py:106-116)."""
        oldH = self._kinetic(oldP) + self.potential(oldQ)
        newH = self._kinetic(newP) + self.potential(newQ)
        d = oldH - newH
        return np.exp(d) if isinstance(d, np.ndarray) else d.exp()

    def print_information(self):
        print("integrator: ", self.integrator)
        print("final integration time: ", self.simulTime)
        print("time step: ", self.stepSize)

    # ------------------------------------------------------------------------------------
    def _flags(self):
        return (_lib.FLAG_BUGCOMPAT_MOMENTUM if self.bugCompat else 0) | (
            _lib.FLAG_REJECT_NONFINITE if (self._inRun if self.rejectNonFinite is None else self.rejectNonFinite) else 0)

    def _args(self, temperature, dynamic=None, reuseEndpoint=False):
        integ = _lib.LEAPFROG if self.method == "Leapfrog" else _lib.STORMER_VERLET
        flags = self._flags() | (_lib.FLAG_REUSE_ENDPOINT if reuseEndpoint else 0)
        return _lib.make_args(self.stepSize, self.stepSize**2, self.integrator.numSteps, boltzmannConst, temperature,
                              integ, flags, self.seed, self.iteration, self.ensemble.particleOffset, dynamic)

    def step(self, temperature, p_out=None, accept=None, stats=None, z=None, u=None, dynamic=None, reuseEndpoint=False):
        """One HMC iteration on ``integrator.q`` in place (the body of getSamples' loop).

        reuseEndpoint=True is the caller's promise that nothing touched ``q`` since the previous step() of
        this driver: families with an endpoint cache (logistic regression) then start the trajectory from the
        gradient and energy kept at the end of the previous one (L instead of L + 1 gradient evaluations)."""
        q = self.integrator.q
        host = isinstance(q, np.ndarray)
        ctx = _lib.Context.get(None if host else q.device.index)
        bits = (q.dtype.itemsize if host else q.element_size()) * 8
        mass = self.integrator.mass
        if host:
            mass = np.ascontiguousarray(mass, dtype=q.dtype)
        args = self._args(temperature, dynamic, reuseEndpoint)
        _lib.hmc_iter(ctx, self.potential.handle(bits, ctx), q, mass, args, p_out=p_out, z=z, u=u, accept=accept,
                      stats=stats, stream=_lib.current_stream_ptr(q))
        self.iteration += 1

    def getSamples(self, numSamples, temperature, qStd):
        """Get samples from HMC (src/HMC.py:123-183).

        Returns (samples_hmc, momentum_hmc), each (numDimensions, numParticles, numSamples),
        NumPy float64 for host ensembles, torch tensors on the device for device ensembles.
        """
        ens = self.ensemble
        D, P = ens.numDimensions, ens.numParticles
        host = not ens.onDevice
        if host:
            samples_hmc = np.zeros((D, P, numSamples))
            momentum_hmc = np.zeros_like(samples_hmc)
        else:
            import torch

            samples_hmc = torch.zeros((D, P, numSamples), dtype=ens.dtype, device=ens.device)
            momentum_hmc = torch.zeros_like(samples_hmc)

        self.print_information()
        self.integrator.q = ens.setPosition(qStd)
        dt = self.integrator.q.dtype

        if host:
            p_buf = np.empty((D, P), dtype=dt)
            acc = np.empty(P, dtype=np.uint8)
        else:
            p_buf = torch.empty((D, P), dtype=dt, device=ens.device)
            acc = torch.empty(P, dtype=torch.uint8, device=ens.device)

        if not host and self.rng == "philox" and numSamples > 0 and self._fused_loop_ok():
            # device ensemble, Philox draws, small-D family: the whole loop is ONE kernel launch
            # (ehmc_hmc_run); every iteration writes its slot of the (D, P, S) arrays directly
            for i in range(0, numSamples, 100):
                print("HMC iteration ", i + 1)
            ctx = _lib.Context.get(ens.device.index)
            bits = ens.q.element_size() * 8
            _lib.hmc_run(ctx, self.potential.handle(bits, ctx), self.integrator.q, self.integrator.mass,
                         self._args(temperature), numSamples, samples_hmc.view(D * P, numSamples),
                         momentum_hmc.view(D * P, numSamples), 0, stream=_lib.current_stream_ptr(ens.q))
            self.iteration += numSamples
            p_buf.copy_(momentum_hmc[:, :, numSamples - 1])
            self.integrator.p = p_buf
            ens.p = p_buf
            ens.q = self.integrator.q
            self.lastAccept = None
            return samples_hmc, momentum_hmc

        for i in range(numSamples):
            if i % 100 == 0:
                print("HMC iteration ", i + 1)
            z = u = None
            if self.rng == "numpy":
                # the reference's draws, in its order: norm.rvs((D,P)) for the momenta
                # (ensemble.py:89-91, == standard_normal * pStd bit for bit), then uniform(P)
                z = np.random.standard_normal((D, P))
                u = np.random.uniform(size=P)
                if host:
                    z = z.astype(dt, copy=False)
                    u = u.astype(dt, copy=False)
                else:
                    z = torch.from_numpy(z).to(device=ens.device, dtype=dt)
                    u = torch.from_numpy(u).to(device=ens.device, dtype=dt)
            # between iterations q is only read (copied into samples_hmc): the endpoint cache may be used
            self.step(temperature, p_out=p_buf, accept=acc, z=z, u=u, reuseEndpoint=i > 0)
            self.integrator.p = p_buf
            ens.p = p_buf
            samples_hmc[:, :, i] = self.integrator.q
            momentum_hmc[:, :, i] = self.integrator.p
        ens.q = self.integrator.q
        self.lastAccept = acc
        return samples_hmc, momentum_hmc


    def getSamplesTempered(self, numSamples, temperature, qStd, betas):
        """getSamples with parallel tempering (replica exchange), for multimodal targets (build-defined).

        The ensemble is cut into P / R systems of R = len(betas) adjacent particles (R in 1, 2, 4, ..., 32; P and
        particleOffset multiples of R).  Slot r of a system samples at inverse temperature betas[r]
        (1 = betas[0] > betas[1] > ... > 0): its momentum std is the usual one over sqrt(beta_r) and its Metropolis
        test uses beta_r (oldH - newH), so with boltzmannConst * temperature = 1 (temperature = 1 / boltzmannConst, as
        for getSamples) slot r targets exp(-beta_r U).  After every iteration neighbouring slots propose to exchange
        their states (deterministic even-odd schedule), so states found at high temperature reach slot 0.  The whole
        loop is one launch (ehmc_hmc_run_tempered): the pairs are R adjacent lanes of a warp and a swap is a few
        register shuffles.  betas = [1] reproduces getSamples bit for bit.

        qStd: positions drawn as in getSamples (Ensemble.setPosition), or None to continue from the ensemble's
        current positions (two calls of n iterations then give the bits of one call of 2 n).
        Device ensembles with Philox draws and small-D families only.

        Returns dict(samples (D, P, S) in level order, coldSamples (D, P / R, S): the view of slot 0, the target's
        samples; acceptRate[R], swapRate[R - 1] (float64 arrays: accepted HMC proposals per slot, accepted swaps of
        slot r with slot r + 1 per attempt); roundTrips (P / R,) int32: per system, the states that went from slot 0
        to the hottest slot and back within the call)."""
        import torch

        ens = self.ensemble
        if not ens.onDevice or self.rng != "philox":
            raise ValueError("getSamplesTempered needs a device ensemble with rng='philox' (the swap uniforms and the "
                             "momenta are drawn inside the kernel)")
        if not self._fused_loop_ok():
            raise ValueError("getSamplesTempered needs a small-D potential family (diagonal or Gaussian mixture up "
                             "to D = 32, funnel, coin toss, hierarchical normal; dense Gaussian up to D = 16)")
        b = np.atleast_1d(np.asarray(betas, dtype=np.float64))
        R = int(b.shape[0])
        D, P, S = ens.numDimensions, ens.numParticles, int(numSamples)
        dev = ens.device
        samples = torch.zeros((D, P, S), dtype=ens.dtype, device=dev)
        accepted = torch.zeros(P, dtype=torch.int32, device=dev)
        swaps = torch.zeros(P, dtype=torch.int32, device=dev)
        trips = torch.zeros(P // max(R, 1), dtype=torch.int32, device=dev)
        self.integrator.q = ens.setPosition(qStd) if qStd is not None else ens.q
        ctx = _lib.Context.get(dev.index)
        bits = ens.q.element_size() * 8
        it0 = self.iteration
        _lib.hmc_run_tempered(ctx, self.potential.handle(bits, ctx), self.integrator.q, self.integrator.mass,
                              self._args(temperature), S, R, torch.as_tensor(b, device=dev),
                              samples.view(D * P, S) if S else None, 0, accepted, swaps, trips,
                              stream=_lib.current_stream_ptr(ens.q))
        self.iteration += S
        ens.q = self.integrator.q
        self.lastAccept = None
        nsys = P // R
        # pair (r, r + 1) is proposed at the iterations k = r (mod 2)
        attempts = np.array([sum(1 for k in range(it0, it0 + S) if k % 2 == r % 2) for r in range(R - 1)], dtype=float)
        acc = accepted.view(nsys, R).sum(0).double().cpu().numpy()
        sw = swaps.view(nsys, R).sum(0).double().cpu().numpy()[:R - 1]
        with np.errstate(invalid="ignore", divide="ignore"):
            return dict(samples=samples, coldSamples=samples.view(D, nsys, R, S)[:, :, 0, :],
                        acceptRate=acc / max(S * nsys, 1), swapRate=sw / (attempts * nsys), roundTrips=trips)

    def _fused_loop_ok(self):
        """Families whose getSamples loop runs as one launch (ehmc_hmc_run)."""
        pot = self.potential
        return pot.family in (_lib.FAMILY_DIAG_GAUSSIAN, _lib.FAMILY_FUNNEL, _lib.FAMILY_COIN_TOSS,
                              _lib.FAMILY_HIERARCHICAL_NORMAL, _lib.FAMILY_GAUSSIAN_MIXTURE) and \
            pot.numDimensions <= 32 or (pot.family == _lib.FAMILY_DENSE_GAUSSIAN and pot.numDimensions <= 16)

    # ------------------------------------------------------------------------------------
    def run(self, numIterations, temperature, *, adapt=False, targetAccept=0.8, adaptIterations=None,
            traceParticles=0, group=None, collectStats=True, keepNumSteps=False, deviceAdapt=False, graph=False,
            fused=None, adaptLag=1, adaptMass=False, massWindows=3, chainDiagnostics=False, superchainSize=1):
        """Production loop for device ensembles (build-defined; scales where getSamples'
        (D, P, S) arrays cannot, SURVEY.md section 7 hard part 7).

        Every iteration is one ehmc_hmc_iter launch on the resident ensemble with in-kernel
        Philox draws.  Per-iteration ensemble statistics (2D+3 float64 sums) are produced by the
        same launch, all-reduced across the ranks of `group` asynchronously and consumed one
        iteration late (step-size adaptation, running moments).  Positions of the first
        `traceParticles` local particles are kept for ESS estimation.

        Adaptation changes the step size; by default the trajectory LENGTH simulTime stays fixed and
        numSteps = int(simulTime / stepSize) follows (src/integrator.py:51).  keepNumSteps=True keeps
        the number of leapfrog steps instead (simulTime = numSteps * stepSize follows).

        deviceAdapt=True keeps the step size and the Philox iteration counter in a device-resident
        control block (ehmc_dynamic): the trajectory kernel reads them at run time and a tiny kernel
        (ehmc_adapt_step) applies the update after the all-reduce, so the host never waits for a value
        (same one-iteration-stale pipeline as the host-side loop, same results); graph=True replays
        blocks of iterations from a CUDA graph.  The number of leapfrog steps stays fixed in this mode.
        Measured at config 5 (profiles/r01_adapt_probe.txt): host loop 285 us / iteration, device blocks
        287 us, graph 373 us -- the cross-stream edges a graph needs for the overlap cost more than the
        Python enqueue they save, so graph replay is off by default.

        fused=True runs the WHOLE call as one persistent cooperative launch (ehmc_hmc_run_ensemble, small-D
        families, Leapfrog, fixed numSteps): trajectory kernel, per-iteration statistics, their all-reduce across the
        ranks of `group` (stores into the peers' mailboxes over NVLink, inside the kernel) and the step-size update,
        with the same one-iteration-stale schedule as the host loop -- no launch, no NCCL call and no host work per
        iteration.  fused=None (default) picks it whenever it applies (statistics wanted, numSteps fixed: adapt=False
        or keepNumSteps=True); it needs CUDA IPC / peer access between the GPUs of `group`.

        adaptLag: the statistics of iteration k set the step size of iteration k + 1 + adaptLag.  1 (default) is the
        one-iteration-stale pipeline described above; 2 .. 4 leave that many iterations for the hand-out of an
        iteration's batches, its last trajectories, the reductions and the all-reduce, which is what small shards on
        many GPUs need (at 2^19 particles per GPU an iteration is 30 us and that span measured 90-100 us: 3).  The
        host loop and the fused launch implement the same schedule for every value; results do not depend on the
        number of GPUs.

        adaptMass=True adds ensemble-based diagonal MASS adaptation to the warm-up (the first adaptIterations
        iterations; needs adapt=True): at the end of each of `massWindows` windows of doubling length the all-reduced
        moments sum q_d, sum q_d^2 of the window give per-dimension scales s_d = sqrt(var_d) (parallel.MassAdapter:
        the same numbers, hence the same masses, on every rank), the ensemble is rescaled to q / s and the potential
        replaced by the same family in those coordinates (Potential.rescaled) -- HMC with the diagonal mass matrix
        M_d = mass / s_d^2, the kernels untouched.  The accumulated scales are kept in self.massScale and applied by
        later run() calls; ensemble.q is in the original coordinates whenever run() returns, and so are the returned
        mean, var (those of the last phase: after the warm-up if the call goes beyond it) and trace.  See
        _run_mass_adapt.

        chainDiagnostics=True accumulates every chain's mean and within-chain variance over the sampling window on the
        GPU (Welford, inside the fused launch or one elementwise kernel per iteration of the host loop) and returns
        nested R-hat over ALL chains of all ranks (diagnostics.py), chains k M .. k M + M - 1 of the global ensemble
        forming superchain k (M = superchainSize; start them with Ensemble.setPosition(qStd, superchainSize=M)).  The
        window is the iterations whose step size is final: adaptIterations + adaptLag .. with adapt=True (the
        non-warm-up phase with adaptMass), the whole call otherwise.  Positions, traces, step sizes and statistics are
        the same bits with and without it.  Not with deviceAdapt=True.

        Returns dict(acceptRate[S], meanAcceptProb[S], meanH[S], stepSize[S], mean[D], var[D],
        trace (D, traceParticles, S) or None); with chainDiagnostics also rhat[D], rhatBetween[D] (B^), rhatWithin[D]
        (W^) as float64 CPU tensors, chainMean and chainVar (D, P local) device tensors in the ensemble's dtype (the
        original coordinates) and rhatDraws (N, the window's length) -- all None when the window is empty.
        """
        o = SimpleNamespace(**locals())  # the options, handed on to the engines as given
        del o.self
        if adaptLag not in (1, 2, 3, 4):
            raise ValueError("adaptLag must be 1, 2, 3 or 4")
        n = int(numIterations)
        # the iterations whose statistics adapt the step size
        nAdapt = 0 if not adapt else (n if adaptIterations is None else min(n, int(adaptIterations)))
        phased = adaptMass or self.massScale is not None
        if chainDiagnostics:
            self._check_chain_diagnostics(o, n, nAdapt, phased)
        if adaptMass and not adapt:
            raise ValueError("adaptMass=True needs adapt=True (the step size must follow the mass)")
        if deviceAdapt and adaptLag != 1:
            raise ValueError("deviceAdapt=True implements adaptLag=1 only")
        if not self.ensemble.onDevice:
            raise TypeError("HMC.run needs a device-backed Ensemble (device='cuda'); use getSamples for host arrays")
        if fused and (self.method != "Leapfrog" or not self._fused_loop_ok()):
            raise ValueError("fused=True needs method='Leapfrog' and a small-D potential family (D <= 32)")
        if deviceAdapt and not fused and graph and traceParticles:
            raise ValueError("traceParticles needs graph=False (the trace slot changes every iteration)")
        # everything below runs with _inRun set: non-finite acceptance ratios are rejected unless the driver was
        # built with an explicit rejectNonFinite=False (see __init__)
        self._inRun = True
        try:
            if phased:
                return self._run_mass_adapt(o, n, nAdapt)
            return self._run_engine(o, n, adapt, nAdapt, chainDiagnostics)
        finally:
            self._inRun = False

    def _run_engine(self, o, n, adapt, nAdapt, chainDiagnostics):
        """n iterations, the first nAdapt of them adapting the step size, on the engine that applies: a whole run()
        call, or one phase of _run_mass_adapt.  n, adapt, nAdapt and chainDiagnostics are the call's or the phase's;
        the other options come from o, run()'s arguments."""
        import torch

        fused = o.fused
        if fused is None:
            fused = (o.collectStats and not o.deviceAdapt and self.method == "Leapfrog" and self._fused_loop_ok()
                     and (o.keepNumSteps or not adapt) and n > 0)
        ens = self.ensemble
        D = ens.numDimensions
        world, Ptot, ranks = self._ensemble_size(o.group)
        trace = (torch.empty((D, o.traceParticles, n), dtype=ens.dtype, device=ens.device)
                 if o.traceParticles else None)
        w0 = self._chain_window(n, nAdapt, o.adaptLag) if chainDiagnostics else n
        chains = self._chain_buffers(n, w0)
        # every engine fills hist (n, 4): acceptance rate, mean acceptance probability and mean H of the iterations
        # whose statistics it collected (the first nstat), step size of every iteration; and mom: the sums of q_d and
        # q_d^2 over those nstat iterations
        if fused:
            hist, numSteps, mom, nstat = self._run_fused(o, n, nAdapt, Ptot, trace, chains)
        elif o.deviceAdapt:
            hist, numSteps, mom, nstat = self._run_device_adapt(o, n, nAdapt, Ptot, trace)
        else:
            hist, numSteps, mom, nstat = self._run_host_loop(o, n, nAdapt, Ptot, trace, chains)
        h, m = hist.cpu().numpy(), mom.cpu().numpy()
        cnt = float(max(nstat, 1)) * Ptot
        mean = torch.from_numpy(m[:D] / cnt)
        out = dict(acceptRate=list(h[:nstat, 0]), meanAcceptProb=list(h[:nstat, 1]), meanH=list(h[:nstat, 2]),
                   stepSize=list(h[:, 3]), numSteps=numSteps, mean=mean, var=torch.from_numpy(m[D:] / cnt) - mean * mean,
                   trace=trace, worldSize=world)
        if fused:
            out["fused"] = True
        if chainDiagnostics:
            out.update(self._chain_result(chains, n - w0, o.superchainSize, ranks))
        return out

    def _ensemble_size(self, group):
        """(world size, particles of all ranks, the ranks that combine the chain diagnostics or None) for `group`.
        The total costs one NCCL all-reduce and a host read-back, so it is taken ONCE per (group, shard size) --
        repeated in every call it put ~2 ms of collective + synchronisation in front of a fused launch that runs 200
        iterations in 7 ms at 8 GPUs."""
        import torch.distributed as dist

        P = self.ensemble.numParticles
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
            return 1, float(P), None
        key = (id(group), P)
        cache = self.__dict__.setdefault("_ptotCache", {})
        if key not in cache:
            import torch

            t = torch.tensor([P], dtype=torch.float64, device=self.ensemble.device)
            dist.all_reduce(t, group=group)
            cache[key] = float(t.item())
        return dist.get_world_size(group), cache[key], group if group is not None else dist.group.WORLD

    def _keep_step_size(self, stepSize):
        """Takes over the step size an engine with a fixed number of leapfrog steps ended with."""
        self.stepSize = float(stepSize)
        self.integrator.stepSize = self.stepSize
        self.simulTime = self.integrator.finalTime = self.integrator.numSteps * self.stepSize

    # ------------------------------------------------------------------------------------
    def _chain_window(self, n, nAdapt, adaptLag, phased=False):
        """First iteration of a run() call of n iterations, nAdapt of them adapting the step size, whose positions
        enter the chain diagnostics: the first one whose step size is final (the statistics of iteration k set the
        step size of iteration k + 1 + adaptLag); with mass adaptation (phased) the first one after the warm-up
        phases."""
        if nAdapt == 0:
            return 0
        return nAdapt if phased else min(n, nAdapt + adaptLag)

    def _check_chain_diagnostics(self, o, n, nAdapt, phased):
        """run(chainDiagnostics=True)'s refusals, raised before any device work."""
        if o.deviceAdapt:
            raise ValueError("chainDiagnostics=True needs deviceAdapt=False (a graph replay would bake in the draw count)")
        ens = self.ensemble
        M = int(o.superchainSize)
        if M < 1 or ens.numParticles % M or ens.particleOffset % M:
            raise ValueError(f"superchainSize {M} must be >= 1 and divide numParticles ({ens.numParticles}) and "
                             f"particleOffset ({ens.particleOffset}): a superchain must not straddle two shards")
        N = n - self._chain_window(n, nAdapt, o.adaptLag, phased)
        if N == 1 and M == 1:
            raise ValueError("nested R-hat needs superchainSize > 1 or a window of more than one iteration")
        import torch.distributed as dist

        single = not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(o.group) == 1
        if single and ens.numParticles // M < 2:
            raise ValueError(f"nested R-hat needs at least 2 superchains, got {ens.numParticles // M}")

    def _chain_buffers(self, n, w0):
        """(mean, m2, w0): the accumulators [D, P] of the chain diagnostics over iterations w0 .. n - 1 of a call (no
        initialisation: draw 1 writes them), or None when that window is empty."""
        if w0 >= n:
            return None
        import torch

        ens = self.ensemble
        mean, m2 = (torch.empty((ens.numDimensions, ens.numParticles), dtype=ens.dtype, device=ens.device)
                    for _ in range(2))
        return mean, m2, w0

    def _chain_result(self, chains, N, M, group):
        """The result keys of run(chainDiagnostics=True) from the accumulators of N draws (group: combine the ranks)."""
        if chains is None:
            return dict(rhat=None, rhatBetween=None, rhatWithin=None, chainMean=None, chainVar=None, rhatDraws=None)
        from .diagnostics import nested_rhat_from_moments

        mean, m2, _ = chains
        var = m2 / (N - 1) if N > 1 else m2.zero_()
        rhat, between, within = nested_rhat_from_moments(mean, var, N, M, group=group)
        return dict(rhat=rhat.cpu(), rhatBetween=between.cpu(), rhatWithin=within.cpu(), chainMean=mean, chainVar=var,
                    rhatDraws=N)


    def _run_mass_adapt(self, o, n, nAdapt):
        """run() in rescaled coordinates (see run(adaptMass=True)).

        The call is cut into phases -- parallel.mass_windows during the warm-up, one phase for the rest -- and every
        phase runs on its engine (one fused launch where that applies) on the ensemble in the coordinates
        q' = q / massScale with the potential Potential.rescaled(massScale).  A window's var (all-reduced over ranks,
        pooled over the window's iterations) is the variance in the CURRENT coordinates, so the scales compose
        multiplicatively.  Step-size adaptation restarts its gain sequence in every phase (each phase starts at
        k = 1), which lets the step size follow a new mass quickly, as Stan does."""
        import torch

        from .parallel import MassAdapter, mass_windows

        ens = self.ensemble
        D = ens.numDimensions
        phases = mass_windows(nAdapt, o.massWindows) if o.adaptMass else ([(nAdapt, False)] if nAdapt else [])
        phases = [(k, upd, True) for k, upd in phases]
        if n - nAdapt > 0:
            phases.append((n - nAdapt, False, False))
        base = self.potential
        scale = np.ones(D) if self.massScale is None else np.asarray(self.massScale, dtype=np.float64)
        adapter = MassAdapter(D)

        def enter(s):
            self.potential = base if np.all(s == 1.0) else base.rescaled(s)
            return torch.as_tensor(s, dtype=ens.q.dtype, device=ens.device)[:, None]

        st = enter(scale)
        ens.q.div_(st)  # into the rescaled coordinates
        out = dict(acceptRate=[], meanAcceptProb=[], meanH=[], stepSize=[], numSteps=[], massScale=[])
        traces = []
        chainOut = dict(rhat=None, rhatBetween=None, rhatWithin=None, chainMean=None, chainVar=None, rhatDraws=None)
        r = None
        try:
            for k, updateMass, adaptive in phases:
                # the chain diagnostics' window is the phase after the warm-up (its step size and mass are final)
                r = self._run_engine(o, k, adaptive, k if adaptive else 0, o.chainDiagnostics and not adaptive)
                for key in ("acceptRate", "meanAcceptProb", "meanH", "stepSize", "numSteps"):
                    out[key].extend(r[key])
                out["massScale"].extend([scale.copy()] * k)
                if r["trace"] is not None:
                    traces.append(r["trace"] * st[:, :, None])  # original coordinates
                if r.get("chainMean") is not None:  # original coordinates; R-hat itself is scale invariant
                    sc2 = torch.from_numpy(scale * scale)
                    chainOut = dict(rhat=r["rhat"], rhatBetween=r["rhatBetween"] * sc2, rhatWithin=r["rhatWithin"] * sc2,
                                    chainMean=r["chainMean"] * st, chainVar=r["chainVar"] * (st * st),
                                    rhatDraws=r["rhatDraws"])
                if updateMass:
                    # local particles x world: not the ensemble's size when the shards are uneven
                    cnt = float(k) * float(ens.numParticles * r["worldSize"])
                    s_new = base.projectScales(adapter.scales(r["mean"].numpy(), r["var"].numpy(), cnt))
                    ens.q.div_(torch.as_tensor(s_new, dtype=ens.q.dtype, device=ens.device)[:, None])
                    scale = scale * s_new
                    st = enter(scale)
        finally:
            ens.q.mul_(st)  # back to the original coordinates
            self.potential = base
        self.massScale = None if np.all(scale == 1.0) else scale
        if r is not None:
            sc = torch.from_numpy(scale)
            out.update(mean=r["mean"] * sc, var=r["var"] * sc * sc, worldSize=r["worldSize"],
                       fused=r.get("fused", False))
        out["trace"] = torch.cat(traces, dim=2) if traces else None
        if o.chainDiagnostics:
            out.update(chainOut)
        return out

    def _run_host_loop(self, o, n, nAdapt, Ptot, trace, chains):
        """One ehmc_hmc_iter launch per iteration; returns (hist, numSteps, mom, nstat) (see _run_engine)."""
        import torch

        from .parallel import StatsReducer, StepSizeAdapter

        ens = self.ensemble
        D, dev = ens.numDimensions, ens.device
        # the options the loop reads every iteration, as locals
        temperature, collectStats, keepNumSteps, adaptLag = o.temperature, o.collectStats, o.keepNumSteps, o.adaptLag
        ntrace = o.traceParticles
        reducer = StatsReducer(o.group)
        # without keepNumSteps the trajectory length is fixed and numSteps follows the step size: a step size above
        # simulTime would mean numSteps = 0 (nothing moves, acceptance 1, the adapter runs away), so it is capped
        adapter = (StepSizeAdapter(self.stepSize, o.targetAccept, maxStep=1e3 if keepNumSteps else min(1e3, self.simulTime))
                   if nAdapt else None)
        # adaptLag + 1 statistics slots (device vector + pinned host copy + "copy done" event).  Iteration k
        # writes slot k % nslot; a side stream all-reduces it and copies it to the host behind an event,
        # so the host only ever waits for iteration k - adaptLag while iteration k is already running:
        # the GPU never idles on the statistics (they are consumed adaptLag iterations late).
        nslot = adaptLag + 1
        stats = [torch.zeros(2 * D + 3, dtype=torch.float64, device=dev) for _ in range(nslot)]
        hosts = [torch.zeros(2 * D + 3, dtype=torch.float64).pin_memory() for _ in range(nslot)]
        hosts_np = [h.numpy() for h in hosts]
        done = [torch.cuda.Event() for _ in range(nslot)]
        main = torch.cuda.current_stream(dev)
        side = torch.cuda.Stream(dev)
        hist = torch.zeros((n, 4), dtype=torch.float64)
        mom = torch.zeros(2 * D, dtype=torch.float64)
        hist_np, mom_np = hist.numpy(), mom.numpy()
        stepSizes, numSteps = [], []
        nstat = 0
        w0 = n if chains is None else chains[2]
        ctx = _lib.Context.get(dev.index)
        self.integrator.q = ens.q
        pending = []  # slots whose statistics are in flight, oldest first (at most adaptLag of them)

        def consume(slot, it):
            nonlocal nstat
            done[slot].synchronize()  # host wait: kernel `it` + all-reduce + D2H of 2D+3 doubles
            h = hosts_np[slot]
            hist_np[it, :3] = h[:3] / Ptot
            mom_np[:] += h[3:]
            nstat += 1
            if adapter is not None and it < nAdapt:
                self.stepSize = adapter.update(float(hist_np[it, 1]))
                self.integrator.stepSize = self.stepSize
                if keepNumSteps:
                    self.simulTime = self.integrator.finalTime = self.integrator.numSteps * self.stepSize
                else:
                    self.integrator.numSteps = max(1, int(self.simulTime / self.stepSize))  # src/integrator.py:51

        for it in range(n):
            slot = it % nslot
            stepSizes.append(self.stepSize)
            numSteps.append(self.integrator.numSteps)
            self.step(temperature, stats=stats[slot] if collectStats else None, reuseEndpoint=it > 0)
            if trace is not None:
                trace[:, :, it] = ens.q[:, :ntrace]
            if it >= w0:
                _lib.chain_moments_update(ctx, ens.q, chains[0], chains[1], it - w0 + 1, _lib.current_stream_ptr(ens.q))
            if collectStats:
                side.wait_stream(main)
                with torch.cuda.stream(side):
                    reducer.reduce(stats[slot])
                    hosts[slot].copy_(stats[slot], non_blocking=True)
                    done[slot].record(side)
                if len(pending) >= adaptLag:
                    consume(*pending.pop(0))  # statistics of iteration it - adaptLag
                pending.append((slot, it))
        for pd in pending:
            consume(*pd)
        main.wait_stream(side)
        hist_np[:, 3] = stepSizes
        return hist, numSteps, mom, nstat

    def _run_fused(self, o, n, nAdapt, Ptot, trace, chains):
        """HMC.run as ONE launch: see run(fused=True) and csrc/k_small_ens.cuh; returns (hist, numSteps, mom, nstat)
        (see _run_engine)."""
        import math

        import torch

        from .parallel import ensemble_comm

        ens = self.ensemble
        D, dev = ens.numDimensions, ens.device
        ctx = _lib.Context.get(dev.index)
        state = torch.tensor([self.stepSize, math.log(self.stepSize), 0.0, 0.0], dtype=torch.float64, device=dev)
        hist = torch.zeros((n, 4), dtype=torch.float64, device=dev)
        mom = torch.zeros(2 * D, dtype=torch.float64, device=dev)
        ntrace = 0 if trace is None else trace.shape[1]
        self.integrator.q = q = ens.q
        _lib.hmc_run_ensemble(ctx, self.potential.handle(q.element_size() * 8, ctx), q, self.integrator.mass,
                              self._args(o.temperature), n,
                              _lib.make_adapt_args(Ptot, nAdapt, target=o.targetAccept, lag=o.adaptLag), state,
                              comm=ensemble_comm(ctx, o.group, dev), history=hist, moments=mom,
                              trace=None if trace is None else trace.view(D * ntrace, n), trace_particles=ntrace,
                              stream=_lib.current_stream_ptr(q), chains=chains)
        self.iteration += n
        self._keep_step_size(state[0].item())  # synchronises
        return hist, [self.integrator.numSteps] * n, mom, n

    def _run_device_adapt(self, o, n, nAdapt, Ptot, trace, graphIterations=10):
        """Two control blocks used alternately: iteration k runs with block k & 1; on a side stream the
        statistics of iteration k are all-reduced and ehmc_adapt_step writes the block iteration k + 2
        will read, taking the adaptation state from the other block.  Iteration k + 1 therefore only
        waits for the update computed from iteration k - 1 (the one-iteration-stale pipeline of the
        host-side loop) and the all-reduce overlaps iteration k + 1.  Returns (hist, numSteps, mom, nstat)
        (see _run_engine)."""
        import torch

        from .parallel import StatsReducer

        ens = self.ensemble
        D, dev = ens.numDimensions, ens.device
        reducer = StatsReducer(o.group)
        ctx = _lib.Context.get(dev.index)
        it0 = self.iteration
        blocks = [_lib.dynamic_to_device(self.stepSize, it0 + b, dev, row=b) for b in range(2)]
        stats = [torch.zeros(2 * D + 3, dtype=torch.float64, device=dev) for _ in range(2)]
        hist = torch.zeros((n, 4), dtype=torch.float64, device=dev)
        mom = torch.zeros(2 * D, dtype=torch.float64, device=dev)
        self.integrator.q = ens.q
        # high priority: the 1-block update kernel and the small all-reduce must not queue behind the
        # thousands of CTAs of the running trajectory kernel
        side = torch.cuda.Stream(dev, priority=-1)

        def enqueue(k0, count, main):
            """Iterations k0 .. k0 + count - 1 on `main` + `side`; joins the two streams at the end."""
            ran = [None, None]      # per parity: event "kernel + statistics of this parity done"
            adapted = [None, None]  # per parity: event "block of this parity rewritten"
            for k in range(k0, k0 + count):
                b = k & 1
                if adapted[b] is not None:
                    main.wait_event(adapted[b])  # block b and stats[b] are free / up to date
                self.step(o.temperature, stats=stats[b], dynamic=blocks[b].data_ptr())
                if trace is not None:
                    trace[:, :, k] = ens.q[:, :o.traceParticles]
                ran[b] = torch.cuda.Event()
                ran[b].record(main)
                with torch.cuda.stream(side):
                    side.wait_event(ran[b])
                    reducer.reduce(stats[b])
                    _lib.adapt_step(ctx, stats[b], Ptot, blocks[b].data_ptr(), target=o.targetAccept,
                                    adapt_rows=nAdapt, state_ptr=blocks[1 - b].data_ptr(), stride=2, history=hist,
                                    moments=mom, stream=_lib.current_stream_ptr(stats[b]))
                    adapted[b] = torch.cuda.Event()
                    adapted[b].record(side)
            main.wait_stream(side)

        main = torch.cuda.current_stream(dev)
        side.wait_stream(main)
        G = int(graphIterations) & ~1
        if o.graph and G >= 2 and n >= 2 + G:
            # eager head: sizes the library's scratch buffers outside the capture and leaves a multiple of G
            head = 2 + (n - 2) % G
            enqueue(0, head, main)
            g = torch.cuda.CUDAGraph()
            cap = torch.cuda.Stream(dev)
            cap.wait_stream(main)
            with torch.cuda.stream(cap):
                # capture executes nothing; step size / iteration / history row advance on the device at replay
                with torch.cuda.graph(g, stream=cap):
                    enqueue(head, G, cap)
            main.wait_stream(cap)
            self.iteration = it0 + head  # the captured calls advanced the host counter; it is reset below anyway
            for _ in range((n - head) // G):
                g.replay()
        else:
            enqueue(0, n, main)
        self.iteration = it0 + n
        self._keep_step_size(_lib.dynamic_from_device(blocks[(n - 1) & 1 if n else 0]).stepSize)  # synchronises
        return hist, [self.integrator.numSteps] * n, mom, n


class GaussianDensity:
    """Density object for the ``density`` argument: a multivariate normal whose
    ``.potential`` is the matching GaussianPotential descriptor (the role played by
    ``lambda q: multivariate_normal.pdf(q, mean, cov)`` in src/tests/test_HMC.py:48)."""

    def __init__(self, mean, cov):
        from .potential import GaussianPotential

        self.mean = np.asarray(mean, dtype=np.float64)
        self.cov = np.asarray(cov, dtype=np.float64)
        self.potential = GaussianPotential(cov=self.cov, mean=self.mean)
        d = self.mean.shape[0]
        self._lognorm = 0.5 * (d * np.log(2 * np.pi) + np.linalg.slogdet(self.cov)[1])

    def __call__(self, q):
        u = self.potential(q)
        return np.exp(-(u + self._lognorm)) if isinstance(u, (np.ndarray, np.floating, float)) else (-(u + self._lognorm)).exp()
