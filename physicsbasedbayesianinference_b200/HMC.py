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


    def _fused_loop_ok(self):
        """Families whose getSamples loop runs as one launch (ehmc_hmc_run)."""
        pot = self.potential
        return pot.family in (_lib.FAMILY_DIAG_GAUSSIAN, _lib.FAMILY_FUNNEL, _lib.FAMILY_COIN_TOSS,
                              _lib.FAMILY_HIERARCHICAL_NORMAL) and \
            pot.numDimensions <= 32 or (pot.family == _lib.FAMILY_DENSE_GAUSSIAN and pot.numDimensions <= 16)

    # ------------------------------------------------------------------------------------
    def run(self, numIterations, temperature, *, adapt=False, targetAccept=0.8, adaptIterations=None,
            traceParticles=0, group=None, collectStats=True, keepNumSteps=False, deviceAdapt=False, graph=False,
            fused=None, adaptLag=1, adaptMass=False, massWindows=3):
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
        with the same one-iteration-stale schedule as the loop below -- no launch, no NCCL call and no host work per
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

        Returns dict(acceptRate[S], meanAcceptProb[S], meanH[S], stepSize[S], mean[D], var[D],
        trace (D, traceParticles, S) or None).
        """
        if adaptLag not in (1, 2, 3, 4):
            raise ValueError("adaptLag must be 1, 2, 3 or 4")
        if not self._inRun:
            # everything below runs with _inRun set: non-finite acceptance ratios are rejected unless the driver was
            # built with an explicit rejectNonFinite=False (see __init__)
            self._inRun = True
            try:
                return self.run(numIterations, temperature, adapt=adapt, targetAccept=targetAccept,
                                adaptIterations=adaptIterations, traceParticles=traceParticles, group=group,
                                collectStats=collectStats, keepNumSteps=keepNumSteps, deviceAdapt=deviceAdapt,
                                graph=graph, fused=fused, adaptLag=adaptLag, adaptMass=adaptMass,
                                massWindows=massWindows)
            finally:
                self._inRun = False
        if adaptMass or getattr(self, "massScale", None) is not None:
            if adaptMass and not adapt:
                raise ValueError("adaptMass=True needs adapt=True (the step size must follow the mass)")
            return self._run_mass_adapt(numIterations, temperature, adaptMass=adaptMass, massWindows=massWindows,
                                        adapt=adapt, targetAccept=targetAccept, adaptIterations=adaptIterations,
                                        traceParticles=traceParticles, group=group, collectStats=collectStats,
                                        keepNumSteps=keepNumSteps, deviceAdapt=deviceAdapt, graph=graph, fused=fused,
                                        adaptLag=adaptLag)
        if deviceAdapt and adaptLag != 1:
            raise ValueError("deviceAdapt=True implements adaptLag=1 only")
        if fused is None:
            fused = (collectStats and not deviceAdapt and self.ensemble.onDevice and self.method == "Leapfrog"
                     and self._fused_loop_ok() and (keepNumSteps or not adapt) and numIterations > 0)
        if fused:
            return self._run_fused(numIterations, temperature, adapt, targetAccept, adaptIterations, traceParticles,
                                   group, adaptLag)
        if deviceAdapt:
            return self._run_device_adapt(numIterations, temperature, adapt, targetAccept, adaptIterations,
                                          traceParticles, group, graph)
        import torch

        from .parallel import StatsReducer, StepSizeAdapter, unpack_stats

        ens = self.ensemble
        if not ens.onDevice:
            raise TypeError("HMC.run needs a device-backed Ensemble (device='cuda'); use getSamples for host arrays")
        D, P = ens.numDimensions, ens.numParticles
        dev = ens.device
        reducer = StatsReducer(group)
        world = reducer.dist.get_world_size(group) if reducer.enabled else 1
        Ptot = float(P)
        if reducer.enabled:
            t = torch.tensor([P], dtype=torch.float64, device=dev)
            reducer.dist.all_reduce(t, group=group)
            Ptot = float(t.item())
        # without keepNumSteps the trajectory length is fixed and numSteps follows the step size: a step size above
        # simulTime would mean numSteps = 0 (nothing moves, acceptance 1, the adapter runs away), so it is capped
        adapter = (StepSizeAdapter(self.stepSize, targetAccept, maxStep=1e3 if keepNumSteps else min(1e3, self.simulTime))
                   if adapt else None)
        adaptIterations = numIterations if adaptIterations is None else adaptIterations
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
        out = dict(acceptRate=[], meanAcceptProb=[], meanH=[], stepSize=[], numSteps=[])
        sum1 = np.zeros(D)
        sum2 = np.zeros(D)
        nstat = 0
        trace = (torch.empty((D, traceParticles, numIterations), dtype=ens.dtype, device=dev)
                 if traceParticles else None)
        self.integrator.q = ens.q
        pending = []  # slots whose statistics are in flight, oldest first (at most adaptLag of them)

        def consume(slot, it):
            nonlocal nstat
            done[slot].synchronize()  # host wait: kernel `it` + all-reduce + D2H of 2D+3 doubles
            h = hosts_np[slot]
            acc_prob = float(h[1]) / Ptot
            out["acceptRate"].append(float(h[0]) / Ptot)
            out["meanAcceptProb"].append(acc_prob)
            out["meanH"].append(float(h[2]) / Ptot)
            sum1[:] += h[3:3 + D]
            sum2[:] += h[3 + D:3 + 2 * D]
            nstat += 1
            if adapter is not None and it < adaptIterations:
                self.stepSize = adapter.update(acc_prob)
                self.integrator.stepSize = self.stepSize
                if keepNumSteps:
                    self.simulTime = self.integrator.finalTime = self.integrator.numSteps * self.stepSize
                else:
                    self.integrator.numSteps = max(1, int(self.simulTime / self.stepSize))  # src/integrator.py:51

        for it in range(numIterations):
            slot = it % nslot
            out["stepSize"].append(self.stepSize)
            out["numSteps"].append(self.integrator.numSteps)
            self.step(temperature, stats=stats[slot] if collectStats else None, reuseEndpoint=it > 0)
            if trace is not None:
                trace[:, :, it] = ens.q[:, :traceParticles]
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
        sum1 = torch.from_numpy(sum1)
        sum2 = torch.from_numpy(sum2)
        n = max(nstat, 1) * Ptot
        mean = sum1 / n
        out.update(mean=mean, var=sum2 / n - mean * mean, trace=trace, worldSize=world)
        return out


    def _run_mass_adapt(self, numIterations, temperature, *, adaptMass, massWindows, adapt, adaptIterations,
                        traceParticles, **kw):
        """run() in rescaled coordinates (see run(adaptMass=True)).

        The call is cut into phases -- parallel.mass_windows during the warm-up, one phase for the rest -- and every
        phase is an ordinary run() (one fused launch where that applies) on the ensemble in the coordinates
        q' = q / massScale with the potential Potential.rescaled(massScale).  A window's var (returned by its run(),
        all-reduced over ranks, pooled over the window's iterations) is the variance in the CURRENT coordinates, so
        the scales compose multiplicatively.  Step-size adaptation restarts its gain sequence in every phase (each
        run() call starts at k = 1), which lets the step size follow a new mass quickly, as Stan does."""
        import torch

        from .parallel import MassAdapter, mass_windows

        ens = self.ensemble
        if not ens.onDevice:
            raise TypeError("HMC.run needs a device-backed Ensemble (device='cuda')")
        D = ens.numDimensions
        n = int(numIterations)
        nAdapt = 0 if not adapt else (n if adaptIterations is None else min(n, int(adaptIterations)))
        phases = mass_windows(nAdapt, massWindows) if adaptMass else ([(nAdapt, False)] if nAdapt else [])
        phases = [(k, upd, True) for k, upd in phases]
        if n - nAdapt > 0:
            phases.append((n - nAdapt, False, False))
        base = self.potential
        scale = np.ones(D) if getattr(self, "massScale", None) is None else np.asarray(self.massScale, dtype=np.float64)
        self.massScale = None  # (the phases below are plain run() calls)
        adapter = MassAdapter(D)

        def enter(s):
            self.potential = base if np.all(s == 1.0) else base.rescaled(s)
            return torch.as_tensor(s, dtype=ens.q.dtype, device=ens.device)[:, None]

        st = enter(scale)
        ens.q.div_(st)  # into the rescaled coordinates
        out = dict(acceptRate=[], meanAcceptProb=[], meanH=[], stepSize=[], numSteps=[], massScale=[])
        traces = []
        r = None
        try:
            for k, updateMass, adaptive in phases:
                r = self.run(k, temperature, adapt=adaptive, adaptIterations=k if adaptive else 0,
                             traceParticles=traceParticles, **kw)
                for key in ("acceptRate", "meanAcceptProb", "meanH", "stepSize", "numSteps"):
                    out[key].extend(r[key])
                out["massScale"].extend([scale.copy()] * k)
                if r["trace"] is not None:
                    traces.append(r["trace"] * st[:, :, None])  # original coordinates
                if updateMass:
                    cnt = float(k) * float(r.get("numParticlesTotal", ens.numParticles * r.get("worldSize", 1)))
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
            out.update(mean=r["mean"] * sc, var=r["var"] * sc * sc, worldSize=r.get("worldSize", 1),
                       fused=r.get("fused", False))
        out["trace"] = torch.cat(traces, dim=2) if traces else None
        return out

    def _run_fused(self, numIterations, temperature, adapt, targetAccept, adaptIterations, traceParticles, group,
                   adaptLag=1):
        """HMC.run as ONE launch: see run(fused=True) and csrc/k_small_ens.cuh."""
        import math

        import torch

        from .parallel import ensemble_comm

        ens = self.ensemble
        if not ens.onDevice:
            raise TypeError("HMC.run needs a device-backed Ensemble (device='cuda')")
        if self.method != "Leapfrog" or not self._fused_loop_ok():
            raise ValueError("fused=True needs method='Leapfrog' and a small-D potential family (D <= 32)")
        D, P, dev = ens.numDimensions, ens.numParticles, ens.device
        ctx = _lib.Context.get(dev.index)
        comm = ensemble_comm(ctx, group, dev)
        world, Ptot = 1, float(P)
        if comm is not None:
            import torch.distributed as dist

            world = dist.get_world_size(group)
            # the ensemble size over all ranks: one NCCL all-reduce and a host read-back, ONCE per (group, shard
            # size) -- repeated in every call it put ~2 ms of collective + synchronisation in front of a launch
            # that runs 200 iterations in 7 ms at 8 GPUs
            key = (id(group), P)
            cache = self.__dict__.setdefault("_ptotCache", {})
            if key not in cache:
                t = torch.tensor([P], dtype=torch.float64, device=dev)
                dist.all_reduce(t, group=group)
                cache[key] = float(t.item())
            Ptot = cache[key]
        n = int(numIterations)
        adaptRows = 0 if not adapt else (n if adaptIterations is None else min(n, int(adaptIterations)))
        state = torch.tensor([self.stepSize, math.log(self.stepSize), 0.0, 0.0], dtype=torch.float64, device=dev)
        hist = torch.zeros((n, 4), dtype=torch.float64, device=dev)
        mom = torch.zeros(2 * D, dtype=torch.float64, device=dev)
        ntrace = int(traceParticles)
        trace = torch.empty((D, ntrace, n), dtype=ens.dtype, device=dev) if ntrace else None
        self.integrator.q = ens.q
        numSteps = self.integrator.numSteps
        q = ens.q
        bits = q.element_size() * 8
        _lib.hmc_run_ensemble(ctx, self.potential.handle(bits, ctx), q, self.integrator.mass, self._args(temperature), n,
                              _lib.make_adapt_args(Ptot, adaptRows, target=targetAccept, lag=adaptLag), state, comm=comm,
                              history=hist,
                              moments=mom, trace=None if trace is None else trace.view(D * ntrace, n),
                              trace_particles=ntrace, stream=_lib.current_stream_ptr(q))
        self.iteration += n
        st = state.cpu().numpy()  # synchronises
        self.stepSize = float(st[0])
        self.integrator.stepSize = self.stepSize
        self.simulTime = self.integrator.finalTime = numSteps * self.stepSize
        h = hist.cpu().numpy()
        m = mom.cpu().numpy()
        cnt = float(max(n, 1)) * Ptot
        mean = torch.from_numpy(m[:D] / cnt)
        return dict(acceptRate=list(h[:, 0]), meanAcceptProb=list(h[:, 1]), meanH=list(h[:, 2]), stepSize=list(h[:, 3]),
                    numSteps=[numSteps] * n, mean=mean, var=torch.from_numpy(m[D:] / cnt) - mean * mean,
                    trace=trace, worldSize=world, fused=True)

    def _run_device_adapt(self, numIterations, temperature, adapt, targetAccept, adaptIterations, traceParticles,
                          group, graph, graphIterations=10):
        """Two control blocks used alternately: iteration k runs with block k & 1; on a side stream the
        statistics of iteration k are all-reduced and ehmc_adapt_step writes the block iteration k + 2
        will read, taking the adaptation state from the other block.  Iteration k + 1 therefore only
        waits for the update computed from iteration k - 1 (the one-iteration-stale pipeline of the
        host-side loop) and the all-reduce overlaps iteration k + 1."""
        import torch

        from .parallel import StatsReducer

        ens = self.ensemble
        if not ens.onDevice:
            raise TypeError("HMC.run needs a device-backed Ensemble (device='cuda')")
        if graph and traceParticles:
            raise ValueError("traceParticles needs graph=False (the trace slot changes every iteration)")
        D, P, dev = ens.numDimensions, ens.numParticles, ens.device
        reducer = StatsReducer(group)
        world = reducer.dist.get_world_size(group) if reducer.enabled else 1
        Ptot = float(P)
        if reducer.enabled:
            t = torch.tensor([P], dtype=torch.float64, device=dev)
            reducer.dist.all_reduce(t, group=group)
            Ptot = float(t.item())
        ctx = _lib.Context.get(dev.index)
        adaptRows = 0 if not adapt else (numIterations if adaptIterations is None else adaptIterations)
        it0 = self.iteration
        blocks = [_lib.dynamic_to_device(self.stepSize, it0 + b, dev, row=b) for b in range(2)]
        stats = [torch.zeros(2 * D + 3, dtype=torch.float64, device=dev) for _ in range(2)]
        hist = torch.zeros((numIterations, 4), dtype=torch.float64, device=dev)
        mom = torch.zeros(2 * D, dtype=torch.float64, device=dev)
        trace = (torch.empty((D, traceParticles, numIterations), dtype=ens.dtype, device=dev)
                 if traceParticles else None)
        self.integrator.q = ens.q
        numSteps = self.integrator.numSteps
        # high priority: the 1-block update kernel and the small all-reduce must not queue behind the
        # thousands of CTAs of the running trajectory kernel
        side = torch.cuda.Stream(dev, priority=-1)

        def enqueue(k0, n, main):
            """Iterations k0 .. k0 + n - 1 on `main` + `side`; joins the two streams at the end."""
            ran = [None, None]      # per parity: event "kernel + statistics of this parity done"
            adapted = [None, None]  # per parity: event "block of this parity rewritten"
            for k in range(k0, k0 + n):
                b = k & 1
                if adapted[b] is not None:
                    main.wait_event(adapted[b])  # block b and stats[b] are free / up to date
                self.step(temperature, stats=stats[b], dynamic=blocks[b].data_ptr())
                if trace is not None:
                    trace[:, :, k] = ens.q[:, :traceParticles]
                ran[b] = torch.cuda.Event()
                ran[b].record(main)
                with torch.cuda.stream(side):
                    side.wait_event(ran[b])
                    reducer.reduce(stats[b])
                    _lib.adapt_step(ctx, stats[b], Ptot, blocks[b].data_ptr(), target=targetAccept,
                                    adapt_rows=adaptRows, state_ptr=blocks[1 - b].data_ptr(), stride=2, history=hist,
                                    moments=mom, stream=_lib.current_stream_ptr(stats[b]))
                    adapted[b] = torch.cuda.Event()
                    adapted[b].record(side)
            main.wait_stream(side)

        main = torch.cuda.current_stream(dev)
        side.wait_stream(main)
        G = int(graphIterations) & ~1
        if graph and G >= 2 and numIterations >= 2 + G:
            # eager head: sizes the library's scratch buffers outside the capture and leaves a multiple of G
            head = 2 + (numIterations - 2) % G
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
            for _ in range((numIterations - head) // G):
                g.replay()
        else:
            enqueue(0, numIterations, main)
        self.iteration = it0 + numIterations
        newest = _lib.dynamic_from_device(blocks[(numIterations - 1) & 1 if numIterations else 0])  # synchronises
        self.stepSize = float(newest.stepSize)
        self.integrator.stepSize = self.stepSize
        self.simulTime = self.integrator.finalTime = numSteps * self.stepSize
        h = hist.cpu().numpy()
        m = mom.cpu().numpy()
        n = float(max(numIterations, 1)) * Ptot
        mean = torch.from_numpy(m[:D] / n)
        return dict(acceptRate=list(h[:, 0]), meanAcceptProb=list(h[:, 1]), meanH=list(h[:, 2]), stepSize=list(h[:, 3]),
                    numSteps=[numSteps] * numIterations, mean=mean, var=torch.from_numpy(m[D:] / n) - mean * mean,
                    trace=trace, worldSize=world)


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
