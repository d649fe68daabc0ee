"""Chain diagnostics on the GPU (pytest -m gpu): the per-chain moments HMC.run(chainDiagnostics=True) accumulates --
inside the fused launch (k_small_ens) or with k_chain_moments after every iteration of the host loop -- against
float64 NumPy over the window of the full trace, nested R-hat against diagnostics.nested_rhat on that trace, the
fused run against the host loop, the absence of any effect on the sampler, mass adaptation's coordinates, the
behaviour of R-hat on a Gaussian, and the combination over two ranks."""
import os

import numpy as np
import pytest

from oracle import hmc_oracle as O

pytestmark = pytest.mark.gpu

KB = O.BOLTZMANN
TEMP = 1 / KB
# the context's defaults (csrc/host_defs.h); the context is one per process, shared with every other test module
DEFAULT_OPTIONS = {"small_waves": 8, "ens_sshift": -1, "ens_groups": 0, "dense_path": 0}
ITERS, ADAPT = 16, 6


@pytest.fixture(scope="module")
def E():
    import physicsbasedbayesianinference_b200 as pkg

    pkg._lib.Context.get()  # fails loudly when the extension or the GPU is missing
    return pkg


@pytest.fixture
def options(E):
    """set_options(name=value, ...) on the context; every option in DEFAULT_OPTIONS is restored afterwards."""
    ctx = E._lib.Context.get()

    def set_options(**kw):
        for name, value in kw.items():
            ctx.set_option(name, value)

    try:
        yield set_options
    finally:
        for name, value in DEFAULT_OPTIONS.items():
            ctx.set_option(name, value)


def host(t):
    return t.double().cpu().numpy()


def small_family(E, name, D, rng):
    """(descriptor, step size, start (D, P) sampler) of a small-D family at width D."""
    if name == "dense":
        A = rng.standard_normal((D, D))
        return E.GaussianPotential(precision=A @ A.T / D + np.eye(D)), 0.15
    if name == "diag":
        return E.HarmonicPotential(rng.uniform(0.5, 4.0, D)), 0.1
    if name == "funnel":
        return E.FunnelPotential(D, 3.0), 0.05
    assert name == "hier" and D == 10
    return E.HierarchicalNormalPotential.eightSchools(centered=False), 0.1


def check_against_trace(r, w0, M, dt, where):
    """chainMean / chainVar against float64 NumPy over iterations w0 .. of the trace, R-hat against
    diagnostics.nested_rhat on the same draws."""
    from physicsbasedbayesianinference_b200 import diagnostics

    tr = host(r["trace"])[:, :, w0:]
    N = tr.shape[2]
    assert r["rhatDraws"] == N, where
    mean_t = tr.mean(axis=2)
    var_t = tr.var(axis=2, ddof=1)
    mean_g, var_g = host(r["chainMean"]), host(r["chainVar"])
    assert r["chainMean"].dtype == r["trace"].dtype and r["chainVar"].dtype == r["trace"].dtype, where
    scale = np.abs(mean_t) + np.sqrt(var_t)
    if dt == np.float64:
        assert np.all(np.abs(mean_g - mean_t) <= 1e-12 * scale), where
        assert np.all(np.abs(var_g - var_t) <= 1e-12 * np.maximum(var_t, 1e-12 * scale * scale)), where
    else:
        assert np.all(np.abs(mean_g - mean_t) <= 1e-5 * scale), where
        # beyond the 1e-4 relative bound: float32 Welford rounds d = q - mean and the mean at |q|, so a chain whose
        # |mean| >> sd carries an absolute error of a few float32 ulps of |mean| times sd in its variance
        assert np.all(np.abs(var_g - var_t) <= 1e-4 * var_t + 1e-5 * scale * np.sqrt(var_t)), where
    ref = diagnostics.nested_rhat(tr, superchainSize=M)
    assert r["rhat"].dtype.is_floating_point and r["rhat"].device.type == "cpu" and r["rhat"].shape == mean_t.shape[:1]
    if dt == np.float64:
        for key, want in zip(("rhat", "rhatBetween", "rhatWithin"), ref):
            np.testing.assert_allclose(r[key].numpy(), want.numpy(), rtol=1e-10, err_msg=f"{where} {key}")
    else:
        np.testing.assert_allclose(r["rhat"].numpy(), ref[0].numpy(), rtol=0, atol=1e-5, err_msg=where)


# (family, D, sshift, P, adaptLag, adapt, superchainSize): exact (funnel, hierarchical: DT = 10) and padded widths
# (dense 3 -> 4, diagonal 17 -> 32), every queue item size, ragged last batches (P not a multiple of 32)
FUSED_CASES = [
    ("dense", 3, 0, 1000, 1, True, 4),
    ("diag", 17, 1, 2080, 4, True, 32),
    ("funnel", 10, 2, 4004, 1, False, 1),
    ("hier", 10, 0, 968, 4, False, 4),
    ("funnel", 10, 1, 1200, 4, True, 4),
    ("hier", 10, 2, 3104, 1, True, 32),
]


@pytest.mark.parametrize("name,D,sshift,P,lag,adapt,M", FUSED_CASES)
def test_fused_run_chain_moments_match_the_trace(E, options, name, D, sshift, P, lag, adapt, M):
    import torch

    L = 5
    options(ens_sshift=sshift)
    assert -(-P // (32 << sshift)) >= 8  # several queue items of the forced size, the last one ragged or not
    rng = np.random.RandomState(P + D + lag)
    pot, h0 = small_family(E, name, D, rng)
    ctx = E._lib.Context.get()
    for dt in (np.float64, np.float32):
        where = f"{name} D={D} sshift={sshift} P={P} lag={lag} adapt={adapt} M={M} {np.dtype(dt).name}"
        ens = E.Ensemble(D, P, dtype=dt, device="cuda", seed=3)
        ens.setPosition(1.0, superchainSize=M)
        hmc = E.HMC(ens, L * h0 + 1e-9, h0, None, potential=pot, seed=3, bugCompat=False)
        n0 = ctx.launch_count()
        r = hmc.run(ITERS, TEMP, adapt=adapt, adaptIterations=ADAPT, keepNumSteps=True, adaptLag=lag, traceParticles=P,
                    chainDiagnostics=True, superchainSize=M)
        assert r.get("fused") and ctx.launch_count() - n0 == 1, where
        w0 = ADAPT + lag if adapt else 0
        if adapt:  # the window starts where the step size is final
            assert r["stepSize"][w0] == r["stepSize"][-1] and r["stepSize"][w0 - 1] != r["stepSize"][-1], where
        check_against_trace(r, w0, M, dt, where)
        assert torch.isfinite(r["rhat"]).all(), where


def host_loop_family(E, name, rng):
    """(descriptor, D, step size, steps, method) of the host-loop families."""
    if name == "dense24":  # the dense kernels (float32: the tensor-core kernel)
        D = 24
        A = rng.standard_normal((D, D))
        return E.GaussianPotential(precision=A @ A.T / D + np.eye(D)), D, 0.15, 6, "Leapfrog"
    if name == "logistic":
        D, Nd = 8, 200
        X = rng.standard_normal((Nd, D))
        y = (rng.uniform(size=Nd) < 1 / (1 + np.exp(-X @ rng.standard_normal(D)))).astype(np.float64)
        return E.LogisticPotential(X, y, priorScale=2.0), D, 0.05, 6, "Leapfrog"
    assert name == "stormer"
    return E.HarmonicPotential(rng.uniform(0.5, 2.0, 6)), 6, 0.1, 6, "Stormer-Verlet"


@pytest.mark.parametrize("name", ["dense24", "logistic", "stormer"])
@pytest.mark.parametrize("adapt", [False, True])
def test_host_loop_chain_moments_match_the_trace(E, name, adapt):
    rng = np.random.RandomState(len(name))
    pot, D, h0, L, method = host_loop_family(E, name, rng)
    P, M, lag = 2000, 4, 2
    for dt in (np.float64, np.float32):
        where = f"{name} adapt={adapt} {np.dtype(dt).name}"
        ens = E.Ensemble(D, P, dtype=dt, device="cuda", seed=7)
        ens.setPosition(0.5, superchainSize=M)
        hmc = E.HMC(ens, L * h0 + 1e-9, h0, None, potential=pot, seed=7, method=method, bugCompat=False)
        r = hmc.run(ITERS, TEMP, adapt=adapt, adaptIterations=ADAPT, adaptLag=lag, fused=False, traceParticles=P,
                    chainDiagnostics=True, superchainSize=M)
        assert not r.get("fused"), where
        check_against_trace(r, ADAPT + lag if adapt else 0, M, dt, where)


@pytest.mark.parametrize("dt,adapt", [(np.float32, True), (np.float64, False)])
def test_fused_run_and_host_loop_give_the_same_bits(E, dt, adapt):
    """float32 with adaptation (every iteration's float32(h) is the same number on both paths) and float64 without:
    the same positions, hence -- one update function for both -- identical accumulators."""
    import torch

    D, P, M, h0, L = 10, 3000, 4, 0.05, 5
    pot = E.FunnelPotential(D, 3.0)
    out = []
    for fused in (True, False):
        ens = E.Ensemble(D, P, dtype=dt, device="cuda", seed=2)
        ens.setPosition(1.0, superchainSize=M)
        hmc = E.HMC(ens, L * h0 + 1e-9, h0, None, potential=pot, seed=2, bugCompat=False)
        r = hmc.run(ITERS, TEMP, adapt=adapt, adaptIterations=ADAPT, keepNumSteps=True, adaptLag=1, fused=fused,
                    chainDiagnostics=True, superchainSize=M)
        assert bool(r.get("fused")) == fused
        out.append((ens.q.clone(), r))
    (qf, rf), (qh, rh) = out
    assert torch.equal(qf, qh)
    assert rf["rhatDraws"] == rh["rhatDraws"] == (ITERS - ADAPT - 1 if adapt else ITERS)
    assert torch.equal(rf["chainMean"], rh["chainMean"]) and torch.equal(rf["chainVar"], rh["chainVar"])
    assert torch.equal(rf["rhat"], rh["rhat"])


@pytest.mark.parametrize("fused", [True, False])
def test_diagnostics_do_not_perturb_the_sampler(E, fused):
    import torch

    D, P, M, h0, L = 10, 5000, 4, 0.05, 5
    pot = E.FunnelPotential(D, 3.0)
    ctx = E._lib.Context.get()
    runs = []
    for on in (False, True):
        ens = E.Ensemble(D, P, dtype=np.float32, device="cuda", seed=4)
        ens.setPosition(1.0, superchainSize=M)
        hmc = E.HMC(ens, L * h0 + 1e-9, h0, None, potential=pot, seed=4, bugCompat=False)
        n0 = ctx.launch_count()
        r = hmc.run(ITERS, TEMP, adapt=True, adaptIterations=ADAPT, keepNumSteps=True, adaptLag=2, fused=fused,
                    traceParticles=64, chainDiagnostics=on, superchainSize=M)
        launches = ctx.launch_count() - n0
        runs.append((ens.q.clone(), r, launches, hmc.stepSize))
    (q0, r0, n_off, h_off), (q1, r1, n_on, h_on) = runs
    assert "rhat" not in r0 and r1["rhat"] is not None
    assert torch.equal(q0, q1) and torch.equal(r0["trace"], r1["trace"])
    assert r0["stepSize"] == r1["stepSize"] and r0["acceptRate"] == r1["acceptRate"] and h_off == h_on
    assert r0["meanH"] == r1["meanH"] and torch.equal(r0["mean"], r1["mean"]) and torch.equal(r0["var"], r1["var"])
    if fused:
        assert n_off == n_on == 1
    else:  # one k_chain_moments launch per iteration of the window
        assert n_on - n_off == ITERS - ADAPT - 2


def test_mass_adaptation_returns_moments_in_the_original_coordinates(E):
    D, P, M, h0, L, n, nAdapt = 10, 4000, 4, 0.05, 5, 40, 24
    ens = E.Ensemble(D, P, dtype=np.float64, device="cuda", seed=6)
    ens.setPosition(1.0, superchainSize=M)
    hmc = E.HMC(ens, L * h0 + 1e-9, h0, None, potential=E.FunnelPotential(D, 3.0), seed=6, bugCompat=False)
    r = hmc.run(n, TEMP, adapt=True, adaptIterations=nAdapt, adaptMass=True, keepNumSteps=True, traceParticles=P,
                chainDiagnostics=True, superchainSize=M)
    assert hmc.massScale is not None and np.any(np.abs(hmc.massScale - 1) > 0.05)
    check_against_trace(r, nAdapt, M, np.float64, "adaptMass")


def test_rhat_flags_separated_superchains_and_passes_converged_chains(E):
    D = 10
    pot = E.HarmonicPotential(np.ones(D))
    # superchains of 64 started 10 standard deviations apart, 5 short trajectories: far from converged
    ens = E.Ensemble(D, 1 << 14, dtype=np.float32, device="cuda", seed=1)
    ens.setPosition(10.0, superchainSize=64)
    hmc = E.HMC(ens, 3 * 0.1 + 1e-9, 0.1, None, potential=pot, seed=1)
    r = hmc.run(5, TEMP, chainDiagnostics=True, superchainSize=64)
    assert r["rhatDraws"] == 5 and bool((r["rhat"] > 1.1).all()), r["rhat"]
    # exact draws of the target and trajectories of about pi / 2 (nearly independent draws): converged
    ens = E.Ensemble(D, 1 << 16, dtype=np.float32, device="cuda", seed=1)
    ens.setPosition(1.0)
    hmc = E.HMC(ens, 8 * 0.2 + 1e-9, 0.2, None, potential=pot, seed=1)
    r = hmc.run(300, TEMP, chainDiagnostics=True)
    assert r["rhatDraws"] == 300 and bool((r["rhat"] < 1.01).all()), r["rhat"]


def test_two_ranks_agree_with_one_process(E, tmp_path):
    import socket
    import subprocess
    import sys

    worker = os.path.join(os.path.dirname(os.path.abspath(__file__)), "chain_rank_worker.py")
    sock = socket.socket()
    sock.bind(("127.0.0.1", 0))
    port = sock.getsockname()[1]
    sock.close()

    def launch(rank, world, out):
        return subprocess.Popen([sys.executable, worker, "--rank", str(rank), "--world", str(world), "--port", str(port),
                                 "--out", out], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)

    single = str(tmp_path / "single.npz")
    p = launch(0, 1, single)
    out, _ = p.communicate(timeout=300)
    assert p.returncode == 0, out
    procs = [launch(r, 2, str(tmp_path / f"rank{r}.npz")) for r in range(2)]
    for p in procs:
        try:
            o, _ = p.communicate(timeout=300)
        except subprocess.TimeoutExpired:
            for k in procs:
                k.kill()
            pytest.fail("the two-rank run did not finish")
        assert p.returncode == 0, o
    ref = np.load(single)
    shards = [np.load(str(tmp_path / f"rank{r}.npz")) for r in range(2)]
    for key in ("rhat", "rhatBetween", "rhatWithin"):
        assert np.array_equal(shards[0][key], shards[1][key]), key  # identical bits on both ranks
        np.testing.assert_allclose(shards[0][key], ref[key], rtol=1e-12, err_msg=key)
    for sh in shards:
        lo, hi = int(sh["lo"]), int(sh["hi"])
        assert np.array_equal(sh["chainMean"], ref["chainMean"][:, lo:hi])
        assert np.array_equal(sh["chainVar"], ref["chainVar"][:, lo:hi])
