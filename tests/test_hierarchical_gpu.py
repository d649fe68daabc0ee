"""The hierarchical normal family on the GPU (pytest -m gpu): HierPot (csrc/k_small.cuh) in every small-D kernel
against the float64 reference of tests/hierarchical_reference.py, and eight schools end to end against the
quadrature of its posterior.

Tolerances are those of tests/test_small_d_engine.py: trajectories within 1e-5 relative in float32 and 1e-12 in
float64, accept decisions identical outside the tie band.
"""
import numpy as np
import pytest

from oracle import hmc_oracle as O
from tests import hierarchical_reference as H
from tests.test_small_d_engine import E, KB, RTOL, TEMP, TIE, host, on_device, rel_err, rounded, run_iteration  # noqa: F401

pytestmark = pytest.mark.gpu

# D = J + 2: exact and padded widths of every instance the launchers pick (DT = 4, 8, 10, 16, 32), every D mod 4
WIDTHS = (3, 4, 5, 7, 8, 9, 10, 11, 16, 17, 31, 32)


def model(E, D, centered, scaled, rng):
    """(engine descriptor, reference, step size, start sampler) of a J = D - 2 group model.  The start covers the bulk
    of the posterior: mu around the data, eta in [0, 2] (centred: the conditional scale of theta is tau) or [-1, 2]."""
    J = D - 2
    if J == 8:
        y, sigma = H.EIGHT_SCHOOLS["y"], H.EIGHT_SCHOOLS["sigma"]
    else:
        y, sigma = rng.normal(5.0, 10.0, J), rng.uniform(5.0, 20.0, J)
    scale = rng.uniform(0.5, 2.0, D) if scaled else None
    pe = E.HierarchicalNormalPotential(y, sigma, 1.0, 5.0, 5.0, centered=centered)
    if scaled:
        pe = pe.rescaled(scale)
    po = H.HierarchicalNormal(y, sigma, 1.0, 5.0, 5.0, centered=centered, scale=scale)

    def start(P):
        x = np.empty((D, P))
        x[0] = rng.normal(4.0, 3.0, P)
        x[1] = rng.uniform(0.0, 2.0, P) if centered else rng.uniform(-1.0, 2.0, P)
        z = rng.standard_normal((J, P))
        x[2:] = x[0] + np.exp(x[1]) * z if centered else z
        return x / po.s[:, None]

    return pe, po, (0.03 if centered else 0.08), start


@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("scaled", [False, True])
@pytest.mark.parametrize("centered", [False, True])
def test_kernel_matrix_vs_reference(E, centered, scaled, dt):
    """hmc_iter with fed z and u (q, stored momentum, accept flags, the 2D+3 statistics), integrate-only Leapfrog and
    Stormer-Verlet, and the descriptor's energy and gradient at every width, against the float64 reference; energy and
    gradient also at eta = -20 and 20, where they must be finite."""
    ctx = E._lib.Context.get()
    bits = 32 if dt == np.float32 else 64
    L = 7
    for D in WIDTHS:
        P = 333
        rng = np.random.RandomState(100 * D + 10 * centered + scaled)
        pe, po, h, start = model(E, D, centered, scaled, rng)
        q0 = rounded(start(P), dt)
        z = rounded(rng.standard_normal((D, P)), dt)
        u = rounded(rng.uniform(size=P), dt)
        mass = rounded(rng.uniform(0.5, 2.0, P), dt)
        for method in ("Leapfrog", "Stormer-Verlet"):
            a = run_iteration(E, pe, po, D, P, dt, method, h, L, q0, mass, z, u, bug=method != "Leapfrog")
            assert a.sum() > P // 4, (D, method)
            p0 = rounded(z * np.sqrt(mass), dt)
            q, p = on_device(q0, dt), on_device(p0, dt)
            E._lib.leapfrog(ctx, pe.handle(bits, ctx), q, p, on_device(mass, dt), h, h * h, L,
                            stormer=method != "Leapfrog")
            integ = O.leapfrog if method == "Leapfrog" else O.stormer_verlet
            qr, pr = integ(q0, p0, mass, h, L, po.grad)
            where = f"integrate D={D} {method} {np.dtype(dt).name}"
            assert rel_err(host(q), qr) < RTOL[dt], where
            assert rel_err(host(p), pr) < (2e-4 if dt == np.float32 and method != "Leapfrog" else RTOL[dt]), where
        etol = RTOL[dt] * (10 if dt == np.float32 else 1)
        qh = np.asarray(q0, dtype=dt)
        assert rel_err(pe(qh), po.energy(q0)) < etol, f"energy D={D}"
        assert rel_err(pe.gradient(qh), po.grad(q0)) < etol, f"gradient D={D}"
        # far into both ends of eta: finite, and the same numbers as the reference
        qx = q0[:, :2].copy()
        qx[1] = np.array([-20.0, 20.0]) / po.s[1]
        qx = rounded(qx, dt)
        e, g = pe(np.asarray(qx, dtype=dt)), pe.gradient(np.asarray(qx, dtype=dt))
        assert np.all(np.isfinite(e)) and np.all(np.isfinite(g)), f"eta = +-20, D={D}"
        for k in range(2):  # per point: the two ends differ by ~40 orders of magnitude
            assert rel_err(e[k], po.energy(qx[:, k])) < etol, f"energy at eta = +-20, D={D}"
            assert rel_err(g[:, k], po.grad(qx[:, k])) < etol, f"gradient at eta = +-20, D={D}"
            # the trajectory kernel's own gradient (float32: the packed form with the fused kick) at the same points:
            # one leapfrog step from rest with h |grad U| = 1, against the reference's step
            q1 = qx[:, k:k + 1]
            hk = 1.0 / np.max(np.abs(po.grad(q1)))
            qd, pd = on_device(q1, dt), on_device(np.zeros((D, 1)), dt)
            E._lib.leapfrog(ctx, pe.handle(bits, ctx), qd, pd, on_device(np.ones(1), dt), hk, hk * hk, 1)
            qr, pr = O.leapfrog(q1, np.zeros((D, 1)), np.ones(1), hk, 1, po.grad)
            assert np.all(np.isfinite(host(qd))) and np.all(np.isfinite(host(pd))), f"step at eta = +-20, D={D}"
            assert rel_err(host(qd), qr) < RTOL[dt], f"step at eta = +-20, D={D}"
            assert rel_err(host(pd), pr) < etol, f"step at eta = +-20, D={D}"


@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("centered", [False, True])
def test_getSamples_one_launch_equals_iteration_by_iteration(E, centered, dt, capsys):
    """getSamples on a device ensemble (ONE k_small_run launch) == one k_small launch per iteration, bit for bit:
    samples, stored momenta and the final state, at the exact width (eight schools) and padded ones."""
    import torch

    P, S = 777, 9
    tdt = torch.float32 if dt == np.float32 else torch.float64
    for D in (10, 5, 17):
        rng = np.random.RandomState(40 + D)
        pot, _, h, start = model(E, D, centered, False, rng)
        q0 = start(P)
        mass = rng.uniform(0.5, 2.0, P)

        def fresh(method):
            ens = E.Ensemble(D, P, dtype=dt, device="cuda", seed=9)
            ens.mass = torch.tensor(mass, dtype=tdt, device="cuda")
            hmc = E.HMC(ens, 7 * h + 1e-9, h, None, potential=pot, seed=9, bugCompat=D % 2 == 0, method=method)
            ens.setPosition = lambda qStd: ens.q.copy_(torch.tensor(q0, dtype=tdt))  # fixed start
            return ens, hmc

        for method in ("Leapfrog", "Stormer-Verlet"):
            ens_a, hmc_a = fresh(method)
            sa, ma = hmc_a.getSamples(S, TEMP, 1.0)  # fused
            ens_b, hmc_b = fresh(method)
            hmc_b._fused_loop_ok = lambda: False
            sb, mb = hmc_b.getSamples(S, TEMP, 1.0)  # one launch per iteration
            assert torch.equal(sa, sb) and torch.equal(ma, mb), (D, method)
            assert torch.equal(ens_a.q, ens_b.q) and torch.equal(ens_a.p, ens_b.p), (D, method)
            moved = (sa[:, :, -1] != torch.tensor(q0, dtype=tdt, device="cuda")).any(0).float().mean().item()
            assert moved > 0.5, (D, method)
    capsys.readouterr()


@pytest.mark.parametrize("lag", [1, 2])
@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("centered", [False, True])
def test_run_fused_matches_host_loop(E, centered, dt, lag):
    """HMC.run as ONE k_small_ens launch against the iteration-by-iteration host loop: step sizes to 1e-12,
    acceptRate exactly, the chains bit for bit in float32 and to 1e-9 in float64."""
    import torch

    P, S, L = 5000, 31, 5
    D = 10
    rng = np.random.RandomState(22)
    pot, _, h0, start = model(E, D, centered, False, rng)
    tdt = torch.float32 if dt == np.float32 else torch.float64
    q0 = torch.tensor(start(P), dtype=tdt, device="cuda")
    ctx = E._lib.Context.get()

    def fresh():
        ens = E.Ensemble(D, P, dtype=dt, device="cuda", seed=5)
        ens.q.copy_(q0)
        return ens, E.HMC(ens, L * h0 + 1e-9, h0, None, potential=pot, seed=5, bugCompat=False)

    kw = dict(adapt=True, targetAccept=0.8, adaptIterations=24, keepNumSteps=True, traceParticles=7, adaptLag=lag)
    ens_h, hmc_h = fresh()
    rh = hmc_h.run(S, TEMP, fused=False, **kw)
    ens_f, hmc_f = fresh()
    n0 = ctx.launch_count()
    rf = hmc_f.run(S, TEMP, **kw)
    assert rf.get("fused") and ctx.launch_count() - n0 == 1
    np.testing.assert_allclose(rf["stepSize"], rh["stepSize"], rtol=1e-12)
    assert all(rf["stepSize"][k] == h0 for k in range(lag + 1)) and rf["stepSize"][lag + 1] != h0
    np.testing.assert_array_equal(rf["acceptRate"], rh["acceptRate"])
    np.testing.assert_allclose(rf["meanAcceptProb"], rh["meanAcceptProb"], rtol=1e-12)
    np.testing.assert_allclose(rf["meanH"], rh["meanH"], rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(rf["mean"].numpy(), rh["mean"].numpy(), rtol=1e-11, atol=1e-13)
    np.testing.assert_allclose(rf["var"].numpy(), rh["var"].numpy(), rtol=1e-10)
    assert 0.3 < np.mean(rf["acceptRate"]) < 1.0
    if dt == np.float32:
        assert torch.equal(ens_f.q, ens_h.q) and torch.equal(rf["trace"], rh["trace"])
    else:
        assert rel_err(host(ens_f.q), host(ens_h.q)) < 1e-9
        assert rel_err(host(rf["trace"]), host(rh["trace"])) < 1e-9


@pytest.mark.parametrize("centered", [False, True])
def test_rescaled_potential_is_hmc_with_diagonal_mass(E, centered):
    """One HMC iteration on rescaled(s) in the coordinates q / s against the reference's leapfrog with the diagonal
    mass matrix mass / s^2 in the original coordinates: same fed z and u, float64, 1e-11.  rescaled composes."""
    rng = np.random.RandomState(31)
    P, L, D = 257, 7, 10
    pe, po, h, start = model(E, D, centered, False, rng)
    s1, s2 = rng.uniform(0.5, 2.0, D), rng.uniform(0.5, 2.0, D)
    s = s1 * s2
    q0 = start(P)
    z = rng.standard_normal((D, P))
    u = rng.uniform(size=P)
    mass = rng.uniform(0.5, 2.0, P)
    qr, accr, oh, nh = O.hmc_iter_diag_mass(q0, z, u, mass, 1.0 / s**2, TEMP, h, L, po)
    ps = pe.rescaled(s1).rescaled(s2)
    assert type(ps) is type(pe) and ps.family == pe.family
    np.testing.assert_allclose(ps(q0 / s[:, None]), po.energy(q0), rtol=1e-12, atol=1e-12)
    ens = E.Ensemble(D, P)
    ens.q[:] = q0 / s[:, None]
    ens.mass[:] = mass
    hmc = E.HMC(ens, L * h + 1e-9, h, None, potential=ps, bugCompat=False)
    acc = np.empty(P, dtype=np.uint8)
    hmc.step(TEMP, accept=acc, z=z, u=u)
    clear = np.abs(u - np.minimum(1, np.exp(oh - nh))) > 1e-9
    assert np.array_equal(acc.astype(bool)[clear], accr[clear])
    same = acc.astype(bool) == accr
    assert rel_err((ens.q * s[:, None])[:, same], qr[:, same]) < 1e-11
    assert 0 < np.sum(accr)


def test_eight_schools_end_to_end():
    """Eight schools, non-centred, float32, 2^16 particles: adapted warm-up (step size and diagonal mass, one fused
    launch per phase), then sampling.  E[mu], E[eta] and E[theta_j] of the final ensemble (theta through
    modelParameters) lie within 5 Monte-Carlo standard errors of the quadrature moments, the particles counted as
    independent draws (SE = posterior sd / sqrt(P)); the sampling run's own running means of mu and eta too (a mean
    over iterations of one chain has at most the variance of one draw).  adaptMass returns everything in the
    original coordinates."""
    import torch

    import physicsbasedbayesianinference_b200 as E

    ref = H.hierarchical_posterior_moments(**H.EIGHT_SCHOOLS)
    P, L, h0, warm, S = 1 << 16, 10, 0.1, 400, 200
    pot = E.HierarchicalNormalPotential.eightSchools(centered=False)
    ens = E.Ensemble(10, P, dtype=np.float32, device="cuda", seed=17)
    gen = torch.Generator(device="cuda").manual_seed(17)
    ens.q.copy_(torch.randn((10, P), dtype=torch.float32, device="cuda", generator=gen))
    hmc = E.HMC(ens, L * h0 + 1e-9, h0, None, potential=pot, seed=17, bugCompat=False)
    rw = hmc.run(warm, TEMP, adapt=True, adaptMass=True, keepNumSteps=True, traceParticles=4)
    assert hmc.potential is pot and hmc.massScale is not None and rw.get("fused")
    # trace and ensemble in the original coordinates
    assert torch.equal(rw["trace"][:, :, -1], ens.q[:, :4])
    r = hmc.run(S, TEMP, traceParticles=4)
    assert r.get("fused") and torch.isfinite(ens.q).all()
    assert torch.equal(r["trace"][:, :, -1], ens.q[:, :4])
    acc = float(np.mean(r["acceptRate"]))
    assert 0.5 < acc < 0.99, acc
    mp = pot.modelParameters(ens.q.double())
    se = 1.0 / np.sqrt(P)
    eta = torch.log(mp["tau"])
    checks = [("mu", mp["mu"].mean().item(), ref["mean_mu"], ref["sd_mu"]),
              ("eta", eta.mean().item(), ref["mean_eta"], ref["sd_eta"]),
              ("mu (run mean)", float(r["mean"][0]), ref["mean_mu"], ref["sd_mu"]),
              ("eta (run mean)", float(r["mean"][1]), ref["mean_eta"], ref["sd_eta"])]
    th = mp["theta"].mean(dim=1).cpu().numpy()
    checks += [(f"theta_{j}", th[j], ref["mean_theta"][j], ref["sd_theta"][j]) for j in range(8)]
    bad = [(n, got, want, abs(got - want) / (sd * se)) for n, got, want, sd in checks if abs(got - want) > 5 * sd * se]
    assert not bad, bad
    # the ensemble's spread is the posterior's
    assert abs(mp["mu"].std().item() / ref["sd_mu"] - 1) < 0.05
    assert abs(float(r["var"][1]) ** 0.5 / ref["sd_eta"] - 1) < 0.05
