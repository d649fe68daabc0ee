"""The hierarchical normal family without a GPU: the float64 reference (tests/hierarchical_reference.py) against
NumPyro's density written with scipy.stats and against finite differences, the quadrature of the posterior, the
descriptor's argument checks, the NumPyro spec adapter and HierarchicalNormalPotential.modelParameters."""
import numpy as np
import pytest
from scipy import stats

from tests import hierarchical_reference as H

ES = H.EIGHT_SCHOOLS


def log_density(pot, q):
    """log p(mu, eta, theta | y) + const as NumPyro's log_density writes it, in the coordinates of pot: Normal prior
    of mu, HalfCauchy prior of tau = e^eta plus log |d tau / d eta| = eta, Normal group effects (theta_j itself, or
    thetaTilde_j ~ N(0, 1) with theta_j = mu + tau thetaTilde_j) and Normal observations."""
    x = pot.s[:, None] * q
    mu, eta, th = x[0], x[1], x[2:]
    tau = np.exp(eta)
    lp = stats.norm.logpdf(mu, pot.mu_loc, pot.mu_scale) + stats.halfcauchy.logpdf(tau, scale=pot.tau_scale) + eta
    if pot.centered:
        theta = th
        lp = lp + np.sum(stats.norm.logpdf(theta, mu, tau), axis=0)
    else:
        theta = mu + tau * th
        lp = lp + np.sum(stats.norm.logpdf(th, 0.0, 1.0), axis=0)
    return lp + np.sum(stats.norm.logpdf(pot.y[:, None], theta, 1.0 / np.sqrt(pot.w)[:, None]), axis=0)


def reference(centered, scaled, J=8, seed=0):
    rng = np.random.RandomState(seed)
    if J == 8:
        y, sigma = ES["y"], ES["sigma"]
    else:
        y, sigma = rng.normal(5.0, 10.0, J), rng.uniform(5.0, 20.0, J)
    scale = rng.uniform(0.5, 2.0, J + 2) if scaled else None
    return H.HierarchicalNormal(y, sigma, 1.5, 5.0, 5.0, centered=centered, scale=scale)


def points(pot, P, rng):
    """Positions over the bulk of the posterior and its tails: mu in +-15, eta in [-4, 3], theta near the data."""
    J = pot.J
    x = np.empty((J + 2, P))
    x[0] = rng.uniform(-15.0, 15.0, P)
    x[1] = rng.uniform(-4.0, 3.0, P)
    x[2:] = (pot.y[:, None] + 10.0 * rng.standard_normal((J, P))) if pot.centered else rng.standard_normal((J, P))
    return x / pot.s[:, None]


@pytest.mark.parametrize("scaled", [False, True])
@pytest.mark.parametrize("centered", [False, True])
def test_energy_differences_equal_the_numpyro_log_density(centered, scaled):
    """U(a) - U(b) == -(log p(a) - log p(b)) to 1e-12: U is minus NumPyro's log density up to a constant."""
    rng = np.random.RandomState(1)
    for J in (8, 1, 3, 30):
        pot = reference(centered, scaled, J, seed=J)
        qa, qb = points(pot, 200, rng), points(pot, 200, rng)
        dU = pot.energy(qa) - pot.energy(qb)
        dlp = log_density(pot, qa) - log_density(pot, qb)
        np.testing.assert_allclose(dU, -dlp, rtol=1e-12, atol=1e-12 * np.max(np.abs(dlp)))


@pytest.mark.parametrize("scaled", [False, True])
@pytest.mark.parametrize("centered", [False, True])
def test_gradient_matches_central_differences(centered, scaled):
    rng = np.random.RandomState(2)
    pot = reference(centered, scaled)
    q = points(pot, 50, rng)
    g = pot.grad(q)
    eps = 1e-6
    for d in range(q.shape[0]):
        e = np.zeros_like(q)
        e[d] = eps
        fd = (pot.energy(q + e) - pot.energy(q - e)) / (2 * eps)
        np.testing.assert_allclose(g[d], fd, rtol=1e-6, atol=1e-6 * max(1.0, np.max(np.abs(fd))))
    # (D,) and (D, P) agree
    np.testing.assert_allclose(pot.grad(q[:, 3]), g[:, 3], rtol=1e-15)
    assert pot.energy(q[:, 3]) == pytest.approx(pot.energy(q)[3], rel=1e-15)


def test_gradient_is_finite_at_extreme_eta():
    for centered in (False, True):
        pot = reference(centered, False)
        q = np.zeros((10, 2))
        q[1] = [-20.0, 20.0]
        q[2:] = 0.5
        assert np.all(np.isfinite(pot.grad(q))) and np.all(np.isfinite(pot.energy(q)))


def test_posterior_quadrature_of_eight_schools():
    """The quadrature reproduces the eight-schools posterior (published: E[mu] 4.4, E[tau] 3.6) and does not move
    when the grid is refined or widened (the mass below eta = -15, about e^-15, moves sd(eta) by 6e-6 relative)."""
    m = H.hierarchical_posterior_moments(**ES)
    assert m["mean_mu"] == pytest.approx(4.397, abs=5e-4)
    assert m["sd_mu"] == pytest.approx(3.318, abs=5e-4)
    assert m["mean_eta"] == pytest.approx(0.802, abs=5e-4)
    assert m["mean_tau"] == pytest.approx(3.598, abs=5e-4)
    assert m["mean_theta"][0] == pytest.approx(6.212, abs=5e-4)
    fine = H.hierarchical_posterior_moments(**ES, mu_range=(-50.0, 60.0), eta_range=(-18.0, 7.0), n_mu=2801, n_eta=2201)
    for k in ("mean_mu", "sd_mu", "mean_eta", "sd_eta", "mean_tau"):
        assert fine[k] == pytest.approx(m[k], rel=2e-5), k
    np.testing.assert_allclose(fine["mean_theta"], m["mean_theta"], rtol=2e-5)
    np.testing.assert_allclose(fine["sd_theta"], m["sd_theta"], rtol=2e-5)


def test_descriptor_checks_adapter_and_model_parameters():
    import physicsbasedbayesianinference_b200 as E
    from physicsbasedbayesianinference_b200 import numpyro_adapter as A

    HN = E.HierarchicalNormalPotential
    es = HN.eightSchools()
    assert es.numDimensions == 10 and es.family == E._lib.FAMILY_HIERARCHICAL_NORMAL and not es.centered
    assert es._scalars() == [0.0, 5.0, 5.0, 0.0] and len(es._params()) == 2
    assert HN.eightSchools(centered=True)._scalars()[3] == 1.0
    for bad in (dict(y=[], sigma=[]), dict(y=np.zeros(31), sigma=np.ones(31)), dict(y=[1.0, 2.0], sigma=[1.0]),
                dict(y=[np.nan], sigma=[1.0]), dict(y=[1.0], sigma=[0.0]), dict(y=[1.0], sigma=[-1.0]),
                dict(y=[1.0], sigma=[1.0], muScale=0.0), dict(y=[1.0], sigma=[1.0], tauScale=-1.0),
                dict(y=[1.0], sigma=[1.0], muLoc=np.inf), dict(y=[1.0], sigma=[1.0], centered=2),
                dict(y=[1.0], sigma=[1.0], scale=[1.0, 1.0]), dict(y=[1.0], sigma=[1.0], scale=[1.0, 0.0, 1.0])):
        with pytest.raises(ValueError):
            HN(**bad)
    assert HN(np.zeros(30), np.ones(30)).numDimensions == 32
    # the spec adapter; the bare model name stays unrecognised
    p = A.potentialFromSpec(dict(family="hierarchical_normal", y=ES["y"], sigma=ES["sigma"], centered=True))
    assert isinstance(p, HN) and p.centered and p.numDimensions == 10 and p.tauScale == 5.0
    assert np.array_equal(p.y, ES["y"]) and np.array_equal(p.sigma, ES["sigma"])
    with pytest.raises(NotImplementedError, match="hierarchical_normal"):
        A.potentialFromSpec(dict(family="eight_schools"))
    # rescaled composes with an existing scale
    s1, s2 = np.linspace(0.5, 2.0, 10), np.linspace(3.0, 1.0, 10)
    r = es.rescaled(s1).rescaled(s2)
    assert type(r) is HN and r.family == es.family and not r.centered
    np.testing.assert_allclose(r.scale, s1 * s2, rtol=1e-15)
    assert len(r._params()) == 3
    # modelParameters: (D,), (D, P), (D, P, S), NumPy and torch, plain and rescaled coordinates
    rng = np.random.RandomState(3)
    for pot in (es, HN.eightSchools(centered=True), es.rescaled(s1), HN.eightSchools(True).rescaled(s1)):
        ref = H.HierarchicalNormal(ES["y"], ES["sigma"], centered=pot.centered, scale=pot.scale)
        for shape in ((10,), (10, 7), (10, 7, 3)):
            q = rng.standard_normal(shape)
            x = (ref.s.reshape((10,) + (1,) * (len(shape) - 1))) * q
            theta = x[2:] if pot.centered else x[0] + np.exp(x[1]) * x[2:]
            mp = pot.modelParameters(q)
            assert mp["theta"].shape == (8,) + shape[1:] and np.shape(mp["mu"]) == shape[1:]
            np.testing.assert_allclose(mp["mu"], x[0], rtol=1e-15)
            np.testing.assert_allclose(mp["tau"], np.exp(x[1]), rtol=1e-15)
            np.testing.assert_allclose(mp["theta"], theta, rtol=1e-14, atol=1e-14)
            import torch

            mt = pot.modelParameters(torch.from_numpy(q))
            for k in ("mu", "tau", "theta"):
                np.testing.assert_allclose(mt[k].numpy(), mp[k], rtol=1e-14, atol=1e-14)
    with pytest.raises(ValueError):
        es.modelParameters(np.zeros(9))
