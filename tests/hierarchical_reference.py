"""Float64 NumPy reference for the hierarchical normal family (EHMC_FAMILY_HIERARCHICAL_NORMAL, include/ehmc.h) --
TEST INFRASTRUCTURE ONLY, used by tests/test_hierarchical_cpu.py and tests/test_hierarchical_gpu.py.  Objects follow
the potential interface of oracle/hmc_oracle.py (energy / grad over q of shape (D,) or (D, P)), so they drive
oracle.hmc_oracle's integrators and HMC iterations.

It lives beside the tests rather than in oracle/hmc_oracle.py: that module is the port of the reference's own code
and the fixture set its golden tests pin, and the reference has no hierarchical model.  This one is pinned instead
against NumPyro's density written with scipy.stats (tests/test_hierarchical_cpu.py), and its posterior against a
quadrature that integrates theta out analytically (hierarchical_posterior_moments).
"""
from __future__ import annotations

import numpy as np

EIGHT_SCHOOLS = dict(y=np.array([28.0, 8.0, -3.0, 7.0, -1.0, 1.0, 18.0, 12.0]),
                     sigma=np.array([15.0, 10.0, 16.0, 11.0, 9.0, 11.0, 10.0, 18.0]),
                     mu_loc=0.0, mu_scale=5.0, tau_scale=5.0)


class HierarchicalNormal:
    """mu ~ N(mu_loc, mu_scale^2), tau ~ HalfCauchy(tau_scale), theta_j ~ N(mu, tau^2), y_j ~ N(theta_j, sigma_j^2) in
    the coordinates q = (mu, eta = ln tau, theta | thetaTilde), theta_j = mu + e^eta thetaTilde_j when not centred.
    U = minus the log density with the Jacobian of eta, additive constants dropped; scale: U'(q) = U(scale q)."""

    family = 7

    def __init__(self, y, sigma, mu_loc=0.0, mu_scale=5.0, tau_scale=5.0, centered=False, scale=None):
        self.y = np.asarray(y, dtype=np.float64)
        self.w = 1.0 / np.asarray(sigma, dtype=np.float64) ** 2
        self.J = self.y.shape[0]
        self.mu_loc, self.mu_scale, self.tau_scale = float(mu_loc), float(mu_scale), float(tau_scale)
        self.centered = bool(centered)
        self.s = np.ones(self.J + 2) if scale is None else np.asarray(scale, dtype=np.float64)

    def _col(self, a, q):
        return a if q.ndim == 1 else a[:, None]

    def energy(self, q):
        x = self._col(self.s, q) * q
        mu, eta, th = x[0], x[1], x[2:]
        z = 2.0 * eta - 2.0 * np.log(self.tau_scale)
        U = (mu - self.mu_loc) ** 2 / (2.0 * self.mu_scale**2) + np.logaddexp(0.0, z) - eta
        if self.centered:
            theta = th
            U = U + self.J * eta + 0.5 * np.exp(-2.0 * eta) * np.sum((theta - mu) ** 2, axis=0)
        else:
            theta = mu + np.exp(eta) * th
            U = U + 0.5 * np.sum(th**2, axis=0)
        return U + 0.5 * np.sum(self._col(self.w, q) * (self._col(self.y, q) - theta) ** 2, axis=0)

    def grad(self, q):
        s = self._col(self.s, q)
        x = s * q
        mu, eta, th = x[0], x[1], x[2:]
        w, y = self._col(self.w, q), self._col(self.y, q)
        z = 2.0 * eta - 2.0 * np.log(self.tau_scale)
        sig = 0.5 * (1.0 + np.tanh(0.5 * z))  # 1 / (1 + e^{-z}) without overflow
        g = np.empty_like(x)
        if self.centered:
            r = th - mu
            ie = np.exp(-2.0 * eta)
            g[0] = (mu - self.mu_loc) / self.mu_scale**2 - ie * np.sum(r, axis=0)
            g[1] = 2.0 * sig - 1.0 + self.J - ie * np.sum(r * r, axis=0)
            g[2:] = ie * r - w * (y - th)
        else:
            t = np.exp(eta)
            e = w * (y - mu - t * th)
            g[0] = (mu - self.mu_loc) / self.mu_scale**2 - np.sum(e, axis=0)
            g[1] = 2.0 * sig - 1.0 - t * np.sum(th * e, axis=0)
            g[2:] = th - t * e
        return s * g


def hierarchical_posterior_moments(y, sigma, mu_loc=0.0, mu_scale=5.0, tau_scale=5.0, mu_range=(-40.0, 50.0),
                                   eta_range=(-15.0, 6.0), n_mu=1801, n_eta=1401):
    """Posterior moments of the hierarchical normal model without HMC: theta is integrated out analytically,
    y_j | mu, tau ~ N(mu, sigma_j^2 + tau^2), and the density of (mu, eta) is summed on a rectangular grid.
    E[theta_j | mu, tau, y] = (y_j / sigma_j^2 + mu / tau^2) / (1 / sigma_j^2 + 1 / tau^2) and
    Var[theta_j | mu, tau, y] = 1 / (1 / sigma_j^2 + 1 / tau^2) give theta's moments by the laws of total expectation
    and variance.  Returns dict(mean_mu, sd_mu, mean_eta, sd_eta, mean_tau, mean_theta [J], sd_theta [J])."""
    y = np.asarray(y, dtype=np.float64)
    s2 = np.asarray(sigma, dtype=np.float64) ** 2
    mu = np.linspace(mu_range[0], mu_range[1], n_mu)[:, None]
    eta = np.linspace(eta_range[0], eta_range[1], n_eta)[None, :]
    tau2 = np.exp(2.0 * eta)
    logp = -0.5 * (mu - mu_loc) ** 2 / mu_scale**2 - np.log1p(tau2 / tau_scale**2) + eta  # prior, Jacobian of eta
    for yj, sj in zip(y, s2):
        v = sj + tau2
        logp = logp - 0.5 * np.log(v) - 0.5 * (yj - mu) ** 2 / v
    p = np.exp(logp - logp.max())
    p /= p.sum()
    pm, pe = p.sum(axis=1), p.sum(axis=0)
    m_mu = float(pm @ mu[:, 0])
    m_eta = float(pe @ eta[0])
    out = dict(mean_mu=m_mu, sd_mu=float(np.sqrt(pm @ (mu[:, 0] - m_mu) ** 2)), mean_eta=m_eta,
               sd_eta=float(np.sqrt(pe @ (eta[0] - m_eta) ** 2)), mean_tau=float(pe @ np.exp(eta[0])))
    mt, st = [], []
    for yj, sj in zip(y, s2):
        prec = 1.0 / sj + 1.0 / tau2
        cm = (yj / sj + mu / tau2) / prec
        m = float(np.sum(p * cm))
        mt.append(m)
        st.append(float(np.sqrt(np.sum(p * (1.0 / prec + (cm - m) ** 2)))))
    out.update(mean_theta=np.array(mt), sd_theta=np.array(st))
    return out
