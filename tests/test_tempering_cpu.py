"""CPU checks (no GPU needed) of the Gaussian-mixture family and the tempered run: the float64 references of
tests/tempering_reference.py, the Python descriptor's validation and rescaling, the ABI declarations, and
getSamplesTempered's refusals that come before any device work."""
import ctypes
import os
import re

import numpy as np
import pytest

import physicsbasedbayesianinference_b200 as E
from oracle import hmc_oracle as O
from physicsbasedbayesianinference_b200 import _lib
from tests import tempering_reference as TR

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def random_mixture(K, D, rng):
    return rng.uniform(0.2, 1.0, K), rng.normal(0.0, 2.0, (K, D)), rng.uniform(0.5, 2.0, (K, D))


def naive_energy(w, mu, sd, q):
    """-log sum_k w_k prod_d N(q_d; mu_kd, sd_kd^2) + (D/2) log 2 pi, term by term (no shift)."""
    D = mu.shape[1]
    dens = sum(w[k] * np.prod(np.exp(-0.5 * ((q - mu[k][:, None]) / sd[k][:, None]) ** 2) / sd[k][:, None], axis=0)
               for k in range(len(w)))
    return -np.log(dens)


@pytest.mark.parametrize("K,D", [(1, 2), (3, 7), (8, 10), (8, 32)])
def test_mixture_reference_energy_and_gradient(K, D):
    rng = np.random.RandomState(K + D)
    w, mu, sd = random_mixture(K, D, rng)
    po = TR.GaussianMixture(w, mu, sd)
    q = rng.normal(0.0, 1.5, (D, 40))
    assert np.allclose(po.energy(q), naive_energy(w, mu, sd, q), rtol=1e-12, atol=1e-12)
    eps = 1e-6
    g = po.grad(q)
    for d in range(D):
        e = np.zeros((D, 1))
        e[d] = eps
        fd = (po.energy(q + e) - po.energy(q - e)) / (2 * eps)
        assert np.max(np.abs(fd - g[d])) < 1e-6 * max(1.0, np.max(np.abs(g[d])))
    far = 1e4 * np.sign(rng.standard_normal((D, 8)))
    assert np.all(np.isfinite(po.energy(far))) and np.all(np.isfinite(po.grad(far)))
    assert np.allclose(po.energy(q[:, 3]), po.energy(q)[3], rtol=1e-14) and po.grad(q[:, 3]).shape == (D,)


def test_descriptor_rescaled_is_the_same_target():
    """rescaled(s): U'(q) = U(s q) + one constant, grad U'(q) = s grad U(s q) (on the reference)."""
    rng = np.random.RandomState(2)
    w, mu, sd = random_mixture(3, 5, rng)
    pe = E.GaussianMixturePotential(w, mu, sd)
    s = rng.uniform(0.3, 3.0, 5)
    ps = pe.rescaled(s)
    assert ps.family == _lib.FAMILY_GAUSSIAN_MIXTURE and ps.numDimensions == 5
    a, b = TR.GaussianMixture(pe.weights, pe.means, pe.stds), TR.GaussianMixture(ps.weights, ps.means, ps.stds)
    q = rng.normal(0.0, 1.0, (5, 100))
    d = b.energy(q) - a.energy(s[:, None] * q)
    assert np.allclose(d, d[0], rtol=0, atol=1e-10) and np.isclose(d[0], -np.sum(np.log(s)))
    assert np.allclose(b.grad(q), s[:, None] * a.grad(s[:, None] * q), rtol=1e-12, atol=1e-12)


def test_descriptor_validation():
    ok = dict(weights=[1.0, 2.0], means=np.zeros((2, 3)), stds=np.ones((2, 3)))
    pe = E.GaussianMixturePotential(**ok)
    assert pe.numDimensions == 3 and pe._params()[1].shape == (2, 3) and pe._scalars() == []
    bad = [dict(ok, weights=np.ones(9), means=np.zeros((9, 3)), stds=np.ones((9, 3))),
           dict(ok, weights=[1.0, 0.0]), dict(ok, weights=[1.0, -1.0]), dict(ok, weights=[1.0, np.inf]),
           dict(ok, stds=np.zeros((2, 3))), dict(ok, stds=np.full((2, 3), np.nan)),
           dict(ok, means=np.full((2, 3), np.inf)), dict(ok, means=np.zeros((3, 3))), dict(ok, stds=np.ones((2, 4)))]
    for kw in bad:
        with pytest.raises(ValueError):
            E.GaussianMixturePotential(**kw)


def test_swap_uniform_block():
    """The replica-exchange uniforms come from their own block: in [0, 1), not the Metropolis uniforms of block
    0xFFFFFFFF, and the float32 form is the float64 one's leading 24 bits."""
    ids = np.arange(1000, dtype=np.uint64) + np.uint64(1 << 33)
    u64 = TR.swap_uniform(12345, 77, ids, np.float64)
    u32 = TR.swap_uniform(12345, 77, ids, np.float32)
    _, um = O.philox_stream(12345, 77, ids, 4, np.float64)
    assert np.all((u64 >= 0) & (u64 < 1)) and not np.any(u64 == um)
    assert np.array_equal(u32, np.floor(u64 * 2.0**24) * 2.0**-24)
    assert abs(u64.mean() - 0.5) < 0.05


def test_tempered_reference_with_one_replica_is_the_plain_loop():
    """tempered_run with betas = [1] is the Philox-driven getSamples loop of the oracle, bit for bit."""
    rng = np.random.RandomState(4)
    D, P, S = 3, 16, 6
    po = TR.GaussianMixture(*random_mixture(2, D, rng))
    q0 = rng.normal(0.0, 1.0, (D, P))
    mass = rng.uniform(0.5, 2.0, P)
    r = TR.tempered_run(q0, mass, po, [1.0], S, 1 / O.BOLTZMANN, 0.1, 5, 9, iteration0=3, particle_offset=32)
    q = q0
    ids = np.arange(P, dtype=np.uint64) + np.uint64(32)
    for k in range(S):
        z, u = O.philox_stream(9, 3 + k, ids, D, np.float64)
        q, _, acc, _, _ = O.hmc_iter(q, z, u, mass, 1 / O.BOLTZMANN, 0.1, 5, po)
        assert np.array_equal(r["samples"][:, :, k], q) and np.array_equal(r["accept"][k], acc)
    assert not r["swaps"].any() and not r["roundtrips"].any()


def test_tempered_reference_round_trips_and_schedule():
    """With R = 2 and a flat target every proposed swap is accepted: pair (0, 1) is proposed at even iterations only,
    so a state crosses every other iteration and each crossing back to slot 0 after a visit to slot 1 is a round
    trip."""
    D, P, S = 2, 4, 8

    class Flat:
        def energy(self, q):
            return np.zeros(q.shape[1:])

        def grad(self, q):
            return np.zeros_like(q)

    r = TR.tempered_run(np.zeros((D, P)), np.ones(P), Flat(), [1.0, 0.5], S, 1 / O.BOLTZMANN, 0.1, 1, 1)
    assert np.array_equal(r["swap"][:, 0], np.arange(S) % 2 == 0) and not r["swap"][:, 1].any()
    assert np.array_equal(r["swaps"], [S // 2, 0, S // 2, 0])
    # the state that starts in slot 1 (labelled hottest) reaches slot 0 at iteration 0, the one from slot 0 returns at
    # iteration 2 after its visit to slot 1, and so on: one round trip per accepted swap
    assert np.array_equal(r["roundtrips"], [S // 2, S // 2])


def test_abi_declarations():
    src = open(os.path.join(ROOT, "include", "ehmc.h")).read()
    assert re.search(r"EHMC_FAMILY_GAUSSIAN_MIXTURE\s*=\s*8\b", src) and _lib.FAMILY_GAUSSIAN_MIXTURE == 8
    assert "ehmc_hmc_run_tempered" in _lib.SYMBOLS
    # struct ehmc_temper_args: u32 struct_size, i32 R, three pointers
    assert ctypes.sizeof(_lib.TemperArgs) == 8 + 3 * ctypes.sizeof(ctypes.c_void_p)
    assert "0xFFFFFFFE" in src


def test_get_samples_tempered_refuses_host_ensembles_and_numpy_draws():
    ens = E.Ensemble(2, 8)
    hmc = E.HMC(ens, 0.5, 0.1, None, potential=E.GaussianMixturePotential([1.0, 1.0], [[-1, 0], [1, 0]], np.ones((2, 2))))
    assert hmc.rng == "numpy"
    with pytest.raises(ValueError, match="device ensemble"):
        hmc.getSamplesTempered(2, 1.0, 1.0, [1.0, 0.5])
