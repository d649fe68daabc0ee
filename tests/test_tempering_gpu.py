"""The Gaussian-mixture family and the tempered run on the GPU (pytest -m gpu).

* MixturePot (csrc/k_small.cuh) against the float64 log-sum-exp reference of tests/tempering_reference.py: energy and
  gradient, finite differences, far from every mode, rescaled coordinates, ehmc_potential_create's refusals, and the
  existing samplers (getSamples, run(fused=True)) on a one-component mixture;
* ehmc_hmc_run_tempered / HMC.getSamplesTempered: R = 1 is getSamples bit for bit, the float64 restatement of the
  tempered loop (positions within 1e-12, every decision identical), per-level distributions and swap rates, a
  bimodal target that plain HMC cannot sample, invariance under call splits and shards, and the refusals.
"""
import numpy as np
import pytest

from tests import tempering_reference as TR
from tests.test_small_d_engine import E, KB, RTOL, TEMP, host, on_device, rel_err, rounded  # noqa: F401

pytestmark = pytest.mark.gpu

INVALID, UNSUPPORTED = -1, -3  # ehmc_status (include/ehmc.h)


def bits_of(dt):
    return 32 if dt == np.float32 else 64


def mixture(E, K, D, rng, spread=2.0):
    w = rng.uniform(0.2, 1.0, K)
    mu = rng.normal(0.0, spread, (K, D))
    sd = rng.uniform(0.5, 2.0, (K, D))
    return E.GaussianMixturePotential(w, mu, sd), TR.GaussianMixture(w, mu, sd)


def status(E, call):
    try:
        call()
    except E._lib.EhmcError as e:
        return e.code
    return E._lib.EHMC_OK


def ensemble(E, D, P, dt, seed=0, offset=0):
    return E.Ensemble(D, P, dtype=dt, device="cuda", seed=seed, particleOffset=offset)


# ---------------------------------------------------------------------------------------------------------------------
# the mixture family
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_mixture_energy_and_gradient(E, dt):
    """U and grad U at random points against the float64 reference (1e-5 / 1e-12 relative), at K = 1, 3, 8 and
    D = 2, 7, 10, 32 (exact and padded widths); finite at |q| = 1e4, where every component's density underflows."""
    for K in (1, 3, 8):
        for D in (2, 7, 10, 32):
            rng = np.random.RandomState(10 * K + D)
            pe, po = mixture(E, K, D, rng)
            q = rounded(rng.normal(0.0, 3.0, (D, 500)), dt)
            qd = on_device(q, dt)
            where = f"K={K} D={D} {np.dtype(dt).name}"
            assert rel_err(host(pe(qd)), po.energy(q)) < RTOL[dt], where
            assert rel_err(host(pe.gradient(qd)), po.grad(q)) < RTOL[dt], where
            far = rounded(1e4 * np.sign(rng.standard_normal((D, 64))), dt)
            Uf, gf = host(pe(on_device(far, dt))), host(pe.gradient(on_device(far, dt)))
            assert np.all(np.isfinite(Uf)) and np.all(np.isfinite(gf)), where
            assert rel_err(Uf, po.energy(far)) < RTOL[dt] and rel_err(gf, po.grad(far)) < RTOL[dt], where


def test_mixture_gradient_matches_finite_differences(E):
    rng = np.random.RandomState(5)
    for K, D in ((1, 2), (3, 7), (8, 10)):
        pe, _ = mixture(E, K, D, rng)
        q = rng.normal(0.0, 2.0, (D, 50))
        g = host(pe.gradient(on_device(q, np.float64)))
        eps = 1e-6
        for d in range(D):
            e = np.zeros((D, 1))
            e[d] = eps
            fd = (host(pe(on_device(q + e, np.float64))) - host(pe(on_device(q - e, np.float64)))) / (2 * eps)
            assert np.max(np.abs(fd - g[d])) < 1e-6 * max(1.0, np.max(np.abs(g[d]))), (K, D, d)


@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_mixture_rescaled(E, dt):
    """rescaled(s): U'(q) = U(s q) up to one constant, grad U'(q) = s grad U(s q)."""
    rng = np.random.RandomState(7)
    pe, _ = mixture(E, 3, 5, rng)
    s = rng.uniform(0.3, 3.0, 5)
    ps = pe.rescaled(s)
    q = rounded(rng.normal(0.0, 1.0, (5, 300)), dt)
    sq = rounded(s[:, None] * q, dt)
    d = host(ps(on_device(q, dt))) - host(pe(on_device(sq, dt)))
    scale = np.max(np.abs(host(pe(on_device(sq, dt)))))
    assert np.max(np.abs(d - d[0])) < 10 * RTOL[dt] * scale
    assert rel_err(host(ps.gradient(on_device(q, dt))), s[:, None] * host(pe.gradient(on_device(sq, dt)))) < 10 * RTOL[dt]


@pytest.mark.parametrize("bits", [32, 64])
def test_mixture_create_refusals(E, bits):
    lib = E._lib
    fam = lib.FAMILY_GAUSSIAN_MIXTURE
    ctx = lib.Context.get()

    def code(w, mu, sd, scalars=()):
        return status(E, lambda: lib.PotentialHandle(ctx, fam, [np.asarray(w, float), np.asarray(mu, float),
                                                                 np.asarray(sd, float)], list(scalars), bits))

    ok = code([1.0, 2.0], np.zeros((2, 3)), np.ones((2, 3)))
    assert ok == lib.EHMC_OK
    assert code(np.ones(8), np.zeros((8, 32)), np.ones((8, 32))) == lib.EHMC_OK  # the largest instance
    assert code(np.zeros(0), np.zeros((0, 3)), np.ones((0, 3))) == INVALID  # K = 0
    assert code(np.ones(9), np.zeros((9, 3)), np.ones((9, 3))) == UNSUPPORTED  # K = 9
    assert code(np.ones(2), np.zeros((2, 33)), np.ones((2, 33))) == UNSUPPORTED  # D = 33
    for bad in (0.0, -1.0, np.inf, np.nan):
        assert code([1.0, bad], np.zeros((2, 3)), np.ones((2, 3))) == INVALID, f"weight {bad}"
        sd = np.ones((2, 3))
        sd[1, 2] = bad
        assert code([1.0, 1.0], np.zeros((2, 3)), sd) == INVALID, f"std {bad}"
    for bad in (np.inf, np.nan):
        mu = np.zeros((2, 3))
        mu[0, 1] = bad
        assert code([1.0, 1.0], mu, np.ones((2, 3))) == INVALID, f"mean {bad}"
    assert code([1.0, 1.0], np.zeros((3, 3)), np.ones((3, 3))) == INVALID  # means rows != K
    assert code([1.0, 1.0], np.zeros((2, 3)), np.ones((2, 4))) == INVALID  # stds shape != means shape
    assert code([1.0, 1.0], np.zeros((2, 3)), np.ones((2, 3)), scalars=(1.0,)) == INVALID
    assert status(E, lambda: lib.PotentialHandle(ctx, fam, [np.ones(2), np.zeros((2, 3))], [], bits)) == INVALID


@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_one_component_mixture_with_existing_samplers(E, dt):
    """K = 1 is a diagonal Gaussian: getSamples (ehmc_hmc_run) and run(fused=True) (k_small_ens) give its mean and
    variance within 5 Monte-Carlo standard errors."""
    D = 3
    m, sd = np.array([1.0, -0.5, 2.0]), np.array([0.5, 1.0, 2.0])
    pe = E.GaussianMixturePotential([0.7], m[None], sd[None])
    P, S, burn = 4096, 300, 100
    ens = ensemble(E, D, P, dt, seed=11)
    hmc = E.HMC(ens, 2.0, 0.2, None, potential=pe)
    x = host(hmc.getSamples(S, TEMP, 1.0)[0][:, :, burn:].contiguous())  # (D, P, S - burn)
    cm = x.mean(axis=2)
    c2 = ((x - m[:, None, None]) ** 2).mean(axis=2)
    for d in range(D):
        assert abs(cm[d].mean() - m[d]) < 5 * cm[d].std() / np.sqrt(P), ("getSamples mean", d)
        assert abs(c2[d].mean() - sd[d] ** 2) < 5 * c2[d].std() / np.sqrt(P), ("getSamples var", d)
    P = 1 << 16
    ens = ensemble(E, D, P, dt, seed=12)
    ens.setPosition(1.0)
    hmc = E.HMC(ens, 2.0, 0.2, None, potential=pe)
    hmc.run(100, TEMP, fused=True)
    r = hmc.run(200, TEMP, fused=True)
    assert r.get("fused")
    mean, var = r["mean"].numpy(), r["var"].numpy()
    # each iteration's ensemble moments have the error of P independent draws; averaging over iterations can only
    # reduce it
    assert np.all(np.abs(mean - m) < 5 * sd / np.sqrt(P)), mean
    assert np.all(np.abs(var - sd**2) < 5 * np.sqrt(2.0) * sd**2 / np.sqrt(P)), var


# ---------------------------------------------------------------------------------------------------------------------
# the tempered run
# ---------------------------------------------------------------------------------------------------------------------
def run_tempered(E, pe, q, mass, args, S, betas, dt, samples=True):
    """ehmc_hmc_run_tempered on q in place: (samples (D, P, S) or None, accepted, swaps, roundtrips) on the host."""
    import torch

    lib = E._lib
    D, P = q.shape
    R = len(betas)
    ctx = lib.Context.get()
    out = torch.zeros((D, P, S), dtype=q.dtype, device=q.device) if samples else None
    acc = torch.zeros(P, dtype=torch.int32, device=q.device)
    sw = torch.zeros(P, dtype=torch.int32, device=q.device)
    rt = torch.zeros(P // R, dtype=torch.int32, device=q.device)
    lib.hmc_run_tempered(ctx, pe.handle(bits_of(dt), ctx), q, mass, args, S, R,
                         torch.tensor(np.asarray(betas, float), dtype=torch.float64, device=q.device),
                         None if out is None else out.view(D * P, S), 0, acc, sw, rt)
    return (None if out is None else out.cpu().numpy()), acc.cpu().numpy(), sw.cpu().numpy(), rt.cpu().numpy()


def args(E, h, L, seed=3, iteration=0, offset=0, integrator=0):
    return E._lib.make_args(h, h * h, L, KB, TEMP, integrator, E._lib.FLAG_BUGCOMPAT_MOMENTUM, seed, iteration, offset)


@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_one_replica_is_get_samples(E, dt):
    """betas = [1]: the samples of getSamplesTempered are those of getSamples, bit for bit, and through the C ABI the
    tempered run gives ehmc_hmc_run's samples and accepted counts (leapfrog and Stormer-Verlet; the packed float32
    path of the diagonal Gaussian and the scalar path of the mixture)."""
    import torch

    lib = E._lib
    ctx = lib.Context.get()
    rng = np.random.RandomState(1)
    D, P, S = 5, 1000, 40
    pots = [E.HarmonicPotential(rng.uniform(0.5, 3.0, D)), mixture(E, 3, D, rng)[0]]
    for pe in pots:
        a = ensemble(E, D, P, dt, seed=9)
        b = ensemble(E, D, P, dt, seed=9)
        sa, _ = E.HMC(a, 1.0, 0.1, None, potential=pe).getSamples(S, TEMP, 1.5)
        r = E.HMC(b, 1.0, 0.1, None, potential=pe).getSamplesTempered(S, TEMP, 1.5, [1.0])
        assert torch.equal(sa, r["samples"]) and torch.equal(a.q, b.q), pe
        assert torch.equal(r["coldSamples"], r["samples"])
        for integ in (lib.LEAPFROG, lib.STORMER_VERLET):
            q0 = on_device(rng.normal(0.0, 1.0, (D, P)), dt)
            mass = on_device(rng.uniform(0.5, 2.0, P), dt)
            q1 = q0.clone()
            ref = torch.zeros((D, P, S), dtype=q0.dtype, device="cuda")
            acc = torch.zeros(P, dtype=torch.int32, device="cuda")
            lib.hmc_run(ctx, pe.handle(bits_of(dt), ctx), q0, mass, args(E, 0.1, 10, integrator=integ), S,
                        ref.view(D * P, S), None, 0, acc)
            st, at, sw, rt = run_tempered(E, pe, q1, mass, args(E, 0.1, 10, integrator=integ), S, [1.0], dt)
            assert np.array_equal(st, ref.cpu().numpy()) and torch.equal(q0, q1), (pe, integ)
            assert np.array_equal(at, acc.cpu().numpy()) and not sw.any() and not rt.any()


@pytest.mark.parametrize("target", ["diag", "mixture"])
def test_float64_tempered_run_vs_reference(E, target):
    """P = 64 particles in 16 systems of R = 4, 30 iterations from Philox iteration 7 with particle offset 128: every
    iteration's positions within 1e-12 of tempering_reference.tempered_run (so every Metropolis and swap decision is
    the same), and the accepted, swap and round-trip counts equal."""
    import torch

    rng = np.random.RandomState(3)
    D, P, S, R = 3, 64, 30, 4
    if target == "diag":
        k = rng.uniform(0.5, 3.0, D)
        pe = E.HarmonicPotential(k)
        from oracle import hmc_oracle as O

        po = O.DiagGaussian(k)
    else:
        w, mu, sd = [0.3, 0.5, 0.2], np.array([[-3.0, 0, 0], [0, 3.0, 1.0], [3.0, 0, -2.0]]), np.full((3, D), 0.8)
        pe, po = E.GaussianMixturePotential(w, mu, sd), TR.GaussianMixture(w, mu, sd)
    betas = [1.0, 0.5, 0.25, 0.1]
    q0 = rng.normal(0.0, 2.0, (D, P))
    mass = rng.uniform(0.5, 2.0, P)
    q = on_device(q0, np.float64)
    s, acc, sw, rt = run_tempered(E, pe, q, on_device(mass, np.float64), args(E, 0.1, 10, seed=77, iteration=7,
                                                                              offset=128), S, betas, np.float64)
    ref = TR.tempered_run(q0, mass, po, betas, S, TEMP, 0.1, 10, 77, iteration0=7, particle_offset=128)
    for k in range(S):
        assert rel_err(s[:, :, k], ref["samples"][:, :, k]) < 1e-12, k
    assert rel_err(host(q), ref["q"]) < 1e-12
    assert np.array_equal(acc, ref["accepted"]) and np.array_equal(sw, ref["swaps"])
    assert np.array_equal(rt, ref["roundtrips"])
    assert sw.sum() > 0 and ref["swap"].any() and (~ref["accept"]).any(), "both decisions must be exercised"
    assert torch.isfinite(q).all()


def test_per_level_distributions_and_swap_rates(E):
    """Diagonal Gaussian k = (1, 4, 0.25, 9), R = 8, geometric ladder down to beta = 0.05: slot r has variance
    1 / (beta_r k_d) within 5 Monte-Carlo standard errors, and the swap rate of slots (r, r + 1) is
    E[min(1, exp(dbeta dU))] over independent draws at the two levels (float64 Monte Carlo here)."""
    k = np.array([1.0, 4.0, 0.25, 9.0])
    D, R = 4, 8
    betas = np.geomspace(1.0, 0.05, R)
    P, S = R * 4096, 300
    ens = ensemble(E, D, P, np.float32, seed=21)
    # trajectory 7 x 0.1: omega T = 0.35 .. 2.1 for omega = sqrt(k), away from multiples of pi, where a fixed-length
    # trajectory maps x to about +-x and the chain's x^2 stops mixing
    hmc = E.HMC(ens, 0.75, 0.1, None, potential=E.HarmonicPotential(k))
    hmc.getSamplesTempered(100, TEMP, 1.0, betas)  # burn-in
    r = hmc.getSamplesTempered(S, TEMP, None, betas)
    x = host(r["samples"]).reshape(D, P // R, R, S)
    rng = np.random.RandomState(0)
    for lv in range(R):
        c2 = (x[:, :, lv, :] ** 2).mean(axis=2)  # (D, systems): per-chain second moments
        want = 1.0 / (betas[lv] * k)
        se = c2.std(axis=1) / np.sqrt(P // R)
        assert np.all(np.abs(c2.mean(axis=1) - want) < 5 * se), (lv, c2.mean(axis=1), want)
        if lv + 1 < R:
            n = 1 << 20
            xa = rng.standard_normal((n, D)) / np.sqrt(betas[lv] * k)
            xb = rng.standard_normal((n, D)) / np.sqrt(betas[lv + 1] * k)
            dU = 0.5 * (xa**2 @ k) - 0.5 * (xb**2 @ k)
            expect = np.mean(np.minimum(1.0, np.exp((betas[lv] - betas[lv + 1]) * dU)))
            assert abs(r["swapRate"][lv] - expect) < 0.01, (lv, r["swapRate"][lv], expect)
    assert r["acceptRate"].shape == (R,) and np.all(r["acceptRate"] > 0.5)


def test_tempering_samples_both_modes(E):
    """D = 4, components at -6 e0 (weight 0.25) and +6 e0 (0.75), sigma = 1, every chain started in the minor mode:
    plain HMC (ehmc_hmc_run, getSamples' kernel) stays there; with R = 8 slots down to beta = 0.02 the cold slot's
    fraction in the minor mode settles at 0.25 within 5 Monte-Carlo standard errors, and states make round trips."""
    import torch

    lib = E._lib
    ctx = lib.Context.get()
    D, R = 4, 8
    mu = np.zeros((2, D))
    mu[0, 0], mu[1, 0] = -6.0, 6.0
    pe = E.GaussianMixturePotential([0.25, 0.75], mu, np.ones((2, D)))
    P = R * 2048
    start = np.random.RandomState(4).normal(0.0, 0.5, (D, P)) + mu[0][:, None]

    ens = ensemble(E, D, P, np.float32, seed=5)
    ens.q.copy_(torch.tensor(start))
    hmc = E.HMC(ens, 3.0, 0.3, None, potential=pe)
    S = 500
    plain = torch.zeros((D, P, S), dtype=torch.float32, device="cuda")
    lib.hmc_run(ctx, pe.handle(32, ctx), ens.q, hmc.integrator.mass, hmc._args(TEMP), S, plain.view(D * P, S))
    assert (plain[0, :, -100:] < 0).float().mean().item() > 0.95

    ens.q.copy_(torch.tensor(start))
    betas = np.geomspace(1.0, 0.02, R)
    hmc.getSamplesTempered(500, TEMP, None, betas)  # burn-in
    r = hmc.getSamplesTempered(1000, TEMP, None, betas)
    minor = (r["coldSamples"][0] < 0).double().mean(dim=1).cpu().numpy()  # per system
    se = minor.std() / np.sqrt(P // R)
    assert abs(minor.mean() - 0.25) < 5 * se, (minor.mean(), se)
    assert int(r["roundTrips"].sum()) > 0


def test_call_splits_and_shards_do_not_change_results(E):
    """Two calls of 50 iterations give the bits of one call of 100 (the swap schedule follows the global iteration),
    and two shards (particleOffset 0 and P / 2) give the bits of one launch."""
    import torch

    rng = np.random.RandomState(8)
    D, P, R = 7, 4096, 4
    pe, _ = mixture(E, 3, D, rng)
    betas = np.geomspace(1.0, 0.1, R)
    for dt in (np.float32, np.float64):
        one = ensemble(E, D, P, dt, seed=31)
        two = ensemble(E, D, P, dt, seed=31)
        h1 = E.HMC(one, 1.0, 0.1, None, potential=pe)
        h2 = E.HMC(two, 1.0, 0.1, None, potential=pe)
        r = h1.getSamplesTempered(100, TEMP, 1.0, betas)
        a = h2.getSamplesTempered(50, TEMP, 1.0, betas)
        b = h2.getSamplesTempered(50, TEMP, None, betas)
        assert torch.equal(r["samples"], torch.cat([a["samples"], b["samples"]], dim=2)) and torch.equal(one.q, two.q)
        assert np.allclose(r["swapRate"], (a["swapRate"] + b["swapRate"]) / 2, rtol=1e-12, atol=0)
        assert np.allclose(r["acceptRate"], (a["acceptRate"] + b["acceptRate"]) / 2, rtol=1e-12, atol=0)

        q0 = on_device(rng.normal(0.0, 1.0, (D, P)), dt)
        mass = on_device(rng.uniform(0.5, 2.0, P), dt)
        qf = q0.clone()
        full = run_tempered(E, pe, qf, mass, args(E, 0.1, 10), 40, betas, dt)
        qs = q0.clone()
        H = P // 2
        parts = [run_tempered(E, pe, qs[:, o:o + H], mass[o:o + H], args(E, 0.1, 10, offset=o), 40, betas, dt)
                 for o in (0, H)]
        assert torch.equal(qs, qf)
        for j in range(4):
            assert np.array_equal(full[j], np.concatenate([p[j] for p in parts], axis=1 if j == 0 else 0)), j


def test_tempered_refusals(E):
    """ehmc_hmc_run_tempered's refusals through the C ABI, and getSamplesTempered's own."""
    import torch

    lib = E._lib
    ctx = lib.Context.get()
    D, P = 3, 64
    pe = E.HarmonicPotential(np.ones(D))
    h = pe.handle(32, ctx)
    q = on_device(np.zeros((D, P)), np.float32)
    mass = on_device(np.ones(P), np.float32)

    def code(R=4, betas=(1.0, 0.5, 0.25, 0.1), q=q, mass=mass, a=None, pot=h, host_betas=False, P=P):
        b = np.asarray(betas, float)
        bt = b if host_betas else torch.tensor(b, device="cuda")
        return status(E, lambda: lib.hmc_run_tempered(ctx, pot, q, mass, a or args(E, 0.1, 5), 2, R, bt))

    assert code() == lib.EHMC_OK
    for R in (0, 3, 6, 64):
        assert code(R=R, betas=np.geomspace(1, 0.1, max(R, 1))) == INVALID, R
    assert code(R=8, betas=np.geomspace(1, 0.1, 8), q=q[:, :60], mass=mass[:60]) == INVALID  # P mod R
    assert code(a=args(E, 0.1, 5, offset=6)) == INVALID  # particleOffset mod R
    for bad in ((0.9, 0.5, 0.25, 0.1), (1.0, 0.5, 0.5, 0.1), (1.0, 0.25, 0.5, 0.1), (1.0, 0.5, 0.25, 0.0),
                (1.0, 0.5, 0.25, -0.1), (1.0, 0.5, np.nan, 0.1), (1.0, 0.5, 0.25)):
        assert code(betas=bad) == INVALID, bad
    assert code(q=q.cpu().numpy(), mass=mass.cpu().numpy()) == INVALID  # host tensors
    assert code(host_betas=True) == INVALID
    dyn = lib.dynamic_to_device(0.1, 0, "cuda")
    assert code(a=lib.make_args(0.1, 0.01, 5, KB, TEMP, dynamic=dyn.data_ptr())) == UNSUPPORTED
    X = np.random.RandomState(0).standard_normal((20, D))
    logistic = E.LogisticPotential(X, (X[:, 0] > 0).astype(float)).handle(32, ctx)
    assert code(pot=logistic) == UNSUPPORTED
    D2 = 20
    dense = E.GaussianPotential(precision=np.eye(D2)).handle(32, ctx)
    assert code(pot=dense, q=on_device(np.zeros((D2, P)), np.float32)) == UNSUPPORTED

    ens = ensemble(E, D, P, np.float32)
    hmc = E.HMC(ens, 0.5, 0.1, None, potential=pe, rng="numpy")
    with pytest.raises(ValueError, match="philox"):
        hmc.getSamplesTempered(2, TEMP, 1.0, [1.0, 0.5])
    hmc = E.HMC(ens, 0.5, 0.1, None, potential=E.LogisticPotential(X, (X[:, 0] > 0).astype(float)))
    with pytest.raises(ValueError, match="small-D"):
        hmc.getSamplesTempered(2, TEMP, 1.0, [1.0, 0.5])
    hmc = E.HMC(ens, 0.5, 0.1, None, potential=pe)
    for R, betas in ((3, [1.0, 0.5, 0.2]), (2, [1.0, 1.0]), (2, [0.5, 0.2])):
        with pytest.raises(lib.EhmcError) as e:
            hmc.getSamplesTempered(2, TEMP, 1.0, betas)
        assert e.value.code == INVALID, betas
