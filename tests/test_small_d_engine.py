"""The small-D engine (pytest -m gpu): the register-resident kernels k_small / k_small_run and the fused adaptive run
k_small_ens (csrc/k_small.cuh, csrc/k_small_ens.cuh) against the float64 NumPy oracle, over every kernel instance the
launchers can pick:

  * every width DT in {2, 4, 8, 10, 16, 32}, both as the EXACT kernel (D == DT) and padded (D < DT), and every D mod 4
    (the float32 Metropolis uniform comes from the last normal block when D mod 4 is 1 or 2: RNG stream version 2);
  * diagonal Gaussian, funnel (plain and rescaled), coin toss and dense (D <= 16) families, Leapfrog and
    Stormer-Verlet, float32 (with the packed leapfrog path) and float64;
  * the route of the diagonal Gaussian above 32 dimensions into the dense kernels;
  * the 2D+3 ensemble statistics, also with several grid-stride rounds per CTA;
  * the work-queue shapes of the fused run (sub-batches per queue item, batches per statistics group, ragged last
    batches, adaptation lags) and config 5's own shape at 2^22 particles.

Tolerances are the suite's (tests/test_gpu_parity.py, DESIGN.md section 2): trajectories within 1e-5 relative in
float32 (L <= 10 here) and 1e-12 in float64, "relative" = max |a - b| / max |b|; accept decisions identical outside
the tie band |u - min(1, ratio)| < TIE.
"""
import numpy as np
import pytest

from oracle import hmc_oracle as O

pytestmark = pytest.mark.gpu

RTOL = {np.float32: 1e-5, np.float64: 1e-12}
TIE = {np.float32: 2e-3, np.float64: 1e-9}
KB = O.BOLTZMANN
TEMP = 1 / KB  # k_B T = 1: unit-variance momenta for unit mass
# every width the small-D launchers instantiate, exact and padded, and every D mod 4
WIDTHS = (1, 2, 3, 4, 5, 7, 8, 9, 10, 11, 16, 17, 31, 32)
# the context's defaults (csrc/host_defs.h); the context is one per process, shared with every other test module
DEFAULT_OPTIONS = {"small_waves": 8, "ens_sshift": -1, "ens_groups": 0, "dense_path": 0}


def rel_err(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


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


def on_device(a, dt):
    import torch

    return torch.tensor(np.asarray(a), dtype=torch.float32 if dt == np.float32 else torch.float64, device="cuda")


def host(t):
    return t.double().cpu().numpy()


def rounded(a, dt):
    """a as the kernel receives it (rounded to the state's precision), back in float64 for the oracle."""
    return np.asarray(a, dtype=dt).astype(np.float64)


def family(E, name, D, rng):
    """(engine descriptor, oracle potential, step size, steps, start sampler) of a small-D family."""
    if name == "diag":
        k = rng.uniform(0.5, 4.0, D)
        return E.HarmonicPotential(k), O.DiagGaussian(k), 0.25, 7, lambda P: rng.standard_normal((D, P))
    if name == "funnel":
        return (E.FunnelPotential(D, 3.0), O.Funnel(D, 3.0), 0.1, 7, lambda P: rng.standard_normal((D, P)))
    if name == "funnel_scaled":  # the funnel in the coordinates mass adaptation produces (a = scaleV, lnb = ln scaleX^2)
        return (E.FunnelPotential(D, 3.0, scaleV=1.7, scaleX=0.6), O.Funnel(D, 3.0, 1.7, 0.6), 0.1, 7,
                lambda P: rng.standard_normal((D, P)))
    if name == "coin":
        # successes 6 .. 14 of 20: the posterior modes stay in 0.3 .. 0.7, away from the 1 / q poles where float32
        # trajectories lose digits to the stiffness rather than to the kernel
        k = rng.randint(6, 15, D).astype(np.float64)
        n = np.full(D, 20.0)
        return E.CoinTossPotential(k, n), O.CoinToss(k, n), 0.02, 7, lambda P: rng.uniform(0.3, 0.7, (D, P))
    assert name == "dense"
    A = rng.standard_normal((D, D))
    prec = A @ A.T / D + np.eye(D)
    mu = 0.5 * rng.standard_normal(D)
    return (E.GaussianPotential(precision=prec, mean=mu), O.DenseGaussian(prec, mu), 0.2, 7,
            lambda P: mu[:, None] + rng.standard_normal((D, P)))


def family_widths(name):
    if name.startswith("funnel"):
        return tuple(d for d in WIDTHS if d >= 2)  # the funnel needs v and at least one x
    if name == "dense":
        return tuple(d for d in WIDTHS if d <= 16)  # larger dense potentials run the dense kernels
    return WIDTHS


def stats_tolerance(dt, cols, scale, P):
    """Per-column bound of |device statistic - oracle statistic|.  float64: 1e-12 of the sum of magnitudes.  float32:
    each particle's value may differ from the oracle's by the trajectory tolerance (RTOL * scale of the column), and
    k_small sums 32 particles at a time in float32 (WarpStats: four partial sums of eight, then two levels) before the
    float64 accumulation, an error below 10 ulp = 6e-7 of the sum of magnitudes: 2e-6 leaves headroom."""
    mag = np.sum(np.abs(cols), axis=1)
    if dt == np.float64:
        return 1e-12 * mag
    return P * RTOL[dt] * scale + 2e-6 * mag


def check_stats(st, q_kept, acc, oh, nh, dt):
    """Device statistics vector against ensemble_stats of the oracle's energies and the kept positions."""
    ref = O.ensemble_stats(q_kept, acc, oh, nh)
    D, P = q_kept.shape
    assert st[0] == ref[0], ("n_accept", st[0], ref[0])
    with np.errstate(over="ignore"):
        accp = np.minimum(1.0, np.exp(oh - nh))
    kept_h = np.where(acc, nh, oh)
    hmax = max(np.max(np.abs(oh)), np.max(np.abs(nh)))
    cols = np.vstack([accp[None], kept_h[None], q_kept, q_kept * q_kept])
    scale = np.concatenate([[2 * hmax, hmax], np.max(np.abs(q_kept), axis=1), 2 * np.max(q_kept * q_kept, axis=1)])
    tol = stats_tolerance(dt, cols, scale, P)
    err = np.abs(st[1:] - ref[1:])
    bad = np.nonzero(err > tol)[0]
    assert bad.size == 0, [(int(j) + 1, float(st[j + 1]), float(ref[j + 1]), float(tol[j])) for j in bad[:4]]


def run_iteration(E, pe, po, D, P, dt, method, h, L, q0, mass, z, u, bug, stats=True):
    """One fed-draw HMC iteration on the device vs O.hmc_iter: q, stored momentum, accept decision, statistics."""
    import torch

    ctx = E._lib.Context.get()
    integ = E._lib.LEAPFROG if method == "Leapfrog" else E._lib.STORMER_VERLET
    args = E._lib.make_args(h, h * h, L, KB, TEMP, integrator=integ, flags=E._lib.FLAG_BUGCOMPAT_MOMENTUM if bug else 0)
    q = on_device(q0, dt)
    p = torch.empty_like(q)
    acc = torch.empty(P, dtype=torch.uint8, device="cuda")
    st = torch.zeros(2 * D + 3, dtype=torch.float64, device="cuda") if stats else None
    E._lib.hmc_iter(ctx, pe.handle(32 if dt == np.float32 else 64, ctx), q, on_device(mass, dt), args, p_out=p,
                    z=on_device(z, dt), u=on_device(u, dt), accept=acc, stats=st)
    torch.cuda.synchronize()
    qr, pr, accr, oh, nh = O.hmc_iter(q0, z, u, mass, TEMP, h, L, po, "Leapfrog" if method == "Leapfrog" else "Stormer",
                                      bug_compat=bug)
    a = acc.cpu().numpy().astype(bool)
    with np.errstate(over="ignore"):
        clear = np.abs(u - np.minimum(1, np.exp(oh - nh))) > TIE[dt]
    where = f"D={D} P={P} {method} {np.dtype(dt).name}"
    assert np.array_equal(a[clear], accr[clear]), "accept/reject differs away from a tie: " + where
    same = a == accr
    # float32: the ratio carries ~1e-6 of error (energies of tens, 6e-8 relative), so about P * 1e-6 uniforms fall
    # between the two ratios
    assert np.sum(~same) <= (1 + P * 1e-5 if dt == np.float32 else 0), where
    qd, pd = host(q), host(p)
    assert rel_err(qd[:, same], qr[:, same]) < RTOL[dt], where
    # Stormer-Verlet forms p as the backward difference (q - qPast) / h: float32 rounding of q divided by h
    # (DESIGN.md section 2 states 2e-4 for it)
    ptol = 2e-4 if (dt == np.float32 and method != "Leapfrog") else RTOL[dt]
    assert rel_err(pd[:, same], pr[:, same]) < ptol, where
    if stats:
        # a particle inside the tie band counts with the kernel's decision and its own kept position
        check_stats(host(st), np.where(same[None, :], qr, qd), a, oh, nh, dt)
    return a


# ---------------------------------------------------------------------------
# 1 + 4. every k_small instance vs the oracle, fed z and u; statistics vs ensemble_stats
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("name", ["diag", "funnel", "funnel_scaled", "coin", "dense"])
def test_kernel_matrix_vs_oracle(E, name, dt):
    """hmc_iter (q, stored momentum, accept, the 2D+3 statistics), integrate-only Leapfrog / Stormer-Verlet and the
    potential's energy and gradient at every width, against the float64 oracle on the same (rounded) inputs."""
    ctx = E._lib.Context.get()
    bits = 32 if dt == np.float32 else 64
    widths = family_widths(name)
    one_particle = 17 if 17 in widths else 11  # P = 1 at one padded width per family
    n_rej = {"Leapfrog": 0, "Stormer-Verlet": 0}
    for D in widths:
        for P in ((333, 1) if D == one_particle else (333,)):
            rng = np.random.RandomState(1000 * D + P)
            pe, po, h, L, start = family(E, name, D, rng)
            q0 = rounded(start(P), dt)
            z = rounded(rng.standard_normal((D, P)), dt)
            u = rounded(rng.uniform(size=P), dt)
            mass = rounded(rng.uniform(0.5, 2.0, P), dt)
            for method in ("Leapfrog", "Stormer-Verlet"):
                # the rejected particles' stored momentum: bugCompat's old position with Stormer-Verlet, the
                # redrawn old momentum with leapfrog (in float32 the packed path's own redraw)
                a = run_iteration(E, pe, po, D, P, dt, method, h, L, q0, mass, z, u, bug=method != "Leapfrog")
                assert a.sum() > 0 or P == 1
                n_rej[method] += int(np.sum(~a))
                # integrate-only
                p0 = rounded(z * np.sqrt(mass), dt)
                q, p = on_device(q0, dt), on_device(p0, dt)
                E._lib.leapfrog(ctx, pe.handle(bits, ctx), q, p, on_device(mass, dt), h, h * h, L,
                                stormer=method != "Leapfrog")
                integ = O.leapfrog if method == "Leapfrog" else O.stormer_verlet
                qr, pr = integ(q0, p0, mass, h, L, po.grad)
                where = f"integrate D={D} P={P} {method} {np.dtype(dt).name}"
                assert rel_err(host(q), qr) < RTOL[dt], where
                assert rel_err(host(p), pr) < (2e-4 if dt == np.float32 and method != "Leapfrog" else RTOL[dt]), where
            # energy and gradient (the float32 bound of test_potential_eval_matches_oracle: a sum of D rounded terms)
            qh = np.asarray(q0, dtype=dt)
            etol = RTOL[dt] * (10 if dt == np.float32 else 1)
            assert rel_err(pe(qh), po.energy(q0)) < etol, f"energy D={D}"
            assert rel_err(pe.gradient(qh), po.grad(q0)) < etol, f"gradient D={D}"
    assert min(n_rej.values()) >= 5, n_rej  # the rejection branch ran (stored momentum, kept H in the statistics)


def test_statistics_over_several_grid_stride_rounds(E, options):
    """small_waves = 1 and 2^20 + 77 particles: every CTA of k_small walks several grid-stride rounds (and the last
    one is ragged), accumulating its WarpStats over them before the one row per CTA; padded width (D = 9 in DT = 10)."""
    ctx = E._lib.Context.get()
    options(small_waves=1)
    D, P = 9, (1 << 20) + 77
    # at most 16 CTAs of 128 threads per SM and one wave: fewer CTAs than blocks of 128 particles by a factor > 3
    assert (P + 127) // 128 > 3 * 16 * ctx.device_info()["sm_count"]
    rng = np.random.RandomState(5)
    pe, po, h, L, start = family(E, "diag", D, rng)
    q_start, z_start = start(P), rng.standard_normal((D, P))
    u_start, m_start = rng.uniform(size=P), rng.uniform(0.5, 2.0, P)
    for dt in (np.float64, np.float32):
        q0, z, u, mass = (rounded(a, dt) for a in (q_start, z_start, u_start, m_start))
        a = run_iteration(E, pe, po, D, P, dt, "Leapfrog", h, L, q0, mass, z, u, bug=False)
        assert 0 < a.sum() < P


# ---------------------------------------------------------------------------
# 2. the diagonal Gaussian above 32 dimensions runs the dense kernels
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("spread", ["moderate", "wide"])
@pytest.mark.parametrize("D", [33, 100])
def test_diag_gaussian_above_32_dims_runs_the_dense_kernels(E, options, D, spread, dt):
    """ehmc_potential_create sends a diagonal Gaussian with 32 < D <= 128 to the dense family with Lambda = diag(k).
    float32: k over [0.5, 4] passes the fp16-split guard (the tensor-core kernel: bit-equal to dense_path = 4), k over
    1e-6 .. 1e6 fails it (the CUDA-core kernel: bit-equal to dense_path = 1).  Coordinates are compared in units of
    their own scale k^-1/2."""
    import torch

    rng = np.random.RandomState(D + (0 if spread == "moderate" else 1))
    P, L = 777, 10
    k = rng.permutation(np.geomspace(0.5, 4.0, D) if spread == "moderate" else np.geomspace(1e-6, 1e6, D))
    mass = rounded(rng.uniform(0.5, 2.0, P), dt)
    h = 0.3 / np.sqrt(k.max() / 0.5)  # h omega <= 0.3 (stable, stiffest dimension, lightest particle)
    sk = np.sqrt(k)[:, None]
    q0 = rounded(rng.standard_normal((D, P)) / sk, dt)
    z = rounded(rng.standard_normal((D, P)), dt)
    u = rounded(rng.uniform(size=P), dt)
    pe, po = E.HarmonicPotential(k), O.DiagGaussian(k)
    # (flags 0: a rejected particle stores its old momentum, as with bugCompat=False)
    qr, pr, accr, oh, nh = O.hmc_iter(q0, z, u, mass, TEMP, h, L, po, bug_compat=False)
    with np.errstate(over="ignore"):
        clear = np.abs(u - np.minimum(1, np.exp(oh - nh))) > TIE[dt]
    ctx = E._lib.Context.get()
    args = E._lib.make_args(h, h * h, L, KB, TEMP)
    forced = 4 if spread == "moderate" else 1
    out = {}
    for path in ((0, forced) if dt == np.float32 else (0,)):
        options(dense_path=path)
        q = on_device(q0, dt)
        p = torch.empty_like(q)
        acc = torch.empty(P, dtype=torch.uint8, device="cuda")
        E._lib.hmc_iter(ctx, pe.handle(32 if dt == np.float32 else 64, ctx), q, on_device(mass, dt), args, p_out=p,
                        z=on_device(z, dt), u=on_device(u, dt), accept=acc)
        torch.cuda.synchronize()
        out[path] = (q.cpu().numpy(), p.cpu().numpy(), acc.cpu().numpy())
    qd, pd, a = out[0]
    a = a.astype(bool)
    assert np.array_equal(a[clear], accr[clear])
    same = a == accr
    assert np.sum(~same) <= 1 and a.sum() > 0
    assert rel_err(sk * qd[:, same], sk * qr[:, same]) < RTOL[dt]
    assert rel_err(pd[:, same], pr[:, same]) < RTOL[dt]
    if dt == np.float32:
        for x, y in zip(out[0], out[forced]):
            assert np.array_equal(x, y), f"the default path is not dense_path = {forced}"


# ---------------------------------------------------------------------------
# 3. production RNG
# ---------------------------------------------------------------------------
RNG_WIDTHS = (1, 2, 3, 4, 5, 9, 10, 16, 17, 32)


@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_philox_fill_matches_the_stream_specification(E, dt):
    """ehmc_philox_fill against oracle.philox_stream at every D mod 4 (stream version 2: the float32 uniform is word z
    of block D / 4 when D mod 4 is 1 or 2, word x of block 0xFFFFFFFF otherwise), with the high words of the seed,
    the iteration and the particle id in play."""
    P, seed, it, off = 300, 0x1234567890ABCDEF, (3 << 32) + 5, (5 << 32) + 1000
    for D in RNG_WIDTHS:
        z = np.empty((D, P), dtype=dt)
        u = np.empty(P, dtype=dt)
        E._lib.philox_fill(E._lib.Context.get(), z, u, seed, it, off)
        zr, ur = O.philox_stream(seed, it, np.arange(P, dtype=np.uint64) + np.uint64(off), D, dt)
        assert np.array_equal(u.astype(np.float64), ur), f"D={D}"  # integer stream -> exact
        assert np.max(np.abs(z - zr)) < (5e-6 if dt == np.float32 else 1e-13), f"D={D}"


@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_in_kernel_draws_equal_fed_draws(E, dt):
    """hmc_iter with z = u = NULL (Philox inside k_small) == hmc_iter fed ehmc_philox_fill's output, bit for bit, at
    every D mod 4 and at exact and padded widths; float32 covers the packed leapfrog path and Stormer-Verlet.  The
    rejected particles' stored momentum is the redrawn old momentum (bugCompat off)."""
    import torch

    ctx = E._lib.Context.get()
    P, seed, it, off = 1000, 99, 3, 12345
    for D in RNG_WIDTHS:
        rng = np.random.RandomState(D)
        pe = E.HarmonicPotential(rng.uniform(0.5, 4.0, D))
        h = pe.handle(32 if dt == np.float32 else 64, ctx)
        q0 = on_device(rng.standard_normal((D, P)), dt)
        mass = on_device(rng.uniform(0.5, 2.0, P), dt)
        for integ in (E._lib.LEAPFROG, E._lib.STORMER_VERLET):
            args = E._lib.make_args(0.3, 0.3**2, 7, KB, TEMP, integrator=integ, seed=seed, iteration=it,
                                    particle_offset=off)
            res = []
            for fed in (False, True):
                z = u = None
                if fed:
                    z, u = torch.empty_like(q0), torch.empty(P, dtype=q0.dtype, device="cuda")
                    E._lib.philox_fill(ctx, z, u, seed, it, off)
                q, p = q0.clone(), torch.empty_like(q0)
                acc = torch.empty(P, dtype=torch.uint8, device="cuda")
                st = torch.zeros(2 * D + 3, dtype=torch.float64, device="cuda")
                E._lib.hmc_iter(ctx, h, q, mass, args, p_out=p, z=z, u=u, accept=acc, stats=st)
                res.append((q, p, acc, st))
            torch.cuda.synchronize()
            for x, y in zip(*res):
                assert torch.equal(x, y), f"D={D} integrator {integ}"
            n = int(res[0][2].sum())
            assert 0 < n, f"D={D}"


@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_getSamples_fused_loop_at_padded_widths(E, dt, capsys):
    """getSamples on a device ensemble (ONE k_small_run launch) == one k_small launch per iteration, bit for bit, at
    padded widths: samples, stored momenta and the final state."""
    import torch

    P, S = 777, 9
    tdt = torch.float32 if dt == np.float32 else torch.float64
    for D in (5, 9, 17, 32):
        rng = np.random.RandomState(40 + D)
        q0 = rng.standard_normal((D, P))
        mass = rng.uniform(0.5, 2.0, P)
        pot = E.FunnelPotential(D, 3.0)

        def fresh(method):
            ens = E.Ensemble(D, P, dtype=dt, device="cuda", seed=9)
            ens.mass = torch.tensor(mass, dtype=tdt, device="cuda")
            hmc = E.HMC(ens, 7 * 0.05 + 1e-9, 0.05, None, potential=pot, seed=9, bugCompat=D % 2 == 0, method=method)
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


# ---------------------------------------------------------------------------
# 5. the fused run's work-queue shapes
# ---------------------------------------------------------------------------
# (ens_sshift, ens_groups, P, D, adaptLag): every pair of values of two axes appears in some case.  Sub-batches per
# queue item 2^sshift; ens_groups caps the statistics groups per iteration (0: auto), which forces 2^bshift > 1
# batches per group at small P.  P = 5000 with sshift 1, 2 or 4 leaves a ragged last batch (157 sub-batches), P = 33
# a last sub-batch of one particle.
ENS_CASES = [
    (0, 0, 33, 3, 1), (0, 0, 5000, 32, 3), (0, 1, 31, 10, 4), (0, 3, 1, 17, 3),
    (1, 0, 1, 10, 3), (1, 0, 31, 17, 1), (1, 1, 5000, 3, 3), (1, 3, 33, 32, 4),
    (2, 0, 33, 10, 3), (2, 0, 5000, 17, 4), (2, 1, 1, 32, 1), (2, 3, 31, 3, 4),
    (4, 0, 1, 3, 4), (4, 1, 31, 32, 3), (4, 1, 33, 17, 3), (4, 3, 5000, 10, 1),
]
ENS_ITERS, ENS_ADAPT, ENS_L = 22, 16, 5  # ENS_ITERS >= 2 ENS_RING + the largest lag (k_small_ens.cuh: ENS_RING = 8)


def ens_shape(P, L, sshift_opt, groups_opt):
    """(sshift, bshift) as ens_launch (csrc/inst_small_ens.cuh) picks them."""
    nrows = (P + 31) // 32
    sshift = sshift_opt if sshift_opt >= 0 else ((2 if L <= 8 else 1) if nrows >= 1 << 16 else 0)
    nbatch = (nrows + (1 << sshift) - 1) >> sshift
    gmax = groups_opt if groups_opt > 0 else (4096 if L > 8 else 2048)
    bshift = 0
    while (nbatch >> bshift) > gmax:
        bshift += 1
    return sshift, bshift


def ens_family(E, D, rng):
    if D == 3:
        A = rng.standard_normal((D, D))
        prec = A @ A.T / D + np.eye(D)
        return E.GaussianPotential(precision=prec), O.DenseGaussian(prec), 0.15
    if D == 17:
        k = rng.uniform(0.5, 4.0, D)
        return E.HarmonicPotential(k), O.DiagGaussian(k), 0.1
    return E.FunnelPotential(D, 3.0), O.Funnel(D, 3.0), 0.05


@pytest.mark.parametrize("sshift,groups,P,D,lag", ENS_CASES)
def test_fused_run_work_queue_shapes(E, options, sshift, groups, P, D, lag):
    """HMC.run(adapt=True, keepNumSteps=True) as ONE k_small_ens launch at forced queue shapes, against
    (a) the iteration-by-iteration host loop (fused=False), in float32 and float64;
    (b) oracle.adaptive_run, in float64: step sizes to 1e-12, acceptRate exactly, meanAcceptProb and meanH to 1e-12,
        positions to 1e-9 (the device's exp(log h) may differ from libm's in the last bit);
    (c) the trace of every particle, in both dtypes: mean and var recomputed from it, and acceptRate[k] * P equal to
        the number of particles whose position changed in iteration k (bugCompat off: a rejection writes nothing)."""
    import torch

    options(ens_sshift=sshift, ens_groups=groups)
    s, b = ens_shape(P, ENS_L, sshift, groups)
    assert s == sshift
    rng = np.random.RandomState(P + 100 * D + 7 * lag)
    pot, po, h0 = ens_family(E, D, rng)
    q_start = rng.standard_normal((D, P))
    m_start = rng.uniform(0.5, 2.0, P)
    ctx = E._lib.Context.get()
    where = f"sshift={sshift} bshift={b} P={P} D={D} lag={lag}"
    for dt in (np.float64, np.float32):
        q0, mass = rounded(q_start, dt), rounded(m_start, dt)

        def fresh():
            ens = E.Ensemble(D, P, dtype=dt, device="cuda", seed=5)
            ens.q.copy_(on_device(q0, dt))
            ens.mass = on_device(mass, dt)
            return ens, E.HMC(ens, ENS_L * h0 + 1e-9, h0, None, potential=pot, seed=5, bugCompat=False)

        kw = dict(adapt=True, targetAccept=0.8, adaptIterations=ENS_ADAPT, keepNumSteps=True, traceParticles=P,
                  adaptLag=lag)
        ens_h, hmc_h = fresh()
        rh = hmc_h.run(ENS_ITERS, TEMP, fused=False, **kw)
        ens_f, hmc_f = fresh()
        n0 = ctx.launch_count()
        rf = hmc_f.run(ENS_ITERS, TEMP, **kw)
        assert rf.get("fused") and ctx.launch_count() - n0 == 1, where
        assert hmc_f.integrator.numSteps == ENS_L
        # (a) the host loop
        np.testing.assert_allclose(rf["stepSize"], rh["stepSize"], rtol=1e-12, err_msg=where)
        assert all(x == h0 for x in rf["stepSize"][:lag + 1]) and rf["stepSize"][lag + 1] != h0, where
        assert rf["stepSize"][ENS_ADAPT + lag] == rf["stepSize"][-1], where  # adaptation stops after adaptIterations
        np.testing.assert_array_equal(rf["acceptRate"], rh["acceptRate"], err_msg=where)
        np.testing.assert_allclose(rf["meanAcceptProb"], rh["meanAcceptProb"], rtol=1e-12, err_msg=where)
        np.testing.assert_allclose(rf["meanH"], rh["meanH"], rtol=1e-12, atol=1e-12, err_msg=where)
        np.testing.assert_allclose(rf["mean"].numpy(), rh["mean"].numpy(), rtol=1e-11, atol=1e-12, err_msg=where)
        np.testing.assert_allclose(rf["var"].numpy(), rh["var"].numpy(), rtol=1e-10, atol=1e-12, err_msg=where)
        assert abs(hmc_f.stepSize - hmc_h.stepSize) <= 1e-12 * hmc_h.stepSize, where
        if dt == np.float32:  # float(h) is the same number every iteration: identical bits
            assert np.array_equal(np.float32(rf["stepSize"]), np.float32(rh["stepSize"])), where
            assert torch.equal(ens_f.q, ens_h.q) and torch.equal(rf["trace"], rh["trace"]), where
        else:
            assert rel_err(host(ens_f.q), host(ens_h.q)) < 1e-9, where
            assert rel_err(host(rf["trace"]), host(rh["trace"])) < 1e-9, where
        # (b) the oracle
        if dt == np.float64:
            ref = O.adaptive_run(q0, mass, po, ENS_ITERS, TEMP, h0, ENS_L, seed=5, adapt_iterations=ENS_ADAPT,
                                 target=0.8, lag=lag)
            np.testing.assert_allclose(rf["stepSize"], ref["stepSize"], rtol=1e-12, err_msg=where)
            np.testing.assert_array_equal(rf["acceptRate"], ref["acceptRate"], err_msg=where)
            np.testing.assert_allclose(rf["meanAcceptProb"], ref["meanAcceptProb"], rtol=1e-12, atol=1e-12,
                                       err_msg=where)
            np.testing.assert_allclose(rf["meanH"], ref["meanH"], rtol=1e-12, atol=1e-12, err_msg=where)
            assert abs(hmc_f.stepSize - ref["finalStepSize"]) <= 1e-12 * ref["finalStepSize"], where
            assert rel_err(host(ens_f.q), ref["q"]) < 1e-9, where
            assert rel_err(host(rf["trace"]), ref["trace"]) < 1e-9, where
            assert 0 < np.sum(ref["acceptRate"]) < ENS_ITERS or P == 1, where
        # (c) the trace
        tr = host(rf["trace"])  # (D, P, S)
        prev = q0
        for k in range(ENS_ITERS):
            changed = int(np.sum(np.any(tr[:, :, k] != prev, axis=0)))
            assert changed == int(np.rint(rf["acceptRate"][k] * P)), (where, k)
            prev = tr[:, :, k]
        n = ENS_ITERS * P
        mean_t = tr.sum(axis=(1, 2)) / n
        msq_t = (tr * tr).sum(axis=(1, 2)) / n
        # float64: sums in another order; float32: per-32-particle float32 sums (see stats_tolerance)
        rt = 1e-12 if dt == np.float64 else 2e-6
        mean_d = rf["mean"].numpy()
        assert np.all(np.abs(mean_d - mean_t) <= rt * np.abs(tr).sum(axis=(1, 2)) / n), where
        np.testing.assert_allclose(rf["var"].numpy() + mean_d * mean_d, msq_t, rtol=rt, err_msg=where)


# ---------------------------------------------------------------------------
# 6. config 5 at full size
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("L", [20, 4])
def test_config5_fused_run_at_full_size(E, options, L):
    """BASELINE config 5's own shape: funnel 10-D, 2^22 particles, float32, adaptLag 3, default queue shapes (items of
    2 or 4 sub-batches, 16 batches per statistics group): the fused run against the host loop, step sizes to 1e-12,
    acceptRate exactly, and -- every iteration's float32(h) being the same number -- bit-equal final positions."""
    import torch

    options(**DEFAULT_OPTIONS)  # automatic queue shapes
    D, P, S, h0, lag = 10, 1 << 22, 8, 0.02, 3
    sshift, bshift = ens_shape(P, L, -1, 0)
    assert sshift in (1, 2) and bshift == 4
    pot = E.FunnelPotential(D, 3.0)
    gen = torch.Generator(device="cuda").manual_seed(L)
    q0 = torch.randn((D, P), dtype=torch.float32, device="cuda", generator=gen)

    def fresh():
        ens = E.Ensemble(D, P, dtype=np.float32, device="cuda", seed=11)
        ens.q.copy_(q0)
        return ens, E.HMC(ens, L * h0 + 1e-9, h0, None, potential=pot, seed=11, bugCompat=False)

    kw = dict(adapt=True, targetAccept=0.8, adaptIterations=S, keepNumSteps=True, adaptLag=lag)
    ens_h, hmc_h = fresh()
    rh = hmc_h.run(S, TEMP, fused=False, **kw)
    ens_f, hmc_f = fresh()
    rf = hmc_f.run(S, TEMP, **kw)
    assert rf.get("fused")
    np.testing.assert_allclose(rf["stepSize"], rh["stepSize"], rtol=1e-12)
    assert rf["stepSize"][lag + 1] != h0  # the adaptation reached the run
    np.testing.assert_array_equal(rf["acceptRate"], rh["acceptRate"])
    np.testing.assert_allclose(rf["meanAcceptProb"], rh["meanAcceptProb"], rtol=1e-12)
    assert np.array_equal(np.float32(rf["stepSize"]), np.float32(rh["stepSize"]))
    assert torch.equal(ens_f.q, ens_h.q)
