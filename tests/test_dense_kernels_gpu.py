"""The dense Gaussian family for 16 < D <= 128 (pytest -m gpu): every instance of its two trajectory kernels against the
float64 NumPy oracle.

  * k_dense<T, TN, MINB> (csrc/k_dense.cuh, CUDA cores): float64, ill-conditioned precision matrices and
    dense_path = 1.  TN = dense_tn(D) output dims per warp; float32 TN = 13 also comes with MINB = 2 (two CTAs per SM,
    dense_occupancy = 2).  Run at the TN edges D = 17, 32, 33, 64, 65, 104, 105, 128.
  * k_dense_tc3<C8> (csrc/k_dense_tc3.cuh, 3xFP16 split on the tensor cores, persistent): the float32 default, one
    instance per C8 = ceil(D / 8) = 3 .. 16.  Run at D = 8 C8 (last 8-dim chunk full) and at one D whose last chunk
    is partly padding; across the sweep D mod 4 takes every value (the float32 Metropolis uniform follows RNG stream
    version 2, which depends on D mod 4).

Per instance: one fed HMC iteration (q, stored momentum, accept, the 2D+3 statistics) for both integrators, L = 0, 1, 7
and both rejected-momentum conventions; production (in-kernel Philox) against fed draws bit for bit, with and without
a momentum output; the kernels' write-back branches against each other; integrate-only; forced against automatic
kernel choice; and step size 0.  Then the persistent tile schedule of k_dense_tc3 over tile counts around the SM
count, config 2's own shape at 2^20 particles, and the host (chunked) path.

Tolerances are the suite's (tests/test_gpu_parity.py, DESIGN.md section 2): trajectories within 1e-5 relative in
float32 and 1e-12 in float64, "relative" = max |a - b| / max |b|; Stormer-Verlet momenta within 2e-4 in float32 (the
backward difference (q_{L+1} - q_L) / h); accept decisions identical outside the tie band |u - min(1, ratio)| < TIE.
Each case keeps P L D^2 small: the oracle's cost is float64 matrix products.
"""
import numpy as np
import pytest

from oracle import hmc_oracle as O

pytestmark = pytest.mark.gpu

RTOL = {np.float32: 1e-5, np.float64: 1e-12}
TIE = {np.float32: 2e-3, np.float64: 1e-9}
SV_PTOL32 = 2e-4  # float32 Stormer-Verlet momentum, see test_dense_tensor_core_stormer_verlet
KB = O.BOLTZMANN
TEMP = 1 / KB  # k_B T = 1: unit-variance momenta for unit mass
METHODS = ("Leapfrog", "Stormer-Verlet")
# the context's defaults (csrc/host_defs.h); the context is one per process, shared with every other test module
DEFAULT_OPTIONS = {"dense_path": 0, "dense_occupancy": 2, "host_chunk_mb": 32}


# ---------------------------------------------------------------------------
# the launchers' instance rules (csrc/inst_dense.cuh, csrc/inst_dense_f32.cu, csrc/inst_dense_tc3.cu), written out
# ---------------------------------------------------------------------------
def dense_tn(D):
    """Output dims per warp of k_dense (dense_tn in csrc/inst_dense_f32.cu)."""
    return 4 if D <= 32 else 8 if D <= 64 else 13 if D <= 104 else 16


def dense_minb(dt, tn, occupancy):
    """__launch_bounds__ min-blocks of the k_dense instance launch_dense picks."""
    return 2 if (dt == np.float32 and tn == 13 and occupancy >= 2) else 1


def tc3_c8(D):
    return (D + 7) // 8


K_DENSE_D = (17, 32, 33, 64, 65, 104, 105, 128)
# D = 8 C8 and D = 8 C8 - (1 + C8 mod 7): the last chunk holds 1 .. 7 padding dims, D mod 4 takes all four values
TC3_D = tuple(d for c8 in range(3, 17) for d in (8 * c8, 8 * c8 - 1 - c8 % 7))

# a case is (kernel, dtype, D, dense_occupancy)
CASES = ([("k_dense", np.float32, D, occ) for D in K_DENSE_D for occ in ((1, 2) if dense_tn(D) == 13 else (2,))] +
         [("k_dense", np.float64, D, 2) for D in K_DENSE_D] +
         [("k_dense_tc3", np.float32, D, 2) for D in TC3_D])


def instance(case):
    """The compiled kernel a case runs: ("k_dense", dtype, TN, MINB) or ("k_dense_tc3", "float32", C8)."""
    kernel, dt, D, occ = case
    if kernel == "k_dense":
        tn = dense_tn(D)
        return (kernel, np.dtype(dt).name, tn, dense_minb(dt, tn, occ))
    return (kernel, np.dtype(dt).name, tc3_c8(D))


def case_id(case):
    inst = instance(case)
    if inst[0] == "k_dense":
        return f"k_dense-{inst[1]}-TN{inst[2]}-MINB{inst[3]}-D{case[2]}"
    return f"k_dense_tc3-C8_{inst[2]}-D{case[2]}"


TC3_CASES = [c for c in CASES if c[0] == "k_dense_tc3"]
by_case = pytest.mark.parametrize("case", CASES, ids=[case_id(c) for c in CASES])
by_tc3_case = pytest.mark.parametrize("case", TC3_CASES, ids=[case_id(c) for c in TC3_CASES])


# ---------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------
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


def tdtype(dt):
    import torch

    return torch.float32 if dt == np.float32 else torch.float64


def on_device(a, dt):
    import torch

    return torch.tensor(np.asarray(a), dtype=tdtype(dt), device="cuda")


def host(t):
    return t.double().cpu().numpy()


def rounded(a, dt):
    """a as the kernel receives it (rounded to the state's precision), back in float64 for the oracle."""
    return np.asarray(a, dtype=dt).astype(np.float64)


def padded(a, dt, ld, col0=0):
    """a (D, P) as a column window [col0, col0 + P) of a device array with row stride ld."""
    import torch

    D, P = a.shape
    base = torch.zeros((D, ld), dtype=tdtype(dt), device="cuda")
    view = base[:, col0:col0 + P]
    view.copy_(torch.as_tensor(np.asarray(a), dtype=tdtype(dt)))
    return view


class Problem:
    """A well-conditioned dense Gaussian (Lambda = A A^T / D + I, nonzero mean) with rounded starting states, masses
    in [0.5, 2] and fed draws."""

    def __init__(self, E, D, P, dt, seed):
        rng = np.random.RandomState(seed)
        A = rng.standard_normal((D, D))
        self.prec = A @ A.T / D + np.eye(D)
        self.mu = 0.5 * rng.standard_normal(D)
        self.pe = E.GaussianPotential(precision=self.prec, mean=self.mu)
        self.po = O.DenseGaussian(self.prec, self.mu)
        self.D, self.P, self.dt = D, P, dt
        self.q0 = rounded(self.mu[:, None] + rng.standard_normal((D, P)), dt)
        self.z = rounded(rng.standard_normal((D, P)), dt)
        self.u = rounded(rng.uniform(size=P), dt)
        self.p0 = rounded(rng.standard_normal((D, P)), dt)  # integrate-only momenta
        self.mass = rounded(rng.uniform(0.5, 2.0, P), dt)
        self.rng = rng

    def handle(self, E):
        ctx = E._lib.Context.get()
        return self.pe.handle(32 if self.dt == np.float32 else 64, ctx)


def integ_code(E, method):
    return E._lib.LEAPFROG if method == "Leapfrog" else E._lib.STORMER_VERLET


def select(E, options, case):
    """Context options that make the launcher pick the case's kernel."""
    kernel, dt, D, occ = case
    if kernel == "k_dense":
        options(dense_path=1, dense_occupancy=occ)
    else:
        options(dense_path=4)


def ld_of(case, P):
    """Row stride of the device arrays: k_dense reads and writes 16-byte vectors when the stride is a multiple of its
    per-thread particle count (4 in float32, 2 in float64) and the base is aligned; a stride that is a multiple of 4
    gives every full thread the vector branch while P stays ragged."""
    return P if case[0] == "k_dense_tc3" else (P + 3) // 4 * 4


def run_hmc(E, prob, args, *, ld=None, col0=0, q0=None, fed=True, p_out=True, stats=True, z=None, u=None):
    """One ehmc_hmc_iter on device views with row stride ld.  Returns (q, p or None, accept, stats or None) on the
    host, and keeps the device results."""
    import torch

    D, P, dt = prob.D, prob.P, prob.dt
    ld = P if ld is None else ld
    q = padded(prob.q0 if q0 is None else q0, dt, ld, col0)
    p = padded(np.zeros((D, P)), dt, ld, col0) if p_out else None
    zz = padded(prob.z, dt, ld, col0) if (fed and z is None) else z
    uu = on_device(prob.u, dt) if (fed and u is None) else u
    acc = torch.empty(P, dtype=torch.uint8, device="cuda")
    st = torch.zeros(2 * D + 3, dtype=torch.float64, device="cuda") if stats else None
    ctx = E._lib.Context.get()
    E._lib.hmc_iter(ctx, prob.handle(E), q, on_device(prob.mass, dt), args, p_out=p, z=zz, u=uu, accept=acc,
                    stats=st)
    torch.cuda.synchronize()
    return (host(q), None if p is None else host(p), acc.cpu().numpy().astype(bool),
            None if st is None else st.cpu().numpy())


def check_stats(st, q, acc, oh, nh, dt):
    """The 2D+3 statistics against O.ensemble_stats of the oracle's energies with the kernel's decisions and q.

    [0] is exactly the accept count.  [3:] are float64 sums of the returned q, within 1e-9 of the sum of magnitudes
    (both kernels sum float64 conversions in float64; only the order differs).  The energy terms are bounded the way
    test_small_d_engine.stats_tolerance bounds them: each particle's min(1, ratio) and kept H may differ from the
    oracle's by the trajectory tolerance RTOL times the column's scale (2 max|H| for the ratio, whose argument is a
    difference of two energies; max|H| for H), plus the float64 sum's own rounding."""
    D, P = q.shape
    ref = O.ensemble_stats(q, acc, oh, nh)
    assert st[0] == acc.sum(), ("n_accept", st[0], acc.sum())
    mag = np.concatenate([np.sum(np.abs(q), axis=1), np.sum(q * q, axis=1)])
    err = np.abs(st[3:] - ref[3:])
    assert np.all(err <= 1e-9 * mag), ("coordinate sums", float(np.max(err / np.maximum(mag, 1e-300))))
    with np.errstate(over="ignore"):
        accp = np.minimum(1.0, np.exp(oh - nh))
    kept_h = np.where(acc, nh, oh)
    hmax = max(np.max(np.abs(oh)), np.max(np.abs(nh)))
    tol = P * RTOL[dt] * np.array([2 * hmax, hmax]) + 1e-12 * np.array([np.sum(accp), np.sum(np.abs(kept_h))])
    assert np.all(np.abs(st[1:3] - ref[1:3]) <= tol), ("energy terms", st[1:3], ref[1:3], tol)


def compare_iteration(prob, res, method, L, h, bug, where, z=None, u=None):
    """A fed HMC iteration's (q, p, accept, stats) against O.hmc_iter on the same rounded inputs (the problem's own
    draws, or z and u)."""
    q, p, a, st = res
    dt = prob.dt
    z = prob.z if z is None else z
    u = prob.u if u is None else u
    qr, pr, accr, oh, nh = O.hmc_iter(prob.q0, z, u, prob.mass, TEMP, h, L, prob.po, method, bug_compat=bug)
    with np.errstate(over="ignore"):
        clear = np.abs(u - np.minimum(1, np.exp(oh - nh))) > TIE[dt]
    assert np.array_equal(a[clear], accr[clear]), "accept/reject differs away from a tie: " + where
    same = a == accr
    assert rel_err(q[:, same], qr[:, same]) < RTOL[dt], where
    ptol = SV_PTOL32 if (dt == np.float32 and method != "Leapfrog") else RTOL[dt]
    if p is not None:
        assert rel_err(p[:, same], pr[:, same]) < ptol, where
    if st is not None:
        check_stats(st, q, a, oh, nh, dt)
    return a


# ---------------------------------------------------------------------------
# 1. the instance table covers what the launchers compile: tests/test_dense_kernels_cpu.py
# 2. per instance, against the oracle
# ---------------------------------------------------------------------------
@by_case
def test_fed_iteration_vs_oracle(E, options, case):
    """(a) + (e): one HMC iteration with fed z and u and a momentum output, both integrators, L = 0, 1, 7, with the
    reference's rejected-row momentum (the old position, EHMC_FLAG_BUGCOMPAT_MOMENTUM) and without (the old momentum),
    against O.hmc_iter; the statistics against O.ensemble_stats.  P is ragged: not a multiple of 128 or of k_dense's
    particles per CTA.  The tensor-core kernel's statistics take the P < 16 D route (k_stats_finalize + k_colstats)
    except at D = 20; test_statistics_many_particles covers the other."""
    kernel, dt, D, occ = case
    P = 333
    prob = Problem(E, D, P, dt, seed=1000 + D)
    select(E, options, case)
    h = 0.1
    n_rej = 0
    for method in METHODS:
        for L in (0, 1, 7):
            for bug in (False, True):
                args = E._lib.make_args(h, h * h, L, KB, TEMP, integrator=integ_code(E, method),
                                        flags=E._lib.FLAG_BUGCOMPAT_MOMENTUM if bug else 0, seed=3, iteration=5,
                                        particle_offset=777)
                res = run_hmc(E, prob, args, ld=ld_of(case, P))
                a = compare_iteration(prob, res, method, L, h, bug, f"{case_id(case)} {method} L={L} bug={bug}")
                n_rej += int((~a).sum())
    assert n_rej > 0  # the rejected-row momentum conventions were exercised


@by_tc3_case
@pytest.mark.parametrize("P_of_D", ["16D-1", "16D+77"])
def test_statistics_many_particles(E, options, case, P_of_D):
    """(e) Both statistics routes of the tensor-core kernel: the per-particle scalars are reduced by k_stats_finalize
    with k_colstats below P = 16 D, and by k_ens_stats_partial from P = 16 D on."""
    kernel, dt, D, occ = case
    P = 16 * D - 1 if P_of_D == "16D-1" else 16 * D + 77
    prob = Problem(E, D, P, dt, seed=2000 + D)
    select(E, options, case)
    h, L = 0.1, 7
    for method in METHODS:
        args = E._lib.make_args(h, h * h, L, KB, TEMP, integrator=integ_code(E, method), seed=3, iteration=5)
        for p_out in (True, False):  # general and fast write-back
            res = run_hmc(E, prob, args, p_out=p_out)
            compare_iteration(prob, res, method, L, h, False, f"{case_id(case)} {method} P={P} p_out={p_out}")


@by_case
def test_production_equals_fed(E, options, case):
    """(b) + (c): with z = u = NULL the kernel draws the Philox stream itself (k_dense_tc3: the producer warpgroup and
    its shared-memory stashes); the result equals feeding ehmc_philox_fill's draws for the same seed, iteration and
    particle offset, bit for bit, with and without a momentum output.  Without one, k_dense_tc3 takes its fast
    write-back, whose q must be bit-equal to the general write-back's.  k_dense's vector branch (aligned base, row
    stride a multiple of 4 or 2) must be bit-equal to its scalar branch (odd stride, misaligned base)."""
    import torch

    kernel, dt, D, occ = case
    P = 333
    prob = Problem(E, D, P, dt, seed=3000 + D)
    select(E, options, case)
    ctx = E._lib.Context.get()
    seed, it, off = 0x9E3779B97F4A7C15, 11, 5 * 128 + 3
    z = padded(np.zeros((D, P)), dt, P)
    u = torch.empty(P, dtype=tdtype(dt), device="cuda")
    E._lib.philox_fill(ctx, z, u, seed, it, off)
    torch.cuda.synchronize()
    zf, uf = host(z), host(u)
    h, L = 0.1, 7
    n_rej = 0
    for method in METHODS:
        for flags in (0, E._lib.FLAG_BUGCOMPAT_MOMENTUM):
            args = E._lib.make_args(h, h * h, L, KB, TEMP, integrator=integ_code(E, method), flags=flags, seed=seed,
                                    iteration=it, particle_offset=off)
            where = f"{case_id(case)} {method} flags={flags}"
            ld = ld_of(case, P)
            prod = run_hmc(E, prob, args, ld=ld, fed=False)
            prod_fast = run_hmc(E, prob, args, ld=ld, fed=False, p_out=False)
            fed = run_hmc(E, prob, args, ld=ld, z=z, u=u)
            fed_fast = run_hmc(E, prob, args, ld=ld, z=z, u=u, p_out=False)
            n_rej += int((~prod[2]).sum())
            for r in (prod_fast, fed, fed_fast):
                assert np.array_equal(r[0], prod[0]), where
                assert np.array_equal(r[2], prod[2]), where
                assert np.array_equal(r[3], prod[3]), where
            assert np.array_equal(fed[1], prod[1]), where
            # the fed run is the oracle's iteration on these draws
            compare_iteration(prob, fed, method, L, h, flags != 0, where, z=zf, u=uf)
            if kernel == "k_dense":
                # scalar loads and stores: odd row stride, base one element past an aligned address
                odd = run_hmc(E, prob, args, ld=P + 2 + (P % 2 == 0), col0=1, z=padded(zf, dt, P + 5, 1), u=u)
                for x, y in zip(odd, fed):
                    assert np.array_equal(x, y), where
    assert n_rej > 0  # rejected rows: the redrawn old momentum (flags 0) and the old position (bugCompat)


@by_case
def test_integrate_only_vs_oracle(E, options, case):
    """(d) ehmc_leapfrog / ehmc_stormer_verlet (no Metropolis step) against O.leapfrog / O.stormer_verlet; the
    tensor-core kernel's overflow counter (rows that left the fp16 operand range) stays 0."""
    import torch

    kernel, dt, D, occ = case
    P = 333
    prob = Problem(E, D, P, dt, seed=4000 + D)
    select(E, options, case)
    ctx = E._lib.Context.get()
    ctx.overflow_count()  # start from 0
    h = 0.1
    for method in METHODS:
        for L in (0, 7):
            integ = O.leapfrog if method == "Leapfrog" else O.stormer_verlet
            qr, pr = integ(prob.q0, prob.p0, prob.mass, h, L, prob.po.grad)
            q, p = on_device(prob.q0, dt), on_device(prob.p0, dt)
            E._lib.leapfrog(ctx, prob.handle(E), q, p, on_device(prob.mass, dt), h, h * h, L,
                            stormer=method != "Leapfrog")
            torch.cuda.synchronize()
            where = f"{case_id(case)} {method} L={L}"
            assert rel_err(host(q), qr) < RTOL[dt], where
            ptol = SV_PTOL32 if (dt == np.float32 and method != "Leapfrog") else RTOL[dt]
            assert rel_err(host(p), pr) < ptol, where
    assert ctx.overflow_count() == 0


def guard_failing_precision(D, rng):
    """A positive definite Lambda whose diagonal spans 2^30: coordinate scales beyond the fp16 split's headroom, so
    the automatic path runs k_dense (csrc/inst_dense_tc3.cu, pack_dense_tc3)."""
    s = np.logspace(0, 4.5, D)
    A = rng.standard_normal((D, D))
    prec = (A @ A.T / D + np.eye(D)) * np.outer(s, s)
    return 0.5 * (prec + prec.T), 1.0 / s


@by_tc3_case
def test_auto_path_equals_forced_path(E, options, case):
    """(f) dense_path = 0 (automatic) is bit-equal to the kernel it should pick: the tensor-core kernel (4) for a
    well-conditioned Lambda, the CUDA-core kernel (1) for one that fails the split guard."""
    kernel, dt, D, occ = case
    P = 333
    prob = Problem(E, D, P, dt, seed=5000 + D)
    h, L = 0.1, 7
    for method in METHODS:
        args = E._lib.make_args(h, h * h, L, KB, TEMP, integrator=integ_code(E, method), seed=8, iteration=2,
                                particle_offset=129)
        out = {}
        for path in (0, 4):
            options(dense_path=path)
            out[path] = run_hmc(E, prob, args, fed=False)
        for x, y in zip(out[0], out[4]):
            assert np.array_equal(x, y), f"{case_id(case)} {method}"
    # a Lambda that fails the guard
    bad = Problem(E, D, P, dt, seed=5100 + D)
    bad.prec, sd = guard_failing_precision(D, bad.rng)
    bad.pe = E.GaussianPotential(precision=bad.prec, mean=bad.mu * sd)
    bad.q0 = rounded(bad.mu[:, None] * sd[:, None] + bad.z * sd[:, None], dt)
    h = 0.3 / np.sqrt(np.linalg.eigvalsh(bad.prec).max())
    args = E._lib.make_args(h, h * h, L, KB, TEMP, seed=8, iteration=2, particle_offset=129)
    out = {}
    for path in (0, 1):
        options(dense_path=path)
        out[path] = run_hmc(E, bad, args, fed=False)
    for x, y in zip(out[0], out[1]):
        assert np.array_equal(x, y), f"{case_id(case)} guard"
    assert 0 < out[0][2].sum()


@pytest.mark.parametrize("D", [D for D in K_DENSE_D if dense_tn(D) == 13])
def test_k_dense_occupancy_variants_agree(E, options, D):
    """(f) float32 k_dense<float, 13, 1> and <float, 13, 2> differ only in __launch_bounds__.  Their PTX (nvcc -ptx
    for sm_100a) holds the same floating-point operations, with the same FMA contraction (1640 fma.rn.f32 each); the
    MINB = 2 body re-computes six products of the step-size factors instead of keeping them live, which changes no
    value.  So both give the same bits, fed and in production."""
    P = 333
    prob = Problem(E, D, P, np.float32, seed=6000 + D)
    h, L = 0.1, 7
    for method in METHODS:
        args = E._lib.make_args(h, h * h, L, KB, TEMP, integrator=integ_code(E, method), seed=8, iteration=2,
                                particle_offset=129)
        out = {}
        for occ in (1, 2):
            options(dense_path=1, dense_occupancy=occ)
            out[occ] = (run_hmc(E, prob, args, ld=ld_of(("k_dense",), P), fed=False),
                        run_hmc(E, prob, args, ld=ld_of(("k_dense",), P)))
        for r1, r2 in zip(out[1], out[2]):
            for x, y in zip(r1, r2):
                assert np.array_equal(x, y), f"D={D} {method}"


@by_case
def test_zero_step_size(E, options, case):
    """(g) stepSize = 0.  Leapfrog on both kernels, and Stormer-Verlet on the tensor-core kernel, are the fixed point:
    q and p unchanged (up to the rounding of the kernels' own coordinate transforms), H unchanged, every proposal
    accepted (outside the tie band at ratio 1).  Stormer-Verlet on k_dense follows the reference: q is unchanged and the
    backward-difference momentum (q - q) / 0 is NaN, so the ratio is NaN -- accepted under the reference's flags (NaN
    momentum written), rejected under EHMC_FLAG_REJECT_NONFINITE (q kept, the old momentum stored).  integrate() does
    the same without the Metropolis step."""
    import torch

    kernel, dt, D, occ = case
    P = 333
    prob = Problem(E, D, P, dt, seed=7000 + D)
    select(E, options, case)
    ctx = E._lib.Context.get()
    eps = np.finfo(dt).eps
    clear = prob.u < 1 - TIE[dt]
    p_old = prob.z * O.momentum_std(prob.mass, TEMP)
    for method in METHODS:
        nan_p = kernel == "k_dense" and method != "Leapfrog"
        if nan_p:  # what the reference computes
            with np.errstate(invalid="ignore", divide="ignore"):
                qr, pr, accr, _, _ = O.hmc_iter(prob.q0, prob.z, prob.u, prob.mass, TEMP, 0.0, 5, prob.po, method,
                                                bug_compat=False)
            assert np.isnan(pr).all() and accr.all() and np.array_equal(qr, prob.q0)
        for flags in (0, E._lib.FLAG_REJECT_NONFINITE):
            args = E._lib.make_args(0.0, 0.0, 5, KB, TEMP, integrator=integ_code(E, method), flags=flags)
            q, p, a, _ = run_hmc(E, prob, args, ld=ld_of(case, P), stats=False)
            where = f"{case_id(case)} {method} flags={flags}"
            assert rel_err(q, prob.q0) < 4 * eps, where
            if nan_p and flags:
                assert not a.any(), where
                assert np.array_equal(q, prob.q0), where
                assert rel_err(p, p_old) < RTOL[dt], where
            elif nan_p:
                assert a.all() and np.isnan(p).all(), where
            else:
                assert a[clear].all(), where
                assert rel_err(p, p_old) < 8 * eps, where
        # integrate-only
        q, p = on_device(prob.q0, dt), on_device(prob.p0, dt)
        E._lib.leapfrog(ctx, prob.handle(E), q, p, on_device(prob.mass, dt), 0.0, 0.0, 5, stormer=method != "Leapfrog")
        torch.cuda.synchronize()
        where = f"{case_id(case)} {method} integrate"
        assert rel_err(host(q), prob.q0) < 4 * eps, where
        if nan_p:
            assert np.isnan(host(p)).all(), where
        else:
            assert rel_err(host(p), prob.p0) < 8 * eps, where
    assert ctx.overflow_count() == 0


# ---------------------------------------------------------------------------
# 3. the persistent tile schedule of k_dense_tc3
# ---------------------------------------------------------------------------
def tc3_tiles(P):
    return (P + 127) // 128


def tc3_schedule(P, S):
    """(CTA, group) of every 128-particle tile: tiles are dealt to min(S, tiles) CTAs in contiguous ranges and
    alternately to the CTA's two consumer groups (csrc/k_dense_tc3.cuh)."""
    T = tc3_tiles(P)
    grid = min(S, T)
    out = {}
    for b in range(grid):
        t0, t1 = T * b // grid, T * (b + 1) // grid
        for t in range(t0, t1):
            out[t] = (b, (t - t0) & 1)
    return out


def fed_pair(E, prob, args, q0, seed, it, off):
    """Production (z = u = NULL) and fed (philox_fill draws) iterations from the same device start q0, no momentum
    output, statistics on: what HMC.run's host loop and bench.py run.  Returns both results as device tensors and
    the draws."""
    import torch

    ctx = E._lib.Context.get()
    D, P, dt = prob.D, prob.P, prob.dt
    mass = on_device(prob.mass, dt)
    z = torch.empty((D, P), dtype=tdtype(dt), device="cuda")
    u = torch.empty(P, dtype=tdtype(dt), device="cuda")
    E._lib.philox_fill(ctx, z, u, seed, it, off)
    out = []
    for zz, uu in ((None, None), (z, u)):
        q = q0.clone()
        acc = torch.empty(P, dtype=torch.uint8, device="cuda")
        st = torch.zeros(2 * D + 3, dtype=torch.float64, device="cuda")
        E._lib.hmc_iter(ctx, prob.handle(E), q, mass, args, z=zz, u=uu, accept=acc, stats=st)
        out.append((q, acc, st))
    torch.cuda.synchronize()
    return out[0], out[1], z, u


def test_persistent_schedule(E, options):
    """Tile counts 1, S - 1, S, S + 1, 2 S + 1 and 5 S + 3 on S SMs, each with a ragged last tile: each consumer group
    runs 0, 1, 2 or more tiles, with odd and even counts per CTA, and waits on its stash of normals again and again.
    For each: production without a momentum output, with statistics, equals fed bit for bit; fed matches the oracle
    over the whole ensemble; two consecutive production iterations equal the fed chain."""
    import torch

    ctx = E._lib.Context.get()
    S = ctx.device_info()["sm_count"]
    D, L, h = 100, 10, 0.05
    seed, off = 77, 1 << 20
    for T in (1, S - 1, S, S + 1, 2 * S + 1, 5 * S + 3):
        P = 128 * (T - 1) + 1 + (37 * T) % 127  # ragged last tile
        sched = tc3_schedule(P, S)
        per_group = {}
        for b, g in sched.values():
            per_group[(b, g)] = per_group.get((b, g), 0) + 1
        prob = Problem(E, D, P, np.float32, seed=T)
        args0 = E._lib.make_args(h, h * h, L, KB, TEMP, seed=seed, iteration=0, particle_offset=off)
        args1 = E._lib.make_args(h, h * h, L, KB, TEMP, seed=seed, iteration=1, particle_offset=off)
        q0 = on_device(prob.q0, np.float32)
        prod, fed, z, u = fed_pair(E, prob, args0, q0, seed, 0, off)
        where = f"T={T} P={P} tiles per group {sorted(set(per_group.values()))}"
        for x, y in zip(prod, fed):
            assert torch.equal(x, y), where
        zf, uf = host(z), host(u)
        qr, _, accr, oh, nh = O.hmc_iter(prob.q0, zf, uf, prob.mass, TEMP, h, L, prob.po)
        q, a, st = host(fed[0]), fed[1].cpu().numpy().astype(bool), fed[2].cpu().numpy()
        with np.errstate(over="ignore"):
            clear = np.abs(uf - np.minimum(1, np.exp(oh - nh))) > TIE[np.float32]
        assert np.array_equal(a[clear], accr[clear]), where
        same = a == accr
        assert rel_err(q[:, same], qr[:, same]) < RTOL[np.float32], where
        check_stats(st, q, a, oh, nh, np.float32)
        # the second iteration from each run's own state: production chain == fed chain
        prod2, fed2, _, _ = fed_pair(E, prob, args1, prod[0], seed, 1, off)
        for x, y in zip(prod2, fed2):
            assert torch.equal(x, y), where
        assert not torch.equal(prod2[0], prod[0])


# ---------------------------------------------------------------------------
# 4. config 2's own shape
# ---------------------------------------------------------------------------
def test_config2_production_shape(E, options):
    """BASELINE config 2 exactly as bench.py and HMC.run run it: D = 100, P = 2^20, L = 50, h = 0.05, float32,
    in-kernel Philox, particle offset 2^19 (rank 1 of 2), statistics on, no momentum output.  q is bit-equal to the
    fed run; a subset of particles (first and last rows of the first and last tiles of both groups of CTA 0 and of
    the last CTA, and random rows) matches the oracle fed with the same draws; the statistics match float64 sums."""
    import torch

    ctx = E._lib.Context.get()
    S = ctx.device_info()["sm_count"]
    D, P, L, h = 100, 1 << 20, 50, 0.05
    seed, it, off = 20221018, 4, 1 << 19
    rng = np.random.RandomState(2)
    A = rng.standard_normal((D, D))
    prec = A @ A.T / D + np.eye(D)
    mu = 0.5 * rng.standard_normal(D)
    pe, po = E.GaussianPotential(precision=prec, mean=mu), O.DenseGaussian(prec, mu)
    gen = torch.Generator(device="cuda").manual_seed(3)
    q0 = torch.randn((D, P), dtype=torch.float32, device="cuda", generator=gen) + torch.tensor(
        mu, dtype=torch.float32, device="cuda")[:, None]
    mass = torch.rand(P, dtype=torch.float32, device="cuda", generator=gen) * 1.5 + 0.5
    z = torch.empty((D, P), dtype=torch.float32, device="cuda")
    u = torch.empty(P, dtype=torch.float32, device="cuda")
    E._lib.philox_fill(ctx, z, u, seed, it, off)
    args = E._lib.make_args(h, h * h, L, KB, TEMP, seed=seed, iteration=it, particle_offset=off)
    hd = pe.handle(32, ctx)
    res = []
    for zz, uu in ((None, None), (z, u)):
        q = q0.clone()
        acc = torch.empty(P, dtype=torch.uint8, device="cuda")
        st = torch.zeros(2 * D + 3, dtype=torch.float64, device="cuda")
        E._lib.hmc_iter(ctx, hd, q, mass, args, z=zz, u=uu, accept=acc, stats=st)
        res.append((q, acc, st))
    torch.cuda.synchronize()
    (qp, ap, sp), (qf, af, sf) = res
    assert torch.equal(qp, qf) and torch.equal(ap, af)
    n_acc = int(af.sum().item())
    assert sp[0].item() == n_acc and 0.2 * P < n_acc < P
    qs = qp.double()
    np.testing.assert_allclose(sp[3:3 + D].cpu().numpy(), qs.sum(1).cpu().numpy(), rtol=1e-9,
                               atol=1e-9 * qs.abs().sum(1).max().item())
    np.testing.assert_allclose(sp[3 + D:].cpu().numpy(), (qs * qs).sum(1).cpu().numpy(), rtol=1e-9)
    del qs
    # the particle subset
    sched = tc3_schedule(P, S)
    last_cta = max(b for b, _ in sched.values())
    cols = set()
    for b in (0, last_cta):
        for g in (0, 1):
            tiles = sorted(t for t, bg in sched.items() if bg == (b, g))
            assert len(tiles) >= 2, (b, g)
            for t in (tiles[0], tiles[-1]):
                cols.update(t * 128 + r for r in (0, 1, 31, 32, 63, 64, 96, 127))
    cols.update(rng.choice(P, 256, replace=False).tolist())
    idx = torch.tensor(sorted(cols), device="cuda")
    assert len(idx) >= 256
    sub = lambda t: t[..., idx].double().cpu().numpy()
    zs, us = sub(z), sub(u)
    qr, _, accr, oh, nh = O.hmc_iter(sub(q0), zs, us, sub(mass), TEMP, h, L, po)
    with np.errstate(over="ignore"):
        clear = np.abs(us - np.minimum(1, np.exp(oh - nh))) > TIE[np.float32]
    a = sub(ap).astype(bool)
    assert np.array_equal(a[clear], accr[clear])
    same = a == accr
    assert rel_err(sub(qp)[:, same], qr[:, same]) < RTOL[np.float32]


# ---------------------------------------------------------------------------
# 5. the host path
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("kernel,dt", [("k_dense_tc3", np.float32), ("k_dense", np.float64)],
                         ids=["k_dense_tc3-float32", "k_dense-float64"])
def test_host_path_equals_device_path(E, options, kernel, dt):
    """Host tensors with host_chunk_mb = 1: the ensemble crosses in many column chunks, each with its own particle
    offset into the Philox stream and its own rows of statistics partials.  q, p and accept are bit-equal to the
    device path's, the statistics agree within 1e-12 relative."""
    import torch

    D, P, L, h = 100, 20011, 7, 0.2  # a step size at which some proposals are rejected
    prob = Problem(E, D, P, dt, seed=8)
    options(host_chunk_mb=1)
    ctx = E._lib.Context.get()
    hd = prob.handle(E)
    for method in METHODS:
        args = E._lib.make_args(h, h * h, L, KB, TEMP, integrator=integ_code(E, method), seed=12, iteration=3,
                                particle_offset=4099)
        qh, ph = prob.q0.astype(dt), np.empty((D, P), dtype=dt)
        acc_h = np.empty(P, dtype=np.uint8)
        st_h = np.zeros(2 * D + 3)
        E._lib.hmc_iter(ctx, hd, qh, prob.mass.astype(dt), args, p_out=ph, accept=acc_h, stats=st_h)
        qd, pd = on_device(prob.q0, dt), torch.empty((D, P), dtype=tdtype(dt), device="cuda")
        acc_d = torch.empty(P, dtype=torch.uint8, device="cuda")
        st_d = torch.zeros(2 * D + 3, dtype=torch.float64, device="cuda")
        E._lib.hmc_iter(ctx, hd, qd, on_device(prob.mass, dt), args, p_out=pd, accept=acc_d, stats=st_d)
        torch.cuda.synchronize()
        assert np.array_equal(qh, qd.cpu().numpy()) and np.array_equal(ph, pd.cpu().numpy()), method
        assert np.array_equal(acc_h, acc_d.cpu().numpy()), method
        assert 0 < acc_h.sum() < P
        std = st_d.cpu().numpy()
        assert st_h[0] == std[0], method
        assert rel_err(st_h, std) < 1e-12, method
        np.testing.assert_allclose(st_h, std, rtol=1e-12, atol=1e-12 * np.abs(std).max())
