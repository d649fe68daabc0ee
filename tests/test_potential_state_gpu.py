"""A potential's parameters after ehmc_potential_create, through the C ABI itself (pytest -m gpu).

  * what ehmc_potential_create refuses, with its status code;
  * the funnel's optional scales default to 1: {D, s} and {D, s, 1, 1} are the same potential, bit for bit;
  * which potentials ehmc_hmc_run, ehmc_hmc_run_ensemble and args.dynamic take: those with a register-resident (small-D)
    kernel -- dense Gaussians up to D = 16, diagonal Gaussians and hierarchical models up to D = 32 -- and not a
    diagonal Gaussian above 32 dimensions, which runs as a dense one.

The calls go through the ctypes layer (physicsbasedbayesianinference_b200._lib), which validates nothing itself, so
these are the library's own checks, not the Python classes'.
"""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

INVALID, UNSUPPORTED = -1, -3  # ehmc_status (include/ehmc.h)


@pytest.fixture(scope="module")
def lib():
    import physicsbasedbayesianinference_b200 as pkg

    pkg._lib.Context.get()  # fails loudly when the extension or the GPU is missing
    return pkg._lib


def create(lib, family, params, scalars, bits):
    return lib.PotentialHandle(lib.Context.get(), family, params, scalars, bits)


def status(lib, call):
    """The ehmc status code of call() (0: EHMC_OK)."""
    try:
        call()
    except lib.EhmcError as e:
        return e.code
    return lib.EHMC_OK


def device(a, bits):
    import torch

    return torch.tensor(np.asarray(a), dtype=torch.float32 if bits == 32 else torch.float64, device="cuda")


@pytest.mark.parametrize("bits", [32, 64])
def test_create_checks_parameters(lib, bits):
    rng = np.random.RandomState(1)
    X, y = rng.standard_normal((64, 3)), (rng.uniform(size=64) < 0.5).astype(np.float64)
    funnel, coin, nbody, logistic = lib.FAMILY_FUNNEL, lib.FAMILY_COIN_TOSS, lib.FAMILY_NBODY, lib.FAMILY_LOGISTIC
    refused = [
        (funnel, [], [4, 0.0]),  # sigma_v <= 0
        (funnel, [], [4, -3.0]),
        (funnel, [], [4, 3.0, 0.0, 1.0]),  # scaleV <= 0
        (funnel, [], [4, 3.0, 1.0, -0.5]),  # scaleX <= 0
        (funnel, [], [4, 3.0, 1.0]),  # three scalars
        (coin, [np.array([2.0, 5.0]), np.array([4.0, 4.0])], []),  # successes > trials
        (nbody, [np.ones(3)], [1.0, -0.1]),  # eps < 0
        (logistic, [X, y], [0.0]),  # priorScale <= 0
        (logistic, [X, y], [-1.0]),
    ]
    for family, params, scalars in refused:
        assert status(lib, lambda: create(lib, family, params, scalars, bits)) == INVALID, (family, scalars)
    accepted = [
        (funnel, [], [4, 3.0]),
        (funnel, [], [4, 3.0, 1.7, 0.6]),
        (coin, [np.array([2.0, 4.0]), np.array([4.0, 4.0])], []),
        (nbody, [np.ones(3)], [1.0, 0.0]),
        (nbody, [np.ones(3)], [1.0, 0.1]),
        (logistic, [X, y], [2.0]),
    ]
    for family, params, scalars in accepted:
        assert status(lib, lambda: create(lib, family, params, scalars, bits)) == lib.EHMC_OK, (family, scalars)


@pytest.mark.parametrize("bits", [32, 64])
def test_funnel_scales_default_to_one(lib, bits):
    import torch

    ctx = lib.Context.get()
    rng = np.random.RandomState(2)
    P = 1000
    for D in (2, 5, 10, 17, 32):
        q = device(rng.standard_normal((D, P)) * np.r_[3.0, np.ones(D - 1)][:, None], bits)
        out = []
        for scalars in ([D, 3.0], [D, 3.0, 1.0, 1.0]):
            e, g = torch.empty(P, dtype=q.dtype, device="cuda"), torch.empty_like(q)
            lib.potential_eval(ctx, create(lib, lib.FAMILY_FUNNEL, [], scalars, bits), q, e, g)
            out.append((e.cpu(), g.cpu()))
        assert torch.isfinite(out[0][0]).all() and torch.isfinite(out[0][1]).all(), D
        assert torch.equal(out[0][0], out[1][0]) and torch.equal(out[0][1], out[1][1]), D


def small_d_case(lib, kind, D, bits):
    rng = np.random.RandomState(D)
    if kind == "dense":
        A = rng.standard_normal((D, D))
        return create(lib, lib.FAMILY_DENSE_GAUSSIAN, [A @ A.T / D + np.eye(D)], [], bits)
    if kind == "diag":  # above D = 32 the library runs it as a dense Gaussian
        return create(lib, lib.FAMILY_DIAG_GAUSSIAN, [rng.uniform(0.5, 2.0, D)], [], bits)
    J = D - 2
    return create(lib, lib.FAMILY_HIERARCHICAL_NORMAL, [rng.normal(5.0, 10.0, J), rng.uniform(5.0, 20.0, J)],
                  [0.0, 5.0, 5.0, 0.0], bits)


# (family, D, whether it has a register-resident kernel); the hierarchical models are J = 1 and J = 30 groups
SMALL_D_BOUNDARY = [("dense", 16, True), ("dense", 17, False), ("diag", 32, True), ("diag", 33, False),
                    ("hierarchical", 3, True), ("hierarchical", 32, True)]


@pytest.mark.parametrize("bits", [32, 64])
@pytest.mark.parametrize("kind,D,small", SMALL_D_BOUNDARY)
def test_fused_runs_and_dynamic_take_small_d_potentials(lib, kind, D, small, bits):
    import torch

    ctx = lib.Context.get()
    pot = small_d_case(lib, kind, D, bits)
    P, h, L = 512, 0.05, 4
    rng = np.random.RandomState(3)
    q = device(0.5 * rng.standard_normal((D, P)), bits)
    mass = device(np.ones(P), bits)
    want = lib.EHMC_OK if small else UNSUPPORTED
    args = lib.make_args(h, h * h, L, 1.0, 1.0, seed=7)
    assert status(lib, lambda: lib.hmc_run(ctx, pot, q, mass, args, 2)) == want, "ehmc_hmc_run"
    state = torch.tensor([h, math.log(h), 0.0, 0.0], dtype=torch.float64, device="cuda")
    adapt = lib.make_adapt_args(P, 2)
    assert status(lib, lambda: lib.hmc_run_ensemble(ctx, pot, q, mass, args, 2, adapt, state)) == want, \
        "ehmc_hmc_run_ensemble"
    if bits == 64:  # float32 dense potentials above D = 16 take args.dynamic on the tensor-core kernel
        dyn = lib.dynamic_to_device(h, 0, q.device)
        dargs = lib.make_args(h, h * h, L, 1.0, 1.0, seed=7, dynamic=dyn.data_ptr())
        assert status(lib, lambda: lib.hmc_iter(ctx, pot, q, mass, dargs)) == want, "ehmc_hmc_iter, args.dynamic"
    torch.cuda.synchronize()
    assert torch.isfinite(q).all()
