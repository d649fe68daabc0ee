"""CPU tests of the chain diagnostics (no GPU needed): nested R-hat (diagnostics.nested_rhat,
nested_rhat_from_moments) against the formulas written out as plain loops, its identities and invariances, the
cross-rank combination over gloo, superchain starts in Ensemble.setPosition, and the refusals of
HMC.run(chainDiagnostics=True) that come before any device work."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import physicsbasedbayesianinference_b200 as E
from physicsbasedbayesianinference_b200 import diagnostics


def nested_rhat_loops(draws, M):
    """Nested R-hat straight from the definitions (diagnostics.py's docstring), one dimension at a time."""
    D, C, N = draws.shape
    K = C // M
    rhat, B, W = np.empty(D), np.empty(D), np.empty(D)
    for d in range(D):
        f_mk = [[np.mean(draws[d, k * M + m]) for m in range(M)] for k in range(K)]
        s2_mk = [[np.var(draws[d, k * M + m], ddof=1) if N > 1 else 0.0 for m in range(M)] for k in range(K)]
        f_k = [sum(f_mk[k]) / M for k in range(K)]
        f_all = sum(f_k) / K
        b = sum((f_k[k] - f_all) ** 2 for k in range(K)) / (K - 1)
        w = 0.0
        for k in range(K):
            bt = sum((f_mk[k][m] - f_k[k]) ** 2 for m in range(M)) / (M - 1) if M > 1 else 0.0
            wt = sum(s2_mk[k]) / M if N > 1 else 0.0
            w += bt + wt
        w /= K
        rhat[d], B[d], W[d] = np.sqrt(1.0 + b / w), b, w
    return rhat, B, W


def draws_of(K, M, N, D=3, seed=0):
    """Superchains with different centres and chains with different offsets: R-hat well away from 1."""
    rng = np.random.RandomState(seed)
    centres = rng.standard_normal((D, K, 1, 1))
    offsets = 0.3 * rng.standard_normal((D, K, M, 1))
    x = centres + offsets + rng.standard_normal((D, K, M, N))
    return x.reshape(D, K * M, N)


@pytest.mark.parametrize("K,M,N", [(2, 1, 5), (5, 1, 7), (4, 3, 6), (3, 4, 1), (6, 2, 2), (7, 5, 9)])
def test_nested_rhat_matches_the_formulas(K, M, N):
    x = draws_of(K, M, N)
    ref = nested_rhat_loops(x, M)
    got = diagnostics.nested_rhat(x, superchainSize=M)
    for g, r in zip(got, ref):
        assert g.dtype == torch.float64 and g.shape == (3,)
        np.testing.assert_allclose(g.numpy(), r, rtol=1e-12, atol=0)
    # the same numbers from the moments, and from torch input
    mean = x.mean(axis=2)
    var = x.var(axis=2, ddof=1) if N > 1 else np.zeros_like(mean)
    got_m = diagnostics.nested_rhat_from_moments(torch.from_numpy(mean), torch.from_numpy(var), N, M)
    for g, r in zip(got_m, ref):
        np.testing.assert_allclose(g.numpy(), r, rtol=1e-12, atol=0)


@pytest.mark.parametrize("N", [2, 5, 40])
def test_superchains_of_one_give_classic_rhat_plus_one_over_n(N):
    x = draws_of(9, 1, N, D=4, seed=N)
    rhat = diagnostics.nested_rhat(x, superchainSize=1)[0].numpy()
    # classic (non-split) Gelman-Rubin: var+ = (N - 1) / N W + B / N, R^2 = var+ / W
    W = x.var(axis=2, ddof=1).mean(axis=1)
    B = N * x.mean(axis=2).var(axis=1, ddof=1)
    classic2 = ((N - 1) / N * W + B / N) / W
    np.testing.assert_allclose(rhat ** 2, classic2 + 1.0 / N, rtol=1e-12)


def test_invariant_to_permuting_superchains_and_affine_maps():
    K, M, N, D = 6, 4, 5, 3
    x = draws_of(K, M, N, D=D, seed=3)
    ref = diagnostics.nested_rhat(x, superchainSize=M)[0].numpy()
    perm = np.random.RandomState(1).permutation(K)
    xp = x.reshape(D, K, M, N)[:, perm].reshape(D, K * M, N)
    np.testing.assert_allclose(diagnostics.nested_rhat(xp, superchainSize=M)[0].numpy(), ref, rtol=1e-12)
    a = np.array([3.0, -0.25, 1e3])[:, None, None]
    b = np.array([-7.0, 2.0, 1e4])[:, None, None]
    np.testing.assert_allclose(diagnostics.nested_rhat(a * x + b, superchainSize=M)[0].numpy(), ref, rtol=1e-10)


def test_refusals():
    x = draws_of(2, 2, 3)
    with pytest.raises(ValueError):  # K = 1
        diagnostics.nested_rhat(x, superchainSize=4)
    with pytest.raises(ValueError):  # M = 1 and N = 1
        diagnostics.nested_rhat(draws_of(5, 1, 1), superchainSize=1)
    with pytest.raises(ValueError):  # M does not divide C
        diagnostics.nested_rhat(x, superchainSize=3)
    with pytest.raises(ValueError):
        diagnostics.nested_rhat_from_moments(np.zeros((2, 6)), np.ones((2, 6)), 4, superchainSize=4)
    diagnostics.nested_rhat(draws_of(2, 3, 1), superchainSize=3)  # M > 1 with one draw is defined
    for P, off, M in ((10, 0, 4), (12, 2, 4), (12, 0, 0)):
        ens = E.Ensemble(2, P, particleOffset=off)
        with pytest.raises(ValueError):
            ens.setPosition(1.0, superchainSize=M)


def test_host_setPosition_keeps_the_reference_draws():
    from scipy.stats import norm

    np.random.seed(12)
    q = E.Ensemble(3, 10).setPosition(2.5)
    np.random.seed(12)
    ref = norm.rvs(scale=2.5, size=(3, 10))  # src/ensemble.py:72-74
    assert np.array_equal(q, ref)


def test_host_setPosition_repeats_each_superchains_first_draw():
    from scipy.stats import norm

    np.random.seed(4)
    ens = E.Ensemble(3, 12)
    q = ens.setPosition(1.5, superchainSize=4)
    assert q.shape == (3, 12) and q is ens.q
    np.random.seed(4)
    first = norm.rvs(scale=1.5, size=(3, 3))
    assert np.array_equal(q, np.repeat(first, 4, axis=1))
    assert len(np.unique(q[0])) == 3


def test_run_refuses_chain_diagnostics_before_device_work():
    ens = E.Ensemble(2, 8)
    hmc = E.HMC(ens, 1.0, 0.1, None, potential=E.HarmonicPotential(np.ones(2)))
    with pytest.raises(ValueError, match="deviceAdapt"):
        hmc.run(10, 1.0, chainDiagnostics=True, deviceAdapt=True)
    with pytest.raises(ValueError, match="superchainSize"):
        hmc.run(10, 1.0, chainDiagnostics=True, superchainSize=3)
    with pytest.raises(ValueError, match="2 superchains"):
        hmc.run(10, 1.0, chainDiagnostics=True, superchainSize=8)
    with pytest.raises(ValueError):  # a window of one draw with M = 1: adapt 5 + lag 1 of 7 iterations
        hmc.run(7, 1.0, adapt=True, adaptIterations=5, chainDiagnostics=True)


def _worker(rank, world, port, mean, var, N, M, bounds, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    lo, hi = bounds[rank], bounds[rank + 1]
    r = diagnostics.nested_rhat_from_moments(torch.from_numpy(mean[:, lo:hi]), torch.from_numpy(var[:, lo:hi]), N, M,
                                             group=dist.group.WORLD)
    torch.save(r, os.path.join(out_dir, f"rank{rank}.pt"))
    dist.destroy_process_group()


def test_ranks_combine_to_the_single_process_numbers_gloo(tmp_path):
    K, M, N, world = 7, 3, 6, 2
    x = draws_of(K, M, N, D=4, seed=8)
    mean, var = x.mean(axis=2), x.var(axis=2, ddof=1)
    bounds = [0, 2 * M, K * M]  # 2 and 5 superchains: shards of unequal size
    sock = socket.socket()
    sock.bind(("127.0.0.1", 0))
    port = sock.getsockname()[1]
    sock.close()
    mp.spawn(_worker, args=(world, port, mean, var, N, M, bounds, str(tmp_path)), nprocs=world, join=True)
    r = [torch.load(str(tmp_path / f"rank{k}.pt")) for k in range(world)]
    ref = diagnostics.nested_rhat(x, superchainSize=M)
    for a, b, want in zip(r[0], r[1], ref):
        assert torch.equal(a, b)  # identical bits on every rank
        np.testing.assert_allclose(a.numpy(), want.numpy(), rtol=1e-12)
