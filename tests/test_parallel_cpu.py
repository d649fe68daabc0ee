"""CPU tests of the multi-rank host logic (gloo, world_size 2): particle sharding, the
statistics all-reduce and the rank-identical step-size adaptation."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from physicsbasedbayesianinference_b200 import diagnostics, parallel
from oracle import hmc_oracle as O


def test_shard_ranges_cover_exactly():
    for P in (1, 7, 1024, (1 << 20) + 3):
        for W in (1, 2, 3, 8):
            r = [parallel.shard_range(P, k, W) for k in range(W)]
            assert r[0][0] == 0 and r[-1][1] == P
            assert all(r[k][1] == r[k + 1][0] for k in range(W - 1))
            sizes = [b - a for a, b in r]
            assert max(sizes) - min(sizes) <= 1


def _worker(rank, world, port, D, P, q, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    lo, hi = parallel.shard_range(P, rank, world)
    x = torch.tensor(q[:, lo:hi])
    acc = (x[0] > 0).double()
    stats = torch.zeros(2 * D + 3, dtype=torch.float64)
    stats[0] = acc.sum()
    stats[1] = acc.sum() * 0.9
    stats[2] = x.pow(2).sum()
    stats[3:3 + D] = x.sum(1)
    stats[3 + D:] = x.pow(2).sum(1)
    red = parallel.StatsReducer()
    assert red.enabled
    red.reduce_async(stats)
    red.wait()
    u = parallel.unpack_stats(stats, D, P)
    ad = parallel.StepSizeAdapter(0.1, target=0.8)
    hs = [ad.update(u["meanAcceptProb"]) for _ in range(3)]
    scales = torch.from_numpy(parallel.MassAdapter(D).scales(u["mean"].numpy(), u["var"].numpy(), P))
    torch.save(dict(stats=stats, hs=hs, mean=u["mean"], var=u["var"], acc=u["acceptRate"], scales=scales),
               os.path.join(out_dir, f"rank{rank}.pt"))
    dist.destroy_process_group()


def test_stats_allreduce_and_adaptation_gloo_world2(tmp_path):
    D, P, world = 5, 1001, 2
    rng = np.random.RandomState(0)
    q = rng.standard_normal((D, P))
    sock = socket.socket()  # a port no other process on the machine holds
    sock.bind(("127.0.0.1", 0))
    port = sock.getsockname()[1]
    sock.close()
    mp.spawn(_worker, args=(world, port, D, P, q, str(tmp_path)), nprocs=world, join=True)
    r = [torch.load(str(tmp_path / f"rank{k}.pt")) for k in range(world)]
    assert torch.equal(r[0]["stats"], r[1]["stats"])  # same sums on every rank
    assert r[0]["hs"] == r[1]["hs"]  # identical step sizes without a broadcast
    np.testing.assert_allclose(r[0]["mean"].numpy(), q.mean(1), rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(r[0]["var"].numpy(), q.var(1), rtol=1e-10)
    assert r[0]["acc"] == pytest.approx((q[0] > 0).mean())
    # mass adaptation consumes the same all-reduced moments: identical masses on every rank, = the ensemble's std
    assert torch.equal(r[0]["scales"], r[1]["scales"])
    np.testing.assert_allclose(r[0]["scales"].numpy(), q.std(1), rtol=1e-2)


def test_mass_adapter_and_windows():
    ad = parallel.MassAdapter(3)
    s = ad.scales(np.zeros(3), np.array([4.0, 0.25, np.nan]), 1e6)
    np.testing.assert_allclose(s, [2.0, 0.5, 1.0], rtol=1e-5)  # non-finite moments leave the scale at 1
    assert ad.scales(np.zeros(1), np.array([0.0]), 10)[0] == pytest.approx(np.sqrt(1e-3 * 5 / 15))  # Stan's shrinkage
    for n in (0, 5, 19, 20, 100, 1000, 1237):
        w = parallel.mass_windows(n, 3)
        assert sum(k for k, _ in w) == n and all(k > 0 for k, _ in w)
        if n >= 100:
            upd = [k for k, u in w if u]
            assert len(upd) == 3 and upd[0] < upd[1] < upd[2]  # doubling windows
            assert not w[0][1] and not w[-1][1]  # step-size-only stretches at both ends


def test_step_size_adapter_moves_towards_target():
    ad = parallel.StepSizeAdapter(0.1, target=0.8)
    h0 = ad.stepSize
    assert ad.update(0.99) > h0  # accepting too often -> larger steps
    ad2 = parallel.StepSizeAdapter(0.1, target=0.8)
    assert ad2.update(0.2) < h0
    assert ad2.update(float("nan")) < ad2.stepSize * 1.0000001


def test_ess_matches_oracle_estimator():
    rng = np.random.RandomState(5)
    x = rng.standard_normal((300, 32))
    y = np.zeros_like(x)
    for t in range(1, 300):
        y[t] = 0.8 * y[t - 1] + rng.standard_normal(32)
    for a in (x, y):
        assert diagnostics.ess(torch.tensor(a)) == pytest.approx(O.ess_geyer(a), rel=1e-9)
    tr = torch.tensor(np.stack([x.T, y.T]))  # (D=2, C=32, S=300)
    m, scaled = diagnostics.ess_min_over_dims(tr, numParticlesTotal=64)
    assert m == pytest.approx(O.ess_geyer(y), rel=1e-9) and scaled == pytest.approx(2 * m)
