"""Cost of the replica-exchange move: milliseconds per iteration of getSamples' one-launch loop without tempering
(ehmc_hmc_run, k_small_run) and with it (ehmc_hmc_run_tempered, k_small_run<..., TEMPER = true>) on the same inputs.

Workload: a 4-component Gaussian mixture in D = 10, float32, 2^20 particles, L = 20 leapfrog steps, 200 iterations per
call, no sample arrays (positions stay on chip; the accepted counts, and with tempering the swap and round-trip counts,
are written at the end).  Legs: ehmc_hmc_run; ehmc_hmc_run_tempered with R = 1 (betas = [1]: no swap move); and with
R = 8 (geometric ladder down to beta = 0.05: a swap proposal after every iteration).  One warm-up call per leg, then
the legs alternate for several repeats; each call is timed with CUDA events around the launch.

With --bench-parent DIR (a built checkout of the parent commit) bench.py runs alternately in that tree and in this
one; the lines show its config-2 step, its config-1 leg with getSamples' one-launch loop (k_small_run) and its config-5
leg (k_small_ens).

    python profiles/temper_probe.py [--repeats 5] [--bench-parent DIR] > profiles/temper_probe_b200.txt
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
KB = 1.380649e-23


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return f"nvidia-smi unavailable: {e}"


def probe(a):
    import torch

    import physicsbasedbayesianinference_b200 as E

    lib = E._lib
    torch.cuda.set_device(0)
    ctx = lib.Context.get(0)
    D, K, P, L, h, n = 10, 4, 1 << 20, 20, 0.1, a.iters
    rng = np.random.RandomState(0)
    pot = E.GaussianMixturePotential(rng.uniform(0.2, 1.0, K), rng.normal(0.0, 2.0, (K, D)),
                                     rng.uniform(0.5, 2.0, (K, D)))
    handle = pot.handle(32, ctx)
    ens = E.Ensemble(D, P, dtype=np.float32, device="cuda:0", seed=1)
    q0 = ens.setPosition(1.0).clone()
    mass = torch.ones(P, dtype=torch.float32, device="cuda:0")
    acc = torch.zeros(P, dtype=torch.int32, device="cuda:0")
    sw = torch.zeros(P, dtype=torch.int32, device="cuda:0")
    ladders = {1: torch.ones(1, dtype=torch.float64, device="cuda:0"),
               8: torch.tensor(np.geomspace(1.0, 0.05, 8), dtype=torch.float64, device="cuda:0")}
    trips = {R: torch.zeros(P // R, dtype=torch.int32, device="cuda:0") for R in ladders}
    state = {"iteration": 0}

    def call(leg):
        q = q0.clone()
        args = lib.make_args(h, h * h, L, KB, 1 / KB, lib.LEAPFROG, 0, 7, state["iteration"], 0)
        state["iteration"] += n
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        if leg == "plain":
            lib.hmc_run(ctx, handle, q, mass, args, n, None, None, 0, acc)
        else:
            R = leg
            lib.hmc_run_tempered(ctx, handle, q, mass, args, n, R, ladders[R], None, 0, acc, sw, trips[R])
        t1.record()
        torch.cuda.synchronize()
        return t0.elapsed_time(t1) / n, acc.double().mean().item() / n, sw.double().sum().item()

    legs = {"plain": "ehmc_hmc_run", 1: "ehmc_hmc_run_tempered R = 1", 8: "ehmc_hmc_run_tempered R = 8"}
    for leg in legs:
        call(leg)  # warm-up (module load, first launch)
    res = {leg: [] for leg in legs}
    info = {}
    for _ in range(a.repeats):
        for leg in legs:
            ms, ar, ns = call(leg)
            res[leg].append(ms)
            info[leg] = (ar, ns)
    print(f"mixture D = {D}, K = {K}, float32, P = 2^20, L = {L}, {n} iterations per call, {a.repeats} repeats, "
          "legs alternated, CUDA events around each call")
    base = np.median(res["plain"])
    for leg, name in legs.items():
        x = np.array(res[leg])
        ar, ns = info[leg]
        extra = "" if leg == "plain" else f", swaps accepted {ns / (P * n):.3f} per particle-iteration"
        print(f"  {name:30s} ms/iteration {' '.join('%.4f' % v for v in x)}   median {np.median(x):.4f} "
              f"({100 * (np.median(x) / base - 1):+.1f} % against ehmc_hmc_run)   acceptance {ar:.3f}{extra}")
    sys.stdout.flush()


def bench(tree, a):
    cmd = [sys.executable, "bench.py", "--gpus", "1", "--steps", str(a.steps), "--warmup", str(a.warmup),
           "--no-cpu-baseline", "--no-e2e", "--no-sustained", "--ess-iters", "0"]
    out = subprocess.run(cmd, cwd=tree, capture_output=True, text=True, timeout=3600)
    line = [l for l in out.stdout.splitlines() if l.startswith("{")]
    if out.returncode != 0 or not line:
        return dict(error=out.returncode, tail=(out.stdout + out.stderr)[-2000:])
    return json.loads(line[-1])


def summarize(j):
    if "error" in j:
        return f"FAILED {j['error']}: {j['tail']}"
    o = j.get("other_configs") or {}
    c1, c5 = o.get("c1", {}), o.get("c5", {})
    fused = c1.get("getSamples_fused_loop") or {}
    return (f"C2 ms/step {j.get('ms_per_step')}   C1 leg ms/step {c1.get('ms_per_step')}   C1 getSamples(1000) "
            f"one launch ms {fused.get('ms_total')}   C5 leg ms/step {c5.get('ms_per_step')}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--bench-parent", default=None, help="a built checkout of the parent commit: bench.py before / after")
    ap.add_argument("--bench-repeats", type=int, default=2)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    print("card (name, power limit, max SM clock):", card())
    probe(a)
    if a.bench_parent:
        for k in range(a.bench_repeats):
            for label, tree in (("before", a.bench_parent), ("after", ROOT)):
                print(f"bench.py {label} #{k}: {summarize(bench(tree, a))}")
                sys.stdout.flush()
    print("card (name, power limit, max SM clock):", card())


if __name__ == "__main__":
    main()
