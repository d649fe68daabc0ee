"""Cost of HMC.run(chainDiagnostics=True) on one GPU: milliseconds per iteration with the per-chain moments off and on,
the two settings alternated within one process, several repeats to show the spread.

  * C5 fused: Neal's funnel 10-D, float32, 2^22 chains, L = 20, one k_small_ens launch per call (the update sits in the
    launch's per-batch epilogue);
  * C2 host loop: 100-D dense Gaussian, float32, 2^20 chains, L = 50, one ehmc_hmc_iter per iteration (+ one
    k_chain_moments launch per iteration when on).

A call is timed from a device synchronise to the end of run() (which reads its results back); the time of the final
nested R-hat reduction over all chains (float64, once per call) is reported on its own.  With --bench-parent DIR,
bench.py of that checkout (built) and of this one run alternately in the same process tree, and so does a
fused run with the diagnostics off on one of the k_small_ens instances whose spill bytes changed.

    python profiles/chain_diag_probe.py [--repeats 3] [--bench-parent DIR] > profiles/chain_diag_probe_b200.txt
"""
import argparse
import json
import os
import subprocess
import sys
import time

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


def timed_run(hmc, n, **kw):
    import torch

    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = hmc.run(n, 1 / KB, **kw)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / n, r


def rhat_ms(r, M):
    import torch

    from physicsbasedbayesianinference_b200.diagnostics import nested_rhat_from_moments

    torch.cuda.synchronize()
    t0 = time.perf_counter()
    nested_rhat_from_moments(r["chainMean"], r["chainVar"], r["rhatDraws"], M)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3


def probe(args):
    import torch

    import physicsbasedbayesianinference_b200 as E

    torch.cuda.set_device(0)
    cases = {}
    # C5: one fused launch per call
    D, P, L, h = 10, 1 << 22, 20, 0.05
    ens5 = E.Ensemble(D, P, dtype=np.float32, device="cuda:0", seed=1)
    ens5.setPosition(1.0, superchainSize=args.M)
    hmc5 = E.HMC(ens5, L * h + 1e-9, h, None, potential=E.FunnelPotential(D, 3.0), seed=1)
    cases["C5 fused (funnel 10-D, 2^22, L=20)"] = (hmc5, args.iters5, dict(keepNumSteps=True, fused=True))
    # C2: the host loop
    D, P, L, h = 100, 1 << 20, 50, 0.05
    rng = np.random.RandomState(0)
    A = rng.standard_normal((D, D))
    ens2 = E.Ensemble(D, P, dtype=np.float32, device="cuda:0", seed=2)
    ens2.setPosition(1.0, superchainSize=args.M)
    hmc2 = E.HMC(ens2, L * h + 1e-9, h, None, potential=E.GaussianPotential(precision=A @ A.T / D + np.eye(D)), seed=2)
    cases["C2 host loop (dense 100-D, 2^20, L=50)"] = (hmc2, args.iters2, dict(fused=False))
    for name, (hmc, n, kw) in cases.items():
        timed_run(hmc, 3, chainDiagnostics=False, **kw)  # warm-up of both settings
        timed_run(hmc, 3, chainDiagnostics=True, superchainSize=args.M, **kw)
        res = {False: [], True: []}
        fin = []
        for _ in range(args.repeats):
            for on in (False, True):
                ms, r = timed_run(hmc, n, chainDiagnostics=on, superchainSize=args.M, **kw)
                res[on].append(ms)
                if on:
                    fin.append(rhat_ms(r, args.M))
        off, on = np.array(res[False]), np.array(res[True])
        print(f"{name}: {n} iterations per call, {args.repeats} repeats, alternated")
        print(f"  off: ms/iteration {' '.join('%.4f' % x for x in off)}   (min {off.min():.4f}, max {off.max():.4f})")
        print(f"  on:  ms/iteration {' '.join('%.4f' % x for x in on)}   (min {on.min():.4f}, max {on.max():.4f})")
        print(f"  on - off (medians): {np.median(on) - np.median(off):+.4f} ms/iteration "
              f"({100 * (np.median(on) / np.median(off) - 1):+.1f} %); nested R-hat over all chains once per call: "
              f"{np.median(fin):.2f} ms (inside the 'on' times)")
        sys.stdout.flush()


# One fused run with the diagnostics off, timed in a fresh process of the given checkout (the parent's package has no
# chainDiagnostics argument): the funnel at D = 12 runs k_small_ens<float, 16, FunnelPot, 0, false>, one of the padded
# instances whose spill bytes moved with the new epilogue (profiles/chain_diag_ptxas.txt).
OFF_LEG = """
import sys, time
sys.path.insert(0, sys.argv[1])
import numpy as np, torch
import physicsbasedbayesianinference_b200 as E
D, P, L, h, n = 12, 1 << 21, 20, 0.05, 200
ens = E.Ensemble(D, P, dtype=np.float32, device="cuda:0", seed=3)
ens.setPosition(1.0)
hmc = E.HMC(ens, L * h + 1e-9, h, None, potential=E.FunnelPotential(D, 3.0), seed=3)
hmc.run(5, 1 / 1.380649e-23, keepNumSteps=True, fused=True)
out = []
for _ in range(3):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    hmc.run(n, 1 / 1.380649e-23, keepNumSteps=True, fused=True)
    torch.cuda.synchronize()
    out.append((time.perf_counter() - t0) * 1e3 / n)
print(" ".join("%.4f" % x for x in out))
"""


def off_leg(tree):
    out = subprocess.run([sys.executable, "-c", OFF_LEG, tree], cwd=tree, capture_output=True, text=True, timeout=1200)
    return out.stdout.strip() if out.returncode == 0 else f"FAILED {out.returncode}: {(out.stdout + out.stderr)[-1500:]}"


def bench(tree, extra):
    cmd = [sys.executable, "bench.py", "--gpus", "1", "--steps", str(extra.steps), "--warmup", str(extra.warmup),
           "--no-cpu-baseline", "--no-e2e", "--no-sustained", "--ess-iters", "0"]
    out = subprocess.run(cmd, cwd=tree, capture_output=True, text=True, timeout=3600)
    line = [l for l in out.stdout.splitlines() if l.startswith("{")]
    if out.returncode != 0 or not line:
        return dict(error=out.returncode, tail=(out.stdout + out.stderr)[-2000:])
    return json.loads(line[-1])


def summarize(j):
    if "error" in j:
        return f"FAILED {j['error']}: {j['tail']}"
    c5 = (j.get("other_configs") or {}).get("c5", {})
    return (f"C2 ms/step {j.get('ms_per_step'):.4f}   C5 leg ms/step {c5.get('ms_per_step')}   "
            f"(C5 value {c5.get('value')}, C2 value {j.get('value')})")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--iters5", type=int, default=200)
    ap.add_argument("--iters2", type=int, default=20)
    ap.add_argument("--M", type=int, default=4, help="superchain size")
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
                print(f"funnel 12-D float32 fused, 2^21 chains, L=20, diagnostics off, {label} #{k}: ms/iteration "
                      f"{off_leg(tree)}")
                sys.stdout.flush()
        for k in range(a.bench_repeats):
            for label, tree in (("before", a.bench_parent), ("after", ROOT)):
                print(f"bench.py {label} #{k}: {summarize(bench(tree, a))}")
                sys.stdout.flush()
    print("card (name, power limit, max SM clock):", card())


if __name__ == "__main__":
    main()
