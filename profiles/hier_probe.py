"""Time per iteration of the fused ensemble run (HMC.run, one k_small_ens launch) for eight schools, centred and
non-centred, beside the 10-D funnel of BASELINE config 5, in one process.

    python profiles/hier_probe.py [--particles 22] [--iters 2000] [--warmup 200]

Float32, 2^22 particles by default, trajectories of L = 20 and L = 4 leapfrog steps, fixed step size, statistics on
(what HMC.run always collects).  Each case is warmed up (module load, first launch, ensemble moved off its start) and
then timed with CUDA events around one run() call of --iters iterations.  Prints the device name and power limit
with the numbers: they are part of them.
"""
import argparse
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def device_line():
    import torch

    name = torch.cuda.get_device_name()
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        extra = out.stdout.strip() or "power limit unknown"
    except (OSError, subprocess.SubprocessError):
        extra = "power limit unknown"
    return f"{name}, power limit / max SM clock: {extra}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--particles", type=int, default=22, help="log2 of the ensemble size")
    ap.add_argument("--iters", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=200)
    a = ap.parse_args()
    import torch

    import physicsbasedbayesianinference_b200 as E

    KB = 1.380649e-23
    P = 1 << a.particles
    cases = [("eight schools, non-centred", E.HierarchicalNormalPotential.eightSchools(centered=False), 0.15),
             ("eight schools, centred", E.HierarchicalNormalPotential.eightSchools(centered=True), 0.05),
             ("funnel D = 10", E.FunnelPotential(10, 3.0), 0.02)]
    print(device_line())
    print(f"float32, P = 2^{a.particles}, {a.iters} timed iterations after {a.warmup} warm-up iterations, fused run")
    gen = torch.Generator(device="cuda").manual_seed(1)
    for L in (20, 4):
        for name, pot, h in cases:
            ens = E.Ensemble(pot.numDimensions, P, dtype=np.float32, device="cuda", seed=3)
            ens.q.copy_(torch.randn((pot.numDimensions, P), dtype=torch.float32, device="cuda", generator=gen))
            hmc = E.HMC(ens, L * h + 1e-9, h, None, potential=pot, seed=3, bugCompat=False)
            r = hmc.run(a.warmup, 1 / KB)
            assert r.get("fused") and hmc.integrator.numSteps == L
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            t0.record()
            r = hmc.run(a.iters, 1 / KB)
            t1.record()
            torch.cuda.synchronize()
            ms = t0.elapsed_time(t1) / a.iters
            print(f"L = {L:2d}  {name:28s} D = {pot.numDimensions:2d}  {ms:.4f} ms / iteration  "
                  f"acceptance {np.mean(r['acceptRate']):.3f}", flush=True)


if __name__ == "__main__":
    main()
