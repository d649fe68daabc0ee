#!/usr/bin/env python
"""Benchmark of the ensemble-HMC leapfrog hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config c2|c1|c3|c4|c5|c5l4]
                    [--no-others] [--no-sustained] [--no-e2e] [--no-cpu-baseline] [--ess-iters I]
                    [--dump-outputs DIR]

Headline workload at every N: BASELINE config 2 -- 100-D correlated Gaussian (dense precision
Lambda = A A^T / D + I), ensemble of 2^20 particles, L = 50 leapfrog steps per HMC iteration, float32 state,
Philox in-kernel RNG, synthetic data.  A "step" is ONE HMC iteration of the whole ensemble (momentum refresh +
L leapfrog steps + Metropolis), i.e. P*L particle-leapfrog-steps in one fused kernel launch.  The 2^20 particles are
sharded over the N ranks (strong scaling, no data-path collective).

value     : particle-leapfrog-steps/s with the ensemble resident in HBM (device path), K timed steps.
sustained : the same loop for >= 700 iterations (>= 2 s at one GPU) with >= 100 NVML samples: the number the roofline
            claims in DESIGN.md quote (`value` over K = 20 steps is a burst number).
e2e       : the same metric through the public drop-in API on HOST buffers (HMC.step on a host-backed Ensemble ->
            ehmc_hmc_iter host path): every step copies q from pinned host memory, runs the kernel, copies q back.
other_configs : short legs of the other BASELINE configs on the same ranks (c1 at one GPU only), each with value,
            ms_per_step, roofline and clocks; c5 / c5l4 run the fused adaptive ensemble run whose statistics
            all-reduce happens inside the kernel over NVLink.
cpu_baseline     : the NumPy float64 oracle port on the host cores (bounded sample), timed in this run.
cpu_baseline_ref : the UNMODIFIED reference under the jax.numpy stand-in at config 1 (and at configs 2 and 5 with a
            reduced ensemble), timed in the build container (it is Python and cannot travel to the GPU box;
            profiles/r02_ref_standin_c1.json, r02_ref_standin_reduced.json).

--dump-outputs DIR writes what the headline leg's last timed step handed its caller to DIR/<name>.npy (see
dump_outputs).  Every input is generated from fixed seeds, so two builds run with the same arguments can be compared
output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

KB = 1.380649e-23
SEED = 20221018

CONFIGS = {
    # name: D, P, L, h, description
    "c2": dict(D=100, P=1 << 20, L=50, h=0.05, desc="config2: 100-D dense-precision Gaussian, P=2^20, L=50"),
    "c5": dict(D=10, P=1 << 22, L=20, h=0.05, desc="config5: Neal's funnel 10-D, P=2^22, L=20, ensemble step-size adaptation"),
    "c5l4": dict(D=10, P=1 << 22, L=4, h=0.05, desc="config5 HBM-bound variant: funnel 10-D, P=2^22, L=4"),
    "c1": dict(D=2, P=1024, L=20, h=0.05, desc="config1: 2-D isotropic Gaussian, P=1024, L=20"),
    "c3": dict(D=256, P=65536, L=10, h=0.01, N=100000,
               desc="config3: Bayesian logistic regression, X 100k x 256, P=65536, L=10"),
    "c4": dict(D=3 * 4096, P=1024, L=10, h=0.01, B=4096,
               desc="config4: pairwise gravitational N-body, 4096 bodies x 3-D per particle, P=1024, L=10, eps=0.05"),
}
OTHER_STEPS = {"c1": 50, "c3": 3, "c4": 4, "c5": 1000, "c5l4": 1000}  # (config 5: one fused launch of that many iterations)
LOGI_PREC = os.environ.get("EHMC_LOGISTIC_PRECISION", "fp16x3")


ADAPT_LAG = int(os.environ.get("EHMC_ADAPT_LAG", "3"))


def flops_per_unit(name, D):
    """Algorithmic flops per particle-leapfrog-step (SURVEY.md section 8d): grad U + 7 D."""
    if name == "c2":
        return 2.0 * D * D + 7.0 * D
    if name.startswith("c5"):
        return 110.0
    if name == "c3":
        return 4.0 * 100000 * D + 7.0 * D  # two GEMMs over the N data rows
    if name == "c4":
        return 20.0 * (D // 3) ** 2 + 7.0 * D  # 20-flop/interaction convention, all pairs
    return 2.0 * D + 7.0 * D


def bytes_per_particle_iter(D, es=4):
    """Algorithmic HBM bytes per particle-iteration in production mode: read q, write q, read mass."""
    return 2.0 * D * es + es


def make_precision(D):
    rng = np.random.RandomState(SEED)
    A = rng.standard_normal((D, D))
    return A @ A.T / D + np.eye(D)


def make_logistic_data(D, N):
    rng = np.random.RandomState(SEED)
    X = rng.standard_normal((N, D)) / np.sqrt(D)
    theta = rng.standard_normal(D)
    y = (rng.uniform(size=N) < 1.0 / (1.0 + np.exp(-X @ theta))).astype(np.float64)
    return X, y


def make_potential(E, name, D):
    if name == "c3":
        X, y = make_logistic_data(D, CONFIGS["c3"]["N"])
        return E.LogisticPotential(X, y, 1.0, precision=LOGI_PREC)
    if name == "c4":
        B = D // 3
        return E.NBodyPotential(np.ones(B) / B, G=1.0, eps=0.05)
    if name == "c2":
        return E.GaussianPotential(precision=make_precision(D))
    if name.startswith("c5"):
        return E.FunnelPotential(D, 3.0)
    return E.HarmonicPotential(np.ones(D))


def make_oracle_potential(O, name, D):
    if name == "c3":
        X, y = make_logistic_data(D, CONFIGS["c3"]["N"])
        return O.Logistic(X, y, 1.0)
    if name == "c4":
        B = D // 3
        return O.NBody(np.ones(B) / B, 1.0, 0.05)
    if name == "c2":
        return O.DenseGaussian(make_precision(D))
    if name.startswith("c5"):
        return O.Funnel(D, 3.0)
    return O.DiagGaussian(np.ones(D))


# ---------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clock, power and throttle reasons of one GPU through NVML (nvidia_ml_py) every
    few ms in a thread while the timed region runs; falls back to one nvidia-smi query."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x2: "applications_clocks_setting", 0x10: "sync_boost", 0x80: "hw_power_brake_slowdown",
               0x100: "display_clock_setting"}  # (0x1 gpu_idle is not a slowdown)

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.samples = []
        self.stop_flag = threading.Event()
        self.thread = None
        self.nvml = None

    def start(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
        except Exception:
            self.nvml = None
            return self
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()
        return self

    def _run(self):
        n = self.nvml
        while not self.stop_flag.is_set():
            try:
                sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                pw = n.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
                try:
                    rs = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                except Exception:
                    rs = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                self.samples.append((sm, pw, rs))
            except Exception:
                pass
            time.sleep(0.004)

    def stop(self):
        if self.nvml is None:
            return self._smi_once()
        self.stop_flag.set()
        self.thread.join(timeout=1)
        n = self.nvml
        try:
            mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
        except Exception:
            mx = None
        sm = [x[0] for x in self.samples]
        reasons = set()
        for _, _, rs in self.samples:
            for bit, name in self.REASONS.items():
                if rs & bit:
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_min_mhz": float(min(sm)) if sm else None,
                "sm_max_mhz": float(mx) if mx else None,
                "power_w_max": max(x[1] for x in self.samples) if self.samples else None,
                "samples": len(sm), "reasons": sorted(reasons),
                "reason_bits_or": hex(int(np.bitwise_or.reduce([int(x[2]) for x in self.samples]))) if self.samples else None,
                "source": "nvml, 4 ms sleep between queries, during the timed region"}

    def _smi_once(self):
        try:
            out = subprocess.run(["nvidia-smi", f"--id={self.gpu}", "--query-gpu=clocks.sm,clocks.max.sm,power.draw",
                                  "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=10).stdout
            f = [float(x) for x in out.strip().split(",")]
            return {"sm_mhz": f[0], "sm_max_mhz": f[1], "power_w_max": f[2], "samples": 1, "reasons": [],
                    "source": "nvidia-smi single query (nvml unavailable)"}
        except Exception:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock query unavailable"]}


# ---------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port on the host cores
# ---------------------------------------------------------------------------
def cpu_port_rate(name, cfg, sample_particles, iters):
    """particle-leapfrog-steps/s of the NumPy float64 oracle (oracle/hmc_oracle.py) on a
    bounded sample of the workload: `sample_particles` particles, `iters` HMC iterations."""
    from oracle import hmc_oracle as O

    D, L, h = cfg["D"], cfg["L"], cfg["h"]
    pot = make_oracle_potential(O, name, D)
    rng = np.random.RandomState(SEED)
    q = rng.standard_normal((D, sample_particles))
    mass = np.ones(sample_particles)
    times = []
    for _ in range(iters):
        z = rng.standard_normal((D, sample_particles))
        u = rng.uniform(size=sample_particles)
        t0 = time.perf_counter()
        q, _, _, _, _ = O.hmc_iter(q, z, u, mass, 1 / KB, h, L, pot)
        times.append(time.perf_counter() - t0)
    return sample_particles * L / float(np.median(times)), times


CPU_SAMPLE = {"c2": 1 << 16, "c3": 64, "c4": 1}


def config_dict(cfg, D, P, L, h, Pl, world, L_mean=None):
    return {"workload": cfg["desc"], "D": D, "P": P, "L": L, "L_executed_mean": L if L_mean is None else L_mean, "h": h,
            "particles_per_gpu": Pl, "rng": "philox in-kernel",
            "l2": "inputs_exceed_l2" if D * Pl * 4 > 126e6 else "resident",
            "parallelism": f"particle-shard x{world}, no data-path collective"}


def run_reference_arm(args, cfg, rank, world):
    if rank != 0:
        return
    name = args.config
    sample = min(cfg["P"], CPU_SAMPLE.get(name, 1 << 17))
    rate, times = cpu_port_rate(name, cfg, sample, args.warmup + args.steps)
    times = times[args.warmup:]
    ms = 1e3 * float(np.mean(times))
    value = sample * cfg["L"] / (ms * 1e-3)
    threads = os.cpu_count()
    D, P, L, h = cfg["D"], cfg["P"], cfg["L"], cfg["h"]
    line = {
        "impl": "reference", "metric": "particle-leapfrog-steps/sec", "value": value,
        "unit": "particle-leapfrog-steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": config_dict(cfg, D, P, L, h, (P + world - 1) // world, world),
        "cpu_baseline": {"value": value, "unit": "particle-leapfrog-steps/s", "cores": threads, "kind": "port",
                         "sample": f"{sample} of {cfg['P']} particles per step (NumPy float64 oracle port of "
                                   "src/integrator.py:105-120 + src/HMC.py:154-176, BLAS threads = host cores); "
                                   "the reference itself is pure Python + JAX and cannot run here (no jax wheel)"},
        "e2e": {"value": value, "unit": "particle-leapfrog-steps/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------
# roofline of one measured leg
# ---------------------------------------------------------------------------
def roofline(name, D, Pl, L, kern_ms, fp32_peak, peaks, ctx, world, sustained=False):
    fl = flops_per_unit(name, D)
    ach_tf = Pl * L * fl / (kern_ms * 1e-3) / 1e12
    by = bytes_per_particle_iter(D) * Pl
    ach_gbs = by / (kern_ms * 1e-3) / 1e9
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    hbm_src = "MEASURED_PEAKS.json" if "hbm_gbs" in peaks else "fallback"
    info = ctx.device_info()
    nominal_fp32 = info["sm_count"] * 128 * 2 * info["sm_clock_mhz"] * 1e6 / 1e12
    dense_tc = name == "c2" and os.environ.get("EHMC_DENSE_PATH", "0") != "1"
    logi_tc = name == "c3" and LOGI_PREC in ("bf16", "fp16x3", "auto")
    compute_bound = ach_tf / fp32_peak > ach_gbs / hbm_peak
    if dense_tc:
        # the gradient GEMM runs on tcgen05 as a 3-pass fp16 split (float32 accuracy from 11-bit operands):
        # tensor-pipe roofline against the measured dense bf16 peak (burst for a short timed region, sustained for
        # the long one).  Executed tensor flops per algorithmic flop = 3 passes x padding to K = N = 112.
        key = "bf16_tflops_sustained" if sustained else "bf16_tflops"
        tpeak = peaks.get(key, peaks.get("bf16_tflops", 1590.0))
        kp = (D + 15) // 16 * 16
        exec_factor = 3.0 * kp * kp / (D * D)
        roof = {"bound": "tensor", "achieved": ach_tf, "peak": tpeak, "unit": "TFLOP/s", "frac": ach_tf / tpeak,
                "traffic": None, "peak_source": f"MEASURED_PEAKS.json {key}" if key in peaks else "fallback",
                "flops_per_unit": fl, "units_per_launch": Pl * L,
                "executed_tensor_tflops": ach_tf * exec_factor, "formulation_ceiling_frac": 1.0 / exec_factor,
                "note": "algorithmic fp32 flops (2 D^2 + 7 D per particle-step) over the measured bf16 peak; the "
                        f"3xFP16 split executes {exec_factor:.2f}x those flops (3 passes x padding to K = N = {kp}), "
                        "so `frac` cannot exceed formulation_ceiling_frac"}
    elif logi_tc:
        tpeak = peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1590.0))
        split = LOGI_PREC != "bf16"
        roof = {"bound": "tensor", "achieved": ach_tf, "peak": tpeak, "unit": "TFLOP/s", "frac": ach_tf / tpeak,
                "traffic": None, "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside "
                "a long step)", "flops_per_unit": fl, "units_per_launch": Pl * L,
                "executed_tensor_tflops": ach_tf * (3.0 if split else 1.0),
                "formulation_ceiling_frac": 1.0 / 3.0 if split else 1.0,
                "note": ("tcgen05 GEMM chain at float32 accuracy (trajectories within 1e-5 of the float64 oracle at "
                         "full size): every operand a 2-term fp16 split, 3 MMA passes per GEMM = 3x the algorithmic "
                         "flops, so `frac` cannot exceed formulation_ceiling_frac" if split else
                         "bf16 tcgen05 GEMM chain, operands rounded to bf16: OUTSIDE the 1e-5 tolerance, opt-in only") +
                        "; kernel_ms is the whole iteration (L gradient launches + kick/drift launches)"}
    elif compute_bound:
        roof = {"bound": "fp32", "achieved": ach_tf, "peak": fp32_peak, "unit": "TFLOP/s",
                "frac": ach_tf / fp32_peak, "traffic": None,
                "peak_source": "measured in this run (ehmc_measure_fp32_peak, register-only FFMA kernel); "
                               f"nominal {nominal_fp32:.1f} = SMs*128*2*max clock",
                "flops_per_unit": fl, "units_per_launch": Pl * L}
    else:
        roof = {"bound": "hbm", "achieved": ach_gbs, "peak": hbm_peak, "unit": "GB/s",
                "frac": ach_gbs / hbm_peak, "traffic": None, "peak_source": hbm_src,
                "bytes_per_unit": bytes_per_particle_iter(D) / L, "units_per_launch": Pl * L}
    for fname in ("r02_traffic.json", "r01_traffic.json"):
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", fname))).get(name)
        except (OSError, ValueError):
            tr = None
        if tr and world == 1:
            roof["traffic"] = tr["dram_bytes_per_launch"]
            roof["traffic_source"] = tr["source"]
            for k_src, k_dst in (("tensor_pipe_active_pct", "ncu_tensor_pipe_active_pct"),
                                 ("issue_active_pct", "ncu_issue_active_pct"), ("fma_pipe_active_pct", "ncu_fma_pipe_active_pct")):
                if tr.get(k_src) is not None:
                    roof[k_dst] = tr[k_src]
            break
    roof["algorithmic_bytes_per_launch"] = by
    roof["kernel_ms"] = kern_ms
    roof["other"] = {"hbm_GBps": ach_gbs, "hbm_frac": ach_gbs / hbm_peak, "fp32_TFLOPs": ach_tf,
                     "fp32_frac": ach_tf / fp32_peak}
    return roof


def dtype_of(name):
    if name == "c2" and os.environ.get("EHMC_DENSE_PATH", "0") != "1":
        return "f32 (3xFP16 tensor-core split, fp32 accumulate)"
    if name == "c3":
        return {"bf16": "f32 state, bf16 tensor-core gradient GEMMs (fp32 accumulate)",
                "fp32": "f32"}.get(LOGI_PREC, "f32 (3xFP16 tensor-core split of both gradient GEMMs, fp32 accumulate)")
    return "f32"


# ---------------------------------------------------------------------------
# one device-resident leg of one config
# ---------------------------------------------------------------------------
class Leg:
    """Ensemble + driver of one config on this rank, and its timed loop."""

    def __init__(self, E, name, rank, world, dev):
        self.E, self.name, self.rank, self.world, self.dev = E, name, rank, world, dev
        cfg = CONFIGS[name]
        self.cfg = cfg
        self.D, self.P, self.L, self.h = cfg["D"], cfg["P"], cfg["L"], cfg["h"]
        self.p_lo = rank * self.P // world
        self.Pl = (rank + 1) * self.P // world - self.p_lo
        self.pot = make_potential(E, name, self.D)
        self.ens = E.Ensemble(self.D, self.Pl, dtype=np.float32, device=dev, seed=SEED, particleOffset=self.p_lo)
        self.ens.setPosition(1.0)
        self.hmc = E.HMC(self.ens, self.L * self.h + 1e-9, self.h, None, potential=self.pot, seed=SEED, bugCompat=False)
        assert self.hmc.integrator.numSteps == self.L
        self.adaptive = name.startswith("c5")  # config 5: ensemble statistics all-reduced every iteration
        self.run_out = None

    def loop(self, n, group):
        """n iterations enqueued on the current stream (config 5: ONE fused launch with the in-kernel all-reduce)."""
        if n <= 0:
            return
        if self.adaptive:
            # the same adaptLag (3) at every N (results must not depend on the GPU count): the reductions and the all-reduce get
            # three iterations, see HMC.run
            self.run_out = self.hmc.run(n, 1 / KB, adapt=True, group=group, keepNumSteps=True, adaptLag=ADAPT_LAG)
        else:
            for _ in range(n):
                self.hmc.step(1 / KB, reuseEndpoint=True)  # q is only touched by the step itself

    def timed(self, steps, warmup, group, barrier, ctx, sample_clocks=True):
        import torch
        import torch.distributed as dist

        self.loop(warmup, group)
        barrier()
        sampler = ClockSampler(self.dev.index).start() if (self.rank == 0 and sample_clocks) else None
        l0 = ctx.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        self.loop(steps, group)
        e1.record()
        barrier()
        launches = ctx.launch_count() - l0
        clocks = sampler.stop() if sampler else None
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
        # leapfrog steps actually executed per iteration (fixed here: the adaptive legs keep numSteps)
        L_mean = float(np.mean(self.run_out["numSteps"])) if self.adaptive else float(self.L)
        return dict(total_ms=total_ms, ms_per_step=total_ms / steps, launches=int(launches), clocks=clocks,
                    value=self.P * L_mean * steps / (total_ms * 1e-3), L_mean=L_mean)


def fused_get_samples(E, leg, dev):
    """The reference's own call on its own runnable configuration: HMC.getSamples, 1000 iterations, whose whole loop is
    one launch for the small-D families (ehmc_hmc_run)."""
    import contextlib
    import io

    import torch

    D, P, L, h = leg.D, leg.P, leg.L, leg.h
    ens_f = E.Ensemble(D, P, dtype=np.float32, device=dev, seed=SEED)
    hmc_f = E.HMC(ens_f, L * h + 1e-9, h, None, potential=leg.pot, seed=SEED)
    with contextlib.redirect_stdout(io.StringIO()):
        hmc_f.getSamples(1000, 1 / KB, 1.0)  # warm-up of the same size: first-use cudaMalloc of the (D, P, S) arrays
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        hmc_f.getSamples(1000, 1 / KB, 1.0)
        torch.cuda.synchronize()
        tf = time.perf_counter() - t0
    return {"value": P * L * 1000 / tf, "unit": "particle-leapfrog-steps/s", "ms_total": 1e3 * tf,
            "iterations": 1000, "api": "HMC.getSamples(1000, ...) on a device ensemble -> ehmc_hmc_run, "
            "one launch, samples and momenta (D, P, S) written by the kernel"}


DUMP_Q_BYTES = 32 << 20


def dump_outputs(leg, out_dir, group):
    """Writes what the leg's last timed call handed its caller to out_dir/<name>.npy (rank 0 writes):
      q.npy  the positions HMC.step / HMC.run updated in place, float32 (D, n): the columns of a fixed, seeded sample of
             n particles in ascending particle order, n the whole ensemble or as many as fit DUMP_Q_BYTES (the full
             config-2 ensemble is 400 MB);
      acceptRate, meanAcceptProb, meanH, stepSize, numSteps (one value per iteration), mean, var (D): what HMC.run
             returned, float64 -- the adaptive legs (config 5) only."""
    import torch
    import torch.distributed as dist

    q_all = leg.ens.q
    n = min(leg.P, DUMP_Q_BYTES // (leg.D * q_all.element_size()))
    cols = np.sort(np.random.RandomState(SEED).choice(leg.P, n, replace=False))
    mine = cols[(cols >= leg.p_lo) & (cols < leg.p_lo + leg.Pl)] - leg.p_lo
    q = q_all[:, torch.from_numpy(mine).to(q_all.device)].cpu().numpy()
    if leg.world > 1:
        parts = [None] * leg.world
        dist.all_gather_object(parts, q, group=group)
        q = np.concatenate(parts, axis=1)
    if leg.rank != 0:
        return
    out = {"q": q}
    if leg.run_out is not None:
        for k in ("acceptRate", "meanAcceptProb", "meanH", "stepSize", "numSteps", "mean", "var"):
            out[k] = np.asarray(leg.run_out[k], dtype=np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--e2e-steps", type=int, default=6)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-others", action="store_true", help="skip the short legs of the other BASELINE configs")
    ap.add_argument("--no-sustained", action="store_true")
    ap.add_argument("--sustained-iters", type=int, default=0, help="0 = enough iterations for ~2.2 s (>= 700)")
    ap.add_argument("--ess-iters", type=int, default=150, help="iterations of the ESS/s phase (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of the headline leg computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    cfg = CONFIGS[args.config]

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference_arm(args, cfg, rank, world)
        return

    import torch
    import torch.distributed as dist

    import physicsbasedbayesianinference_b200 as E
    from physicsbasedbayesianinference_b200 import _lib

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    ctx = _lib.Context.get(local_rank)
    if os.environ.get("EHMC_DENSE_PATH"):
        ctx.set_option("dense_path", float(os.environ["EHMC_DENSE_PATH"]))
    if os.environ.get("EHMC_TC_DEBUG"):
        ctx.set_option("tc_debug", float(os.environ["EHMC_TC_DEBUG"]))
    if os.environ.get("EHMC_ENS_DEBUG"):  # phase stamps of the fused ensemble run (dumped to stderr after the headline leg)
        ctx.set_option("ens_debug", float(os.environ["EHMC_ENS_DEBUG"]))
    if os.environ.get("EHMC_DENSE_OCC"):
        ctx.set_option("dense_occupancy", float(os.environ["EHMC_DENSE_OCC"]))
    group = dist.group.WORLD if world > 1 else None
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    fp32_peak = ctx.measure_fp32_peak(60.0)

    # ---- headline leg --------------------------------------------------------------------------
    leg = Leg(E, args.config, rank, world, dev)
    D, P, L, h, Pl = leg.D, leg.P, leg.L, leg.h, leg.Pl
    main_t = leg.timed(args.steps, args.warmup, group, barrier, ctx)
    value, ms_per_step = main_t["value"], main_t["ms_per_step"]
    main_adapt = leg.run_out
    if args.dump_outputs:
        dump_outputs(leg, args.dump_outputs, group)
    if os.environ.get("EHMC_ENS_DEBUG") and rank == 0:
        ctx.set_option("ens_debug_dump", max(0.0, float(os.environ["EHMC_ENS_DEBUG"]) - 24))

    # ---- sustained: the same loop for >= 2 s -----------------------------------------------------
    sustained = None
    if not args.no_sustained:
        n_sus = args.sustained_iters or max(700, int(2200.0 / max(ms_per_step, 1e-3)))
        n_sus = min(n_sus, 100000)
        st = leg.timed(n_sus, 0, group, barrier, ctx)
        if rank == 0:
            ck = st["clocks"] or {}
            sustained = {"iters": n_sus, "ms_per_step": st["ms_per_step"], "value": st["value"],
                         "seconds": st["total_ms"] * 1e-3, "sm_mhz_median": ck.get("sm_mhz"),
                         "power_w_max": ck.get("power_w_max"), "nvml_samples": ck.get("samples"),
                         "reasons": ck.get("reasons"),
                         "roofline": roofline(args.config, D, Pl, st["L_mean"], st["ms_per_step"], fp32_peak, peaks, ctx,
                                              world, sustained=True)}

    # ---- ESS/s: min over dimensions of the ESS of traced chains, scaled to the ensemble ------
    ess = None
    if args.ess_iters > 0:
        from physicsbasedbayesianinference_b200 import diagnostics

        ntrace = min(256, Pl)
        leg.hmc.run(30, 1 / KB, collectStats=False)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = leg.hmc.run(args.ess_iters, 1 / KB, traceParticles=ntrace, collectStats=False)
        e1.record()
        barrier()
        tsec = torch.tensor([e0.elapsed_time(e1) * 1e-3], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tsec, op=dist.ReduceOp.MAX)
        if rank == 0:
            m, scaled = diagnostics.ess_min_over_dims(r["trace"], numParticlesTotal=P)
            ess = {"ess_per_sec": scaled / float(tsec.item()), "iterations": args.ess_iters,
                   "ess_per_chain_per_iter_min_dim": m / (ntrace * args.ess_iters), "traced_chains": ntrace,
                   "estimator": "FFT autocovariance averaged over traced chains + Geyer initial positive "
                                "sequence, min over dimensions, scaled by P/traced"}

    # ---- e2e through the host-facing API ------------------------------------------------
    e2e = None
    if not args.no_e2e:
        qh_t = torch.empty((D, Pl), dtype=torch.float32, pin_memory=True)
        qh_t.copy_(leg.ens.q)
        ens_h = E.Ensemble(D, Pl, dtype=np.float32, seed=SEED, particleOffset=leg.p_lo)
        ens_h.q = qh_t.numpy()
        ens_h.mass = torch.ones(Pl, dtype=torch.float32, pin_memory=True).numpy()
        hmc_h = E.HMC(ens_h, L * h + 1e-9, h, None, potential=leg.pot, rng="philox", seed=SEED, bugCompat=False)
        acc_h = torch.empty(Pl, dtype=torch.uint8, pin_memory=True).numpy()
        hmc_h.step(1 / KB, accept=acc_h)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            hmc_h.step(1 / KB, accept=acc_h)  # returns after q and accept are back in host memory
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
        te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e_s = float(te.item())
        e2e = {"value": P * L * args.e2e_steps / e2e_s, "unit": "particle-leapfrog-steps/s",
               "h2d_bytes_per_step": int(D * Pl * 4 + Pl * 4), "d2h_bytes_per_step": int(D * Pl * 4 + Pl),
               "steps": args.e2e_steps, "ms_per_step": 1e3 * e2e_s / args.e2e_steps,
               "api": "HMC.step on a host-backed Ensemble -> ehmc_hmc_iter (host path, pinned buffers)"}
        del ens_h, hmc_h, qh_t

    fused = fused_get_samples(E, leg, dev) if (args.config == "c1" and world == 1 and rank == 0) else None

    # ---- the other BASELINE configs, short legs ---------------------------------------------------
    others = None
    if not args.no_others:
        others = {}
        for name in ("c1", "c3", "c4", "c5", "c5l4"):
            if name == args.config:
                continue
            if name == "c1" and world > 1:
                others[name] = {"skipped": "1024 particles: measured at one GPU only"}
                continue
            try:
                lg = Leg(E, name, rank, world, dev)
                steps = OTHER_STEPS[name]
                t = lg.timed(steps, 3, group, barrier, ctx)
                if rank == 0:
                    o = {"workload": lg.cfg["desc"], "value": t["value"], "unit": "particle-leapfrog-steps/s",
                         "ms_per_step": t["ms_per_step"], "steps": steps, "warmup": 3, "dtype": dtype_of(name),
                         "particles_per_gpu": lg.Pl, "gpu_launches": t["launches"], "clocks": t["clocks"],
                         "roofline": roofline(name, lg.D, lg.Pl, t["L_mean"], t["ms_per_step"], fp32_peak, peaks, ctx, world)}
                    if lg.adaptive:
                        ro = lg.run_out
                        o["adaptation"] = {"final_step_size": ro["stepSize"][-1], "accept_rate_last": ro["acceptRate"][-1],
                                           "fused_launch": bool(ro.get("fused")), "adapt_lag": ADAPT_LAG,
                                           "collective": ("statistics all-reduce inside the kernel: 2D+3 float64 stored into "
                                                          f"each of {world - 1} peer mailboxes over NVLink per iteration"
                                                          if world > 1 else "single GPU: no collective")}
                    if name == "c1":
                        o["getSamples_fused_loop"] = fused_get_samples(E, lg, dev)
                    others[name] = o
                del lg
                torch.cuda.empty_cache()
            except Exception as exc:  # one leg must not take the headline down
                others[name] = {"error": f"{type(exc).__name__}: {exc}"}

    if rank == 0:
        roof = roofline(args.config, D, Pl, main_t["L_mean"], ms_per_step, fp32_peak, peaks, ctx, world)
        cpu = None
        if not args.no_cpu_baseline:
            sample = min(P, CPU_SAMPLE.get(args.config, 1 << 17))
            rate, times = cpu_port_rate(args.config, cfg, sample, 3)
            cpu = {"value": rate, "unit": "particle-leapfrog-steps/s", "cores": os.cpu_count(), "kind": "port",
                   "sample": f"{sample} of {P} particles x 3 iterations, median (NumPy float64 oracle port, "
                             f"BLAS on all host cores; {sum(times):.1f} s of CPU wall time)"}
        cpu_ref = None
        try:
            cpu_ref = json.load(open(os.path.join(ROOT, "profiles", "r02_ref_standin_c1.json")))
            # the same unmodified reference loop on configs 2 and 5 at reduced ensemble size (its rate per
            # particle-leapfrog-step does not depend on P: a serial Python loop over particles)
            red = json.load(open(os.path.join(ROOT, "profiles", "r02_ref_standin_reduced.json")))
            cpu_ref["reduced_configs"] = {k: red[k] for k in ("c2", "c5")}
        except (OSError, ValueError, KeyError):
            pass
        line = {
            "metric": "particle-leapfrog-steps/sec", "value": value, "unit": "particle-leapfrog-steps/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": dtype_of(args.config),
            "data": "synthetic", "config": config_dict(cfg, D, P, L, h, Pl, world, main_t["L_mean"]),
            "gpu_launches": main_t["launches"], "clocks": main_t["clocks"], "e2e": e2e, "roofline": roof,
            "sustained": sustained, "cpu_baseline": cpu, "cpu_baseline_ref": cpu_ref, "ess": ess,
            "other_configs": others, "getSamples_fused_loop": fused,
            "adaptation": ({"final_step_size": main_adapt["stepSize"][-1], "accept_rate_last": main_adapt["acceptRate"][-1],
                            "fused_launch": bool(main_adapt.get("fused"))} if main_adapt else None),
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
