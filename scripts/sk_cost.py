"""Cost of the density modes (ljmd_density_modes, csrc/sk.cu) on the GPU, the kernel behind S(k).

Workloads (snapshots of a lattice-jitter cell-list run, one snapshot per step):
    N = 4,096      S = 100   every vector with 0 < |k| <= 8
    N = 65,536     S = 100   every vector with 0 < |k| <= 8
    N = 4,194,304  S = 10    k_max = 8, at most 64 vectors per shell
Device time of one call (CUDA events on the handle's stream), median of --reps calls after one warm-up call.
Reported: (particle, vector) evaluations/s and their share of the XU bound (2 MUFU per evaluation at
16 MUFU/clk/SM, taken at the card's maximum SM clock).  Then the driver's end-to-end "S(k) Analysis" time at
4 M particles (10 snapshots, --sk_kmax 8 --sk_per_shell 64) from a separate process.

    python scripts/sk_cost.py [--reps 5] [--skip-driver]
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from jax_tpus_benchmark_physics_simulation_b200 import lattice_jitter  # noqa: E402
from jax_tpus_benchmark_physics_simulation_b200.md import LJSimulation, structure_factor_vectors  # noqa: E402

WORKLOADS = [(4096, 100, 8.0, None), (65536, 100, 8.0, None), (4194304, 10, 8.0, 64)]
MUFU_PER_CLK_PER_SM = 16
MUFU_PER_EVAL = 2


def gpu_info():
    name = torch.cuda.get_device_name(0)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    power, clock = "unknown", None
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        if q:
            p, c = [x.strip() for x in q[0].split(",")]
            power, clock = f"{p} W", float(c) * 1e6
    except (OSError, subprocess.SubprocessError, ValueError):
        pass
    return name, sms, power, clock


def timed(fn, out):
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    fn()
    ev1.record()
    ev1.synchronize()
    out.append(ev0.elapsed_time(ev1) * 1e-3)


def driver_4m():
    with tempfile.TemporaryDirectory() as d:
        cmd = [sys.executable, "-m", "jax_tpus_benchmark_physics_simulation_b200.driver", "--N", "4194304",
               "--rc", "2.5", "--path", "cells", "--ic", "lattice", "--eq_steps", "100", "--prod_steps", "1000",
               "--sample_every", "100", "--gr_rmax", "5", "--sk_kmax", "8", "--sk_per_shell", "64",
               "--output", os.path.join(d, "g_r_plot.png")]
        out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, check=True).stdout
    lines = [ln.strip() for ln in out.splitlines() if "S(k)" in ln and ("Analysis" in ln or "peak" in ln)]
    t = float(re.search(r"S\(k\) Analysis\s+([0-9.]+) s", out).group(1))
    return t, lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--skip-driver", action="store_true")
    args = ap.parse_args()
    name, sms, power, clock = gpu_info()
    xu_rate = sms * MUFU_PER_CLK_PER_SM * clock / MUFU_PER_EVAL if clock else None
    print(f"GPU: {name}, {sms} SMs, power limit {power}")
    if xu_rate:
        print(f"max SM clock {clock / 1e6:.0f} MHz -> XU bound {xu_rate:.3e} evaluations/s")
    results = []
    for N, S, k_max, per_shell in WORKLOADS:
        R, V, box = lattice_jitter(N, seed=0)
        sim = LJSimulation(N, rc=2.5, dt=0.001, path="cells" if N > 131072 else "allpairs")
        (_, _), traj = sim.run((R, V), S, sample_every=1)
        Rh = traj.tensor
        nvec, _ = structure_factor_vectors(float(box), k_max, per_shell)
        nv = torch.from_numpy(nvec).cuda()
        K = nv.shape[0]
        rho = torch.empty((S, K, 2), dtype=torch.float64, device="cuda")

        def call():
            assert sim.lib.ljmd_density_modes(sim._h, Rh.data_ptr(), S, nv.data_ptr(), K, rho.data_ptr()) == 0

        l0 = sim.launch_count()
        timed(call, [])
        launches = sim.launch_count() - l0
        ts = []
        for _ in range(args.reps):
            timed(call, ts)
        sim.check()
        t = float(np.median(ts))
        evals = S * N * K
        rate = evals / t
        r = {"N": N, "S": S, "K": K, "k_max": k_max, "max_per_shell": per_shell, "launches_per_call": launches,
             "s_median": t, "s_runs": ts, "evaluations": evals, "evaluations_per_s": rate,
             "xu_share": rate / xu_rate if xu_rate else None}
        results.append(r)
        share = f"{rate / xu_rate:.1%} of the XU bound" if xu_rate else "XU bound unknown"
        print(f"N={N:9d} S={S:4d} K={K:7d}  {t * 1e3:10.2f} ms  ({min(ts) * 1e3:.2f} .. {max(ts) * 1e3:.2f})  "
              f"{rate:.3e} evaluations/s  {share}  launches/call {launches}")
        del Rh, traj, rho
        sim.close()
        torch.cuda.empty_cache()
    drv = None
    if not args.skip_driver:
        t, lines = driver_4m()
        drv = {"sk_analysis_s": t, "lines": lines}
        print("driver N=4194304, 10 snapshots, --sk_kmax 8 --sk_per_shell 64:")
        for ln in lines:
            print("   ", ln)
    print(json.dumps({"gpu": name, "sms": sms, "power_limit": power, "max_sm_clock_hz": clock,
                      "xu_bound_evaluations_per_s": xu_rate, "results": results, "driver_4m": drv}))


if __name__ == "__main__":
    main()
