"""Cost of the bond-orientational order psi_6 (ljmd_bond_order, csrc/bond.cu) and of its pair correlation g_6(r)
(ljmd_bond_corr) on the GPU.

Workloads (snapshots of a lattice-jitter run, one snapshot per step; m = 6, r_nb = 1.5):
    N = 4,096       S = 100
    N = 65,536      S = 100
    N = 4,194,304   S = 10
    N = 16,777,216  S = 2
Device time of one call (CUDA events on the handle's stream), median of --reps calls after one warm-up call.
ljmd_bond_order is reported against two bounds: bytes moved / 7.7 TB/s of HBM, with the bytes of its four
launches counted from the shapes (bond_bytes), and FP64-pipe instructions / the data sheet's 37 TFLOP/s FP64
(1.85e13 DFMA-class instructions/s), with the instructions per bond term counted from cuobjdump -sass of
bond_order_kernel (fp64_per_term) times the measured neighbour count.  ljmd_bond_corr and ljmd_gr_hist_rmax (r_max = 5, 100 bins) are
timed alternately in the same process.  Then the driver's end-to-end "psi_6 Analysis" time at 4 M particles (10
snapshots, --gr_rmax 5 --bond_m 6) from a separate process.

    python scripts/bond_cost.py [--reps 5] [--skip-driver] [--skip-corr]
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
from jax_tpus_benchmark_physics_simulation_b200.md import LJSimulation  # noqa: E402

WORKLOADS = [(4096, 100), (65536, 100), (4194304, 10), (16777216, 2)]
HBM_BYTES_PER_S = 7.7e12
FP64_INSTR_PER_S = 1.85e13


def fp64_per_term(m):
    """FP64-pipe instructions of one bond term on its fast path (cuobjdump -sass of bond_order_kernel): 2 F2F and
    2 DMUL + DADD for r_d^2, 9 for the square root (MUFU.RSQ64H and its DMUL / DFMA refinement), 9 for each of the
    two divisions (MUFU.RCP64H and its refinement), 4 DMUL + 2 DADD per complex product, 2 DMUL and 2 F2I.S64.F64
    for the fixed point."""
    return 5 + 9 + 2 * 9 + 6 * (m - 1) + 4


def gpu_info():
    name = torch.cuda.get_device_name(0)
    power = "unknown"
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        if q:
            power = f"{q[0].strip()} W"
    except (OSError, subprocess.SubprocessError):
        pass
    return name, power


def bond_bytes(N, S, ncell):
    """HBM bytes of ljmd_bond_order if every array is touched once per pass (neighbour re-reads hit the caches):
    count (R 8, rank 4), scan (cell starts twice), scatter (R 8, rank 4, start 4, P 8, idx 4), bond kernel (P 8,
    idx 4, psi 16, n 4) per particle."""
    return S * (N * (12 + 28 + 32) + 2 * 4 * (ncell + 1))


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
               "--sample_every", "100", "--gr_rmax", "5", "--bond_m", "6", "--output", os.path.join(d, "g_r_plot.png")]
        out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, check=True).stdout
    lines = [ln.strip() for ln in out.splitlines() if "Analysis" in ln or "Psi_6" in ln]
    t = float(re.search(r"psi_6 Analysis\s+([0-9.]+) s", out).group(1))
    return t, lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--skip-driver", action="store_true")
    ap.add_argument("--skip-corr", action="store_true")
    args = ap.parse_args()
    name, power = gpu_info()
    print(f"GPU: {name}, power limit {power}")
    results = []
    for N, S in WORKLOADS:
        R, V, box = lattice_jitter(N, seed=0)
        sim = LJSimulation(N, rc=2.5, dt=0.001, path="cells" if N > 131072 else "allpairs")
        (_, _), traj = sim.run((R, V), S, sample_every=1)
        Rh = traj.tensor
        psi = torch.empty((S, N, 2), dtype=torch.float64, device="cuda")
        nnb = torch.empty((S, N), dtype=torch.int32, device="cuda")
        b32 = np.float32(box)
        nc = max(1, int(np.floor(float(b32) / (1.5 + float(b32) * 2.0 ** -20))))
        nc = min(nc, int(np.sqrt(N)))
        ncell = nc * nc if nc >= 3 else 1

        def order():
            assert sim.lib.ljmd_bond_order(sim._h, Rh.data_ptr(), S, 6, 1.5, psi.data_ptr(), nnb.data_ptr()) == 0

        l0 = sim.launch_count()
        timed(order, [])
        launches = sim.launch_count() - l0
        ts = []
        for _ in range(args.reps):
            timed(order, ts)
        sim.check()
        t = float(np.median(ts))
        nbytes = bond_bytes(N, S, ncell)
        nmean = float(nnb.double().mean())
        t_hbm = nbytes / HBM_BYTES_PER_S
        t_fp64 = S * N * nmean * fp64_per_term(6) / FP64_INSTR_PER_S
        r = {"N": N, "S": S, "cells": ncell, "launches_per_call": launches, "bond_order_s_median": t,
             "bond_order_s_runs": ts, "bytes": nbytes, "bytes_per_s": nbytes / t,
             "hbm_share": t_hbm / t, "mean_neighbours": nmean, "hbm_bound_s": t_hbm, "fp64_bound_s": t_fp64,
             "fp64_share": t_fp64 / t}
        print(f"bond_order N={N:9d} S={S:4d}  {t * 1e3:9.3f} ms  ({min(ts) * 1e3:.3f} .. {max(ts) * 1e3:.3f})  "
              f"{nbytes / t / 1e9:8.1f} GB/s = {t_hbm / t:.1%} of 7.7 TB/s  FP64 bound {t_fp64 * 1e3:.3f} ms "
              f"= {t_fp64 / t:.1%}  <n> = {nmean:.3f}  launches/call {launches}")
        if not args.skip_corr:
            nbins = 100
            edges = torch.from_numpy(np.linspace(0, np.float32(5.0), nbins + 1, dtype=np.float32)).cuda()
            counts = torch.empty((S, nbins), dtype=torch.int64, device="cuda")
            counts_g = torch.empty((S, nbins), dtype=torch.int64, device="cuda")
            wsum = torch.empty((S, nbins), dtype=torch.int64, device="cuda")

            def corr():
                assert sim.lib.ljmd_bond_corr(sim._h, Rh.data_ptr(), psi.data_ptr(), S, nbins, edges.data_ptr(),
                                              5.0, counts.data_ptr(), wsum.data_ptr()) == 0

            def gr():
                assert sim.lib.ljmd_gr_hist_rmax(sim._h, Rh.data_ptr(), S, nbins, edges.data_ptr(), 5.0,
                                                 counts_g.data_ptr()) == 0

            timed(corr, [])
            timed(gr, [])
            tc, tg = [], []
            for _ in range(args.reps):
                timed(corr, tc)
                timed(gr, tg)
            sim.check()
            assert torch.equal(counts, counts_g)
            c, g = float(np.median(tc)), float(np.median(tg))
            r.update({"bond_corr_s_median": c, "bond_corr_s_runs": tc, "gr_hist_rmax_s_median": g,
                      "gr_hist_rmax_s_runs": tg, "corr_over_gr": c / g})
            print(f"bond_corr  N={N:9d} S={S:4d}  {c * 1e3:9.3f} ms   gr_hist_rmax {g * 1e3:9.3f} ms   "
                  f"ratio {c / g:.2f}  (r_max 5, 100 bins; counts equal)")
        results.append(r)
        del Rh, traj, psi, nnb
        sim.close()
        torch.cuda.empty_cache()
    drv = None
    if not args.skip_driver:
        t, lines = driver_4m()
        drv = {"psi_analysis_s": t, "lines": lines}
        print("driver N=4194304, 10 snapshots, --gr_rmax 5 --bond_m 6:")
        for ln in lines:
            print("   ", ln)
    print(json.dumps({"gpu": name, "power_limit": power, "results": results, "driver_4m": drv}))


if __name__ == "__main__":
    main()
