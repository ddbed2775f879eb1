"""Cost of the g(r) pair-distance histogram on the GPU: the all-pairs kernel (ljmd_gr_hist) against the
cell-grid kernel (ljmd_gr_hist_rmax), alternated in one process, on S = 100 snapshots of a lattice-jitter
cell-list run with r_max = 5 and dr = 0.05 (100 bins).  Device time of one call (CUDA events on the
handle's stream), median of --reps calls.  Where the all-pairs kernel cannot run in reasonable time
(N = 4 M: ~8.8e12 pairs per snapshot; N = 16 M: its grid exceeds gridDim.x) its time is extrapolated
from its measured pair rate and marked as an estimate.  A torch.profiler pass then splits the cell-grid
call into binning (count, scan, scatter) and histogram kernels.  At the largest N one snapshot is checked
bit for bit against the CPU cell recount (tests/gr_reference.c).

    python scripts/gr_cost.py [--reps 5] [--sizes 4096,65536,4194304,16777216]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from jax_tpus_benchmark_physics_simulation_b200 import lattice_jitter  # noqa: E402
from jax_tpus_benchmark_physics_simulation_b200.md import LJSimulation  # noqa: E402

S, R_MAX, NBINS = 100, 5.0, 100
ALLPAIRS_RUNS_UP_TO = 65536      # beyond: extrapolated


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        power = q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def candidate_pairs(Rh, box, r_max):
    """Pairs the cell-grid kernel evaluates: per cell, its own pairs plus its particles times those of its
    E, NE, N and NW neighbours, with the grid and fp32 binning of csrc/gr.cu (gr_grid_side, gr_cell)."""
    N = Rh.shape[1]
    eff = r_max + np.ldexp(float(box), -20)
    nc = int(np.floor(float(box) / eff))
    while nc > 0 and float(box) / nc < eff:
        nc -= 1
    nc = min(nc, int(np.floor(np.sqrt(N))))
    inv = float(np.float32(nc) / np.float32(box))
    total = 0
    for R in Rh:                                    # fp32 multiply and truncation on the GPU, as gr_cell
        c = torch.clamp((R * torch.tensor(inv, dtype=torch.float32, device=R.device)).to(torch.int64), 0, nc - 1)
        n = torch.bincount(c[:, 1] * nc + c[:, 0], minlength=nc * nc).reshape(nc, nc)   # [y, x]
        e = torch.roll(n, -1, dims=1)
        nb = e + torch.roll(e, -1, dims=0) + torch.roll(n, -1, dims=0) + torch.roll(torch.roll(n, 1, dims=1), -1, dims=0)
        total += int((n * (n - 1) // 2).sum() + (n * nb).sum())
    return total, nc


def timed(sim, fn, args, reps_out):
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    rc = fn(*args)
    ev1.record()
    assert rc == 0, sim.lib.ljmd_last_error()
    ev1.synchronize()
    reps_out.append(ev0.elapsed_time(ev1) * 1e-3)


def profile_split(sim, args):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        assert sim.lib.ljmd_gr_hist_rmax(*args) == 0
        torch.cuda.synchronize()
    binning = hist = 0.0
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if "gr_cells_kernel" in e.key:
            hist += t
        elif any(k in e.key for k in ("gr_count_kernel", "gr_scan_kernel", "gr_scatter_kernel")):
            binning += t
    return binning * 1e-6, hist * 1e-6


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sizes", default="4096,65536,4194304,16777216")
    args = ap.parse_args()
    name, power = gpu_info()
    print(f"GPU: {name}, power limit {power}")
    sizes = [int(x) for x in args.sizes.split(",")]
    results = {}
    ap_rate = None
    for N in sizes:
        R, V, box = lattice_jitter(N, seed=0)
        sim = LJSimulation(N, rc=2.5, dt=0.001, path="cells")
        (_, _), traj = sim.run((R, V), S, sample_every=1)
        Rh = traj.tensor
        assert Rh.shape[0] == S
        edges = torch.from_numpy(np.linspace(0, np.float32(R_MAX), NBINS + 1, dtype=np.float32)).cuda()
        c_new = torch.zeros((S, NBINS), dtype=torch.int64, device="cuda")
        c_ap = torch.zeros((S, NBINS), dtype=torch.int64, device="cuda")
        new_args = (sim._h, Rh.data_ptr(), S, NBINS, edges.data_ptr(), float(np.float32(R_MAX)), c_new.data_ptr())
        ap_args = (sim._h, Rh.data_ptr(), S, NBINS, edges.data_ptr(), c_ap.data_ptr())
        run_ap = N <= ALLPAIRS_RUNS_UP_TO
        t_new, t_ap = [], []
        timed(sim, sim.lib.ljmd_gr_hist_rmax, new_args, [])           # warm-up (scratch allocation)
        if run_ap:
            timed(sim, sim.lib.ljmd_gr_hist, ap_args, [])
        for _ in range(args.reps):
            timed(sim, sim.lib.ljmd_gr_hist_rmax, new_args, t_new)
            if run_ap:
                timed(sim, sim.lib.ljmd_gr_hist, ap_args, t_ap)
        sim.check()
        cand, nc = candidate_pairs(Rh, box, R_MAX)
        tn = float(np.median(t_new))
        binning, hist = profile_split(sim, new_args)
        all_pairs = S * N * (N - 1) // 2
        r = {"N": N, "S": S, "nc": nc, "cells_s": tn, "cells_runs_s": t_new,
             "cells_pair_distances": cand, "cells_distances_per_s": cand / tn,
             "binning_s_profiled": binning, "histogram_s_profiled": hist,
             "binning_share": binning / (binning + hist) if binning + hist > 0 else None}
        if run_ap:
            ta = float(np.median(t_ap))
            same = bool(torch.equal(c_new, c_ap))
            ap_rate = all_pairs / ta
            r.update({"allpairs_s": ta, "allpairs_runs_s": t_ap, "allpairs_distances_per_s": ap_rate,
                      "counts_equal": same})
            print(f"N={N:9d} nc={nc:5d}  all-pairs {ta * 1e3:10.3f} ms ({ap_rate:.3e} dist/s)   "
                  f"cell grid {tn * 1e3:9.3f} ms ({cand / tn:.3e} dist/s)   speed-up {ta / tn:8.1f}x   "
                  f"counts equal: {same}")
        else:
            why = "gridDim.x limit" if (N + 255) // 256 * ((N + 255) // 256 + 1) // 2 > 2**31 - 1 else "too slow"
            est = all_pairs / ap_rate if ap_rate else None
            r.update({"allpairs_s": None, "allpairs_cannot_run": why, "allpairs_s_estimate": est})
            est_txt = f"~{est:.0f} s (estimate from its 65,536 rate)" if est else "n/a"
            print(f"N={N:9d} nc={nc:5d}  all-pairs cannot run ({why}; {est_txt})   "
                  f"cell grid {tn * 1e3:9.3f} ms ({cand / tn:.3e} dist/s)")
        print(f"          cell grid split (profiler): binning {binning * 1e3:.3f} ms, histogram {hist * 1e3:.3f} ms"
              f" -> binning share {r['binning_share']:.1%}")
        if N == max(sizes):
            from gr_reference import c_gr_hist_cells
            ref = c_gr_hist_cells(Rh[0].cpu().numpy(), box, NBINS, R_MAX)
            r["cpu_recount_match_snapshot0"] = bool(np.array_equal(c_new[0].cpu().numpy(), ref))
            print(f"          snapshot 0 against the CPU cell recount: "
                  f"{'match' if r['cpu_recount_match_snapshot0'] else 'MISMATCH'}")
        results[N] = r
        del Rh, traj, c_new, c_ap
        sim.close()
        torch.cuda.empty_cache()
    print(json.dumps({"gpu": name, "power_limit": power, "S": S, "r_max": R_MAX, "nbins": NBINS,
                      "results": results}))


if __name__ == "__main__":
    main()
