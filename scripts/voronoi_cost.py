"""Cost of the Voronoi tessellation (ljmd_voronoi, csrc/voronoi.cu) on the GPU, against ljmd_bond_order (r_nb = 1.5)
on the same snapshots: both bin the snapshots into the g(r) cell grid and run one thread per particle.

Workloads:
    N = 4,096       S = 100
    N = 65,536      S = 100
    N = 4,194,304   S = 10
    N = 16,777,216  S = 2
each on lattice-jitter snapshots (one step apart) and on uniform random snapshots at rho = 0.3.  Device time of
one call (CUDA events on the handle's stream), median of --reps calls after one warm-up call, the two calls
alternated.  Outputs: nvor, area, adjacency (adj_cap 16) and psi_6.

Bounds, each reported as a share (bound / measured time):
  bytes  the arrays each launch touches once over 7.7 TB/s of HBM (voronoi_bytes);
  FP64   the FP64-pipe instructions the kernel must issue over 148 SMs x 64 FP64 lanes x 1.965 GHz.  Per particle
         they are counted as 11 per scanned candidate (the displacement's two subtractions and four image compares,
         two products and a sum for r2, two key compares: the minimum the loop body of voronoi_kernel issues) plus
         8 per polygon vertex and clip call (the f pass and the R^2 pass).  Scanned candidates, clip calls and
         vertices per particle come from a host emulation of the kernel's walk on --sample particles of the first
         snapshot (emulate).
Then the driver's end-to-end "Voronoi Analysis" line at 4 M particles (10 snapshots) from a separate process.

    python scripts/voronoi_cost.py [--reps 5] [--sample 300] [--skip-driver]
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
FP64_INSTR_PER_S = 148 * 64 * 1.965e9
VOR_CELL = 2.0                      # csrc/voronoi.cu
ADJ_CAP, M = 16, 6


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


def voronoi_bytes(N, S, ncell):
    """HBM bytes if every array is touched once: count (R 8, rank 4), scan (cell starts twice), scatter (R 8, rank 4,
    start 4, P 8, idx 4), voronoi (P 8, idx 4; nvor 4, area 8, adj 4 ADJ_CAP, psi 16) per particle."""
    return S * (N * (12 + 28 + 12 + 28 + 4 * ADJ_CAP) + 2 * 4 * (ncell + 1))


def grid_side(N):
    nc = int(np.floor(np.sqrt(N) / VOR_CELL))
    return nc if nc >= 3 else 1


def emulate(X, box, sample, seed=0):
    """The kernel's walk (selection scans, ring growth, clips) for `sample` particles of X, in double on the host:
    mean scanned candidates, clip calls and polygon vertices per clip call."""
    N = X.shape[0]
    nc = grid_side(N)
    inv = np.float32(nc) / np.float32(box)
    c = np.minimum(np.maximum((X * inv).astype(np.int64), 0), nc - 1)          # gr_cell (fp32 product, truncation)
    cid = c[:, 1] * nc + c[:, 0]
    by_cell = np.argsort(cid, kind="stable")
    starts = np.searchsorted(cid[by_cell], np.arange(nc * nc + 1))
    w = box / nc
    half = 0.5 * box
    K = min(6, nc // 2)                              # rings gathered around a sampled particle (the walk stays within)
    rng = np.random.default_rng(seed)
    scanned = clips = verts = 0
    for i in rng.choice(N, size=min(sample, N), replace=False):
        if 2 * K + 1 >= nc:
            near = np.arange(N)
        else:
            cells = [((c[i, 1] + oy) % nc) * nc + (c[i, 0] + ox) % nc
                     for oy in range(-K, K + 1) for ox in range(-K, K + 1)]
            near = np.concatenate([by_cell[starts[q]:starts[q + 1]] for q in cells])
        d = X[near].astype(np.float64) - X[i].astype(np.float64)
        d = np.where(d > half, d - box, np.where(d < -half, d + box, d))
        r2 = d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]
        cn = c[near]
        ring = np.maximum(np.minimum((cn[:, 0] - c[i, 0]) % nc, (c[i, 0] - cn[:, 0]) % nc),
                          np.minimum((cn[:, 1] - c[i, 1]) % nc, (c[i, 1] - cn[:, 1]) % nc))
        order = np.lexsort((near, r2))
        order = order[r2[order] > 0]
        poly = [(-half, -half), (half, -half), (half, half), (-half, half)]
        R2 = 2 * half * half
        k, allp, pos = 1, nc < 3, 0
        while True:
            assert allp == (2 * K + 1 >= nc) or k <= K, "the walk left the gathered rings"
            scanned += N if allp else int((ring <= k).sum())
            cover = np.inf if allp else max(k * w - box * 2.0 ** -20, 0.0) ** 2
            stop = min(4 * R2, half * half)
            j = order[pos] if pos < order.size else -1
            if j >= 0 and r2[j] < cover:
                if r2[j] >= stop:
                    break
                clips += 1
                verts += len(poly)
                h = 0.5 * r2[j]
                f = [px * d[j, 0] + py * d[j, 1] - h for px, py in poly]
                out = []
                for a in range(len(poly)):
                    b = (a + 1) % len(poly)
                    if f[a] <= 0:
                        out.append(poly[a])
                    if (f[a] <= 0) != (f[b] <= 0):
                        t = f[a] / (f[a] - f[b])
                        out.append((poly[a][0] + t * (poly[b][0] - poly[a][0]),
                                    poly[a][1] + t * (poly[b][1] - poly[a][1])))
                poly = out
                R2 = max(px * px + py * py for px, py in poly)
                pos += 1
                continue
            if cover >= stop:
                break
            k += 1
            allp = allp or 2 * k + 1 >= nc
    n = min(sample, N)
    return scanned / n, clips / n, verts / max(clips, 1)


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
               "--sample_every", "100", "--gr_rmax", "5", "--bond_m", "6", "--voronoi",
               "--output", os.path.join(d, "g_r_plot.png")]
        out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, check=True).stdout
    lines = [ln.strip() for ln in out.splitlines()
             if "Analysis" in ln or "<n> =" in ln or "Voronoi-weighted" in ln]
    t = {k: float(re.search(re.escape(k) + r" Analysis\s+([0-9.]+) s", out).group(1))
         for k in ("g(r)", "psi_6", "Voronoi")}
    return t, lines


def measure(sim, Rh, N, S, box, kind, reps, sample):
    nvor = torch.empty((S, N), dtype=torch.int32, device="cuda")
    area = torch.empty((S, N), dtype=torch.float64, device="cuda")
    adj = torch.empty((S, N, ADJ_CAP), dtype=torch.int32, device="cuda")
    psi = torch.empty((S, N, 2), dtype=torch.float64, device="cuda")
    bpsi = torch.empty((S, N, 2), dtype=torch.float64, device="cuda")
    nc = grid_side(N)

    def vor():
        assert sim.lib.ljmd_voronoi(sim._h, Rh.data_ptr(), S, nvor.data_ptr(), area.data_ptr(), adj.data_ptr(),
                                    ADJ_CAP, M, psi.data_ptr()) == 0

    def order():
        assert sim.lib.ljmd_bond_order(sim._h, Rh.data_ptr(), S, M, 1.5, bpsi.data_ptr(), None) == 0

    l0 = sim.launch_count()
    timed(vor, [])
    launches = sim.launch_count() - l0
    timed(order, [])
    tv, tb = [], []
    for _ in range(reps):
        timed(vor, tv)
        timed(order, tb)
    sim.check()
    incomplete = int((nvor < 0).sum())
    n_mean = float(nvor[nvor >= 0].double().mean())
    v, b = float(np.median(tv)), float(np.median(tb))
    nbytes = voronoi_bytes(N, S, nc * nc)
    t_hbm = nbytes / HBM_BYTES_PER_S
    scanned, clips, verts = emulate(Rh[0].cpu().numpy(), float(box), sample)
    fp64 = (11 * scanned + 8 * clips * verts) * N * S
    t_fp64 = fp64 / FP64_INSTR_PER_S
    r = {"N": N, "S": S, "kind": kind, "cells": nc * nc, "launches_per_call": launches, "voronoi_s_median": v,
         "voronoi_s_runs": tv, "bond_order_s_median": b, "bond_order_s_runs": tb, "ratio": v / b,
         "bytes": nbytes, "hbm_share": t_hbm / v, "scanned_per_particle": scanned, "clips_per_particle": clips,
         "vertices_per_clip": verts, "fp64_instr": fp64, "fp64_share": t_fp64 / v, "mean_n": n_mean,
         "incomplete": incomplete}
    print(f"{kind:8s} N={N:9d} S={S:4d}  voronoi {v * 1e3:9.3f} ms ({min(tv) * 1e3:.3f} .. {max(tv) * 1e3:.3f})  "
          f"bond_order {b * 1e3:8.3f} ms  ratio {v / b:5.2f}  HBM {t_hbm / v:.2%}  FP64 {t_fp64 / v:.1%}  "
          f"scanned {scanned:.1f} clips {clips:.2f} verts/clip {verts:.1f}  <n> {n_mean:.4f}  "
          f"incomplete {incomplete}  launches/call {launches}")
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sample", type=int, default=300)
    ap.add_argument("--skip-driver", action="store_true")
    args = ap.parse_args()
    name, power = gpu_info()
    print(f"GPU: {name}, power limit {power}")
    results = []
    for N, S in WORKLOADS:
        R, V, box = lattice_jitter(N, seed=0)
        sim = LJSimulation(N, rc=2.5, dt=0.001, path="cells" if N > 131072 else "allpairs")
        (_, _), traj = sim.run((R, V), S, sample_every=1)
        results.append(measure(sim, traj.tensor, N, S, box, "lattice", args.reps, args.sample))
        del traj
        sim.close()
        sim = LJSimulation(N, rho=0.3, rc=2.5, dt=0.001, path="cells" if N > 131072 else "allpairs")
        g = torch.Generator(device="cuda").manual_seed(1)
        box3 = float(sim.box_size)
        Rh = torch.rand((S, N, 2), generator=g, device="cuda", dtype=torch.float32) * np.float32(box3)
        results.append(measure(sim, Rh.contiguous(), N, S, box3, "rho0.3", args.reps, args.sample))
        del Rh
        sim.close()
        torch.cuda.empty_cache()
    drv = None
    if not args.skip_driver:
        t, lines = driver_4m()
        drv = {"analysis_s": t, "lines": lines}
        print("driver N=4194304, 10 snapshots, --gr_rmax 5 --bond_m 6 --voronoi:")
        for ln in lines:
            print("   ", ln)
    print(json.dumps({"gpu": name, "power_limit": power, "results": results, "driver_4m": drv}))


if __name__ == "__main__":
    main()
