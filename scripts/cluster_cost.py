"""Cost of the cluster analysis (ljmd_clusters, csrc/cluster.cu) on the GPU, against ljmd_bond_order on the same
snapshots: both bin the snapshots into the same cell grid and walk the same 9-cell stencil once, so their ratio
isolates the cost of the union-find.

Workloads (r_link = 1.5; psi_6 with r_nb = 1.5):
    N = 4,096       S = 100
    N = 65,536      S = 100
    N = 4,194,304   S = 10
    N = 16,777,216  S = 2
each on lattice-jitter snapshots (one step apart: one percolating cluster, the most contention at the roots) and
on uniform random snapshots at rho = 0.3 (many small clusters).  Device time of one call (CUDA events on the
handle's stream), median of --reps calls after one warm-up call, the two calls alternated.  The bytes bound counts
the arrays each launch touches once (cluster_bytes) over 7.7 TB/s of HBM.  Then the driver's end-to-end "Cluster
Analysis", "g(r) Analysis" and "psi_6 Analysis" times at 4 M particles (10 snapshots) from a separate process.

    python scripts/cluster_cost.py [--reps 5] [--skip-driver]
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
R_LINK = 1.5


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


def cluster_bytes(N, S, ncell):
    """HBM bytes of ljmd_clusters if every array is touched once per pass (neighbour re-reads and forest walks hit
    the caches): sizes memset 4, count (R 8, rank 4), scan (cell starts twice), scatter (R 8, rank 4, start 4, P 8,
    idx 4), init (R 8, labels 4), hook (P 8, idx 4, labels 4 read + 4 written), flatten (labels 4 + 4, sizes 4)
    per particle."""
    return S * (N * (4 + 12 + 28 + 12 + 20 + 12) + 2 * 4 * (ncell + 1))


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
               "--sample_every", "100", "--gr_rmax", "5", "--bond_m", "6", "--cluster_rlink", str(R_LINK),
               "--output", os.path.join(d, "g_r_plot.png")]
        out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, check=True).stdout
    lines = [ln.strip() for ln in out.splitlines() if "Analysis" in ln or "<clusters>" in ln]
    t = {k: float(re.search(re.escape(k) + r" Analysis\s+([0-9.]+) s", out).group(1))
         for k in ("g(r)", "psi_6", "Cluster")}
    return t, lines


def measure(sim, Rh, N, S, box, kind, reps):
    labels = torch.empty((S, N), dtype=torch.int32, device="cuda")
    sizes = torch.empty((S, N), dtype=torch.int32, device="cuda")
    psi = torch.empty((S, N, 2), dtype=torch.float64, device="cuda")
    b32 = np.float32(box)
    nc = max(1, int(np.floor(float(b32) / (R_LINK + float(b32) * 2.0 ** -20))))
    nc = min(nc, int(np.sqrt(N)))
    ncell = nc * nc if nc >= 3 else 1

    def clus():
        assert sim.lib.ljmd_clusters(sim._h, Rh.data_ptr(), S, R_LINK, None, labels.data_ptr(),
                                     sizes.data_ptr()) == 0

    def order():
        assert sim.lib.ljmd_bond_order(sim._h, Rh.data_ptr(), S, 6, R_LINK, psi.data_ptr(), None) == 0

    l0 = sim.launch_count()
    timed(clus, [])
    launches = sim.launch_count() - l0
    timed(order, [])
    tc, tb = [], []
    for _ in range(reps):
        timed(clus, tc)
        timed(order, tb)
    sim.check()
    ncl = (sizes > 0).sum(dim=1).double()
    largest = sizes.max(dim=1).values.double()
    c, b = float(np.median(tc)), float(np.median(tb))
    nbytes = cluster_bytes(N, S, ncell)
    t_hbm = nbytes / HBM_BYTES_PER_S
    r = {"N": N, "S": S, "kind": kind, "cells": ncell, "launches_per_call": launches, "clusters_s_median": c,
         "clusters_s_runs": tc, "bond_order_s_median": b, "bond_order_s_runs": tb, "ratio": c / b,
         "bytes": nbytes, "bytes_per_s": nbytes / c, "hbm_share": t_hbm / c, "hbm_bound_s": t_hbm,
         "mean_clusters": float(ncl.mean()), "mean_largest": float(largest.mean())}
    print(f"{kind:8s} N={N:9d} S={S:4d}  clusters {c * 1e3:9.3f} ms ({min(tc) * 1e3:.3f} .. {max(tc) * 1e3:.3f})  "
          f"bond_order {b * 1e3:9.3f} ms  ratio {c / b:.2f}  {nbytes / c / 1e9:7.1f} GB/s = {t_hbm / c:.1%} of "
          f"7.7 TB/s  <clusters> {float(ncl.mean()):.1f}  <largest> {float(largest.mean()):.1f}  "
          f"launches/call {launches}")
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--skip-driver", action="store_true")
    args = ap.parse_args()
    name, power = gpu_info()
    print(f"GPU: {name}, power limit {power}")
    results = []
    for N, S in WORKLOADS:
        R, V, box = lattice_jitter(N, seed=0)
        sim = LJSimulation(N, rc=2.5, dt=0.001, path="cells" if N > 131072 else "allpairs")
        (_, _), traj = sim.run((R, V), S, sample_every=1)
        results.append(measure(sim, traj.tensor, N, S, box, "lattice", args.reps))
        del traj
        sim.close()
        sim = LJSimulation(N, rho=0.3, rc=2.5, dt=0.001, path="cells" if N > 131072 else "allpairs")
        g = torch.Generator(device="cuda").manual_seed(1)
        box3 = float(sim.box_size)
        Rh = torch.rand((S, N, 2), generator=g, device="cuda", dtype=torch.float32) * np.float32(box3)
        results.append(measure(sim, Rh.contiguous(), N, S, box3, "rho0.3", args.reps))
        del Rh
        sim.close()
        torch.cuda.empty_cache()
    drv = None
    if not args.skip_driver:
        t, lines = driver_4m()
        drv = {"analysis_s": t, "lines": lines}
        print(f"driver N=4194304, 10 snapshots, --gr_rmax 5 --bond_m 6 --cluster_rlink {R_LINK}:")
        for ln in lines:
            print("   ", ln)
    print(json.dumps({"gpu": name, "power_limit": power, "results": results, "driver_4m": drv}))


if __name__ == "__main__":
    main()
