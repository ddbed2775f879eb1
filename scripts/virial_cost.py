"""Cost of the pair virial on the GPU: 1000-step calls with energy_every = 1 (every step an energy step),
without and with the virial, alternated in one process; device time of the step loop (CUDA events,
ljmd_last_run_ms) in us per step.

    python scripts/virial_cost.py [--steps 1000] [--reps 5]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from jax_tpus_benchmark_physics_simulation_b200 import lattice_jitter  # noqa: E402
from jax_tpus_benchmark_physics_simulation_b200.md import LJSimulation  # noqa: E402

WORKLOADS = {  # name: (N, rc, path)
    "ap400": (400, None, "allpairs"),
    "ap4096": (4096, 2.5, "allpairs"),
    "cells4m": (4194304, 2.5, "cells"),
}


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        power = q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--dt", type=float, default=0.001)
    args = ap.parse_args()
    name, power = gpu_info()
    print(f"GPU: {name}, power limit {power}")
    results = {}
    for wl, (N, rc, path) in WORKLOADS.items():
        R, V, _ = lattice_jitter(N, seed=0)
        sim = LJSimulation(N, rc=rc, dt=args.dt, path=path)
        Rd, Vd = torch.from_numpy(R).cuda(), torch.from_numpy(V).cuda()
        for vir in (False, True):                        # warm-up of both instantiations
            sim.run((Rd, Vd), 20, energy_every=1, virial=vir)
            sim.check()
        t = {False: [], True: []}
        for _ in range(args.reps):
            for vir in (False, True):
                sim.run((Rd, Vd), args.steps, energy_every=1, virial=vir)
                t[vir].append(1e3 * sim.last_run_ms() / args.steps)
        off, on = float(np.median(t[False])), float(np.median(t[True]))
        results[wl] = {"N": N, "us_per_step_energy_steps": off, "us_per_step_with_virial": on,
                       "overhead_pct": 100.0 * (on - off) / off,
                       "runs_off": t[False], "runs_on": t[True]}
        print(f"{wl:8s} N={N:8d}  energy every step: {off:9.2f} us/step   + virial: {on:9.2f} us/step"
              f"   ({100.0 * (on - off) / off:+.2f} %)  [medians of {args.reps}]")
        sim.close()
    print(json.dumps({"gpu": name, "power_limit": power, "steps": args.steps, "results": results}))


if __name__ == "__main__":
    main()
