#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native LJ-MD hot path.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload NAME] [--no-extra]
                    [--dump-outputs DIR]

Metric (BASELINE.json): particle-steps/s (and pair-interactions/s).  One bench "step" is one
pass of the hot path over one batch: ``md_steps_per_step`` velocity-Verlet steps of the named
system issued as ONE device dispatch (like equilibrate_fn, MD:77-83).

Workloads (BASELINE.json configs):
  cells16m cell-list N=16,777,216 rho=0.8 rc=2.5 (configs[4]; THE DEFAULT for every --gpus N: the
                                                  largest config, fits one GPU, and --gpus N shards
                                                  it (row slabs + halo pushes over NVLink) -> the
                                                  driver's 1/2/4/8 curve is STRONG scaling)
  cells4m  cell-list N=4,194,304                  (configs[3]; the >=60 % of HBM target)
  ap65536  all-pairs N=65,536 rc=2.5 dt=0.005     (configs[2]; --gpus N shards it: atom
                                                  decomposition, Newton's-third-law tiles dealt to
                                                  the ranks; the >=1e12 pairs/s target)
  ap4096   all-pairs N=4,096  rc=2.5 dt=0.005     (configs[1]; single GPU: a step is ~15 us)
  ap400    the reference script's default run     (configs[0]; single GPU)

The JSON line is the default workload's.  The other configs are measured in the same invocation
(a few seconds each) and attached under ``extra.workloads``: at N = 1 cells4m, ap65536, ap4096,
ap400; at N > 1 the sharded ap65536.

Before anything is timed the run checks itself (``parity_check`` in the line; a mismatch exits
non-zero): forces and potential energy of the timed handle against the CPU oracle, and for N > 1
the sharded handle against a single-GPU handle on every rank (forces, energies, short
trajectory) — `pytest -m gpu` runs on one GPU, so this is where multi-GPU correctness is shown.

The reference arm (--impl reference) times the CPU restatement of the reference's own
verlet_step (two force evaluations per step, MD:66-75) on the same config with all host threads —
JAX itself is not installable in this image (SURVEY.md §8c), so kind = "port".
"""
from __future__ import annotations

import os
import sys

# torchrun exports OMP_NUM_THREADS=1 to its workers.  The CPU arm (rank 0 only) and the oracle
# checks (rank 0 only, the other ranks wait) are meant to use every host core, so the variable is
# set before torch / numpy / the oracle's OpenMP runtime are loaded.
_NCPU = os.cpu_count() or 1
os.environ["OMP_NUM_THREADS"] = str(_NCPU)
os.environ.setdefault("MKL_NUM_THREADS", str(_NCPU))
# The benchmark writes nothing into the source tree, which may be read-only.
sys.dont_write_bytecode = True

import argparse
import json
import statistics
import subprocess
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    "ap400":    dict(N=400, rc=None, dt=1e-3, path="allpairs", md_steps=2000,
                     desc="default 2D LJ run of the reference script (N=400, no cutoff, dt=1e-3)"),
    "ap4096":   dict(N=4096, rc=2.5, dt=0.005, path="allpairs", md_steps=1000,
                     desc="2D LJ all-pairs N=4096 rc=2.5 dt=0.005"),
    "ap65536":  dict(N=65536, rc=2.5, dt=0.005, path="allpairs", md_steps=20,
                     desc="2D LJ all-pairs N=65536 rc=2.5 dt=0.005"),
    "cells4m":  dict(N=4194304, rc=2.5, dt=0.005, path="cells", md_steps=1000, skin=0.5,
                     desc="2D LJ cell-list N=4194304 rho=0.8 rc=2.5 dt=0.005 (skin 0.5)"),
    "cells16m": dict(N=16777216, rc=2.5, dt=0.005, path="cells", md_steps=1000, skin=0.5,
                     desc="2D LJ cell-list N=16777216 rho=0.8 rc=2.5 dt=0.005 (skin 0.5)"),
}
DEFAULT_WORKLOAD = "cells16m"
SHARD_MIN_N = 16384              # smaller systems do not shard (a step is a few microseconds)
FLOP_PER_PAIR_FORCE = 25.0      # SURVEY.md §8d (fixed for builder and judge): one ORDERED pair
FLOP_PER_UNORDERED_N3L = 33.0   # Newton's-third-law tiles: one evaluation (25) + the reaction on j (4 FMA)
BYTES_PER_PARTICLE_STEP = 32.0  # SURVEY.md §8d: read+write R,V as float2
DUMP_ROWS = 1 << 20             # --dump-outputs: at most 2^20 particles (2 x 8 MiB of float32)


def workload_config(wl_name, wl, world):
    """The `config` object of the JSON line: the same for this arm and for --impl reference."""
    N = wl["N"]
    sharded = world > 1 and N >= SHARD_MIN_N
    parallelism = "single GPU" if world == 1 else (f"sharded x{world}" if sharded else f"replicas x{world}")
    return {"workload": wl_name, "desc": wl["desc"], "N": N, "rc": wl["rc"], "dt": wl["dt"],
            "md_steps_per_step": wl["md_steps"], "path": wl["path"], "parallelism": parallelism,
            "l2": "flushed (256 MiB write) between timed steps; inputs of the cell workloads "
                  "(256 MiB+) are larger than L2"}


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "sm_max_mhz": 1965.0}, "fallback"


def load_traffic():
    """DRAM traffic per unit of work of each workload's kernel, extracted from the committed
    ``ncu --set full`` captures by scripts/ncu_summary.py (profiles/traffic.json).  Missing file or
    entry -> roofline.traffic is null."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f)
    except Exception:
        return {}


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-i", str(self.index), "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        def pump():
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                smax.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------
# CPU restatement of the reference's step (the oracle; used here only as the reported baseline,
# the reference arm, and the checker)
def _cpu_step_fn(N, rc, box, path):
    """Returns (step(state) -> state, description): the reference's verlet_step (MD:66-75: F is not
    carried, so TWO force evaluations per step) on the CPU restatement."""
    import numpy as np
    from oracle import lj_oracle as O
    if path == "cells":
        # the dense N x N form does not exist at N >= 4M (1.8e13 pairs / evaluation): the C
        # restatement's cell-grid force evaluation (same pair arithmetic, OpenMP) stands in
        def force(R):
            return O.c_forces_cells(R, box, rc)[0]
        what = "C restatement, cell-grid forces (OpenMP)"
    else:
        import torch
        if N <= 8192:
            def force(R):
                return O.force_autodiff(torch.from_numpy(R), float(box), rc=rc).numpy()
            what = "torch CPU fp32, dense autodiff forces"
        else:   # N x N does not fit: row-chunked restatement of the same formulas
            def force(R):
                return O.force_analytic(torch.from_numpy(R), float(box), rc=rc)[0].numpy()
            what = "torch CPU fp32, row-chunked dense forces"

    def step(state, dt):
        R, V = state
        f32 = np.float32
        F = force(R)
        Vh = V + (f32(0.5) * F) * f32(dt)                       # MD:70
        Rn = np.mod(R + Vh * f32(dt), f32(box)).astype(f32)     # MD:71-72
        Fn = force(Rn)                                          # MD:73
        return Rn, (Vh + (f32(0.5) * Fn) * f32(dt)).astype(f32)  # MD:74
    return step, what


def cpu_baseline_sample(wl, nsteps):
    """Bounded sample: `nsteps` reference steps after one warm-up.  (seconds per step, threads, what)"""
    import torch
    from jax_tpus_benchmark_physics_simulation_b200 import lattice_jitter
    torch.set_num_threads(_NCPU)
    N, rc, dt = wl["N"], wl["rc"], wl["dt"]
    R, V, box = lattice_jitter(N, seed=0)
    step, what = _cpu_step_fn(N, rc, box, wl["path"])
    state = step((R, V), dt)
    t0 = time.perf_counter()
    for _ in range(nsteps):
        state = step(state, dt)
    return (time.perf_counter() - t0) / nsteps, _NCPU, what


def run_reference(args, wl_name, wl):
    """--impl reference: the CPU restatement timed on this box's host cores (rank 0 only; under
    torchrun the other ranks exit at once)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import torch
    from jax_tpus_benchmark_physics_simulation_b200 import lattice_jitter
    torch.set_num_threads(_NCPU)
    N, rc, dt = wl["N"], wl["rc"], wl["dt"]
    R, V, box = lattice_jitter(N, seed=0)
    step, what = _cpu_step_fn(N, rc, box, wl["path"])
    state = (R, V)
    times = []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        state = step(state, dt)
        if i >= args.warmup:
            times.append(time.perf_counter() - t0)
    t = sum(times)
    value = N * args.steps / t
    sample = (f"1 verlet_step (2 force evaluations, MD:66-75) per bench step; {what}; "
              "restatement, JAX unavailable")
    line = {
        "impl": "reference", "metric": "particle-steps/sec", "value": value,
        "unit": "particle-steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True,
        "scaling": "strong" if N >= SHARD_MIN_N else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic lattice+jitter (seed 0, jitter 0.05, kT 1.0)",
        # the arm's own config (the workload as the B200 arm defines it); what one bench step of THIS arm
        # covers is stated in cpu_baseline.sample: a bounded sample, normalised by the metric
        "config": workload_config(wl_name, wl, args.gpus),
        "sample_md_steps_per_step": 1,
        "cpu_baseline": {"value": value, "unit": "particle-steps/s", "cores": _NCPU,
                         "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "particle-steps/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "pair_interactions_per_s": value * (N - 1) if wl["path"] == "allpairs" else None,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------
class Env:
    """What every measurement needs: ranks, device, peaks."""
    def __init__(self):
        import torch
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a GPU (no CPU fallback on the product path)")
        torch.cuda.set_device(self.local_rank)
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
        self.peaks, self.peaks_src = load_peaks()
        self.traffic = load_traffic()
        self.flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")  # > 126 MB L2

    def barrier(self):
        import torch
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, x: float) -> float:
        import torch
        if self.world == 1:
            return x
        import torch.distributed as dist
        tt = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    def all_ok(self, ok: bool) -> bool:
        import torch
        if self.world == 1:
            return ok
        import torch.distributed as dist
        tt = torch.tensor([0 if ok else 1], dtype=torch.int32, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return int(tt.item()) == 0


def parity_check(env, wl, sim, R, V, box, sharded):
    """Correctness of the handle that is about to be timed, on the workload's own inputs.
      (1) N > 1: the sharded handle against a single-GPU handle on every rank — forces, potential
          energy, and a short trajectory with energies and a sample (bounds as scripts/dist_*check.py);
      (2) rank 0: forces + potential energy against the CPU oracle (cell path: the C cell-grid
          restatement over all particles; all-pairs: the C restatement on a row subset, all j).
    Tolerances: forces 1e-5 of max|F| vs the oracle (north_star), 2e-6 sharded vs single; energy 1e-6
    vs the oracle (2e-6 between summation orders)."""
    import numpy as np
    from jax_tpus_benchmark_physics_simulation_b200.md import LJSimulation
    N, rc, dt, path = wl["N"], wl["rc"], wl["dt"], wl["path"]
    out = {}
    ok = True
    F, pe = sim.force_and_energy(R)
    Fn = F.numpy()
    pe = float(pe)
    if sharded:
        one = LJSimulation(N, rc=rc, dt=dt, path=path, device=env.local_rank, skin=wl.get("skin", 0.3))
        F1, pe1 = one.force_and_energy(R)
        F1n, pe1 = F1.numpy(), float(pe1)
        ferr = float(np.abs(Fn - F1n).max() / np.abs(F1n).max())
        steps = 60 if path == "cells" else 20
        se = steps // 2
        (Rs, Vs), traj = sim.run((R, V), steps, sample_every=se, energy_every=se)
        es = sim.last_energies.numpy()
        (Ro, Vo), traj1 = one.run((R, V), steps, sample_every=se, energy_every=se)
        eo = one.last_energies.numpy()
        d = np.abs(Rs.numpy() - Ro.numpy()); d = np.minimum(d, float(box) - d)
        terr = np.abs(traj.numpy() - traj1.numpy()); terr = np.minimum(terr, float(box) - terr)
        # the summation order of a few warps depends on P: a few ulp(box) after 60 steps (DESIGN 6)
        ptol = max(1e-4, 4.0 * float(np.spacing(np.float32(box))))
        derr, terr = float(d.max()), float(terr.max())
        eerr = float(np.abs(es.sum(1) - eo.sum(1)).max() / np.abs(eo.sum(1)).max())
        rebuilds = (sim.last_rebuilds(), one.last_rebuilds()) if path == "cells" else None
        ok_s = (ferr < 2e-6 and abs(pe - pe1) <= 2e-6 * abs(pe1) and derr < ptol and terr < ptol
                and eerr < 2e-6 and (rebuilds is None or rebuilds[0] == rebuilds[1]))
        # the block-distributed convention (ljmd_run_blocked: every rank passes / receives only its index block)
        lo, hi = sim.block_range()
        Rb, Vb = sim.run_blocked((R[lo:hi], V[lo:hi]), steps)
        db = np.abs(Rb.numpy() - Ro.numpy()[lo:hi]); db = np.minimum(db, float(box) - db)
        blk_err = float(db.max())
        vb_err = float(np.abs(Vb.numpy() - Vo.numpy()[lo:hi]).max())
        ok_s = ok_s and blk_err < ptol and vb_err < max(1e-3, 20.0 * ptol)
        out["blocked_io_vs_single"] = {"ok": bool(blk_err < ptol and vb_err < max(1e-3, 20.0 * ptol)),
                                       "max_dR": blk_err, "max_dV": vb_err, "block": [int(lo), int(hi)]}
        out["sharded_vs_single"] = {"ok": bool(ok_s), "force_err": ferr, "pe_rel": abs(pe - pe1) / abs(pe1),
                                    "steps": steps, "max_dR": derr, "traj_err": terr, "pos_tol": ptol,
                                    "energy_rel": eerr, "rebuilds": rebuilds}
        ok = ok and ok_s
        one.close()
        del one, F1, Rs, Vs, Ro, Vo, traj, traj1
    if env.rank == 0:
        from oracle import lj_oracle as O
        t0 = time.perf_counter()
        if path == "cells":
            Fo, pe_o = O.c_forces_cells(R, box, rc)
            ferr = float(np.abs(Fn - Fo).max() / np.abs(Fo).max())
            rows = N
        else:
            rng = None if N <= 8192 else (N // 2 - 128, N // 2 + 128)     # row subset, against all j
            Fo, pe_o = O.c_forces(R, box, rc=rc, rows=rng)
            ferr = float(np.abs((Fn if rng is None else Fn[rng[0]:rng[1]]) - Fo).max() / np.abs(Fo).max())
            rows = N if rng is None else rng[1] - rng[0]
        pe_rel = None
        ok_o = ferr <= 1e-5
        if pe_o is not None and np.isfinite(pe_o) and (path == "cells" or N <= 8192):
            pe_rel = abs(pe - pe_o) / abs(pe_o)
            ok_o = ok_o and pe_rel <= 1e-6
        out["vs_oracle"] = {"ok": bool(ok_o), "force_err": ferr, "pe_rel": pe_rel, "rows_checked": int(rows),
                            "oracle": "C restatement (oracle/lj_oracle.c)", "seconds": time.perf_counter() - t0}
        ok = ok and ok_o
    sim.check()
    ok = env.all_ok(ok)
    out["ok"] = bool(ok)
    return out


def dump_outputs(out_dir, state):
    """Writes the state a timed step returned, positions and velocities (N, 2), as float32
    ``positions.npy`` / ``velocities.npy``.  Above DUMP_ROWS particles both hold the same fixed rows
    (a seed-0 sample, in ascending order), so runs of two builds with the same arguments compare
    file for file."""
    import numpy as np
    import torch
    R, V = state
    N = R.shape[0]
    rows = np.arange(N) if N <= DUMP_ROWS else \
        np.sort(np.random.default_rng(0).choice(N, DUMP_ROWS, replace=False))
    idx = torch.from_numpy(rows).to(R.tensor.device)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("positions", R), ("velocities", V)):
        np.save(os.path.join(out_dir, f"{name}.npy"), a.tensor.index_select(0, idx).cpu().numpy())


def measure(env, wl_name, args, steps, warmup, cpu_steps=0, check=True, dump_dir=None):
    """One workload: parity check, `value` (device-resident), `e2e` (host buffers), roofline.
    With `dump_dir`, rank 0 writes what the last timed step returned there (dump_outputs)."""
    import numpy as np
    import torch
    from jax_tpus_benchmark_physics_simulation_b200 import lattice_jitter
    from jax_tpus_benchmark_physics_simulation_b200.md import LJSimulation, fp32_peak_probe, make_dist_arg

    wl = dict(WORKLOADS[wl_name])
    if args.md_steps and wl_name == (args.workload or DEFAULT_WORKLOAD):
        wl["md_steps"] = args.md_steps
    N, rc, dt, md_steps = wl["N"], wl["rc"], wl["dt"], wl["md_steps"]
    world, rank = env.world, env.rank
    R, V, box = lattice_jitter(N, seed=0)
    sharded = world > 1 and N >= SHARD_MIN_N
    dist_arg = make_dist_arg(rank, world) if sharded else None
    parallelism = "single GPU" if world == 1 else (f"sharded x{world}" if sharded else f"replicas x{world}")
    sim = LJSimulation(N, rc=rc, dt=dt, path=wl["path"], device=env.local_rank, dist=dist_arg,
                       skin=wl.get("skin", 0.3))

    parity = parity_check(env, wl, sim, R, V, box, sharded) if check else None
    if parity is not None and not parity["ok"]:
        return {"workload": wl_name, "parity_check": parity, "failed": True}

    Rd = torch.from_numpy(R).cuda()
    Vd = torch.from_numpy(V).cuda()
    # e2e buffers: a sharded run moves block-distributed state (every rank its own index block of the arrays,
    # LJSimulation.run_blocked), a single-GPU / replica run the whole arrays
    blocked_io = sharded and N % world == 0
    lo, hi = sim.block_range() if blocked_io else (0, N)
    Rh = torch.from_numpy(R[lo:hi].copy()).pin_memory()
    Vh = torch.from_numpy(V[lo:hi].copy()).pin_memory()
    Rh_out = torch.empty_like(Rh).pin_memory()
    Vh_out = torch.empty_like(Vh).pin_memory()
    E_out = torch.empty((1, 2), dtype=torch.float32).pin_memory()

    state = (Rd, Vd)
    for _ in range(warmup):
        state, _ = sim.run(state, md_steps)
    env.barrier()

    # ---- timed region: K steps, device-resident state, L2 flushed between steps ----------------
    sampler = ClockSampler(env.local_rank)
    sampler.start()
    launches0 = sim.launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    env.barrier()
    wall0 = time.perf_counter()
    for k in range(steps):
        env.flush.zero_()                                # evict L2 between timed steps
        ev[k][0].record()
        state, _ = sim.run(state, md_steps)
        ev[k][1].record()
    env.barrier()
    wall = time.perf_counter() - wall0
    launches = sim.launch_count() - launches0
    t_dev = env.max_over_ranks(sum(a.elapsed_time(b) for a, b in ev) * 1e-3)
    clocks = sampler.stop()
    total_particles = N if (world == 1 or sharded) else N * world
    value = total_particles * md_steps * steps / t_dev

    # ---- e2e: host buffers in, host buffers out, copies inside the timed region -----------------
    env.barrier()
    e0 = time.perf_counter()
    for k in range(steps):
        Rk = Rh.to("cuda", non_blocking=True)
        Vk = Vh.to("cuda", non_blocking=True)
        if blocked_io:
            Ro, Vo = sim.run_blocked((Rk, Vk), md_steps, energy_every=md_steps)
        else:
            (Ro, Vo), _ = sim.run((Rk, Vk), md_steps, energy_every=md_steps)
        Rh_out.copy_(Ro.tensor, non_blocking=True)
        Vh_out.copy_(Vo.tensor, non_blocking=True)
        E_out.copy_(sim.last_energies.tensor, non_blocking=True)
        torch.cuda.synchronize()
    env.barrier()
    t_e2e = env.max_over_ranks(time.perf_counter() - e0)
    e2e_value = total_particles * md_steps * steps / t_e2e
    nio = world if blocked_io else 1                 # whole-job bytes: every rank moves its own block
    h2d = (Rh.numel() * 4 + Vh.numel() * 4) * nio
    d2h = (Rh_out.numel() * 4 + Vh_out.numel() * 4) * nio + E_out.numel() * 4

    # one more run on EVERY rank (a sharded run is collective) for the per-launch kernel time
    env.barrier()
    sim.run(state, md_steps)
    launch_ms = env.max_over_ranks(sim.last_run_ms())
    rebuilds = sim.last_rebuilds() if wl["path"] == "cells" else 0
    sim.check()                                          # device status of the timed handle
    env.barrier()
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, state)                    # runs are pure: `state` is still the last timed step's

    res = {"workload": wl_name, "desc": wl["desc"], "N": N, "rc": rc, "dt": dt, "path": wl["path"],
           "md_steps_per_step": md_steps, "parallelism": parallelism, "sharded": sharded,
           "value": value, "us_per_md_step": 1e6 * t_dev / (steps * md_steps),
           "ms_per_step": 1e3 * t_dev / steps, "steps": steps, "warmup": warmup,
           "pair_interactions_per_s": (value * (N - 1)) if wl["path"] == "allpairs" else None,
           "e2e": {"value": e2e_value, "unit": "particle-steps/s", "h2d_bytes_per_step": h2d,
                   "d2h_bytes_per_step": d2h,
                   "io": "block-distributed (run_blocked): bytes summed over the ranks" if blocked_io
                         else "whole arrays per call"},
           "gpu_launches": int(launches), "wall_s": wall, "clocks": clocks, "parity_check": parity}
    if rank != 0:
        sim.close()
        return res

    # ---- roofline of the dominant kernel ----------------------------------------------------------
    peaks = env.peaks
    sm_max = float(peaks.get("sm_max_mhz", 1965.0))
    tr = env.traffic.get(wl_name) if world == 1 else None
    if wl["path"] == "allpairs":
        evals = md_steps + 1                       # one launch = md_steps steps + the prologue evaluation
        pairs = float(N) * float(N - 1) * evals / (world if sharded else 1)      # ORDERED pairs per rank
        ap_mode = sim.allpairs_mode()
        n3l = ap_mode == 3
        # executed work: the N3L kernel evaluates each unordered pair once (SURVEY 8d: report that count
        # for roofline.achieved; the headline pair rate keeps the ordered-pair denominator)
        executed_flop = (FLOP_PER_UNORDERED_N3L * pairs / 2.0) if n3l else (FLOP_PER_PAIR_FORCE * pairs)
        achieved = executed_flop / (launch_ms * 1e-3) / 1e12
        peak = 148 * 128 * 2 * sm_max * 1e6 / 1e12      # one GPU (the cluster kernel uses 16 of its 148 SMs)
        try:
            probe = {"ffma_tflops": fp32_peak_probe(env.local_rank, False),
                     "ffma2_tflops": fp32_peak_probe(env.local_rank, True)}
        except Exception as e:  # pragma: no cover
            probe = {"error": str(e)}
        roofline = {"bound": "fp32", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                    "frac": achieved / peak, "traffic": None,
                    "peak_source": f"148 SM x 128 lanes x 2 x sm_max_mhz={sm_max:.0f} from "
                                   f"MEASURED_PEAKS.json ({env.peaks_src}); CUDA-core FP32, no tensor cores; per GPU",
                    "measured_fp32_probe": probe,
                    "kernel": "ap_cluster_kernel" if ap_mode == 4 else "ap_persistent_kernel",
                    "mode": "newton3 tiles (each unordered pair once)" if n3l
                            else ("ordered pairs, one 16-CTA cluster, state in distributed shared memory"
                                  if ap_mode == 4 else "ordered pairs"),
                    "flop_per_evaluation": FLOP_PER_UNORDERED_N3L if n3l else FLOP_PER_PAIR_FORCE,
                    "ordered_pairs_per_launch": pairs,
                    "ordered_pair_equivalent_tflops": FLOP_PER_PAIR_FORCE * pairs / (launch_ms * 1e-3) / 1e12,
                    "launch_ms": launch_ms}
        if tr and "dram_bytes_per_force_evaluation" in tr:
            roofline["traffic"] = tr["dram_bytes_per_force_evaluation"] * evals
            roofline["traffic_source"] = tr.get("source")
    else:
        bytes_ = BYTES_PER_PARTICLE_STEP * N * md_steps
        achieved = bytes_ / (launch_ms * 1e-3) / 1e9
        peak = float(peaks["hbm_gbs"]) * (world if sharded else 1)     # aggregate over the sharded GPUs
        roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "traffic": None,
                    "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({env.peaks_src})" +
                                   (f" x {world} GPUs" if sharded else ""),
                    "bytes_per_particle_step": BYTES_PER_PARTICLE_STEP,
                    "kernel": "cells_persistent_kernel", "run_ms": launch_ms, "rebuilds": rebuilds}
        if world == 1:
            # SURVEY 8d: the HBM measure is the contract, but the pair loop is FP32-issue bound; report the
            # second roofline and the logically gathered bytes next to it (neighbour statistics of the
            # initial configuration, counted on the device by the library's own recount entry point)
            skin = wl.get("skin", 0.3)
            n_cut = float(sim.neighbor_count(Rd, rc).float().mean().item())
            n_list = float(sim.neighbor_count(Rd, rc + skin).float().mean().item())
            fp32_peak = 148 * 128 * 2 * sm_max * 1e6 / 1e12
            per_s = N * md_steps / (launch_ms * 1e-3)
            roofline["fp32"] = {
                "neighbours_within_rc": n_cut, "neighbours_in_list": n_list,
                "useful_tflops": FLOP_PER_PAIR_FORCE * n_cut * per_s / 1e12,
                "evaluated_tflops": FLOP_PER_PAIR_FORCE * n_list * per_s / 1e12,
                "peak": fp32_peak, "frac_evaluated": FLOP_PER_PAIR_FORCE * n_list * per_s / 1e12 / fp32_peak,
                "binding": "FP32 issue (see DESIGN.md 4.2 and profiles/)"}
            # state + one list byte + one 8-byte position per listed neighbour (positions come from the
            # warp's shared-memory windows, staged once per 32 particles)
            roofline["gathered_bytes_per_particle_step"] = BYTES_PER_PARTICLE_STEP + n_list * (1.0 + 8.0)
            roofline["gathered_GBps"] = roofline["gathered_bytes_per_particle_step"] * per_s / 1e9
            if tr and "dram_bytes_per_particle_step" in tr:
                roofline["traffic"] = tr["dram_bytes_per_particle_step"] * N * md_steps
                roofline["traffic_source"] = tr.get("source")
    res["roofline"] = roofline

    # ---- CPU baseline: bounded sample of the same workload on this box's host cores ------------
    res["cpu_baseline"] = None
    if cpu_steps > 0 and world == 1:
        try:
            per, cores, what = cpu_baseline_sample(wl, cpu_steps)
            res["cpu_baseline"] = {"value": N / per, "unit": "particle-steps/s", "cores": cores, "kind": "port",
                                   "sample": f"{cpu_steps} verlet_step (2 force evaluations each, MD:66-75) "
                                             f"after 1 warm-up step; {what}; restatement, JAX unavailable"}
        except Exception as e:  # pragma: no cover
            res["cpu_baseline"] = {"error": str(e)}
    sim.close()
    return res


# ------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=None, choices=list(WORKLOADS))
    ap.add_argument("--md-steps", type=int, default=None, help="MD steps per bench step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the other configs (extra.workloads)")
    ap.add_argument("--no-check", action="store_true", help="skip the in-run parity check")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the positions and velocities of the last timed step of the named "
                         "workload as DIR/<name>.npy (float32; a fixed sample of 2^20 rows above that size)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    wl_name = args.workload or DEFAULT_WORKLOAD
    if args.impl == "reference":
        run_reference(args, wl_name, dict(WORKLOADS[wl_name]))
        return

    import torch
    env = Env()
    cpu_steps = 0 if args.no_cpu_baseline else (1 if WORKLOADS[wl_name]["N"] > 4096 else 4)
    main_res = measure(env, wl_name, args, args.steps, args.warmup, cpu_steps=cpu_steps, check=not args.no_check,
                       dump_dir=args.dump_outputs)
    if main_res.get("failed"):
        if env.rank == 0:
            print(json.dumps({"error": "parity check failed", **main_res}), flush=True)
        sys.exit(1)

    extras = {}
    if not args.no_extra and args.workload is None:
        names = ["cells4m", "ap65536", "ap4096", "ap400"] if env.world == 1 else ["ap65536"]
        for name in names:
            try:
                r = measure(env, name, args, min(args.steps, 5), 3, cpu_steps=0, check=not args.no_check)
            except Exception as e:  # an extra workload must not take the headline down with it
                r = {"workload": name, "error": f"{type(e).__name__}: {e}"}
            if r.get("failed") and env.rank == 0:
                print(json.dumps({"error": "parity check failed", **r}), flush=True)
            if r.get("failed"):
                sys.exit(1)
            extras[name] = r

    if env.rank == 0:
        m = main_res
        line = {
            "metric": "particle-steps/sec", "value": m["value"], "unit": "particle-steps/s",
            "n_gpus": env.world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": m["ms_per_step"], "higher_is_better": True,
            "scaling": "strong" if m["N"] >= SHARD_MIN_N else "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic lattice+jitter (seed 0, jitter 0.05, kT 1.0)",
            "config": workload_config(wl_name, dict(WORKLOADS[wl_name], md_steps=m["md_steps_per_step"]), env.world),
            "pair_interactions_per_s": m["pair_interactions_per_s"],
            "us_per_md_step": m["us_per_md_step"], "wall_s": m["wall_s"], "clocks": m["clocks"],
            "e2e": m["e2e"], "gpu_launches": m["gpu_launches"],
            "roofline": m["roofline"], "cpu_baseline": m["cpu_baseline"],
            "parity_check": m["parity_check"],
            "extra": {"workloads": {k: {kk: vv for kk, vv in v.items() if kk not in ("desc", "wall_s")}
                                    for k, v in extras.items()}},
        }
        print(json.dumps(line), flush=True)
    if env.world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
