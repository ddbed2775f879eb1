"""CLI driver: the reference script's ``main()`` with the hot path swapped for the B200 library.

    python -m jax_tpus_benchmark_physics_simulation_b200.driver [--N 400 --rho 0.8 --kT 1.0 ...]

Same flags and defaults as molecular_dynamics_jax_single-host_workload.py (MD:196-213) and the
same three dispatch/sync points (MD:142-145, 151-152, 162-163).  Additions (all default to the
reference's behaviour): ``--rc`` (cutoff, default none), ``--path`` (auto|allpairs|cells),
``--ic`` (uniform|lattice; ``uniform`` = the reference's own placement, MD:133-135, and therefore
the default: like the reference's run it overflows fp32 within a few steps - SURVEY.md §0 - and
finishes with non-finite positions; ``lattice`` is the physical lattice+jitter state that the
parity tests and bench.py use), ``--energy_every``, ``--pressure`` (records the pair virial on the
energy rows and reports the mean and spread of P over the production).  matplotlib is imported
lazily (absent in this image): without it g(r) is written as ``.npy``/``.csv`` next to
``--output``.
"""
from __future__ import annotations

import argparse
import time

import numpy as np


def main(args):
    import torch
    from . import ic as ic_mod
    from .md import LJSimulation

    N, rho, kT, dt = args.N, args.rho, args.kT, args.dt
    sim = LJSimulation(N, rho=rho, dt=dt, eq_steps=args.eq_steps, prod_steps=args.prod_steps,
                       sample_every=args.sample_every, rc=args.rc, path=args.path,
                       energy_every=args.energy_every, virial=args.pressure)
    box_size = sim.box_size                                                    # MD:30
    print(f"Molecular Dynamics Simulation (B200 native)\n"
          f"Particles (N): {N}\nDensity (rho): {rho:.2f}\nTemperature (kT): {kT:.1f}\n"
          f"Box Size: {float(box_size):.2f} x {float(box_size):.2f}\n"
          f"Backend: {torch.cuda.get_device_name(sim.device_index)}\n"
          f"Steps (Eq/Prod): {args.eq_steps:,} / {args.prod_steps:,}\nTime Step (dt): {dt}\n"
          f"PRNG Seed: {args.seed}")

    if args.ic == "uniform":                                                   # MD:133-135
        R_initial, V_initial, _ = ic_mod.reference_style_uniform(N, rho, kT, args.seed)
    else:
        R_initial, V_initial, _ = ic_mod.lattice_jitter(N, rho, kT, args.seed)
    state_initial = (R_initial, V_initial)

    print("\n--- Starting Equilibration ---")
    start_time_eq = time.time()
    state_eq = sim.equilibrate_fn(state_initial)                               # MD:142
    state_eq[0].block_until_ready()                                            # MD:145
    time_eq = time.time() - start_time_eq
    print(f"Equilibration finished in {time_eq:.2f} s")

    print("\n--- Starting Production (sampling) ---")
    start_time_prod = time.time()
    state_final, R_history = sim.production_fn(state_eq)                       # MD:151
    R_history.block_until_ready()                                              # MD:152
    time_prod = time.time() - start_time_prod
    print(f"Production finished in {time_prod:.2f} s")

    print("\n--- Calculating g(r) ---")
    dr_g = 0.05                                                                # MD:157-159
    r_max_g = box_size / np.float32(2.0)
    nbins_g = int(r_max_g / dr_g)
    start_time_g_r = time.time()
    r_bins_g, g_r = sim.calculate_g_r(R_history, N, box_size, nbins_g, r_max_g)   # MD:162
    g_r.block_until_ready()                                                    # MD:163
    time_g_r = time.time() - start_time_g_r
    print(f"g(r) calculation complete in {time_g_r:.2f} s")

    print("\nSimulation Summary")
    print(f"  Equilibration  {time_eq:8.2f} s   {args.eq_steps:,} steps")
    print(f"  Production     {time_prod:8.2f} s   {args.prod_steps:,} steps")
    print(f"  g(r) Analysis  {time_g_r:8.2f} s   Collected {R_history.shape[0]} snapshots")
    print(f"  Total          {time_eq + time_prod + time_g_r:8.2f} s")
    if sim.last_energies is not None:
        e = sim.last_energies.numpy()
        print(f"  Energy (KE+PE) first/last sample: {e[0].sum():.4f} / {e[-1].sum():.4f}")
    if sim.last_pressure is not None:
        P = sim.last_pressure.numpy()
        print(f"  Pressure (production): mean {P.mean():.4f}  std {P.std():.4f}  over {P.size} samples")

    r_np, g_np = np.asarray(r_bins_g), np.asarray(g_r)
    try:
        import matplotlib
        matplotlib.use("Agg")
        import matplotlib.pyplot as plt
        plt.figure(figsize=(10, 6))                                            # MD:180-188
        plt.plot(r_np, g_np, marker="o", markersize=4, linestyle="-")
        plt.title(f"Radial Distribution Function (g(r)) - B200 - N={N}, rho={rho}, kT={kT}")
        plt.xlabel(r"Distance r (in units of $\sigma$)")
        plt.ylabel("g(r)")
        plt.grid(True, linestyle="--", alpha=0.6)
        plt.axhline(1.0, color="grey", linestyle="--")
        plt.savefig(args.output, dpi=300, bbox_inches="tight")
        print(f"Plot saved as '{args.output}'")
    except ImportError:
        stem = args.output.rsplit(".", 1)[0]
        np.save(stem + ".npy", np.stack([r_np, g_np]))
        np.savetxt(stem + ".csv", np.stack([r_np, g_np], axis=1), delimiter=",", header="r,g_r")
        print(f"matplotlib unavailable: g(r) saved as '{stem}.npy' and '{stem}.csv'")
    return state_final, R_history, (r_np, g_np)


def build_parser():
    parser = argparse.ArgumentParser(description="B200-native Molecular Dynamics Simulation")
    parser.add_argument("--N", type=int, default=400, help="Number of particles (default: 400)")
    parser.add_argument("--rho", type=float, default=0.8, help="Density (default: 0.8)")
    parser.add_argument("--kT", type=float, default=1.0, help="Temperature (kT) (default: 1.0)")
    parser.add_argument("--dt", type=float, default=1e-3, help="Time step (default: 1e-3)")
    parser.add_argument("--eq_steps", type=int, default=10000, help="Equilibration steps (default: 10000)")
    parser.add_argument("--prod_steps", type=int, default=10000, help="Production steps (default: 10000)")
    parser.add_argument("--sample_every", type=int, default=100, help="Sample every N steps (default: 100)")
    parser.add_argument("--seed", type=int, default=42, help="PRNG seed (default: 42)")
    parser.add_argument("--output", type=str, default="g_r_plot.png", help="Output plot filename")
    # additions (defaults reproduce the reference)
    parser.add_argument("--rc", type=float, default=None, help="cutoff radius (default: none, as the reference)")
    parser.add_argument("--path", choices=["auto", "allpairs", "cells"], default="auto")
    parser.add_argument("--ic", choices=["uniform", "lattice"], default="uniform",
                        help="initial positions: uniform = the reference's (MD:133-135, default); "
                             "lattice = square lattice + 5%% jitter (physical)")
    parser.add_argument("--energy_every", type=int, default=0)
    parser.add_argument("--pressure", action="store_true",
                        help="record the pair virial on the energy rows and report the pressure "
                             "(needs --energy_every > 0)")
    return parser


def parse_args(argv=None):
    parser = build_parser()
    args = parser.parse_args(argv)
    if args.pressure and args.energy_every <= 0:
        parser.error("--pressure needs --energy_every > 0")
    return args


if __name__ == "__main__":
    main(parse_args())
