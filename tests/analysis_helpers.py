"""TEST INFRASTRUCTURE ONLY — what the GPU tests of the snapshot analyses (g(r), S(k), psi_m and g_m(r), clusters,
Voronoi) share: the handle they run on, their snapshots, the raw ljmd_gr_hist_rmax call and a bit comparison."""
import numpy as np
import torch

from gr_reference import edges_for
from jax_tpus_benchmark_physics_simulation_b200 import lattice_jitter
from jax_tpus_benchmark_physics_simulation_b200.md import LJSimulation

E_INVALID = -1                          # LJMD_E_INVALID


def make_sim(N, path="auto", **kw):
    return LJSimulation(N, rc=2.5, dt=0.005, path=path, device=0, **kw)


def md_snapshots(sim, N, nsteps=30, every=10, seed=0):
    """The snapshots (S, N, 2) of an nsteps run of sim from lattice_jitter(N, seed), and the box as a float."""
    R, V, box = lattice_jitter(N, seed=seed)
    (_, _), traj = sim.run((R, V), nsteps, sample_every=every)
    return traj.numpy(), float(box)


def uniform_snapshots(sim, S, seed=0):
    """S uniformly random fp32 snapshots (S, N, 2) in sim's box, and the box as a float."""
    rng = np.random.default_rng(seed)
    box = np.float32(sim.box_size)
    return (rng.random((S, sim.N, 2), dtype=np.float32) * box).astype(np.float32), float(box)


def hist_call(sim, fn, Rs, nbins, r_edges, *extra):
    """fn (ljmd_gr_hist or ljmd_gr_hist_rmax) on the snapshots Rs with edges linspace(0, r_edges, nbins + 1) and the
    arguments extra before counts.  Returns (counts (S, nbins), launches)."""
    Rs = np.ascontiguousarray(Rs, dtype=np.float32).reshape(-1, sim.N, 2)
    Rh = torch.from_numpy(Rs).cuda()
    edges = torch.from_numpy(edges_for(r_edges, nbins)).cuda()
    counts = torch.full((Rs.shape[0], nbins), -1, dtype=torch.int64, device="cuda")
    l0 = sim.launch_count()
    rc = fn(sim._h, Rh.data_ptr(), Rs.shape[0], nbins, edges.data_ptr(), *extra, counts.data_ptr())
    assert rc == 0, sim.lib.ljmd_last_error()
    torch.cuda.synchronize()
    return counts.cpu().numpy(), sim.launch_count() - l0


def hist_rmax(sim, Rs, nbins, r_edges, r_max=None):
    """ljmd_gr_hist_rmax with edges linspace(0, r_edges, nbins + 1) and r_max (default: the last edge).
    Returns (counts (S, nbins), launches)."""
    r_max = edges_for(r_edges, nbins)[-1] if r_max is None else np.float32(r_max)
    return hist_call(sim, sim.lib.ljmd_gr_hist_rmax, Rs, nbins, r_edges, float(r_max))


def same_bits(a, b):
    return np.array_equal(np.asarray(a).view(np.int64), np.asarray(b).view(np.int64))
