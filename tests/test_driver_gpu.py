"""The reference's main() with the hot path swapped (driver.py) and the multi-GPU check."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_driver_default_flags_small(tmp_path):
    """Same CLI as MD:196-213; runs equilibrate -> production -> g(r) with the three syncs."""
    from jax_tpus_benchmark_physics_simulation_b200 import driver
    out = str(tmp_path / "g_r_plot.png")
    args = driver.build_parser().parse_args(
        ["--N", "400", "--eq_steps", "300", "--prod_steps", "300", "--sample_every", "100",
         "--output", out, "--energy_every", "100", "--ic", "lattice"])
    assert args.rho == 0.8 and args.kT == 1.0 and args.dt == 1e-3 and args.seed == 42   # MD defaults
    state_final, R_history, (r, g) = driver.main(args)
    assert R_history.shape == (3, 400, 2)
    assert np.isfinite(g).all() and g[:10].max() == 0.0 and 0.5 < g[-20:].mean() < 1.5
    assert os.path.exists(out) or os.path.exists(out.rsplit(".", 1)[0] + ".npy")
    pos = state_final[0].numpy()
    assert np.isfinite(pos).all()


def test_driver_reference_uniform_ic_completes(tmp_path):
    """--ic uniform is the default, as MD:133-135: overlapping particles, fp32 overflow within a
    few steps (SURVEY.md §0).  Like the reference's run it must finish (no hang, no exception) even
    though the state goes non-finite."""
    from jax_tpus_benchmark_physics_simulation_b200 import driver
    out = str(tmp_path / "g_r_plot.png")
    args = driver.build_parser().parse_args(
        ["--N", "400", "--eq_steps", "200", "--prod_steps", "200", "--sample_every", "100", "--output", out])
    assert args.ic == "uniform"
    state_final, R_history, (r, g) = driver.main(args)
    assert R_history.shape == (2, 400, 2) and g.shape == r.shape
    # and on the cell-list path (clumps overflow a Verlet list: reported, not hidden)
    from jax_tpus_benchmark_physics_simulation_b200 import reference_style_uniform
    from jax_tpus_benchmark_physics_simulation_b200._lib import LjmdError
    from jax_tpus_benchmark_physics_simulation_b200.md import LJSimulation
    R, V, box = reference_style_uniform(16384, seed=42)
    sim = LJSimulation(16384, rc=2.5, dt=1e-3, path="cells")
    (R1, _), _ = sim.run((R, V), 20)
    try:
        R1.block_until_ready()
    except LjmdError as e:
        assert e.code in (-6, -7)


def test_reference_defaults_match_parser():
    from jax_tpus_benchmark_physics_simulation_b200 import driver
    a = driver.build_parser().parse_args([])
    assert (a.N, a.eq_steps, a.prod_steps, a.sample_every, a.output) == (400, 10000, 10000, 100, "g_r_plot.png")
    assert a.rc is None          # the reference has no cutoff


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("N,port", [(16384, 29541), (3364, 29545), (4356, 29547)])
def test_sharded_allpairs_matches_single_gpu(N, port):
    """N = 16384: the tile mode on 8192 particles per rank.  N = 3364 = 58^2: 1682 < 2048 per rank, so the ordered
    ipt 2 kernel with a partly filled i-block.  N = 4356 = 66^2: 2178 per rank, the tile mode with a partly filled
    last 64-particle block."""
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(ROOT, "scripts", "dist_check.py"), str(N), "30"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert r.stdout.count("-> OK") == 2


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_sharded_cells_matches_single_gpu():
    """Row slabs + halo exchange over NVLink: forces, energies and a 60-step trajectory (several
    rebuilds, particles migrating between slabs) equal the single-GPU cell-list run."""
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", "29543",
           os.path.join(ROOT, "scripts", "dist_cells_check.py"), "65536", "60"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert r.stdout.count("-> OK") == 2


def test_run_blocked_single_rank_is_run():
    """ljmd_run_blocked with one rank: the block is everything, the result is ljmd_run's bit for bit."""
    import numpy as np
    from jax_tpus_benchmark_physics_simulation_b200 import lattice_jitter
    from jax_tpus_benchmark_physics_simulation_b200.md import LJSimulation
    for path, N in (("allpairs", 1024), ("cells", 16384)):
        R, V, box = lattice_jitter(N, seed=1)
        sim = LJSimulation(N, rc=2.5, dt=0.005, path=path)
        assert sim.block_range() == (0, N)
        (R1, V1), _ = sim.run((R, V), 25, energy_every=5)
        e1 = sim.last_energies.numpy()
        R2, V2 = sim.run_blocked((R, V), 25, energy_every=5)
        assert np.array_equal(R1.numpy(), R2.numpy()) and np.array_equal(V1.numpy(), V2.numpy())
        assert np.array_equal(e1, sim.last_energies.numpy())
