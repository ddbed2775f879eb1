"""The cell-grid g(r) histogram (ljmd_gr_hist_rmax, csrc/gr.cu): int64 counts bit for bit against the
dense CPU recount (oracle.c_gr_hist), the cell-grid CPU recount (tests/gr_reference.c) and the all-pairs
kernel (ljmd_gr_hist).  Which kernel ran is read from the launch counter: the cell grid makes four
launches per batch of snapshots, the all-pairs histogram one."""
import numpy as np
import pytest
import torch

from analysis_helpers import E_INVALID, hist_call, hist_rmax, make_sim, md_snapshots
from gr_reference import adversarial, c_gr_hist_cells, edges_for
from jax_tpus_benchmark_physics_simulation_b200 import lattice_jitter

pytestmark = pytest.mark.gpu

CELLS, ALLPAIRS = 4, 1                  # launches of one call with one batch of snapshots


@pytest.mark.parametrize("N", [400, 4096])
def test_counts_match_dense_oracle(oracle, N):
    sim = make_sim(N)
    th, box = md_snapshots(sim, N)
    b32 = np.float32(box)
    for r_max in (2.5, 5.0, float(b32 / np.float32(3)) * (1 - 1e-5), float(b32 / np.float32(2))):
        nbins = int(np.float32(r_max) / 0.05)
        states = np.concatenate([th, adversarial(N, box, r_max, seed=N)[None]])
        counts, launches = hist_rmax(sim, states, nbins, r_max)
        assert launches == (ALLPAIRS if r_max * 3 > box * (1 - 1e-6) else CELLS)
        for s in range(states.shape[0]):
            assert np.array_equal(counts[s], oracle.c_gr_hist(states[s], box, nbins, r_max)), (r_max, s)


def test_calculate_g_r_uses_the_grid(oracle):
    N = 4096
    sim = make_sim(N)
    th, box = md_snapshots(sim, N)
    l0 = sim.launch_count()
    centers, g = sim.calculate_g_r(th, N, box, 100, 5.0)
    assert sim.launch_count() - l0 == CELLS
    c_ref, g_ref, hists, _ = oracle.g_r(torch.from_numpy(th), N, box, 100, 5.0)
    assert np.array_equal(sim.last_gr_counts.numpy(), hists)
    assert np.allclose(g.numpy(), g_ref, rtol=1e-6, atol=0)
    assert np.array_equal(centers.numpy(), c_ref)


def test_grid_equals_all_pairs_kernel_65536():
    N = 65536
    sim = make_sim(N, path="allpairs")
    th, box = md_snapshots(sim, N, nsteps=20)
    cells, launches = hist_rmax(sim, th, 100, 5.0)
    assert launches == CELLS
    dense = hist_call(sim, sim.lib.ljmd_gr_hist, th, 100, 5.0)[0]
    assert np.array_equal(cells, dense) and dense.sum() > 0


@pytest.mark.parametrize("N", [400, 4096])
def test_adversarial_geometry(oracle, N):
    sim = make_sim(N)
    box = float(lattice_jitter(N)[2])
    b32 = np.float32(box)
    k = int(box // 5.0)
    # box / r_max just above and just below an integer, and a grid of exactly 3 cells
    rmaxes = [2.5, 5.0, float(b32 / np.float32(k)) * (1 - 2e-7), float(b32 / np.float32(k)) * (1 + 2e-7),
              float(b32 / np.float32(k + 1)), float(b32 / np.float32(3)) * (1 - 1e-5)]
    for r_max in rmaxes:
        nbins = max(1, int(np.float32(r_max) / 0.05))
        X = adversarial(N, box, r_max, seed=7)
        counts, launches = hist_rmax(sim, X, nbins, r_max)
        assert launches == CELLS
        assert np.array_equal(counts[0], oracle.c_gr_hist(X, box, nbins, r_max)), r_max


def test_clumped_state(oracle):
    """Many particles in one cell and empty cells elsewhere: big cells are walked in chunks."""
    N = 4096
    sim = make_sim(N)
    box = float(lattice_jitter(N)[2])
    rng = np.random.default_rng(11)
    X = np.zeros((N, 2), np.float32)
    X[:3000] = 20.5 + 3.0 * rng.random((3000, 2))            # one cell of edge >= 5
    X[3000:] = rng.random((N - 3000, 2)) * 0.25 * box        # a quarter of the box; the rest stays empty
    X = X.astype(np.float32)
    counts, launches = hist_rmax(sim, X, 100, 5.0)
    assert launches == CELLS
    assert np.array_equal(counts[0], oracle.c_gr_hist(X, box, 100, 5.0))


def test_huge_clump_overflows_to_global_counts():
    """A cell with 30,000 particles: one warp bins more pairs than its share of the CTA's 32-bit
    counters may hold, and the rest goes straight to the 64-bit counts."""
    N = 65536
    sim = make_sim(N, path="allpairs")
    box = float(lattice_jitter(N)[2])
    rng = np.random.default_rng(12)
    X = (rng.random((N, 2)) * box).astype(np.float32)
    X[:30000] = (21.0 + 3.0 * rng.random((30000, 2))).astype(np.float32)
    counts, launches = hist_rmax(sim, X, 100, 5.0)
    assert launches == CELLS
    ref = c_gr_hist_cells(X, box, 100, 5.0)
    assert ref.sum() > 30000 * 29999 // 2
    assert np.array_equal(counts[0], ref)


def test_rmax_below_last_edge_drops_longer_pairs():
    N = 4096
    sim = make_sim(N)
    th, box = md_snapshots(sim, N, nsteps=20)
    X = np.concatenate([th, adversarial(N, box, 3.3, seed=2)[None]])
    half = float(np.float32(box) / np.float32(2))
    for r_edges, r_max, path in ((5.0, 3.3, CELLS), (5.0, 2.5, CELLS), (half, half * 0.9, ALLPAIRS)):
        counts, launches = hist_rmax(sim, X, 100, r_edges, r_max)
        assert launches == path
        for s in range(X.shape[0]):
            assert np.array_equal(counts[s], c_gr_hist_cells(X[s], box, 100, r_edges, r_cap=r_max)), (r_max, s)
        assert counts[:, -1].sum() == 0 and counts.sum() > 0


def test_config4_scale(oracle):
    """Cell-list run at N = 4,194,304; g(r) to r_max = 5 with 100 bins."""
    N = 4194304
    sim = make_sim(N, path="cells")
    th, box = md_snapshots(sim, N, nsteps=20)
    assert th.shape[0] == 2
    l0 = sim.launch_count()
    centers, g = sim.calculate_g_r(th, N, box, 100, 5.0)
    assert sim.launch_count() - l0 == CELLS
    counts = sim.last_gr_counts.numpy()
    for s in range(th.shape[0]):
        assert np.array_equal(counts[s], c_gr_hist_cells(th[s], box, 100, 5.0))
    edges = edges_for(5.0, 100)                                              # oracle.g_r's normalisation
    shell = np.float32(np.pi) * (edges[1:] ** 2 - edges[:-1] ** 2)
    ideal = np.float32(N * (N - 1) / 2.0) / (np.float32(box) ** 2) * shell
    g_ref = counts.astype(np.float32).mean(axis=0) / ideal
    assert np.allclose(g.numpy(), g_ref, rtol=1e-6, atol=0)
    assert np.array_equal(centers.numpy(), (edges[:-1] + edges[1:]) / np.float32(2.0))


def test_empty_history_and_argument_errors():
    N = 4096
    sim = make_sim(N)
    counts, _ = hist_rmax(sim, np.zeros((0, N, 2), np.float32), 100, 5.0)
    assert counts.shape == (0, 100)
    _, g = sim.calculate_g_r(np.zeros((0, N, 2), np.float32), N, None, 100, 5.0)
    assert np.array_equal(g.numpy(), np.zeros(100, np.float32))
    lib, h = sim.lib, sim._h
    R = torch.zeros((1, N, 2), dtype=torch.float32, device="cuda")
    e = torch.from_numpy(edges_for(5.0, 100)).cuda()
    c = torch.zeros((1, 100), dtype=torch.int64, device="cuda")
    ok = (h, R.data_ptr(), 1, 100, e.data_ptr(), 5.0, c.data_ptr())
    assert lib.ljmd_gr_hist_rmax(*ok) == 0
    bad = [
        (None,) + ok[1:],                                     # null handle
        ok[:1] + (None,) + ok[2:],                            # null positions with S > 0
        ok[:4] + (None,) + ok[5:],                            # null edges
        ok[:6] + (None,),                                     # null counts
        ok[:2] + (-1,) + ok[3:],                              # S < 0
        ok[:3] + (0,) + ok[4:],                               # nbins out of [1, 8192]
        ok[:3] + (8193,) + ok[4:],
        ok[:5] + (0.0,) + ok[6:],                             # r_max <= 0 or not finite
        ok[:5] + (-1.0,) + ok[6:],
        ok[:5] + (float("nan"),) + ok[6:],
        ok[:5] + (float("inf"),) + ok[6:],
    ]
    for args in bad:
        assert lib.ljmd_gr_hist_rmax(*args) == E_INVALID, args
        assert lib.ljmd_last_error()
    assert lib.ljmd_gr_hist_rmax(h, None, 0, 100, e.data_ptr(), 5.0, c.data_ptr()) == 0   # S = 0


def test_driver_gr_rmax(tmp_path):
    from jax_tpus_benchmark_physics_simulation_b200 import driver
    out = str(tmp_path / "g_r_plot.png")
    args = driver.parse_args(
        ["--N", "16384", "--rc", "2.5", "--path", "cells", "--ic", "lattice", "--eq_steps", "200",
         "--prod_steps", "300", "--sample_every", "100", "--gr_rmax", "5", "--output", out])
    _, R_history, (r, g) = driver.main(args)
    assert R_history.shape == (3, 16384, 2)
    assert g.shape == (100,) and r.shape == (100,)
    assert np.isfinite(g).all() and g[:10].max() == 0.0 and 0.5 < g[-20:].mean() < 1.5
    assert driver.build_parser().parse_args([]).gr_rmax is None
