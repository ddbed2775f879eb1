"""The bond-orientational order (ljmd_bond_order, csrc/bond.cu) and its pair correlation (ljmd_bond_corr): psi_m,
n_i and wsum bit for bit against the fp64 CPU restatement (tests/bond_reference.c), counts against
ljmd_gr_hist_rmax, determinism across calls and batches, the NaN rule, argument errors and the driver.  Which
histogram kernel ran is read from the launch counter: the cell grid makes four launches per batch of snapshots,
the all-pairs histogram one."""
import numpy as np
import pytest
import torch

import bond_reference as ref
from analysis_helpers import E_INVALID, hist_rmax, make_sim, md_snapshots, same_bits
from gr_reference import adversarial, edges_for
from jax_tpus_benchmark_physics_simulation_b200 import lattice_jitter

pytestmark = pytest.mark.gpu

CELLS, ALLPAIRS = 4, 1


def order(sim, Rs, m, r_nb):
    """ljmd_bond_order of the snapshots Rs: (psi (S, N, 2), n (S, N), launches)."""
    l0 = sim.launch_count()
    psi, n = sim.bond_order(Rs, m, r_nb)
    return psi.numpy(), n.numpy(), sim.launch_count() - l0


def corr(sim, Rs, psi, nbins, r_max):
    """ljmd_bond_corr with edges linspace(0, r_max, nbins + 1): (counts, wsum, launches)."""
    Rs = np.ascontiguousarray(Rs, np.float32).reshape(-1, sim.N, 2)
    Rh = torch.from_numpy(Rs).cuda()
    P = torch.from_numpy(np.ascontiguousarray(psi, np.float64).reshape(-1, sim.N, 2)).cuda()
    e = torch.from_numpy(edges_for(r_max, nbins)).cuda()
    c = torch.full((Rs.shape[0], nbins), -1, dtype=torch.int64, device="cuda")
    w = torch.full((Rs.shape[0], nbins), -1, dtype=torch.int64, device="cuda")
    l0 = sim.launch_count()
    rc = sim.lib.ljmd_bond_corr(sim._h, Rh.data_ptr(), P.data_ptr(), Rs.shape[0], nbins, e.data_ptr(),
                                float(edges_for(r_max, nbins)[-1]), c.data_ptr(), w.data_ptr())
    assert rc == 0, sim.lib.ljmd_last_error()
    torch.cuda.synchronize()
    return c.cpu().numpy(), w.cpu().numpy(), sim.launch_count() - l0


@pytest.mark.parametrize("N", [400, 4096, 65536])
def test_psi_matches_reference(N):
    sim = make_sim(N)
    th, box = md_snapshots(sim, N)
    if N == 65536:
        th = th[:1]                                       # the reference visits all N^2 pairs below 65,536 + 1
    for m in (4, 6):
        for r_nb in (1.2, 1.5, 2.5):
            psi, n, launches = order(sim, th, m, r_nb)
            assert launches == 4
            for s in range(th.shape[0]):
                p_ref, n_ref = ref.bond_order(th[s], box, m, r_nb)
                assert np.array_equal(n[s], n_ref), (m, r_nb, s)
                assert same_bits(psi[s], p_ref), (m, r_nb, s)


def test_psi_matches_reference_4m():
    N = 4194304
    sim = make_sim(N, path="cells")
    R, _, box = lattice_jitter(N, seed=3)
    psi, n, _ = order(sim, R, 6, 1.5)
    p_ref, n_ref = ref.bond_order(R, box, 6, 1.5)
    assert np.array_equal(n[0], n_ref) and same_bits(psi[0], p_ref)


@pytest.mark.parametrize("N", [400, 4096])
def test_adversarial_placements(N):
    sim = make_sim(N)
    box = float(lattice_jitter(N)[2])
    for r_nb in (1.2, 1.5, 2.5, 5.0, 8.0):               # 8.0 at N = 400: one cell, all pairs
        X = adversarial(N, box, r_nb, seed=5)
        for m in (3, 6):
            psi, n, _ = order(sim, X, m, r_nb)
            p_ref, n_ref = ref.bond_order(X, box, m, r_nb)
            assert np.array_equal(n[0], n_ref) and same_bits(psi[0], p_ref), (r_nb, m)


@pytest.mark.parametrize("N,r_max,path", [(4096, 5.0, CELLS), (400, None, ALLPAIRS), (4096, None, ALLPAIRS)])
def test_corr_counts_and_wsum(N, r_max, path):
    sim = make_sim(N)
    th, box = md_snapshots(sim, N)
    r_max = float(np.float32(box) / np.float32(2)) if r_max is None else r_max
    nbins = int(np.float32(r_max) / 0.05)
    psi, _, _ = order(sim, th, 6, 1.5)
    counts, wsum, launches = corr(sim, th, psi, nbins, r_max)
    assert launches == path
    assert np.array_equal(counts, hist_rmax(sim, th, nbins, r_max)[0])
    for s in range(th.shape[0]):
        c_ref, w_ref = ref.bond_corr(th[s], psi[s], box, nbins, r_max)
        assert np.array_equal(counts[s], c_ref) and np.array_equal(wsum[s], w_ref), s


@pytest.mark.parametrize("N", [400, 4096])
def test_neighbour_count_is_twice_the_gr_count(N):
    sim = make_sim(N)
    th, box = md_snapshots(sim, N)
    # 8.0 at N = 400: fewer than 3 cells per side, so psi_m uses one cell and g(r) the all-pairs kernel
    for r_nb in (1.2, 1.5, 2.5, 8.0):
        _, n, _ = order(sim, th, 6, r_nb)
        counts, launches = hist_rmax(sim, th, 1, r_nb)
        assert launches == (ALLPAIRS if N == 400 and r_nb == 8.0 else CELLS)
        assert np.array_equal(n.sum(axis=1, dtype=np.int64), 2 * counts[:, 0]), r_nb


def test_bond_correlation_api_and_lattice_physics():
    N = 4096
    sim = make_sim(N)
    R, V, box = lattice_jitter(N, seed=1)
    a = float(box) / 64
    r_nb = 1.2 * a                                        # between a and the diagonal a sqrt(2)
    psi, _, _ = order(sim, R, 4, r_nb)
    start = np.hypot(psi[0, :, 0], psi[0, :, 1]).mean()
    assert start > 0.9
    Psi = sim.last_bond_global.numpy()
    assert Psi.shape == (1, 2) and np.allclose(Psi[0], psi[0].mean(axis=0), rtol=0, atol=1e-15)
    (_, _), traj = sim.run((R, V), 4000, sample_every=2000)
    later, _, _ = order(sim, traj.numpy()[-1], 4, r_nb)
    assert np.hypot(later[0, :, 0], later[0, :, 1]).mean() < start - 0.2
    th = traj.numpy()
    centers, g = sim.bond_correlation(th, 5.0, 100, 6, 1.5)
    counts, wsum = sim.last_bond_counts.numpy(), sim.last_bond_wsum.numpy()
    assert np.array_equal(counts, hist_rmax(sim, th, 100, 5.0)[0])
    assert np.array_equal(centers.numpy(), (edges_for(5.0, 100)[:-1] + edges_for(5.0, 100)[1:]) / np.float32(2))
    g_ref = ref.g_m(counts.sum(axis=0), wsum.astype(np.float64).sum(axis=0))
    assert np.array_equal(np.isnan(g.numpy()), np.isnan(g_ref))
    assert np.allclose(g.numpy(), g_ref, rtol=1e-15, atol=0, equal_nan=True)


def test_determinism_and_batches():
    N = 4096
    sim = make_sim(N)
    th, box = md_snapshots(sim, N, nsteps=60, every=10)
    psi, n, _ = order(sim, th, 6, 1.5)
    psi2, n2, _ = order(sim, th, 6, 1.5)
    assert same_bits(psi, psi2) and np.array_equal(n, n2)
    for s in range(th.shape[0]):
        p1, n1, _ = order(sim, th[s], 6, 1.5)
        assert same_bits(p1[0], psi[s]) and np.array_equal(n1[0], n[s])
    c, w, _ = corr(sim, th, psi, 100, 5.0)
    c2, w2, _ = corr(sim, th, psi, 100, 5.0)
    assert np.array_equal(c, c2) and np.array_equal(w, w2)
    for s in range(th.shape[0]):
        c1, w1, _ = corr(sim, th[s], psi[s], 100, 5.0)
        assert np.array_equal(c1[0], c[s]) and np.array_equal(w1[0], w[s])


def test_batches_at_4m():
    """Eight snapshots of 4 M particles do not fit one 512 MiB batch of the grid scratch (16 B per particle for
    psi_m, 28 B for g_m(r))."""
    N = 4194304
    sim = make_sim(N, path="cells")
    R, _, box = lattice_jitter(N, seed=4)
    rng = np.random.default_rng(0)
    th = np.stack([np.clip(R + rng.uniform(-0.02, 0.02, R.shape).astype(np.float32), 0, box) for _ in range(8)])
    th = th.astype(np.float32)
    psi, n, launches = order(sim, th, 6, 1.5)
    assert launches > 4                                   # several batches
    c, w, launches = corr(sim, th, psi, 100, 5.0)
    assert launches > CELLS
    for s in (0, 7):
        p1, n1, _ = order(sim, th[s], 6, 1.5)
        assert same_bits(p1[0], psi[s]) and np.array_equal(n1[0], n[s])
        c1, w1, _ = corr(sim, th[s], psi[s], 100, 5.0)
        assert np.array_equal(c1[0], c[s]) and np.array_equal(w1[0], w[s])
    assert np.array_equal(c, hist_rmax(sim, th, 100, 5.0)[0])


def test_nan_particle_rule():
    N = 4096
    sim = make_sim(N)
    th, box = md_snapshots(sim, N, nsteps=20)
    X = th.copy()
    X[0, 17] = (np.nan, 1.0)
    X[1, 99, 1] = np.inf
    psi, n, _ = order(sim, X, 6, 1.5)
    assert np.isnan(psi[0, 17]).all() and n[0, 17] == 0 and np.isnan(psi[1, 99]).all() and n[1, 99] == 0
    for s in range(X.shape[0]):
        p_ref, n_ref = ref.bond_order(X[s], box, 6, 1.5)
        assert np.array_equal(n[s], n_ref) and same_bits(psi[s], p_ref)
    c, w, _ = corr(sim, X, psi, 100, 5.0)
    assert np.array_equal(c, hist_rmax(sim, X, 100, 5.0)[0])
    for s in range(X.shape[0]):
        c_ref, w_ref = ref.bond_corr(X[s], psi[s], box, 100, 5.0)
        assert np.array_equal(c[s], c_ref) and np.array_equal(w[s], w_ref)
    assert sim.lib.ljmd_check(sim._h) == 0


def test_handles_agree():
    N = 4096
    a, b = make_sim(N, path="allpairs"), make_sim(N, path="cells")
    th, _ = md_snapshots(a, N, nsteps=20)
    pa, na, _ = order(a, th, 6, 1.5)
    pb, nb, _ = order(b, th, 6, 1.5)
    assert same_bits(pa, pb) and np.array_equal(na, nb)
    ca, wa, _ = corr(a, th, pa, 100, 5.0)
    cb, wb, _ = corr(b, th, pb, 100, 5.0)
    assert np.array_equal(ca, cb) and np.array_equal(wa, wb)


def test_empty_history_and_argument_errors():
    N = 4096
    sim = make_sim(N)
    psi, n = sim.bond_order(np.zeros((0, N, 2), np.float32))
    assert psi.shape == (0, N, 2) and n.shape == (0, N)
    _, g = sim.bond_correlation(np.zeros((0, N, 2), np.float32), 5.0)
    assert np.isnan(g.numpy()).all()
    lib, h = sim.lib, sim._h
    R = torch.zeros((1, N, 2), dtype=torch.float32, device="cuda")
    P = torch.zeros((1, N, 2), dtype=torch.float64, device="cuda")
    nn = torch.zeros((1, N), dtype=torch.int32, device="cuda")
    ok = (h, R.data_ptr(), 1, 6, 1.5, P.data_ptr(), nn.data_ptr())
    assert lib.ljmd_bond_order(*ok) == 0
    assert lib.ljmd_bond_order(*ok[:6], None) == 0                     # nnb may be NULL
    bad = [
        (None,) + ok[1:],
        ok[:1] + (None,) + ok[2:],                                     # null positions with S > 0
        ok[:5] + (None,) + ok[6:],                                     # null psi
        ok[:2] + (-1,) + ok[3:],                                       # S < 0
        ok[:3] + (0,) + ok[4:], ok[:3] + (13,) + ok[4:],               # m out of [1, 12]
        ok[:4] + (0.0,) + ok[5:], ok[:4] + (-1.0,) + ok[5:],           # r_nb <= 0 or not finite
        ok[:4] + (float("nan"),) + ok[5:], ok[:4] + (float("inf"),) + ok[5:],
        ok[:1] + (R.data_ptr() + 4,) + ok[2:],                         # R_hist not 8-byte aligned
        ok[:5] + (P.data_ptr() + 8,) + ok[6:],                         # psi not 16-byte aligned
    ]
    for args in bad:
        assert lib.ljmd_bond_order(*args) == E_INVALID, args
        assert lib.ljmd_last_error()
    assert lib.ljmd_bond_order(h, None, 0, 6, 1.5, None, None) == 0    # S = 0
    e = torch.from_numpy(edges_for(5.0, 100)).cuda()
    c = torch.zeros((1, 100), dtype=torch.int64, device="cuda")
    w = torch.zeros((1, 100), dtype=torch.int64, device="cuda")
    ok = (h, R.data_ptr(), P.data_ptr(), 1, 100, e.data_ptr(), 5.0, c.data_ptr(), w.data_ptr())
    assert lib.ljmd_bond_corr(*ok) == 0
    bad = [
        (None,) + ok[1:],
        ok[:1] + (None,) + ok[2:],                                     # null positions
        ok[:2] + (None,) + ok[3:],                                     # null psi
        ok[:5] + (None,) + ok[6:],                                     # null edges
        ok[:7] + (None,) + ok[8:], ok[:8] + (None,),                   # null counts / wsum
        ok[:3] + (-1,) + ok[4:],                                       # S < 0
        ok[:4] + (0,) + ok[5:], ok[:4] + (8193,) + ok[5:],             # nbins out of [1, 8192]
        ok[:6] + (0.0,) + ok[7:], ok[:6] + (-1.0,) + ok[7:],           # r_max <= 0 or not finite
        ok[:6] + (float("nan"),) + ok[7:], ok[:6] + (float("inf"),) + ok[7:],
        ok[:1] + (R.data_ptr() + 4,) + ok[2:],                         # R_hist not 8-byte aligned
        ok[:2] + (P.data_ptr() + 8,) + ok[3:],                         # psi not 16-byte aligned
    ]
    for args in bad:
        assert lib.ljmd_bond_corr(*args) == E_INVALID, args
        assert lib.ljmd_last_error()
    assert lib.ljmd_bond_corr(h, None, None, 0, 100, None, 5.0, None, None) == 0   # S = 0


@pytest.mark.parametrize("N,extra", [(400, []), (4096, ["--gr_rmax", "5"])])
def test_driver_bond_m(tmp_path, capsys, N, extra):
    from jax_tpus_benchmark_physics_simulation_b200 import driver
    out = str(tmp_path / "g_r_plot.png")
    args = driver.parse_args(
        ["--N", str(N), "--rc", "2.5", "--ic", "lattice", "--eq_steps", "200", "--prod_steps", "300",
         "--sample_every", "100", "--bond_m", "6", "--output", out] + extra)
    res = driver.main(args)
    assert len(res) == 3
    text = capsys.readouterr().out
    assert "psi_6 Analysis" in text and "<|Psi_6|> = " in text and "chi_6 = " in text
    stem = str(tmp_path / "g_r_plot")
    Psi = np.load(stem + "_psi6.npy")
    assert Psi.shape == (3, 2) and np.isfinite(Psi).all()
    saved = np.load(stem + "_g6.npy")
    r, g = res[2]
    assert saved.shape == (2, r.size) and np.array_equal(saved[0], r)
    assert np.allclose(np.loadtxt(stem + "_g6.csv", delimiter=","), saved.T, equal_nan=True)
    assert np.array_equal(np.isfinite(saved[1]), g > 0)                # g_6 is finite exactly where g(r) counts
    assert np.nanmax(np.abs(saved[1])) <= 1.0
    assert driver.build_parser().parse_args([]).bond_m is None
