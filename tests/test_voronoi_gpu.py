"""The Voronoi tessellation (ljmd_voronoi, csrc/voronoi.cu): nvor and the adjacency exactly, area and the
edge-weighted psi_m within 1e-9 of the Qhull reference (tests/voronoi_reference.py) on MD snapshots and uniform
states, the exact square lattice, 4 M and 16 M particles (windows against Qhull and global invariants),
determinism across calls, batches, handles and snapshots, the incomplete / NaN / coincident rules, launches,
argument errors and the driver.  A call makes four launches per batch of snapshots: the grid's three and one."""
import numpy as np
import pytest
import torch

import voronoi_reference as ref
from analysis_helpers import E_INVALID, make_sim, md_snapshots, uniform_snapshots
from jax_tpus_benchmark_physics_simulation_b200 import lattice_jitter
from jax_tpus_benchmark_physics_simulation_b200.md import topological_defects

pytestmark = pytest.mark.gpu

LAUNCHES = 4
TOL = 1e-9


def run(sim, Rs, m=None, adj_cap=64):
    """voronoi() of the snapshots Rs: (nvor, area, adj, psi or None, launches) as numpy arrays."""
    l0 = sim.launch_count()
    nvor, area = sim.voronoi(Rs, m=m, adj_cap=adj_cap)
    psi = sim.last_voronoi_psi.numpy() if m is not None else None
    adj = sim.last_voronoi_adj.numpy() if adj_cap else None
    return nvor.numpy(), area.numpy(), adj, psi, sim.launch_count() - l0


def compare(got, r, sel=None, ms=(4, 6)):
    """Exact nvor / adjacency, area and psi within TOL, on the particles the reference determined (sel)."""
    nvor, area, adj, psis = got
    det = r["nvor"] != -2 if sel is None else sel
    assert r["tau_ratio"] >= 2.0, r["tau_ratio"]                 # no ridge within a factor 2 of the threshold
    assert np.array_equal(nvor[det], r["nvor"][det])
    assert np.array_equal(adj[det], r["adj"][det][:, :adj.shape[1]])
    ok = det & (r["nvor"] >= 0)
    assert np.all(np.isnan(area[det & ~ok]))
    ea = float(np.max(np.abs(area[ok] - r["area"][ok]) / r["area"][ok])) if ok.any() else 0.0
    assert ea <= TOL, ea
    ep = 0.0
    for m in ms:
        ep = max(ep, float(np.max(np.abs(psis[m][ok] - r["psi"][m][ok]))) if ok.any() else 0.0)
    assert ep <= TOL, ep
    return ea, ep


def check_ref(sim, Rs, box, ms=(4, 6)):
    Rs = np.asarray(Rs, np.float32).reshape(-1, sim.N, 2)
    runs = {m: run(sim, Rs, m) for m in ms}
    nvor, area, adj, _, launches = runs[ms[0]]
    worst = (0.0, 0.0)
    for s in range(Rs.shape[0]):
        r = ref.tessellate(Rs[s], box, ms)
        ea, ep = compare((nvor[s], area[s], adj[s], {m: runs[m][3][s] for m in ms}), r, ms=ms)
        worst = (max(worst[0], ea), max(worst[1], ep))
    print(f"N = {sim.N}: max relative area error {worst[0]:.3e}, max psi error {worst[1]:.3e}")
    return nvor, area, adj, launches


@pytest.mark.parametrize("N", [400, 4096, 65536])
def test_matches_reference(N):
    sim = make_sim(N)
    th, box = md_snapshots(sim, N, nsteps=20)
    _, _, _, launches = check_ref(sim, th, box)
    assert launches == LAUNCHES
    for rho in (0.05, 0.3, 0.8):
        sr = make_sim(N, rho=rho)
        X, b = uniform_snapshots(sr, 1, seed=int(rho * 100))
        check_ref(sr, X, b)


def test_exact_square_lattice():
    N = 4096
    sim = make_sim(N, rho=1.0)
    assert sim.box_size == 64.0
    g = np.arange(64, dtype=np.float32) + np.float32(0.5)
    X = np.stack(np.meshgrid(g, g), axis=-1).reshape(N, 2).astype(np.float32)
    X = X[np.random.default_rng(1).permutation(N)]
    nvor, area, _, psi, _ = run(sim, X, m=4)
    assert np.all(nvor == 4) and np.all(area == 1.0)
    assert np.max(np.abs(psi[0] - np.array([1.0, 0.0]))) <= 1e-12


def _symmetric(adj):
    """adj (N, cap) device tensor: every (i, j) has its (j, i)."""
    N, cap = adj.shape
    i = torch.arange(N, device=adj.device, dtype=torch.int64)[:, None].expand(N, cap)
    j = adj.to(torch.int64)
    on = j >= 0
    a = torch.sort(i[on] * N + j[on]).values
    b = torch.sort(j[on] * N + i[on]).values
    return torch.equal(a, b)


@pytest.mark.parametrize("N,path", [(4194304, "cells"), (16777216, "cells")])
def test_large(N, path):
    sim = make_sim(N, path=path)
    if N == 4194304:
        th, box = md_snapshots(sim, N, nsteps=10, every=10, seed=3)
        X = th[0]
    else:
        R, _, box = lattice_jitter(N, seed=3)
        X, box = np.asarray(R, np.float32), float(box)
    nvor_d, area_d = sim.voronoi(X, m=6, adj_cap=16)
    nv = nvor_d.tensor[0]
    assert int(nv.min()) >= 3                                     # every cell complete, n >= 3
    assert int(nv.sum()) == 6 * N
    d = topological_defects(nvor_d, sim.last_voronoi_adj)
    assert int(d["charge"][0]) == 0 and int(d["incomplete"][0]) == 0
    tot = float(area_d.tensor[0].sum())
    assert abs(tot / box ** 2 - 1.0) <= 1e-9, tot / box ** 2
    assert _symmetric(sim.last_voronoi_adj.tensor[0])
    nvor, area = nv.cpu().numpy(), area_d.numpy()[0]
    adj, psi = sim.last_voronoi_adj.numpy()[0], sim.last_voronoi_psi.numpy()[0]
    a = box / np.sqrt(N)
    for lo in (0.0, 0.37 * box, box - 60 * a):                   # windows of 60 x 60 spacings, one at the edge
        hi = lo + 60 * a
        r = ref.tessellate(X, box, (6,), window=(lo, hi), margin=8 * a)
        sel = r["nvor"] != -2
        assert sel.sum() > 2000
        r["adj"] = r["adj"][:, :16]
        compare((nvor, area, adj, {6: psi}), r, sel, ms=(6,))


def test_determinism_handles_and_snapshots():
    N = 4096
    a, b = make_sim(N, path="allpairs"), make_sim(N, path="cells")
    th, _ = md_snapshots(a, N, nsteps=60, every=10)
    ra = run(a, th, 6)
    ra2 = run(a, th, 6)
    rb = run(b, th, 6)
    for x, y, z in zip(ra[:4], ra2[:4], rb[:4]):
        assert np.array_equal(x, y, equal_nan=True) and np.array_equal(x, z, equal_nan=True)
    for s in range(th.shape[0]):
        r1 = run(a, th[s], 6)
        for x, y in zip(r1[:4], ra[:4]):
            assert np.array_equal(x[0], y[s], equal_nan=True)


def test_batches_at_4m():
    """Ten snapshots of 4 M particles do not fit one 512 MiB batch of the grid scratch (16 B per particle)."""
    N = 4194304
    sim = make_sim(N, path="cells")
    R, _, box = lattice_jitter(N, seed=4)
    rng = np.random.default_rng(0)
    th = np.stack([np.clip(R + rng.uniform(-0.05, 0.05, R.shape).astype(np.float32), 0, box)
                   for _ in range(10)]).astype(np.float32)
    nvor, area, adj, psi, launches = run(sim, th, 6, adj_cap=8)
    assert launches > LAUNCHES and launches % LAUNCHES == 0        # several batches
    for s in (0, 9):
        n1, a1, j1, p1, _ = run(sim, th[s], 6, adj_cap=8)
        assert np.array_equal(n1[0], nvor[s]) and np.array_equal(a1[0], area[s])
        assert np.array_equal(j1[0], adj[s]) and np.array_equal(p1[0], psi[s])


def test_nan_rule():
    N = 4096
    sim = make_sim(N)
    th, box = md_snapshots(sim, N, nsteps=20)
    X = th.copy()
    X[0, 17] = (np.nan, 1.0)
    X[1, 99, 1] = np.inf
    nvor, area, adj, _ = check_ref(sim, X, box)
    assert nvor[0, 17] == -1 and np.isnan(area[0, 17]) and np.all(adj[0, 17] == -1)
    assert not np.any(adj[0] == 17) and not np.any(adj[1] == 99)
    assert sim.lib.ljmd_check(sim._h) == 0


def test_vertex_cap():
    """A particle at the centre of a ring of 70 sites would need 70 vertices: incomplete; the rest as Qhull."""
    N = 4096
    sim = make_sim(N, rho=0.3)
    X, box = uniform_snapshots(sim, 1, seed=5)
    X = X[0]
    c = np.float32(box / 2)
    far = np.hypot(X[:, 0] - c, X[:, 1] - c) > 6.0
    X[~far] = X[far][: (~far).sum()] * np.float32(0.25)          # clear a disc around the centre
    t = 2 * np.pi * np.arange(70) / 70
    X[0] = (c, c)
    X[1:71, 0] = (c + 3.0 * np.cos(t)).astype(np.float32)
    X[1:71, 1] = (c + 3.0 * np.sin(t)).astype(np.float32)
    nvor, area, adj, psi, _ = run(sim, X, 6)
    assert nvor[0, 0] == -1 and np.isnan(area[0, 0]) and np.all(adj[0, 0] == -1)
    r = ref.tessellate(X, box, (6,))
    assert r["nvor"][0] == 70
    sel = np.ones(N, bool)
    sel[0] = False
    compare((nvor[0], area[0], adj[0], {6: psi[0]}), r, sel, ms=(6,))


def test_tiny_box_and_void():
    sim = make_sim(16)
    X, box = uniform_snapshots(sim, 4, seed=2)
    nvor, _, _, _ = check_ref(sim, X, box)
    assert (nvor == -1).any() and (nvor > 0).any()               # both kinds of rows occur
    sim = make_sim(400)
    X, box = uniform_snapshots(sim, 1, seed=6)
    X = X[0] * np.float32(0.5)                                    # everything in one quarter of the box ...
    X[7] = (np.float32(0.75) * box, np.float32(0.75) * box)      # ... but one particle
    nvor, _, _, _ = check_ref(sim, X, box)
    assert nvor[0, 7] == -1


def test_coincident_sites():
    """Coincident particles share one cell; their neighbours list only the smallest index of the group."""
    N = 4096
    sim = make_sim(N)
    X, box = uniform_snapshots(sim, 1, seed=9)
    X[0, 100:105] = X[0, 3000]
    nvor, area, adj, _ = check_ref(sim, X, box)
    for k in list(range(100, 105)):
        assert nvor[0, k] == nvor[0, 3000] and area[0, k] == area[0, 3000]
        assert np.array_equal(adj[0, k], adj[0, 3000])
    assert not np.isin(np.arange(101, 105), adj[0]).any() and not np.isin(3000, adj[0]).any()


def test_empty_history_and_argument_errors():
    N = 4096
    sim = make_sim(N)
    nvor, area = sim.voronoi(np.zeros((0, N, 2), np.float32), m=6)
    assert nvor.shape == (0, N) and area.shape == (0, N)
    lib, h = sim.lib, sim._h
    R = torch.zeros((1, N, 2), dtype=torch.float32, device="cuda")
    nv = torch.zeros((1, N), dtype=torch.int32, device="cuda")
    ar = torch.zeros((1, N), dtype=torch.float64, device="cuda")
    adj = torch.zeros((1, N, 8), dtype=torch.int32, device="cuda")
    psi = torch.zeros((1, N, 2), dtype=torch.float64, device="cuda")
    ok = (h, R.data_ptr(), 1, nv.data_ptr(), ar.data_ptr(), adj.data_ptr(), 8, 6, psi.data_ptr())
    assert lib.ljmd_voronoi(*ok) == 0
    assert lib.ljmd_voronoi(h, R.data_ptr(), 1, nv.data_ptr(), None, None, 0, 0, None) == 0   # optional outputs
    bad = [
        (None,) + ok[1:],
        ok[:1] + (None,) + ok[2:],                                 # null positions with S > 0
        ok[:3] + (None,) + ok[4:],                                 # null nvor
        ok[:2] + (-1,) + ok[3:],                                   # S < 0
        ok[:6] + (0,) + ok[7:], ok[:6] + (65,) + ok[7:],           # adj_cap out of range with adj
        ok[:7] + (0,) + ok[8:], ok[:7] + (13,) + ok[8:],           # m out of range with psi
        ok[:1] + (R.data_ptr() + 4,) + ok[2:],                     # R_hist not 8-byte aligned
        ok[:3] + (nv.data_ptr() + 2,) + ok[4:],                    # nvor not 4-byte aligned
        ok[:4] + (ar.data_ptr() + 4,) + ok[5:],                    # area not 8-byte aligned
        ok[:5] + (adj.data_ptr() + 2,) + ok[6:],                   # adj not 4-byte aligned
        ok[:8] + (psi.data_ptr() + 8,),                            # psi not 16-byte aligned
    ]
    for args in bad:
        assert lib.ljmd_voronoi(*args) == E_INVALID, args
        assert b"ljmd_voronoi" in lib.ljmd_last_error()
    assert lib.ljmd_voronoi(h, None, 0, None, None, None, 0, 0, None) == 0   # S = 0


@pytest.mark.parametrize("N,extra", [(400, []), (400, ["--bond_m", "6"]), (4096, []), (4096, ["--bond_m", "6"])])
def test_driver_voronoi(tmp_path, capsys, N, extra):
    from jax_tpus_benchmark_physics_simulation_b200 import driver
    out = str(tmp_path / "g_r_plot.png")
    args = driver.parse_args(
        ["--N", str(N), "--rc", "2.5", "--ic", "lattice", "--eq_steps", "200", "--prod_steps", "300",
         "--sample_every", "100", "--voronoi", "--output", out] + extra)
    state, R_history, _ = driver.main(args)
    text = capsys.readouterr().out
    assert "Voronoi Analysis" in text and "<n> = " in text and "<dislocations> = " in text
    assert ("Voronoi-weighted" in text) == bool(extra)
    stem = str(tmp_path / "g_r_plot")
    saved = np.load(stem + "_voronoi.npy")
    assert np.array_equal(np.loadtxt(stem + "_voronoi.csv", delimiter=",", dtype=np.int64).reshape(-1, 8), saved)
    sim = make_sim(N)
    nvor, _ = sim.voronoi(R_history, adj_cap=16)
    d = topological_defects(nvor, sim.last_voronoi_adj)
    assert np.array_equal(saved[:, 0], d["n5"].cpu().numpy()) and np.array_equal(saved[:, 6],
                                                                                   d["dislocations"].cpu().numpy())
    assert np.all(saved[:, 3] == 0)                               # total charge of the torus
