"""The cluster analysis (ljmd_clusters, csrc/cluster.cu): labels and sizes bit for bit against the CPU restatement
(tests/cluster_reference.{c,py}), adversarial placements, masks, the NaN rule, invariants, the link count against
ljmd_gr_hist_rmax, determinism across calls, batches and handles, argument errors and the driver.  A call makes
six launches per batch of snapshots: the grid's three, then init, hook and flatten."""
import numpy as np
import pytest
import torch

import cluster_reference as ref
from analysis_helpers import E_INVALID, hist_rmax, make_sim, md_snapshots, uniform_snapshots
from gr_reference import adversarial
from jax_tpus_benchmark_physics_simulation_b200 import lattice_jitter

pytestmark = pytest.mark.gpu

LAUNCHES = 6


def run(sim, Rs, r_link, mask=None):
    """clusters() of the snapshots Rs: (labels (S, N), sizes (S, N), launches)."""
    l0 = sim.launch_count()
    labels, sizes = sim.clusters(Rs, r_link, mask)
    return labels.numpy(), sizes.numpy(), sim.launch_count() - l0


def check_ref(sim, Rs, box, r_link, mask=None):
    Rs = np.asarray(Rs, np.float32).reshape(-1, sim.N, 2)
    labels, sizes, launches = run(sim, Rs, r_link, mask)
    for s in range(Rs.shape[0]):
        m = None if mask is None else np.broadcast_to(np.asarray(mask), Rs.shape[:2])[s]
        l_ref, s_ref = ref.clusters(Rs[s], box, r_link, m)
        assert np.array_equal(labels[s], l_ref), (r_link, s)
        assert np.array_equal(sizes[s], s_ref), (r_link, s)
    return labels, sizes, launches


@pytest.mark.parametrize("N", [400, 4096, 65536])
def test_matches_reference(N):
    sim = make_sim(N)
    th, box = md_snapshots(sim, N)
    for r_link in (1.1, 1.5, 2.5):
        _, _, launches = check_ref(sim, th, box, r_link)
        assert launches == LAUNCHES
    for rho in (0.05, 0.3, 0.8):
        s = make_sim(N, rho=rho)
        X, b = uniform_snapshots(s, 2, seed=int(rho * 100))
        for r_link in (1.1, 1.5, 2.5):
            check_ref(s, X, b, r_link)


@pytest.mark.parametrize("r_link", [1.5, 1.05])
def test_matches_reference_4m(r_link):
    N = 4194304
    sim = make_sim(N, path="cells")
    R, _, box = lattice_jitter(N, seed=3)
    labels, sizes, _ = check_ref(sim, R, box, r_link)
    n = int((sizes[0] > 0).sum())
    assert (n == 1) if r_link == 1.5 else (n > 1)                 # one giant cluster / fragments
    assert sim.last_cluster_count.numpy()[0] == n


def test_one_cell():
    sim = make_sim(400)
    th, box = md_snapshots(sim, 400)
    assert 8.0 > box / 3
    check_ref(sim, th, box, 8.0)
    check_ref(sim, th, box, 0.9)


@pytest.mark.parametrize("N", [400, 4096])
def test_adversarial_placements(N):
    sim = make_sim(N)
    box = float(lattice_jitter(N)[2])
    for r_link in (1.2, 1.5, 2.5, 5.0, 8.0):
        X = adversarial(N, box, r_link, seed=5)
        check_ref(sim, X, box, r_link)
        up = float(np.nextafter(np.float32(r_link), np.float32(0)))   # the pairs at exactly r_link now apart
        check_ref(sim, X, box, up)


def test_exact_distance_and_one_ulp():
    sim = make_sim(4096)
    box = np.float32(sim.box_size)
    X, _ = uniform_snapshots(sim, 1, seed=3)
    X = X[0] * np.float32(0.5)                                      # leave the upper half free
    y = np.float32(0.75) * box
    X[10] = (np.float32(3.0), y)
    X[20] = (np.float32(4.5), y)                                    # exactly 1.5 apart in fp32
    X[30] = (np.float32(box - np.float32(0.5)), y + 3)
    X[40] = (np.float32(1.0), y + 3)                                # about 1.5 apart through the periodic edge
    X[50] = (box, y + 6)
    X[60] = (np.float32(1.5), y + 6)                                # x == box
    X[70] = (np.float32(3.0), y + 9)
    X[80] = (np.nextafter(np.float32(4.5), np.float32(9)), y + 9)   # one ulp of 4.5 above 1.5 apart
    labels, _, _ = check_ref(sim, X, box, 1.5)
    assert labels[0, 20] == 10 and labels[0, 80] == 80
    labels, _, _ = check_ref(sim, X, box, float(np.nextafter(np.float32(1.5), np.float32(0))))
    assert labels[0, 20] == 20


def test_permuted_chain_and_periodic_ring():
    N = 65536
    sim = make_sim(N)
    box = np.float32(sim.box_size)
    rng = np.random.default_rng(7)
    X = (rng.random((N, 2), dtype=np.float32) * box * np.float32(0.4)).astype(np.float32)
    X[:, 1] += np.float32(0.5) * box                                # background in the upper half
    L = 20000                                                       # chain in the lower half, random indices
    perm = rng.permutation(N)[:L]
    t = np.arange(L, dtype=np.float32)
    X[perm, 0] = np.float32(0.9) * t % box
    X[perm, 1] = np.float32(0.25) * box + np.float32(1.0) * np.floor(np.float32(0.9) * t / box)
    xs = np.linspace(0, box, int(box) + 1, endpoint=False, dtype=np.float32)
    xs = xs[np.abs(xs - box / 2) > 1.0]                             # a gap of 2 in the middle: joined only
    ring = rng.permutation(np.setdiff1d(np.arange(N), perm))[:xs.size]   # through x = 0 == box
    X[ring, 0] = xs
    X[ring, 1] = np.float32(0.1) * box
    X = np.clip(X, 0, box).astype(np.float32)
    labels, _, _ = check_ref(sim, X, float(box), 1.0)
    assert np.unique(labels[0, ring]).size == 1 and labels[0, ring[0]] == ring.min()


def test_coincident_particles():
    N = 4096
    sim = make_sim(N)
    X, box = uniform_snapshots(sim, 1, seed=9)
    X[0, :1000] = X[0, 123]                                         # 1000 particles on one point
    labels, sizes, _ = check_ref(sim, X, box, 1.1)
    assert np.all(labels[0, :1000] == 0) and sizes[0, 0] >= 1000


def test_masks():
    N = 4096
    sim = make_sim(N)
    th, box = md_snapshots(sim, N)
    rng = np.random.default_rng(2)
    check_ref(sim, th, box, 1.5, rng.random(th.shape[:2]) < 0.5)
    check_ref(sim, th, box, 1.5, (rng.random(N) < 0.3).astype(np.uint8))            # broadcast (N,)
    labels, sizes, _ = run(sim, th, 1.5, np.zeros(N, bool))
    assert np.all(labels == -1) and np.all(sizes == 0)
    assert np.array_equal(sim.last_cluster_count.numpy(), np.zeros(th.shape[0]))
    la, sa, _ = run(sim, th, 1.5, np.ones(th.shape[:2], bool))
    lb, sb, _ = run(sim, th, 1.5)
    assert np.array_equal(la, lb) and np.array_equal(sa, sb)
    psi, _ = sim.bond_order(th, 6, 1.5)
    p = psi.numpy()
    solid = np.hypot(p[..., 0], p[..., 1]) >= 0.7
    check_ref(sim, th, box, 1.5, solid)


def test_nan_rule():
    N = 4096
    sim = make_sim(N)
    th, box = md_snapshots(sim, N, nsteps=20)
    X = th.copy()
    X[0, 17] = (np.nan, 1.0)
    X[1, 99, 1] = np.inf
    labels, sizes, _ = check_ref(sim, X, box, 1.5)
    assert labels[0, 17] == -1 and labels[1, 99] == -1
    keep = np.ones(N, bool)
    keep[17] = False
    la, _, _ = run(sim, th[0], 1.5, keep)                        # the snapshot without particle 17
    assert np.array_equal(la[0], labels[0])
    assert sim.lib.ljmd_check(sim._h) == 0


@pytest.mark.parametrize("N", [400, 65536])
def test_invariants_and_link_count(N):
    sim = make_sim(N)
    th, box = md_snapshots(sim, N)
    for r_link in (1.1, 1.5):
        labels, sizes, _ = run(sim, th, r_link)
        for s in range(th.shape[0]):
            on = labels[s][labels[s] >= 0]
            assert sizes[s].sum() == on.size == N
            assert np.array_equal(labels[s][on], on)
            assert np.array_equal(np.nonzero(sizes[s])[0], np.unique(on))
        assert np.array_equal(sim.last_cluster_largest.numpy(), sizes.max(axis=1))
        n_links = np.array([len(ref.links(th[s], box, r_link)) for s in range(th.shape[0])])
        assert np.array_equal(n_links, hist_rmax(sim, th, 1, r_link)[0][:, 0]), r_link


def test_determinism_and_handles():
    N = 4096
    a, b = make_sim(N, path="allpairs"), make_sim(N, path="cells")
    th, _ = md_snapshots(a, N, nsteps=60, every=10)
    la, sa, _ = run(a, th, 1.5)
    la2, sa2, _ = run(a, th, 1.5)
    lb, sb, _ = run(b, th, 1.5)
    assert np.array_equal(la, la2) and np.array_equal(sa, sa2)
    assert np.array_equal(la, lb) and np.array_equal(sa, sb)
    for s in range(th.shape[0]):
        l1, s1, _ = run(a, th[s], 1.5)
        assert np.array_equal(l1[0], la[s]) and np.array_equal(s1[0], sa[s])


def test_batches_at_4m():
    """Ten snapshots of 4 M particles do not fit one 512 MiB batch of the grid scratch (16 B per particle)."""
    N = 4194304
    sim = make_sim(N, path="cells")
    R, _, box = lattice_jitter(N, seed=4)
    rng = np.random.default_rng(0)
    th = np.stack([np.clip(R + rng.uniform(-0.05, 0.05, R.shape).astype(np.float32), 0, box)
                   for _ in range(10)]).astype(np.float32)
    labels, sizes, launches = run(sim, th, 1.05)
    assert launches > LAUNCHES and launches % LAUNCHES == 0        # several batches
    for s in (0, 9):
        l1, s1, _ = run(sim, th[s], 1.05)
        assert np.array_equal(l1[0], labels[s]) and np.array_equal(s1[0], sizes[s])


def test_distribution():
    N = 4096
    sim = make_sim(N, rho=0.3)
    X, _ = uniform_snapshots(sim, 3, seed=11)
    _, sizes = sim.clusters(X, 1.5)
    s, n_s = sim.cluster_distribution(sizes)
    sz = sizes.numpy()
    vals, cnt = np.unique(sz[sz > 0], return_counts=True)
    assert np.array_equal(s.numpy(), vals) and np.allclose(n_s.numpy(), cnt / 3, rtol=1e-15, atol=0)
    assert np.isclose((s.numpy() * n_s.numpy()).sum(), N)


def test_empty_history_and_argument_errors():
    N = 4096
    sim = make_sim(N)
    labels, sizes = sim.clusters(np.zeros((0, N, 2), np.float32), 1.5)
    assert labels.shape == (0, N) and sizes.shape == (0, N)
    lib, h = sim.lib, sim._h
    R = torch.zeros((1, N, 2), dtype=torch.float32, device="cuda")
    lab = torch.zeros((1, N), dtype=torch.int32, device="cuda")
    siz = torch.zeros((1, N), dtype=torch.int32, device="cuda")
    ok = (h, R.data_ptr(), 1, 1.5, None, lab.data_ptr(), siz.data_ptr())
    assert lib.ljmd_clusters(*ok) == 0
    assert lib.ljmd_clusters(*ok[:6], None) == 0                   # sizes may be NULL
    bad = [
        (None,) + ok[1:],
        ok[:1] + (None,) + ok[2:],                                 # null positions with S > 0
        ok[:5] + (None,) + ok[6:],                                 # null labels
        ok[:2] + (-1,) + ok[3:],                                   # S < 0
        ok[:3] + (0.0,) + ok[4:], ok[:3] + (-1.0,) + ok[4:],       # r_link <= 0 or not finite
        ok[:3] + (float("nan"),) + ok[4:], ok[:3] + (float("inf"),) + ok[4:],
        ok[:1] + (R.data_ptr() + 4,) + ok[2:],                     # R_hist not 8-byte aligned
        ok[:5] + (lab.data_ptr() + 2,) + ok[6:],                   # labels not 4-byte aligned
        ok[:6] + (siz.data_ptr() + 2,),                            # sizes not 4-byte aligned
    ]
    for args in bad:
        assert lib.ljmd_clusters(*args) == E_INVALID, args
        assert b"ljmd_clusters" in lib.ljmd_last_error()
    assert lib.ljmd_clusters(h, None, 0, 1.5, None, None, None) == 0   # S = 0


@pytest.mark.parametrize("extra", [[], ["--bond_m", "6", "--cluster_psi_min", "0.7"]])
def test_driver_clusters(tmp_path, capsys, extra):
    from jax_tpus_benchmark_physics_simulation_b200 import driver
    out = str(tmp_path / "g_r_plot.png")
    args = driver.parse_args(
        ["--N", "400", "--rc", "2.5", "--ic", "lattice", "--eq_steps", "200", "--prod_steps", "300",
         "--sample_every", "100", "--cluster_rlink", "1.5", "--output", out] + extra)
    state, R_history, _ = driver.main(args)
    text = capsys.readouterr().out
    assert "Cluster Analysis" in text and "<clusters> = " in text and "<largest> = " in text
    stem = str(tmp_path / "g_r_plot")
    saved = np.load(stem + "_clusters.npy")
    assert np.allclose(np.loadtxt(stem + "_clusters.csv", delimiter=",").reshape(-1, 2), saved.T)
    sim = make_sim(400)
    mask = None
    if extra:
        psi, _ = sim.bond_order(R_history, 6, 1.5)
        p = psi.numpy()
        mask = np.hypot(p[..., 0], p[..., 1]) >= 0.7
    _, sizes = sim.clusters(R_history, 1.5, mask)
    s, n_s = sim.cluster_distribution(sizes)
    assert np.array_equal(saved[0], s.numpy()) and np.array_equal(saved[1], n_s.numpy())
    assert driver.build_parser().parse_args([]).cluster_rlink is None
    with pytest.raises(SystemExit):
        driver.parse_args(["--cluster_rlink", "1.5", "--cluster_psi_min", "0.7"])
