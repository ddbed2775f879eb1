"""CPU side of the Voronoi tessellation: the Qhull reference (tests/voronoi_reference.py) checked against the
invariants of a tessellation of the torus, topological_defects on hand-built inputs, and the driver's flag."""
import numpy as np
import pytest
import torch

import voronoi_reference as ref
from jax_tpus_benchmark_physics_simulation_b200.md import topological_defects


def _uniform(N, rho, seed):
    box = np.sqrt(np.float32(N / rho), dtype=np.float32)
    rng = np.random.default_rng(seed)
    return (rng.random((N, 2), dtype=np.float32) * box).astype(np.float32), float(box)


@pytest.mark.parametrize("N,rho", [(400, 0.8), (4096, 0.3), (4096, 0.05)])
def test_reference_invariants(N, rho):
    X, box = _uniform(N, rho, seed=N)
    r = ref.tessellate(X, box, (6,))
    n, adj = r["nvor"], r["adj"]
    assert n.min() >= 3 and n.sum() == 6 * N                       # Euler on the torus, no degenerate vertex
    assert abs(r["area"].sum() / box ** 2 - 1) <= 1e-12
    assert r["tau_ratio"] >= 2.0
    pairs = {(i, int(j)) for i in range(N) for j in adj[i][adj[i] >= 0]}
    assert all((j, i) in pairs for i, j in pairs)
    assert np.all(np.hypot(r["psi"][6][:, 0], r["psi"][6][:, 1]) <= 1 + 1e-12)


def test_reference_square_lattice():
    g = np.arange(64, dtype=np.float32) + np.float32(0.5)
    X = np.stack(np.meshgrid(g, g), axis=-1).reshape(-1, 2).astype(np.float32)
    r = ref.tessellate(X, 64.0, (4,))
    assert np.all(r["nvor"] == 4) and np.allclose(r["area"], 1.0, rtol=0, atol=1e-12)
    assert np.allclose(r["psi"][4], [1.0, 0.0], rtol=0, atol=1e-12)
    d = ref.min_image(X[r["adj"][:, :4], 0], X[:, None, 0], 64.0)
    assert np.all(np.diff(np.arctan2(ref.min_image(X[r["adj"][:, :4], 1], X[:, None, 1], 64.0), d), axis=1) > 0)


def test_reference_rules():
    X, box = _uniform(400, 0.8, seed=6)
    X[5] = (np.nan, 1.0)
    X[10:13] = X[200]                                               # coincident group {10, 11, 12, 200}
    r = ref.tessellate(X, box, (6,))
    assert r["nvor"][5] == -1 and np.isnan(r["area"][5]) and not np.isin(5, r["adj"]).any()
    assert np.all(r["nvor"][[10, 11, 12]] == r["nvor"][200]) and np.isin(10, r["adj"]).any()
    assert not np.isin([11, 12, 200], r["adj"]).any()
    Y = X[~np.isin(np.arange(400), [5, 11, 12, 200])]               # the same tessellation without them
    s = ref.tessellate(Y, box)
    assert np.array_equal(np.sort(s["nvor"]), np.sort(r["nvor"][~np.isin(np.arange(400), [5, 11, 12, 200])]))
    Z = X[:16] * np.float32(0.2)                                    # 16 particles in a box of 4.47: big cells
    t = ref.tessellate(np.nan_to_num(Z), float(np.sqrt(np.float32(20.0))))
    assert (t["nvor"] == -1).any()


def _defects(nv, edges, cap=8):
    nv = torch.tensor([nv])
    adj = torch.full((1, nv.shape[1], cap), -1)
    fill = [0] * nv.shape[1]
    for i, j in edges:
        for a, b in ((i, j), (j, i)):
            adj[0, a, fill[a]] = b
            fill[a] += 1
    return {k: int(v[0]) for k, v in topological_defects(nv, adj).items()}


def test_topological_defects():
    six = [6] * 12
    d = _defects(six, [])
    assert d == dict(n5=0, n7=0, other=0, charge=0, incomplete=0, disclinations=0, dislocations=0, defect_clusters=0)
    nv = six.copy(); nv[3] = 5
    d = _defects(nv, [(3, 4)])
    assert d["n5"] == 1 and d["disclinations"] == 1 and d["charge"] == 1
    nv = six.copy(); nv[3] = 7
    d = _defects(nv, [(3, 4)])
    assert d["n7"] == 1 and d["disclinations"] == 1 and d["charge"] == -1
    nv = six.copy(); nv[3], nv[4] = 5, 7
    d = _defects(nv, [(3, 4), (4, 5)])
    assert d["dislocations"] == 1 and d["disclinations"] == 0 and d["charge"] == 0
    nv = six.copy(); nv[1], nv[2], nv[3], nv[4] = 5, 7, 5, 7             # a 5-7-5-7 chain
    d = _defects(nv, [(1, 2), (2, 3), (3, 4)])
    assert d["defect_clusters"] == 1 and d["dislocations"] == 0 and d["disclinations"] == 0
    nv = six.copy(); nv[1], nv[2], nv[8] = 5, 5, 4                       # a 5-5 pair is a cluster, not a dislocation
    nv[9], nv[10] = -1, -1
    d = _defects(nv, [(1, 2)])
    assert d["defect_clusters"] == 1 and d["disclinations"] == 1 and d["other"] == 1
    assert d["incomplete"] == 2 and d["charge"] == 1 + 1 + 2
    with pytest.raises(ValueError):
        _defects([9] + six[1:], [], cap=8)                          # a defect with more neighbours than adj holds
    # several snapshots at once, components do not leak between them
    a = torch.tensor([[5, 7, 6], [5, 6, 7]])
    adj = torch.tensor([[[1, -1], [0, -1], [-1, -1]], [[1, -1], [0, 2], [1, -1]]])
    adj = torch.nn.functional.pad(adj, (0, 6), value=-1)
    d = topological_defects(a, adj)
    assert d["dislocations"].tolist() == [1, 0] and d["disclinations"].tolist() == [0, 2]


def test_driver_flag():
    from jax_tpus_benchmark_physics_simulation_b200 import driver
    assert driver.parse_args([]).voronoi is False
    args = driver.parse_args(["--voronoi", "--bond_m", "6"])
    assert args.voronoi and args.bond_m == 6
    with pytest.raises(SystemExit):
        driver.parse_args(["--voronoi", "1"])
