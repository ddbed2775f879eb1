"""CPU checks for S(k): the fp64 density-mode reference (tests/sk_reference.c) against analytic answers, the host
wave-vector generator of LJSimulation.structure_factor (md.structure_factor_vectors), and the driver's flags."""
import math

import numpy as np
import pytest

from jax_tpus_benchmark_physics_simulation_b200.ic import box_size, lattice_jitter
from jax_tpus_benchmark_physics_simulation_b200.md import structure_factor_vectors
from sk_reference import bound, c_density_modes


def _all_vectors(nmax):
    return np.array([(x, y) for y in range(-nmax, nmax + 1) for x in range(-nmax, nmax + 1)], dtype=np.int32)


def test_reference_one_pair():
    box = np.float32(10.0)
    R = np.array([[1.25, 2.5], [7.0, 3.75]], dtype=np.float32)
    nv = _all_vectors(6)
    rho = c_density_modes(R, box, nv)[0]
    k = 2 * np.pi / float(box) * nv.astype(np.float64)
    dr = R[0].astype(np.float64) - R[1].astype(np.float64)
    want = 2.0 + 2.0 * np.cos(k @ dr)
    assert np.allclose(rho[:, 0] ** 2 + rho[:, 1] ** 2, want, rtol=0, atol=1e-12)


def test_reference_square_lattice():
    m = 8
    box = np.float32(m * 1.5)
    ii, jj = np.meshgrid(np.arange(m), np.arange(m), indexing="ij")
    R = (np.stack([ii.ravel(), jj.ravel()], axis=1) * 1.5 + 0.25).astype(np.float32)
    nv = _all_vectors(2 * m)
    rho = c_density_modes(R, box, nv)[0]
    bragg = (nv[:, 0] % m == 0) & (nv[:, 1] % m == 0)
    assert bragg.sum() == 25
    mag = np.hypot(rho[:, 0], rho[:, 1])
    assert np.allclose(mag[bragg], m * m, rtol=0, atol=1e-9)
    assert mag[~bragg].max() < 1e-9


def test_reference_pair_sum_identity():
    N = 64
    R, _, box = lattice_jitter(N, seed=4, jitter=0.3)
    nv, _ = structure_factor_vectors(float(box), 6.0)
    rho = c_density_modes(R, box, nv)[0]
    sk = (rho[:, 0] ** 2 + rho[:, 1] ** 2) / N
    k = 2 * np.pi / float(box) * nv.astype(np.float64)
    i, j = np.triu_indices(N, k=1)
    d = R[i].astype(np.float64) - R[j].astype(np.float64)
    want = 1.0 + 2.0 / N * np.cos(d @ k.T).sum(axis=0)
    assert np.allclose(sk, want, rtol=0, atol=1e-11)


def test_reference_is_periodic_and_batched():
    N = 256
    R, _, box = lattice_jitter(N, seed=1)
    nv, _ = structure_factor_vectors(float(box), 4.0)
    shifted = (R + np.float32(box) * np.array([1, -2], np.float32)).astype(np.float32)
    a = c_density_modes(np.stack([R, shifted]), box, nv)
    # x + box is rounded in fp32, so the shifted positions are off by up to half an ulp of 3 box
    tol = N * np.abs(nv).sum(axis=1).max() * 2 * np.pi * 3 * float(box) * 2.0 ** -24 / float(box)
    assert np.abs(a[0] - a[1]).max() < tol


def test_bound_is_the_documented_formula():
    b = bound(4096, np.array([[0, 1], [8192, -8192]]))
    eps0 = math.pi * (2 ** -25 + 2 ** -24) + 2 ** -23 + 2 ** -20.5
    assert abs(eps0 - 1.074e-6) < 1e-9
    assert b[0] == pytest.approx(4096 * (eps0 + math.pi * 2 ** -32 + 16.5 * 2 ** -24) + (128 + 1024) * 4096 * 2 ** -53)
    assert b[1] > b[0]


# ---------------------------------------------------------------- wave vectors
def _brute(box, k_max):
    dk = 2 * math.pi / box
    nmax = int(k_max / dk) + 2
    out = []
    for ny in range(0, nmax + 1):
        for nx in range(-nmax, nmax + 1):
            if ny == 0 and nx <= 0:
                continue
            if dk * math.sqrt(nx * nx + ny * ny) <= k_max:
                out.append((nx, ny, math.isqrt(nx * nx + ny * ny)))
    return out


@pytest.mark.parametrize("N,k_max", [(400, 8.0), (4096, 3.0), (4096, 8.0), (1024, 0.3)])
def test_vectors_match_brute_force(N, k_max):
    box = float(box_size(N, 0.8))
    nv, shell = structure_factor_vectors(box, k_max)
    ref = _brute(box, k_max)
    assert nv.dtype == np.int32 and nv.shape == (len(ref), 2) and shell.shape == (len(ref),)
    assert sorted(zip(nv[:, 0].tolist(), nv[:, 1].tolist(), shell.tolist())) == sorted(ref)
    assert np.all(np.diff(shell) >= 0)                                  # grouped by shell
    for m in np.unique(shell):                                         # by angle inside a shell
        v = nv[shell == m]
        assert np.all(np.diff(np.arctan2(v[:, 1], v[:, 0])) > 0)


def test_vectors_cover_each_pair_once():
    box = float(box_size(4096, 0.8))
    nv, _ = structure_factor_vectors(box, 5.0)
    s = set(map(tuple, nv.tolist()))
    assert len(s) == nv.shape[0] and (0, 0) not in s
    assert not any((-x, -y) in s for x, y in s)                        # never both k and -k
    full = [(x, y) for x, y, _ in _brute(box, 5.0)]
    full += [(-x, -y) for x, y in full]
    assert {v for v in full if v in s or (-v[0], -v[1]) in s} == set(full)


def test_shells_are_exact_at_integer_norm():
    box = 2 * math.pi * 10                       # dk = 0.1: |k| = |n| / 10
    nv, shell = structure_factor_vectors(box, 0.65)
    d = {tuple(v): m for v, m in zip(nv.tolist(), shell.tolist())}
    assert d[(3, 4)] == 5 and d[(5, 0)] == 5 and d[(0, 5)] == 5 and d[(-4, 3)] == 5
    assert d[(4, 4)] == 5 and d[(1, 4)] == 4 and d[(6, 0)] == 6
    big = [(3 * 1000, 4 * 1000), (5000, 0), (2999, 4000)]                # exact isqrt where floats could slip
    n2 = np.array([x * x + y * y for x, y in big], dtype=np.int64)
    from jax_tpus_benchmark_physics_simulation_b200.md import _isqrt
    assert _isqrt(n2).tolist() == [math.isqrt(int(v)) for v in n2]
    sq = np.arange(0, 1 << 20, dtype=np.int64) ** 2
    assert np.array_equal(_isqrt(sq), np.arange(0, 1 << 20)) and np.array_equal(_isqrt(sq[1:] - 1), np.arange(0, (1 << 20) - 1))


def test_max_per_shell_is_deterministic_and_even():
    box = float(box_size(65536, 0.8))
    full, fshell = structure_factor_vectors(box, 2.0)
    M = 16
    a, sa = structure_factor_vectors(box, 2.0, M)
    b, sb = structure_factor_vectors(box, 2.0, M)
    assert np.array_equal(a, b) and np.array_equal(sa, sb)
    for m in np.unique(fshell):
        f = full[fshell == m]
        got = a[sa == m]
        if f.shape[0] <= M:
            assert np.array_equal(got, f)
            continue
        assert got.shape[0] == M
        L = f.shape[0]
        assert np.array_equal(got, f[(2 * np.arange(M) + 1) * L // (2 * M)])
        ang = np.arctan2(got[:, 1], got[:, 0])
        # evenly spread over [0, pi): a shell's lattice points are not quite uniform in angle, hence 3 pi / M
        assert np.diff(ang).max() < 3 * math.pi / M and ang[0] < 2 * math.pi / M and ang[-1] > math.pi - 2 * math.pi / M
    assert np.array_equal(np.unique(sa), np.unique(fshell))           # no shell lost
    assert structure_factor_vectors(box, 2.0, 10 ** 9)[0].shape == full.shape


def test_vector_arguments():
    for bad in (0.0, -1.0, float("nan"), float("inf")):
        with pytest.raises(ValueError):
            structure_factor_vectors(10.0, bad)
    with pytest.raises(ValueError):
        structure_factor_vectors(10.0, 1.0, 0)
    nv, shell = structure_factor_vectors(10.0, 0.1)                    # below the smallest |k| = 2 pi / box
    assert nv.shape == (0, 2) and shell.shape == (0,)


def test_driver_sk_flags():
    from jax_tpus_benchmark_physics_simulation_b200 import driver
    a = driver.parse_args([])
    assert a.sk_kmax is None and a.sk_per_shell is None                  # off by default
    a = driver.parse_args(["--sk_kmax", "8", "--sk_per_shell", "64"])
    assert a.sk_kmax == 8.0 and a.sk_per_shell == 64
    for bad in (["--sk_kmax", "0"], ["--sk_kmax", "-1"], ["--sk_kmax", "nan"], ["--sk_kmax", "inf"],
                ["--sk_kmax", "8", "--sk_per_shell", "0"], ["--sk_kmax", "8", "--sk_per_shell", "-3"]):
        with pytest.raises(SystemExit):
            driver.parse_args(bad)
