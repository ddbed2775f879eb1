"""The ragged-N inputs and the float64 per-particle force reference (tests/ragged_reference.py): shape and spacing of
the inputs, agreement with the C oracle, and the power of the per-particle criterion that the GPU tests
(tests/test_ragged_gpu.py) apply: a dropped pair, a doubled pair and a zeroed partial block must all fail it."""
import numpy as np
import pytest

from ragged_reference import (check_forces, check_rows, forces_f64, lj_force, pair_forces,
                              ragged_lattice)

TOL = 1e-5                              # the GPU files' per-particle tolerance (in units of S_i)
GPU_N = [2, 3, 17, 31, 33, 58, 75, 99, 401, 639, 641, 1021, 1025, 2047, 2049, 4097, 5003, 16385, 33331, 70001]


@pytest.mark.parametrize("N", [2, 3, 17, 1021, 5003])
def test_ragged_lattice_shape_range_and_seed(N):
    R, V, box = ragged_lattice(N, seed=3)
    assert R.shape == V.shape == (N, 2) and R.dtype == V.dtype == np.float32 and box.dtype == np.float32
    assert R.min() >= 0.0 and R.max() <= box
    R2, V2, _ = ragged_lattice(N, seed=3)
    assert np.array_equal(R, R2) and np.array_equal(V, V2)
    R3, _, _ = ragged_lattice(N, seed=4)
    assert not np.array_equal(R, R3)
    if N >= 1000:                       # the index tail is spread over the box, not packed into its last rows
        tail = R[-N // 8:]
        assert (tail.max(axis=0) - tail.min(axis=0)).min() > 0.8 * float(box)


def test_ragged_lattice_min_distance(oracle):
    """No pair closer than 0.7 sigma (minimum image) in any input of the GPU tests."""
    for N in GPU_N:
        R, _, box = ragged_lattice(N)
        assert oracle.c_neighbor_count(R, box, 0.7).max() == 0, N


@pytest.mark.parametrize("N,rc", [(3, 2.5), (33, None), (639, None), (639, 2.5), (2049, 2.5), (2049, None)])
def test_reference_matches_c_oracle(oracle, N, rc):
    R, _, box = ragged_lattice(N)
    F, S, pe = forces_f64(R, box, rc=rc)
    Fc, pe_c = oracle.c_forces(R, box, rc=rc)
    ok, worst, i = check_forces(Fc, F, S, 2e-6)
    assert ok, (worst, i)
    if N >= 600:                        # one fp32 pair energy alone is only good to ~1e-7
        assert abs(pe - pe_c) <= 1e-8 * abs(pe)
    # the row form gives the same rows
    Fr, Sr, _ = forces_f64(R, box, rc=rc, rows=(N // 3, N))
    assert np.array_equal(Fr, F[N // 3:]) and np.array_equal(Sr, S[N // 3:])


def test_reference_rows_at_large_n(oracle):
    N = 33331
    R, _, box = ragged_lattice(N)
    for lo, hi in check_rows(N):
        F, S, _ = forces_f64(R, box, rc=2.5, rows=(lo, hi))
        Fc, _ = oracle.c_forces(R, box, rc=2.5, rows=(lo, hi))
        ok, worst, i = check_forces(Fc, F, S, 2e-6)
        assert ok, (lo, worst, i)
    assert check_rows(N)[-1] == (N - 256, N)


def _weakest_pair(R, box, rc, S, i):
    """Partner j and F_ij of the in-cutoff pair of i with the smallest |F_ij| outside the band 10 tol S_i around
    the zero of the force (a pair there is within the criterion's resolution)."""
    j, f = pair_forces(R, box, i, rc=rc)
    mag = np.abs(f).max(axis=1)
    ok = mag >= 10 * TOL * S[i]
    k = np.flatnonzero(ok)[np.argmin(mag[ok])]
    return int(j[k]), f[k]


@pytest.mark.parametrize("N,rc", [(2, 2.5), (17, 2.5), (639, 2.5), (1021, None), (2049, 2.5), (5003, 2.5)])
def test_criterion_rejects_wrong_pair_sets(N, rc):
    R, _, box = ragged_lattice(N)
    F, S, _ = forces_f64(R, box, rc=rc)
    assert check_forces(F, F, S, TOL)[0]
    i = N - 1
    j, fij = _weakest_pair(R, box, rc, S, i)
    dropped = F.copy()
    dropped[i] -= fij
    dropped[j] += fij
    assert not check_forces(dropped, F, S, TOL)[0], "a dropped pair passes"
    doubled = F.copy()
    doubled[i] += fij
    doubled[j] -= fij
    assert not check_forces(doubled, F, S, TOL)[0], "a doubled pair passes"
    if N % 64:
        zeroed = F.copy()
        zeroed[N - N % 64:] = 0.0
        assert not check_forces(zeroed, F, S, TOL)[0], "a zeroed partial 64-block passes"


def test_criterion_resolves_a_pair_at_the_cutoff():
    """TOL * S_i below the force of one pair at rc = 2.5 for every input of the GPU tests (the large N on the row
    blocks those tests check), so no in-cutoff pair can hide inside the tolerance."""
    f_rc = lj_force(2.5)
    for N in GPU_N:
        R, _, box = ragged_lattice(N)
        rows = check_rows(N) if N > 20000 else [None]
        smax = max(forces_f64(R, box, rc=2.5, rows=r)[1].max() for r in rows)
        assert TOL * smax < f_rc, (N, smax)
