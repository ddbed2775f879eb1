"""The CPU restatement of the bond-orientational order (tests/bond_reference.c) against analytic answers: the
square lattice (psi_4, psi_6 and the neighbour counts at two radii), a triangular lattice (psi_6 and g_6) and the
x <-> y mirror, which maps psi_m to i^m conj(psi_m)."""
import numpy as np
import pytest

from bond_reference import bond_corr, bond_order, g_m, square_lattice, triangular_lattice


@pytest.mark.parametrize("n", [16, 17])
def test_square_lattice_first_shell(n):
    R, box = square_lattice(n)
    psi4, n4 = bond_order(R, box, 4, 1.2)
    psi6, n6 = bond_order(R, box, 6, 1.2)
    assert (n4 == 4).all() and (n6 == 4).all()
    assert (psi4[:, 0] == 1.0).all() and (psi4[:, 1] == 0.0).all()
    assert (psi6 == 0.0).all()


def test_square_lattice_second_shell():
    R, box = square_lattice(16)
    psi4, n = bond_order(R, box, 4, 1.5)
    assert (n == 8).all()
    assert np.abs(psi4).max() < 1e-12                     # 4 axis bonds (+1) and 4 diagonal ones (-1)


def test_triangular_lattice_psi6_and_g6():
    R, box = triangular_lattice(26, 30)
    assert abs(30 * np.sqrt(3) / 2 / 26 - 1) < 1e-3    # strained by under 0.1 % to fit the square box
    psi, n = bond_order(R, box, 6, 1.2)
    assert (n == 6).all()
    assert np.hypot(psi[:, 0], psi[:, 1]).min() > 0.99
    counts, wsum = bond_corr(R, psi, box, 100, 5.0)
    g = g_m(counts, wsum)
    assert counts.sum() > 0 and (g[counts > 0] > 0.98).all() and np.isnan(g[counts == 0]).all()


@pytest.mark.parametrize("m", [1, 4, 5, 6, 12])
def test_mirror_x_y(m):
    rng = np.random.default_rng(m)
    R, box = square_lattice(32)
    R = (R + np.float32(0.5) + rng.uniform(-0.15, 0.15, R.shape)).astype(np.float32)
    psi, n = bond_order(R, box, m, 1.5)
    psi_s, n_s = bond_order(R[:, ::-1], box, m, 1.5)
    assert np.array_equal(n, n_s) and n.min() > 0
    z = (psi[:, 0] + 1j * psi[:, 1])
    zs = psi_s[:, 0] + 1j * psi_s[:, 1]
    assert np.abs(zs - (1j ** m) * np.conj(z)).max() < 1e-12


def test_nan_particle_and_isolated_particle():
    R, box = square_lattice(16)
    R = R.copy()
    R[5] = (np.nan, 3.0)
    R[100, 0] = np.inf
    psi, n = bond_order(R, box, 6, 1.2)
    assert np.isnan(psi[[5, 100]]).all() and (n[[5, 100]] == 0).all()
    assert np.isfinite(np.delete(psi, [5, 100], axis=0)).all()
    # the lattice neighbours of the two lost particles have one bond fewer
    assert (n == 4).sum() == R.shape[0] - 2 - 8 and (n == 3).sum() == 8
    psi, n = bond_order(R, box, 6, 0.5)                   # nobody within r_nb: psi = 0
    assert (n == 0).all() and (psi[np.isfinite(psi[:, 0])] == 0.0).all()
