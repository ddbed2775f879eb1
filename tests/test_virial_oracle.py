"""CPU checks of the pair-virial references (tests/virial_reference.py): known answers, the fp32 C
restatement against the fp64 autodiff referee W = -dE(lambda R, lambda box)/dlambda, and the cell-grid
variant against the dense one."""
import numpy as np
import pytest

from jax_tpus_benchmark_physics_simulation_b200 import lattice_jitter

import virial_reference as vref   # tests/virial_reference.py


def _w_exact(r):
    return 24.0 * (2.0 * r ** -12 - r ** -6)


@pytest.mark.parametrize("r", [1.0, 2.0 ** (1.0 / 6.0), 1.5])
@pytest.mark.parametrize("x0", [3.0, 9.6])          # the second pair straddles the periodic seam x = box
def test_two_particles_known_answer(oracle, r, x0):
    box = np.float32(10.0)
    R = np.array([[x0, 5.0], [np.float32((x0 + r) % 10.0), 5.0]], dtype=np.float32)
    rr = float(np.float32(R[1, 0]) - np.float32(R[0, 0]))
    rr = abs(rr - 10.0 * round(rr / 10.0))
    w, wabs = vref.c_virial(R, box, rc=None)
    ref = _w_exact(rr)
    assert abs(w - ref) <= 1e-5 * max(1.0, abs(ref))
    assert wabs == pytest.approx(abs(w), abs=1e-12)
    # (fp64 minimum image of the fp32 positions: r differs from rr in the last fp32 bits, and dW/dr ~ 60)
    assert abs(vref.virial_autodiff(R, box, rc=None) - ref) <= 1e-4 * max(1.0, abs(ref))


def test_zero_at_force_minimum(oracle):
    """At r = 2^(1/6) sigma the force, and so the virial, vanishes."""
    r = np.float32(2.0 ** (1.0 / 6.0))
    R = np.array([[1.0, 1.0], [1.0 + r, 1.0]], dtype=np.float32)
    w, _ = vref.c_virial(R, np.float32(10.0))
    assert abs(w) <= 1e-5
    assert abs(vref.virial_autodiff(R, np.float32(10.0))) <= 1e-5


def test_cutoff_excludes_pair(oracle):
    R = np.array([[1.0, 1.0], [3.0, 1.0]], dtype=np.float32)
    assert vref.c_virial(R, np.float32(10.0), rc=1.5) == (0.0, 0.0)
    assert vref.virial_autodiff(R, np.float32(10.0), rc=1.5) == 0.0


@pytest.mark.parametrize("N", [400, 1024])
@pytest.mark.parametrize("rc", [None, 2.5])
@pytest.mark.parametrize("seed", [0, 1])
def test_c_virial_vs_autodiff(oracle, N, rc, seed):
    R, _, box = lattice_jitter(N, seed=seed)
    w, wabs = vref.c_virial(R, box, rc=rc)
    wd = vref.virial_autodiff(R, box, rc=rc)
    assert abs(w - wd) <= 1e-6 * wabs


@pytest.mark.parametrize("N,seed", [(16384, 0), (65536, 1)])
def test_cell_grid_matches_dense(oracle, N, seed):
    R, _, box = lattice_jitter(N, seed=seed)
    w, wabs = vref.c_virial(R, box, rc=2.5)
    wc, wabsc = vref.c_virial_cells(R, box, 2.5)
    assert abs(w - wc) <= 1e-9 * wabs
    assert abs(wabs - wabsc) <= 1e-9 * wabs
