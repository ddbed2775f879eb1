"""CPU checks of the cell-grid g(r) recount (tests/gr_reference.c) that the GPU tests of the cell-grid
histogram compare against: bit for bit equal to oracle/lj_oracle.c's dense orc_gr_hist.  Also the driver's
--gr_rmax flag."""
import numpy as np
import pytest

from gr_reference import adversarial, c_gr_hist_cells, edges_for
from jax_tpus_benchmark_physics_simulation_b200.ic import lattice_jitter


def _dense_capped(R, box, nbins, r_max, r_cap):
    """fp32 numpy restatement: every pair i < j, r <= min(edges[-1], r_cap), bins against the fp32 edges."""
    R = np.asarray(R, dtype=np.float32)
    box = np.float32(box)
    i, j = np.triu_indices(R.shape[0], k=1)
    d = R[i] - R[j]
    d = d - box * np.rint(d / box)
    r = np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1])
    e = edges_for(r_max, nbins)
    r = r[(r >= e[0]) & (r <= min(e[-1], np.float32(r_cap)))]
    b = np.minimum(np.searchsorted(e, r, side="right") - 1, nbins - 1)
    return np.bincount(b, minlength=nbins).astype(np.int64)


@pytest.mark.parametrize("N", [400, 4096])
def test_cell_recount_matches_dense_oracle(oracle, N):
    R, _, box = lattice_jitter(N, seed=3)
    box = float(box)
    for r_max in (2.5, 5.0, box / 3 * (1 - 1e-6), box / 5 * 1.0001, box / 2):
        nbins = max(1, int(np.float32(r_max) / 0.05))
        for X in (R, adversarial(N, box, r_max, seed=N)):
            assert np.array_equal(c_gr_hist_cells(X, box, nbins, r_max), oracle.c_gr_hist(X, box, nbins, r_max))


def test_cell_recount_cap_drops_longer_pairs(oracle):
    N = 400
    R, _, box = lattice_jitter(N, seed=5)
    X = adversarial(N, float(box), 2.5, seed=1)
    for r_max, cap in ((5.0, 2.5), (5.0, 3.3), (float(box) / 2, 2.5), (2.5, 100.0)):
        got = c_gr_hist_cells(X, box, 100, r_max, r_cap=cap)
        assert np.array_equal(got, _dense_capped(X, box, 100, r_max, cap))
    # the cap at the last edge changes nothing
    assert np.array_equal(c_gr_hist_cells(X, box, 100, 5.0, r_cap=5.0), oracle.c_gr_hist(X, box, 100, 5.0))


def test_adversarial_state_has_the_placements():
    box, r_max = 71.55, 5.0
    X = adversarial(4096, box, r_max)
    assert X.dtype == np.float32 and X.min() == 0.0 and X.max() == np.float32(box)
    d = np.abs(X[:, None, 0] - X[None, :, 0])[np.abs(X[:, None, 1] - X[None, :, 1]) == 0]
    assert (d == np.float32(r_max)).any()            # a pair exactly r_max apart in fp32


def test_driver_gr_rmax_flag():
    from jax_tpus_benchmark_physics_simulation_b200 import driver
    assert driver.parse_args([]).gr_rmax is None                       # default: box/2, as the reference
    assert driver.parse_args(["--gr_rmax", "5"]).gr_rmax == 5.0
    for bad in ("0", "-1", "nan", "inf"):
        with pytest.raises(SystemExit):
            driver.parse_args(["--gr_rmax", bad])
