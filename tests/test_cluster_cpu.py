"""The CPU restatement of the cluster analysis (tests/cluster_reference.{c,py}) against answers known in advance:
lattices below and above their spacing, separated blobs, a strip joined only through the periodic edge, the
x <-> y mirror, and a plain Python union-find over all pairs."""
import numpy as np
import pytest

import cluster_reference as ref
from bond_reference import square_lattice


def _check_convention(labels, sizes, act):
    assert np.array_equal(labels < 0, ~act)
    on = labels[act]
    assert np.array_equal(labels[on], on)                        # every label is its own cluster's label
    assert np.all(on <= np.nonzero(act)[0])                      # ... and the smallest index in it
    assert sizes.sum() == act.sum()
    assert np.array_equal(np.nonzero(sizes)[0], np.unique(on))


@pytest.mark.parametrize("n", [4, 16, 80])                        # 4: every pair; 16, 80: the grid
def test_square_lattice(n):
    R, box = square_lattice(n)
    labels, sizes = ref.clusters(R, box, 0.9)
    assert np.array_equal(labels, np.arange(n * n)) and np.array_equal(sizes, np.ones(n * n))
    labels, sizes = ref.clusters(R, box, 1.1)
    assert np.array_equal(labels, np.zeros(n * n)) and sizes[0] == n * n and sizes[1:].sum() == 0
    assert len(ref.links(R, box, 1.0)) == 2 * n * n               # r == r_link is a link
    assert len(ref.links(R, box, np.nextafter(np.float32(1.0), np.float32(0)))) == 0


def test_two_blobs():
    rng = np.random.default_rng(0)
    box = np.float32(40.0)
    a = rng.uniform(5, 8, (60, 2))
    b = rng.uniform(25, 28, (70, 2))
    R = np.concatenate([a, b]).astype(np.float32)
    perm = rng.permutation(R.shape[0])
    R = R[perm]
    labels, sizes = ref.clusters(R, box, 1.5)
    assert sorted(sizes[sizes > 0].tolist()) == [60, 70]
    blob_a = perm < 60
    assert np.unique(labels[blob_a]).size == 1 and labels[blob_a][0] == np.nonzero(blob_a)[0][0]
    _check_convention(labels, sizes, np.ones(R.shape[0], bool))


def test_strip_joined_through_the_periodic_edge():
    box = np.float32(20.0)
    xs = np.arange(0.5, 20.0, 1.0, dtype=np.float32)                # 0.5 .. 19.5: the edge gap is 1.0
    R = np.stack([xs, np.full_like(xs, 7.0)], axis=1)
    labels, _ = ref.clusters(R, box, 1.0)
    assert np.all(labels == 0)
    cut = R[(xs < 9) | (xs > 10)]                                   # remove 9.5: still one through the edge
    labels, sizes = ref.clusters(cut, box, 1.0)
    assert np.all(labels == 0) and sizes[0] == cut.shape[0]
    labels, sizes = ref.clusters(cut, box, 0.99)
    assert sizes[sizes > 0].size == cut.shape[0]


def test_mirror_invariance_and_mask():
    rng = np.random.default_rng(1)
    N, box = 3000, np.float32(60.0)
    R = (rng.random((N, 2)) * box).astype(np.float32)
    for r_link in (0.8, 1.2, 2.0):
        la, sa = ref.clusters(R, box, r_link)
        lb, sb = ref.clusters(R[:, ::-1], box, r_link)
        assert np.array_equal(la, lb) and np.array_equal(sa, sb)
        _check_convention(la, sa, np.ones(N, bool))
    mask = rng.random(N) < 0.6
    lm, sm = ref.clusters(R, box, 1.2, mask)
    _check_convention(lm, sm, mask)
    sub, _ = ref.clusters(R[mask], box, 1.2)                        # the same graph on the active particles
    idx = np.nonzero(mask)[0]
    assert np.array_equal(lm[mask], idx[sub])


def test_nan_particle_is_inactive():
    R, box = square_lattice(12)
    R = R.copy()
    R[5] = (np.nan, 3.0)
    labels, sizes = ref.clusters(R, box, 1.1)
    assert labels[5] == -1 and sizes.sum() == R.shape[0] - 1


@pytest.mark.parametrize("seed,r_link", [(0, 1.0), (1, 1.6), (2, 2.5)])
def test_dilute_random_matches_brute_force(seed, r_link):
    rng = np.random.default_rng(seed)
    N, box = 300, np.float32(30.0)
    R = (rng.random((N, 2)) * box).astype(np.float32)
    labels, sizes = ref.clusters(R, box, r_link)
    lb, sb = ref.brute_force(R, box, r_link)
    assert np.array_equal(labels, lb) and np.array_equal(sizes, sb)
