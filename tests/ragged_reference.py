"""TEST INFRASTRUCTURE ONLY — inputs at any particle count and a float64 per-particle force reference.

* ``ragged_lattice``: a jittered square lattice with N of its sites kept, for any N >= 2.  ``ic.lattice_jitter``
  needs a perfect square; the kernels pad particles that do not fill their tiles (64-particle blocks, 8-particle
  j units, 32-slot cell-list units, cluster CTAs), and only counts that are not multiples of those sizes reach the
  padding.  The kept sites are in a seeded random order, so the index tail (the padded tiles) is spread over space.
* ``forces_f64``: forces, per-particle force scale S_i = sum_j |F_ij| and PE.  The pair set is decided exactly as
  the kernels and oracle/lj_oracle.c decide it (fp32 displacement, fp32 minimum image, unfused fp32 r^2 against
  fl32(rc * rc), i != j); the pair terms and the sums are float64 from those fp32 displacements.
* ``check_forces``: the worst |F_i - F_ref,i|_inf / S_i.  At tol = 1e-5 a dropped or doubled in-cutoff pair fails it
  for every particle (1e-5 S_i stays below |F(2.5)| = 0.039), including particles whose net force is small.

The product package never imports this module.
"""
from __future__ import annotations

import math

import numpy as np

from jax_tpus_benchmark_physics_simulation_b200.ic import box_size

ROW_BLOCK = 256                         # rows of one block of check_rows


def ragged_lattice(N: int, rho: float = 0.8, seed: int = 0, jitter: float = 0.05, kT: float = 1.0):
    """N sites of the n x n lattice (n = ceil(sqrt(N)), spacing a = box / n) chosen by a seeded permutation and kept
    in that order, positions (i + 1/2, j + 1/2) a + U(-jitter, jitter) a clipped to [0, box], velocities
    N(0, 1) sqrt(kT).  Generated in float64 and cast once to float32.  Returns (R (N, 2), V (N, 2), box) as
    ``ic.lattice_jitter``."""
    N = int(N)
    if N < 2:
        raise ValueError(f"ragged_lattice needs N >= 2, got {N}")
    n = math.isqrt(N - 1) + 1
    box = box_size(N, rho)
    a = float(box) / n
    rng = np.random.default_rng(seed)
    site = rng.permutation(n * n)[:N]
    R = np.stack([(site // n + 0.5) * a, (site % n + 0.5) * a], axis=1)
    R = R + rng.uniform(-jitter, jitter, size=(N, 2)) * a
    V = rng.standard_normal((N, 2)) * np.sqrt(kT)
    R32 = R.astype(np.float32)
    np.clip(R32, np.float32(0.0), box, out=R32)
    return R32, V.astype(np.float32), box


def _rc2(rc) -> np.float32:
    if rc is None or not math.isfinite(rc) or rc <= 0:
        return np.float32(np.inf)
    return np.float32(rc) * np.float32(rc)


def _pairs(R, box, rc, i0, i1):
    """Displacements (float64 of the fp32 values) and the pair mask of rows [i0, i1) against all j."""
    box = np.float32(box)
    d = R[i0:i1, None, :] - R[None, :, :]                               # fp32
    d = d - box * np.round(d / box)                                     # fp32 minimum image, half-to-even
    r2 = d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]                  # fp32, unfused
    mask = r2 < _rc2(rc)
    mask[np.arange(i1 - i0), np.arange(i0, i1)] = False
    return d.astype(np.float64), mask


def _terms(d, mask):
    """Pair force factor f (F_ij = f d_ij) and pair energy, float64, zero outside the mask."""
    r2 = np.where(mask, d[..., 0] ** 2 + d[..., 1] ** 2, 1.0)
    s2 = 1.0 / r2
    s6 = s2 * s2 * s2
    f = np.where(mask, 24.0 * (2.0 * s6 * s6 - s6) * s2, 0.0)
    e = np.where(mask, 4.0 * (s6 * s6 - s6), 0.0)
    return f, e, np.sqrt(r2)


def forces_f64(R, box, rc=None, rows=None):
    """(F, S, pe) of rows [i0, i1) (``rows`` = (i0, i1), default all): F (n, 2) and S (n,) float64 with
    S_i = sum_j |F_ij|, pe = 1/2 sum of the pair energies of those rows (the total PE when rows is None)."""
    R = np.ascontiguousarray(R, dtype=np.float32)
    N = R.shape[0]
    i0, i1 = (0, N) if rows is None else (int(rows[0]), int(rows[1]))
    F = np.zeros((i1 - i0, 2))
    S = np.zeros(i1 - i0)
    pe = 0.0
    chunk = max(1, (1 << 22) // N)
    for a in range(i0, i1, chunk):
        b = min(i1, a + chunk)
        d, mask = _pairs(R, box, rc, a, b)
        f, e, r = _terms(d, mask)
        F[a - i0:b - i0] = np.einsum("ij,ijk->ik", f, d)
        S[a - i0:b - i0] = np.sum(np.abs(f) * r, axis=1)
        pe += float(np.sum(e))
    return F, S, 0.5 * pe


def pair_forces(R, box, i, rc=None):
    """The in-cutoff partners j of particle i and the pair forces F_ij (k, 2) on i, float64."""
    R = np.ascontiguousarray(R, dtype=np.float32)
    d, mask = _pairs(R, box, rc, i, i + 1)
    f, _, _ = _terms(d, mask)
    j = np.flatnonzero(mask[0])
    return j, f[0, j, None] * d[0, j]


def check_forces(F, F_ref, S, tol):
    """(ok, worst, i): worst = max_i |F_i - F_ref,i|_inf / S_i at particle i, ok = worst <= tol."""
    err = np.abs(np.asarray(F, dtype=np.float64) - F_ref).max(axis=1)
    ratio = np.divide(err, S, out=np.where(err > 0, np.inf, 0.0), where=S > 0)
    i = int(np.argmax(ratio))
    return bool(ratio[i] <= tol), float(ratio[i]), i


def check_rows(N: int, nblocks: int = 4, seed: int = 0):
    """nblocks disjoint row ranges of ROW_BLOCK rows for the large-N checks: the last is [N - ROW_BLOCK, N),
    the others are seeded and in [0, N - ROW_BLOCK)."""
    rng = np.random.default_rng(seed)
    starts = rng.choice((N - ROW_BLOCK) // ROW_BLOCK, size=nblocks - 1, replace=False) * ROW_BLOCK
    return [(int(s), int(s) + ROW_BLOCK) for s in sorted(starts)] + [(N - ROW_BLOCK, N)]


def lj_force(r: float) -> float:
    """|F(r)| of the Lennard-Jones pair (sigma = epsilon = 1)."""
    return abs(24.0 * (2.0 * r ** -13 - r ** -7))
