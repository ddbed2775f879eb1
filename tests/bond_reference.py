"""TEST INFRASTRUCTURE ONLY — fp64 CPU restatement of the bond-orientational order psi_m (ljmd_bond_order) and of
its pair-correlation histogram (ljmd_bond_corr), with the library's neighbour and fixed-point rules.

``bond_order`` and ``bond_corr`` call tests/bond_reference.c, compiled on first use (tests/cref.py).  The product
package never imports this module.
"""
from __future__ import annotations

import ctypes

import numpy as np

import cref
from gr_reference import edges_for

def _lib():
    vp, i64, i32, f32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_float
    return cref.load("bond_reference", {"bref_bond_order": ([i64, vp, f32, i32, f32, vp, vp], None),
                                        "bref_bond_corr": ([i64, vp, vp, f32, i32, vp, f32, vp, vp], None)})


def bond_order(R, box, m, r_nb):
    """(psi (N, 2) float64, n (N,) int32) of one snapshot R (N, 2)."""
    R = np.ascontiguousarray(R, dtype=np.float32)
    N = R.shape[0]
    psi = np.zeros((N, 2), np.float64)
    nnb = np.zeros(N, np.int32)
    _lib().bref_bond_order(N, R.ctypes.data, float(np.float32(box)), int(m), float(np.float32(r_nb)),
                           psi.ctypes.data, nnb.ctypes.data)
    return psi, nnb


def bond_corr(R, psi, box, nbins, r_max, r_cap=None):
    """(counts, wsum) int64 (nbins,) of one snapshot with edges_for(r_max, nbins) and pairs up to r_cap (default:
    the last edge), as ljmd_bond_corr."""
    R = np.ascontiguousarray(R, dtype=np.float32)
    psi = np.ascontiguousarray(psi, dtype=np.float64)
    edges = edges_for(r_max, nbins)
    cap = float(edges[-1]) if r_cap is None else float(np.float32(r_cap))
    counts = np.zeros(nbins, np.int64)
    wsum = np.zeros(nbins, np.int64)
    _lib().bref_bond_corr(R.shape[0], R.ctypes.data, psi.ctypes.data, float(np.float32(box)), nbins,
                          edges.ctypes.data, cap, counts.ctypes.data, wsum.ctypes.data)
    return counts, wsum


def g_m(counts, wsum):
    """g_m(r) = wsum / (2^24 counts), NaN where the count is 0 (as LJSimulation.bond_correlation)."""
    c = np.asarray(counts, np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        return np.where(c > 0, np.asarray(wsum, np.float64) / (c * 2.0 ** 24), np.nan)


def square_lattice(n, a=1.0):
    """n x n square lattice of spacing a (exact in fp32 for a = 1) in the box n a."""
    i, j = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    R = (np.stack([i.ravel(), j.ravel()], axis=1) * a).astype(np.float32)
    return R, np.float32(n * a)


def triangular_lattice(nx, ny, a=1.0):
    """nx x ny triangular lattice (ny even) of spacing a, its rows squeezed so that ny rows fill the square box
    nx a exactly; the strain is |ny sqrt(3) / 2 / nx - 1|."""
    box = nx * a
    hy = box / ny                                     # row spacing, about a sqrt(3) / 2
    i, j = np.meshgrid(np.arange(nx), np.arange(ny), indexing="ij")
    x = (i + 0.5 * (j % 2) + 0.25) * a
    y = (j + 0.5) * hy
    return np.stack([x.ravel(), y.ravel()], axis=1).astype(np.float32), np.float32(box)
