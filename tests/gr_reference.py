"""TEST INFRASTRUCTURE ONLY — CPU recount of the g(r) pair-distance histogram for N in the millions.

``c_gr_hist_cells`` is tests/gr_reference.c: oracle/lj_oracle.c's orc_gr_hist (the same fp32 r and binary
search against the fp32 edges) through an OpenMP cell grid with a +-2-cell stencil, optionally dropping
pairs with r > r_cap.  The C file is compiled on first use into a temporary directory (the source tree may
be read-only).  The product package never imports this module.
"""
from __future__ import annotations

import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def _build() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    cc = shutil.which("/usr/bin/gcc") or shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        raise RuntimeError("no C compiler found for tests/gr_reference.c")
    out = os.path.join(tempfile.mkdtemp(prefix="gr_reference_"), "libgr_reference.so")
    src = os.path.join(_HERE, "gr_reference.c")
    flags = ["-O2", "-fPIC", "-shared", "-std=c11", "-ffp-contract=off", "-fno-fast-math"]
    try:
        subprocess.check_call([cc, *flags, "-fopenmp", "-o", out, src, "-lm"], stderr=subprocess.DEVNULL)
    except subprocess.CalledProcessError:             # no OpenMP runtime: serial build
        subprocess.check_call([cc, *flags, "-Wno-unknown-pragmas", "-o", out, src, "-lm"])
    lib = ctypes.CDLL(out)
    f32p = ctypes.POINTER(ctypes.c_float)
    lib.gref_gr_hist.argtypes = [ctypes.c_int64, f32p, ctypes.c_float, ctypes.c_int32, f32p, ctypes.c_float,
                                 ctypes.POINTER(ctypes.c_int64)]
    lib.gref_gr_hist.restype = None
    _lib = lib
    return lib


def edges_for(r_max, nbins):
    """The fp32 edges calculate_g_r and oracle.c_gr_hist use: linspace(0, r_max, nbins + 1) (MD:110)."""
    return np.linspace(0, np.float32(r_max), nbins + 1, dtype=np.float32)


def c_gr_hist_cells(R, box, nbins, r_max, r_cap=None):
    """int64 counts (nbins,) of the pairs of one snapshot R (N, 2) with edges_for(r_max, nbins), dropping
    pairs with r > r_cap as well (r_cap None: none dropped beyond the last edge)."""
    R = np.ascontiguousarray(R, dtype=np.float32)
    edges = edges_for(r_max, nbins)
    cap = float(edges[-1]) if r_cap is None else float(np.float32(r_cap))
    counts = np.zeros(nbins, dtype=np.int64)
    _build().gref_gr_hist(R.shape[0], R.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), float(np.float32(box)),
                          nbins, edges.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), cap,
                          counts.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)))
    return counts


def adversarial(N, box, r_max, seed=0):
    """A lattice-jitter-like state of N particles in [0, box] with the placements that a cell grid of edge
    >= r_max could get wrong: particles on the fp32 grid lines fl(k box / nc) and the fp32 values next to
    them (for the nc a grid of edge r_max would use and its neighbours), pairs exactly r_max apart in fp32
    across a grid line and across the periodic edge, and coordinates 0 and box."""
    rng = np.random.default_rng(seed)
    box = np.float32(box)
    r_max = np.float32(r_max)
    R = (rng.random((N, 2), dtype=np.float32) * box).astype(np.float32)
    pts = []
    nc0 = max(1, int(float(box) // float(r_max)))
    for nc in {max(1, nc0 - 1), nc0, nc0 + 1}:
        for k in range(nc + 1):
            g = np.float32(np.float32(k) * box / np.float32(nc))
            for v in (np.nextafter(g, np.float32(-1)), g, np.nextafter(g, np.float32(2 * box))):
                v = np.float32(min(max(float(v), 0.0), float(box)))
                pts.append((v, np.float32(rng.random() * box)))
                pts.append((np.float32(rng.random() * box), v))
    # pairs exactly r_max apart along an axis, straddling a grid line, and straddling the periodic edge
    for nc in (nc0, nc0 + 1):
        g = np.float32(box / np.float32(nc))
        y = np.float32(rng.random() * box)
        a = np.float32(np.floor((g - r_max / np.float32(2)) * 1024) / 1024)    # a + r_max is exact
        pts += [(a, y), (np.float32(a + r_max), y)]
    y = np.float32(rng.random() * box)
    a = np.float32(box - r_max / np.float32(2))
    b = np.float32(a + r_max - box)
    if b >= 0:
        pts += [(a, y), (b, y)]
    pts += [(np.float32(0), np.float32(0)), (box, box), (np.float32(0), box), (box, np.float32(0)),
            (np.float32(0), y), (box, y)]
    P = np.array(pts, dtype=np.float32)[:N]
    R[:P.shape[0]] = P
    return np.clip(R, 0, box).astype(np.float32)
