"""TEST INFRASTRUCTURE ONLY — fp64 CPU reference of the density modes rho_k and the accuracy bound of the GPU
kernel (csrc/sk.cu, ljmd_density_modes).

``c_density_modes`` is tests/sk_reference.c: the direct sum of exp(i k.r_j) in double over the fp32 positions,
OpenMP over the wave vectors.  The C file is compiled on first use into a temporary directory (the source tree
may be read-only).  The product package never imports this module.
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

U32 = 2.0 ** -24              # fp32 unit roundoff
SK_CHUNK = 32                 # particles per fp32 partial sum in csrc/sk.cu


def _build() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    cc = shutil.which("/usr/bin/gcc") or shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        raise RuntimeError("no C compiler found for tests/sk_reference.c")
    out = os.path.join(tempfile.mkdtemp(prefix="sk_reference_"), "libsk_reference.so")
    src = os.path.join(_HERE, "sk_reference.c")
    flags = ["-O2", "-fPIC", "-shared", "-std=c11", "-ffp-contract=off", "-fno-fast-math"]
    try:
        subprocess.check_call([cc, *flags, "-fopenmp", "-o", out, src, "-lm"], stderr=subprocess.DEVNULL)
    except subprocess.CalledProcessError:             # no OpenMP runtime: serial build
        subprocess.check_call([cc, *flags, "-Wno-unknown-pragmas", "-o", out, src, "-lm"])
    lib = ctypes.CDLL(out)
    lib.skref_modes.argtypes = [ctypes.c_int64, ctypes.POINTER(ctypes.c_float), ctypes.c_double, ctypes.c_int64,
                                ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_double)]
    lib.skref_modes.restype = None
    _lib = lib
    return lib


def c_density_modes(R, box, nvec):
    """float64 (S, K, 2) = (Re, Im) of rho_k for the snapshots R ((N, 2) or (S, N, 2) float32) and the integer
    vectors nvec (K, 2), with k = (2 pi / box) n and box taken as its float32 value."""
    R = np.asarray(R, dtype=np.float32)
    R = np.ascontiguousarray(R[None] if R.ndim == 2 else R)
    nv = np.ascontiguousarray(np.asarray(nvec, dtype=np.int32).reshape(-1, 2))
    out = np.zeros((R.shape[0], nv.shape[0], 2), dtype=np.float64)
    lib = _build()
    for s in range(R.shape[0]):
        lib.skref_modes(R.shape[1], R[s].ctypes.data_as(ctypes.POINTER(ctypes.c_float)), float(np.float32(box)),
                        nv.shape[0], nv.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)),
                        out[s].ctypes.data_as(ctypes.POINTER(ctypes.c_double)))
    return out


def eps_term(nvec):
    """Per-term error bound of one component (cos or sin) of the GPU kernel, per vector (K,): phase words
    (|n_x| + |n_y|) pi 2^-32, I2FP pi 2^-25, the fp32 angle multiply pi 2^-24 + 2^-23, MUFU sin/cos 2^-20.5."""
    n1 = np.abs(np.asarray(nvec, dtype=np.float64).reshape(-1, 2)).sum(axis=1)
    return n1 * np.pi * 2.0 ** -32 + np.pi * (2.0 ** -25 + 2.0 ** -24) + 2.0 ** -23 + 2.0 ** -20.5


def bound(N, nvec):
    """|rho_k(GPU) - rho_k(exact)| bound of each component, per vector (K,) (csrc/sk.cu)."""
    acc = U32 * (SK_CHUNK + 1) / 2
    return N * (eps_term(nvec) + acc) + (N / SK_CHUNK + 1024) * N * 2.0 ** -53
