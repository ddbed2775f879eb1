"""TEST INFRASTRUCTURE ONLY — reference values of the pair virial W = sum_{i<j} r_ij . f_ij.

* ``c_virial`` / ``c_virial_cells``: the fp32 C restatement of tests/virial_reference.c (pair_term's
  arithmetic of oracle/lj_oracle.c, pair terms summed in double), dense and through a CPU cell grid.
  Both return (W, sum_{i<j} |w_ij|); the second number sets the tolerance scale.  The C file is compiled
  on first use (tests/cref.py).
* ``virial_autodiff``: an independent fp64 referee, W = -d/dlambda total_energy(lambda R, lambda box) at
  lambda = 1 with torch autodiff on oracle/lj_oracle.py's restatement of total_energy_fn.

The product package never imports this module.
"""
from __future__ import annotations

import ctypes
import math

import numpy as np
import torch

import cref

def _lib():
    f32p, f64p = ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_double)
    args = [ctypes.c_int64, f32p, ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_float, f64p, f64p]
    return cref.load("virial_reference", {"vref_virial": (args, None), "vref_virial_cells": (args, None)})


def _rc2(rc):
    if rc is None or not math.isfinite(rc) or rc <= 0:
        return float("inf")
    return float(np.float32(rc) * np.float32(rc))


def _call(fn, R, box, last, sigma, epsilon):
    R = np.ascontiguousarray(R, dtype=np.float32)
    w, wa = ctypes.c_double(0.0), ctypes.c_double(0.0)
    fn(R.shape[0], R.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), float(box), sigma, epsilon, last,
       ctypes.byref(w), ctypes.byref(wa))
    return w.value, wa.value


def c_virial(R, box, rc=None, sigma=1.0, epsilon=1.0):
    """Dense fp32 restatement of the pair virial.  Returns (W, sum_{i<j} |w_ij|)."""
    return _call(_lib().vref_virial, R, box, _rc2(rc), sigma, epsilon)


def c_virial_cells(R, box, rc, sigma=1.0, epsilon=1.0):
    """c_virial through a CPU cell grid (needs a finite rc), for N in the millions."""
    return _call(_lib().vref_virial_cells, R, box, float(rc), sigma, epsilon)


def virial_autodiff(R, box, sigma=1.0, epsilon=1.0, rc=None) -> float:
    """W = -d/dlambda total_energy(lambda R, lambda box) at lambda = 1, in float64.  Scaling positions and
    box together scales every minimum-image displacement by lambda (round() has zero gradient) and the
    cutoff indicator has none, so this is sum_{i<j} r_ij . f_ij of the truncated pair potential."""
    from oracle.lj_oracle import total_energy
    R64 = torch.as_tensor(np.asarray(R, dtype=np.float64))
    lam = torch.ones((), dtype=torch.float64, requires_grad=True)
    box64 = torch.as_tensor(float(box), dtype=torch.float64)
    E = total_energy(lam * R64, lam * box64, sigma, epsilon, rc)
    (g,) = torch.autograd.grad(E, lam)
    return -float(g)
