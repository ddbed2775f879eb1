"""ctypes binding of the C ABI declared in include/ljmd.h (the drop-in boundary).

This is the stub a maintainer of the reference script would add (INTEGRATION.md).  There is
no fallback: if ``libljmd.so`` has not been built (``python -c "import __graft_entry__ as g;
g.build()"``) or no sm_100a GPU is present, calls fail loudly.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LJMD_LIB", os.path.join(_HERE, "libljmd.so"))   # LJMD_LIB: developer override

LJMD_PATH_AUTO, LJMD_PATH_ALLPAIRS, LJMD_PATH_CELLS = 0, 1, 2
LJMD_E_OVERFLOW, LJMD_E_TIMEOUT = -6, -7
LJMD_LAW_GRAVITY_NBODY, LJMD_LAW_GRAVITY_EM3 = 0, 1

# every symbol include/ljmd.h declares (checked by tests/test_abi.py)
EXPORTS = (
    "ljmd_abi_version", "ljmd_last_error", "ljmd_create", "ljmd_destroy", "ljmd_energy",
    "ljmd_forces", "ljmd_run", "ljmd_gr_hist", "ljmd_cell_geometry", "ljmd_cell_assign",
    "ljmd_neighbor_count", "ljmd_last_rebuilds", "ljmd_get_unique_id", "ljmd_create_dist",
    "ljmd_last_run_ms", "ljmd_launch_count", "ljmd_fp32_peak_probe", "ljmd_allpairs_mode",
    "ljmd_check", "ljmd_pair_accel", "ljmd_run_blocked", "ljmd_virial", "ljmd_run_virial",
)


class LjmdParams(ctypes.Structure):
    """struct ljmd_params (include/ljmd.h)."""
    _fields_ = [
        ("N", ctypes.c_int64),
        ("box", ctypes.c_float),
        ("sigma", ctypes.c_float),
        ("epsilon", ctypes.c_float),
        ("rc", ctypes.c_float),
        ("dt", ctypes.c_float),
        ("skin", ctypes.c_float),
        ("path", ctypes.c_int32),
        ("device", ctypes.c_int32),
        ("stream", ctypes.c_void_p),
    ]


class LjmdError(RuntimeError):
    """A call of the C ABI failed; ``code`` is its return value (LJMD_E_* / cudaError_t)."""

    def __init__(self, msg, code=None):
        super().__init__(msg)
        self.code = code


_lib = None


def load() -> ctypes.CDLL:
    """Load libljmd.so and declare the prototypes.  Raises if the library is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise LjmdError(
            f"{LIB_PATH} not found: build the CUDA extension first "
            "(python -c 'import __graft_entry__ as g; g.build()').  There is no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    vp, i64, i32, f32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_float
    lib.ljmd_abi_version.restype = ctypes.c_int
    lib.ljmd_abi_version.argtypes = []
    lib.ljmd_last_error.restype = ctypes.c_char_p
    lib.ljmd_last_error.argtypes = []
    lib.ljmd_create.argtypes = [ctypes.POINTER(vp), ctypes.POINTER(LjmdParams)]
    lib.ljmd_destroy.argtypes = [vp]
    lib.ljmd_destroy.restype = None
    lib.ljmd_energy.argtypes = [vp, vp, vp]
    lib.ljmd_forces.argtypes = [vp, vp, vp, vp]
    lib.ljmd_run.argtypes = [vp, vp, vp, vp, vp, i64, i64, vp, i64, vp, f32, i64]
    lib.ljmd_virial.argtypes = [vp, vp, vp]
    lib.ljmd_run_virial.argtypes = [vp, vp, vp, vp, vp, i64, i64, vp, i64, vp, f32, i64, vp]
    lib.ljmd_run_blocked.argtypes = [vp, vp, vp, vp, vp, i64, i64, vp]
    lib.ljmd_gr_hist.argtypes = [vp, vp, i64, i32, vp, vp]
    lib.ljmd_cell_geometry.argtypes = [vp, ctypes.POINTER(i32), ctypes.POINTER(i32), ctypes.POINTER(i32),
                                       ctypes.POINTER(f32), ctypes.POINTER(f32)]
    lib.ljmd_cell_assign.argtypes = [vp, vp, vp, vp]
    lib.ljmd_neighbor_count.argtypes = [vp, vp, f32, vp]
    lib.ljmd_last_rebuilds.argtypes = [vp, ctypes.POINTER(i64)]
    lib.ljmd_get_unique_id.argtypes = [vp]
    lib.ljmd_create_dist.argtypes = [ctypes.POINTER(vp), ctypes.POINTER(LjmdParams), vp, i32, i32]
    lib.ljmd_check.argtypes = [vp]
    lib.ljmd_last_run_ms.argtypes = [vp, ctypes.POINTER(f32)]
    lib.ljmd_launch_count.argtypes = [vp, ctypes.POINTER(i64)]
    lib.ljmd_allpairs_mode.argtypes = [vp, ctypes.POINTER(i32)]
    lib.ljmd_fp32_peak_probe.argtypes = [i32, i32, ctypes.POINTER(f32)]
    lib.ljmd_pair_accel.argtypes = [i32, vp, vp, i64, f32, vp, vp]
    for name in EXPORTS:
        fn = getattr(lib, name)
        if name not in ("ljmd_last_error", "ljmd_destroy"):
            fn.restype = ctypes.c_int
    _lib = lib
    return lib


def check(code: int, what: str) -> None:
    if code != 0:
        msg = load().ljmd_last_error().decode("utf-8", "replace")
        raise LjmdError(f"{what} failed with code {code}: {msg}", code)
