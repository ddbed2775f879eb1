"""TEST INFRASTRUCTURE ONLY — builds and loads the C references of the tests (tests/<stem>.c).

Each is compiled once per process into a temporary directory (the source tree may be read-only) with
-ffp-contract=off -fno-fast-math, so every floating-point operation rounds once, and with OpenMP where the
compiler has it.  The product package never imports this module.
"""
from __future__ import annotations

import ctypes
import os
import shutil
import subprocess
import tempfile

_HERE = os.path.dirname(os.path.abspath(__file__))
_libs: dict = {}


def load(stem: str, prototypes: dict) -> ctypes.CDLL:
    """The library of tests/<stem>.c with prototypes {name: (argtypes, restype)} declared."""
    lib = _libs.get(stem)
    if lib is not None:
        return lib
    cc = shutil.which("/usr/bin/gcc") or shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        raise RuntimeError(f"no C compiler found for tests/{stem}.c")
    out = os.path.join(tempfile.mkdtemp(prefix=stem + "_"), f"lib{stem}.so")
    src = os.path.join(_HERE, stem + ".c")
    flags = ["-O2", "-fPIC", "-shared", "-std=c11", "-ffp-contract=off", "-fno-fast-math", "-I", _HERE]
    try:
        subprocess.check_call([cc, *flags, "-fopenmp", "-o", out, src, "-lm"], stderr=subprocess.DEVNULL)
    except subprocess.CalledProcessError:             # no OpenMP runtime: serial build
        subprocess.check_call([cc, *flags, "-Wno-unknown-pragmas", "-o", out, src, "-lm"])
    lib = ctypes.CDLL(out)
    for name, (argtypes, restype) in prototypes.items():
        fn = getattr(lib, name)
        fn.argtypes, fn.restype = argtypes, restype
    _libs[stem] = lib
    return lib
