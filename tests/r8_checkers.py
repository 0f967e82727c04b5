"""TEST INFRASTRUCTURE: the two binary64 checkers of the real*8 kernels, both derived from the pinned oracle.

* ``oracle_c_r8``      -- oracle/advance_mu_t_oracle.c compiled with ``float`` read as ``double``
                         (tests/advance_mu_t_checker_r8.c), built once per process into a temporary directory
                         with the oracle's flags.
* ``oracle_numpy_r8``  -- oracle/oracle_np.py evaluated with every ``np.float32`` read as ``np.float64``
                         (its only precision-dependent token), so each numpy ufunc is one binary64 rounding.
Arrays: numpy float64, C order [j,k,i] / [j,i] / [k].
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
import tempfile
import types

import numpy as np

from oracle import loader

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SOURCE = os.path.join(ROOT, "tests", "advance_mu_t_checker_r8.c")
CFLAGS = ["-std=c99", "-O3", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-fopenmp", "-shared"]
_ARGS = [C.c_void_p] * 18 + [C.c_double] * 4 + [C.c_void_p] * 8 + [C.c_int] * 3 + [C.c_int] * 17

_state = {}


def _cc():
    return "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else (shutil.which("gcc") or "cc")


def c_library() -> C.CDLL:
    """The compiled binary64 C checker (built on first use; nothing is written inside the repository)."""
    if "c" not in _state:
        d = tempfile.mkdtemp(prefix="wrfb200_r8_checker_")
        so = os.path.join(d, "libchecker_r8.so")
        subprocess.run([_cc()] + CFLAGS + ["-o", so, SOURCE], check=True)
        _state["c"] = C.CDLL(so)
    return _state["c"]


def _pack(fields, grid, scalars):
    for n in loader.ORDER_A + loader.ORDER_B:
        a = fields[n]
        assert isinstance(a, np.ndarray) and a.dtype == np.float64 and a.flags["C_CONTIGUOUS"], n
    return ([fields[n].ctypes.data for n in loader.ORDER_A] + [float(x) for x in scalars]
            + [fields[n].ctypes.data for n in loader.ORDER_B]
            + [int(grid.periodic_x), int(grid.specified), int(grid.nested)]
            + [int(x) for x in grid.index_args()])


def oracle_c_r8(fields, grid, scalars, tiles: int = 0) -> None:
    """The binary64 C checker, in place on ``fields``.  tiles>0: OpenMP over that many j-tiles."""
    lib = c_library()
    if tiles > 0:
        fn = lib.oracle_advance_mu_t_tiled_r8
        fn.restype, fn.argtypes = C.c_int, _ARGS + [C.c_int]
        rc = fn(*_pack(fields, grid, scalars), int(tiles))
    else:
        fn = lib.oracle_advance_mu_t_r8
        fn.restype, fn.argtypes = C.c_int, _ARGS
        rc = fn(*_pack(fields, grid, scalars))
    if rc != 0:
        raise RuntimeError(f"oracle_advance_mu_t_r8 returned {rc}")


def numpy_module() -> types.ModuleType:
    if "np" not in _state:
        src = open(os.path.join(ROOT, "oracle", "oracle_np.py")).read()
        assert "float64" not in src
        mod = types.ModuleType("oracle_np_r8")
        exec(compile(src.replace("np.float32", "np.float64"), "oracle_np.py (binary64)", "exec"), mod.__dict__)
        _state["np"] = mod
    return _state["np"]


def oracle_numpy_r8(fields, grid, scalars) -> None:
    """The binary64 numpy checker, in place on ``fields``."""
    rdx, rdy, dts, epssm = scalars
    a = [fields[n] for n in loader.ORDER_A]
    b = [fields[n] for n in loader.ORDER_B]
    numpy_module().advance_mu_t(*a, rdx, rdy, dts, epssm, *b, grid.periodic_x, grid.specified, grid.nested,
                                *grid.index_args())
