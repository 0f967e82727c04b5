"""oracle/loader.py -- TEST INFRASTRUCTURE, NOT PRODUCT.

ctypes access to the checkers:
  * ``liboracle.so``                      our C restatement (oracle/advance_mu_t_oracle.c)
  * ``_ref/libref_advance_mu_t.so``       the reference's own C translation, unmodified, compiled in place
  * ``_ref/libref_cuda_kernel.so``        the reference's own CUDA-C kernel TU, unmodified, for sm_100a
All take the Fortran argument list (module_small_step_em.f90:7-18) with config_flags as three ints.
Arrays: numpy float32, C order [j,k,i] / [j,i] / [k].
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_SO = os.path.join(HERE, "liboracle.so")
REF_SO = os.path.join(HERE, "_ref", "libref_advance_mu_t.so")
REF_CUDA_SO = os.path.join(HERE, "_ref", "libref_cuda_kernel.so")

ORDER_A = ("ww", "ww_1", "u", "u_1", "v", "v_1", "mu", "mut", "muave", "muts", "muu", "muv",
           "mudf", "t", "t_1", "t_ave", "ft", "mu_tend")
ORDER_B = ("dnw", "fnm", "fnp", "rdnw", "msfuy", "msfvx_inv", "msftx", "msfty")
OUTPUTS = ("ww", "t", "t_ave", "mu", "muave", "muts", "mudf")

_P = C.c_void_p
_ARGS = [_P] * 18 + [C.c_float] * 4 + [_P] * 8 + [C.c_int] * 3 + [C.c_int] * 17

_cache = {}


def _load(path):
    if path not in _cache:
        if not os.path.exists(path):
            raise FileNotFoundError(f"{path} missing: run `make -C oracle` (_ref/ needs REF=<reference checkout>)")
        _cache[path] = C.CDLL(path)
    return _cache[path]


def have_ref() -> bool:
    return os.path.exists(REF_SO)


def have_ref_cuda() -> bool:
    return os.path.exists(REF_CUDA_SO)


def _pack(fields, grid, scalars):
    for n in ORDER_A + ORDER_B:
        a = fields[n]
        assert isinstance(a, np.ndarray) and a.dtype == np.float32 and a.flags["C_CONTIGUOUS"], n
    rdx, rdy, dts, epssm = scalars
    return ([fields[n].ctypes.data for n in ORDER_A] + [float(rdx), float(rdy), float(dts), float(epssm)]
            + [fields[n].ctypes.data for n in ORDER_B]
            + [int(grid.periodic_x), int(grid.specified), int(grid.nested)]
            + [int(x) for x in grid.index_args()])


def oracle_c(fields, grid, scalars, tiles: int = 0) -> None:
    """Our C restatement, in place on ``fields``.  tiles>0: OpenMP over that many j-tiles."""
    lib = _load(ORACLE_SO)
    if tiles > 0:
        fn = lib.oracle_advance_mu_t_tiled
        fn.restype, fn.argtypes = C.c_int, _ARGS + [C.c_int]
        rc = fn(*_pack(fields, grid, scalars), int(tiles))
    else:
        fn = lib.oracle_advance_mu_t
        fn.restype, fn.argtypes = C.c_int, _ARGS
        rc = fn(*_pack(fields, grid, scalars))
    if rc != 0:
        raise RuntimeError(f"oracle_advance_mu_t returned {rc}")


def reference_c(fields, grid, scalars, tiles: int = 0) -> None:
    """The reference's own advance_mu_t.c, in place on ``fields``.  tiles>0: OpenMP over j-tiles."""
    lib = _load(REF_SO)
    if tiles > 0:
        fn = lib.ref_advance_mu_t_tiled
        fn.restype, fn.argtypes = None, _ARGS + [C.c_int]
        fn(*_pack(fields, grid, scalars), int(tiles))
    else:
        fn = lib.ref_advance_mu_t
        fn.restype, fn.argtypes = None, _ARGS
        fn(*_pack(fields, grid, scalars))


def oracle_numpy(fields, grid, scalars) -> None:
    from . import oracle_np
    rdx, rdy, dts, epssm = scalars
    a = [fields[n] for n in ORDER_A]
    b = [fields[n] for n in ORDER_B]
    oracle_np.advance_mu_t(*a, rdx, rdy, dts, epssm, *b, grid.periodic_x, grid.specified, grid.nested,
                           *grid.index_args())


def reference_cuda_kernel(dev_ptrs: dict, scratch: dict, grid, scalars, stream: int = 0) -> None:
    """Launch the reference's own CUDA-C kernel on device pointers (ints), dense Fortran layout."""
    lib = _load(REF_CUDA_SO)
    fn = lib.ref_cuda_kernel_launch
    fn.restype = C.c_int
    fn.argtypes = [_P] * 18 + [C.c_float] * 4 + [_P] * 8 + [_P] * 3 + [C.c_int] * 3 + [C.c_int] * 17 + [_P]
    rdx, rdy, dts, epssm = scalars
    rc = fn(*[dev_ptrs[n] for n in ORDER_A], float(rdx), float(rdy), float(dts), float(epssm),
            *[dev_ptrs[n] for n in ORDER_B], scratch["wdtn"], scratch["dvdxi"], scratch["dmdt"],
            int(grid.periodic_x), int(grid.specified), int(grid.nested),
            *[int(x) for x in grid.index_args()], C.c_void_p(stream))
    if rc != 0:
        raise RuntimeError(f"reference CUDA kernel launch failed: cudaError {rc}")
