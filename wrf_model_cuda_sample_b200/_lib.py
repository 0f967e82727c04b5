"""ctypes binding of libwrfb200.so (the C ABI declared in include/wrfb200.h).

The library is built in-tree by ``__graft_entry__.build()`` (nvcc, sm_100a).  There is no Python or CPU
fallback: if the shared object is missing, importing this module's ``lib()`` raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("WRFB200_LIB") or os.path.join(_HERE, "libwrfb200.so")   # override: A/B builds

# enum wrfb200_field (include/wrfb200.h)
FIELDS_3D = ("ww", "ww_1", "u", "u_1", "v", "v_1", "t", "t_1", "t_ave", "ft")
FIELDS_2D = ("mu", "mut", "muave", "muts", "muu", "muv", "mudf", "mu_tend",
             "msfuy", "msfvx_inv", "msftx", "msfty")
FIELDS_1D = ("dnw", "fnm", "fnp", "rdnw")
FIELDS = FIELDS_3D + FIELDS_2D + FIELDS_1D
FIELD_ID = {name: i for i, name in enumerate(FIELDS)}

# Order of the array arguments in the Fortran subroutine (module_small_step_em.f90:7-18)
FORTRAN_ARRAY_ORDER_A = ("ww", "ww_1", "u", "u_1", "v", "v_1", "mu", "mut", "muave", "muts", "muu", "muv",
                         "mudf", "t", "t_1", "t_ave", "ft", "mu_tend")
FORTRAN_ARRAY_ORDER_B = ("dnw", "fnm", "fnp", "rdnw", "msfuy", "msfvx_inv", "msftx", "msfty")

OK, ERR_INVALID_ARG, ERR_UNSUPPORTED, ERR_CUDA, ERR_NOMEM, ERR_STATE = range(6)
KERNEL_AUTO, KERNEL_COLUMN, KERNEL_TILE, KERNEL_PIPE = 0, 1, 2, 3
# wrfb200_default_last_transfer: every array copied directly / some staged through bounce buffers / all staged
TRANSFER_DIRECT, TRANSFER_MIXED, TRANSFER_STAGED = 0, 1, 2
WEST, EAST, SOUTH, NORTH = 0, 1, 2, 3


class Domain(C.Structure):
    """struct wrfb200_domain."""
    _fields_ = [(n, C.c_int) for n in
                ("ids", "ide", "jds", "jde", "kde", "ims", "ime", "jms", "jme", "kms", "kme",
                 "periodic_x", "specified", "nested")]


class CompareResult(C.Structure):
    """struct wrfb200_compare_result."""
    _fields_ = [("n", C.c_long), ("n_equal", C.c_long), ("n_different", C.c_long),
                ("max_rel", C.c_float), ("max_abs", C.c_float), ("rmse", C.c_float),
                ("max_ulp", C.c_long)]


class CompareResultR8(C.Structure):
    """struct wrfb200_compare_result_r8."""
    _fields_ = [("n", C.c_long), ("n_equal", C.c_long), ("n_different", C.c_long),
                ("max_rel", C.c_double), ("max_abs", C.c_double), ("rmse", C.c_double),
                ("max_ulp", C.c_long)]


class WrfB200Error(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"wrfb200 status {status}: {message}")
        self.status = status


_P = C.c_void_p
_ADV_ARGS = ([_P] * 18 + [C.c_float] * 4 + [_P] * 8 + [C.c_int] * 3 + [C.c_int] * 5 + [C.c_int] * 6 + [C.c_int] * 6)
_ADV_ARGS_R8 = ([_P] * 18 + [C.c_double] * 4 + [_P] * 8 + [C.c_int] * 3 + [C.c_int] * 5 + [C.c_int] * 6 + [C.c_int] * 6)

# every symbol include/wrfb200.h declares, with its ctypes prototype
PROTOTYPES = {
    "wrfb200_advance_mu_t": (C.c_int, _ADV_ARGS),
    "wrfb200_advance_mu_t_loop": (C.c_int, _ADV_ARGS + [C.c_int]),
    "wrfb200_advance_mu_t_r8": (C.c_int, _ADV_ARGS_R8),
    "wrfb200_advance_mu_t_loop_r8": (C.c_int, _ADV_ARGS_R8 + [C.c_int]),
    "wrfb200_set_default_stream": (C.c_int, [_P]),
    "wrfb200_set_default_kernel": (C.c_int, [C.c_int]),
    "wrfb200_release_cache": (C.c_int, []),
    "wrfb200_acoustic_loop_begin": (C.c_int, []),
    "wrfb200_acoustic_loop_end": (C.c_int, []),
    "wrfb200_set_host_pinning": (C.c_int, [C.c_int]),
    "wrfb200_host_register": (C.c_int, [_P, C.c_size_t]),
    "wrfb200_host_unregister_all": (C.c_int, []),
    "wrfb200_default_last_kernel": (C.c_int, [C.POINTER(C.c_int)]),
    "wrfb200_default_last_transfer": (C.c_int, [C.POINTER(C.c_int)]),
    "wrfb200_set_default_devices": (C.c_int, [C.POINTER(C.c_int), C.c_int]),
    "wrfb200_set_shared_tiles": (C.c_int, [C.c_int]),
    "wrfb200_host_split_plan": (C.c_int, [C.POINTER(Domain)] + [C.c_int] * 7 + [C.POINTER(C.c_int)]),
    "wrfb200_upload_constants": (C.c_int, [_P] + [_P] * 17),
    "wrfb200_upload_state": (C.c_int, [_P, _P, _P, _P]),
    "wrfb200_set_uv": (C.c_int, [_P, _P, _P]),
    "wrfb200_download_outputs": (C.c_int, [_P] + [C.c_int] * 6 + [_P] * 7),
    "wrfb200_upload_constants_r8": (C.c_int, [_P] + [_P] * 17),
    "wrfb200_upload_state_r8": (C.c_int, [_P, _P, _P, _P]),
    "wrfb200_set_uv_r8": (C.c_int, [_P, _P, _P]),
    "wrfb200_download_outputs_r8": (C.c_int, [_P] + [C.c_int] * 6 + [_P] * 7),
    "wrfb200_last_kernel": (C.c_int, [_P, C.POINTER(C.c_int)]),
    "wrfb200_create": (C.c_int, [C.POINTER(_P), C.POINTER(Domain), C.c_int, C.c_int]),
    "wrfb200_destroy": (C.c_int, [_P]),
    "wrfb200_set_stream": (C.c_int, [_P, _P]),
    "wrfb200_set_scalars": (C.c_int, [_P, C.c_float, C.c_float, C.c_float, C.c_float]),
    "wrfb200_set_kernel": (C.c_int, [_P, C.c_int]),
    "wrfb200_bind_device": (C.c_int, [_P, C.c_int, _P, C.c_long]),
    "wrfb200_device_ptr": (C.c_int, [_P, C.c_int, C.POINTER(_P), C.POINTER(C.c_long)]),
    "wrfb200_upload": (C.c_int, [_P, C.c_int, _P]),
    "wrfb200_download": (C.c_int, [_P, C.c_int, _P]),
    "wrfb200_upload_range": (C.c_int, [_P, C.c_int, _P] + [C.c_int] * 6),
    "wrfb200_download_range": (C.c_int, [_P, C.c_int, _P] + [C.c_int] * 6),
    "wrfb200_create_r8": (C.c_int, [C.POINTER(_P), C.POINTER(Domain), C.c_int, C.c_int]),
    "wrfb200_set_scalars_r8": (C.c_int, [_P, C.c_double, C.c_double, C.c_double, C.c_double]),
    "wrfb200_bind_device_r8": (C.c_int, [_P, C.c_int, _P, C.c_long]),
    "wrfb200_device_ptr_r8": (C.c_int, [_P, C.c_int, C.POINTER(_P), C.POINTER(C.c_long)]),
    "wrfb200_upload_r8": (C.c_int, [_P, C.c_int, _P]),
    "wrfb200_download_r8": (C.c_int, [_P, C.c_int, _P]),
    "wrfb200_upload_range_r8": (C.c_int, [_P, C.c_int, _P] + [C.c_int] * 6),
    "wrfb200_download_range_r8": (C.c_int, [_P, C.c_int, _P] + [C.c_int] * 6),
    "wrfb200_step": (C.c_int, [_P] + [C.c_int] * 6),
    "wrfb200_step_graph": (C.c_int, [_P] + [C.c_int] * 7),
    "wrfb200_sync": (C.c_int, [_P]),
    "wrfb200_launch_count": (C.c_int, [_P, C.POINTER(C.c_long)]),
    "wrfb200_pack_halo": (C.c_int, [_P, C.c_int, C.c_int, C.c_int] + [C.c_int] * 4 + [_P]),
    "wrfb200_unpack_halo": (C.c_int, [_P, C.c_int, C.c_int, C.c_int] + [C.c_int] * 4 + [_P]),
    "wrfb200_pack_halo_r8": (C.c_int, [_P, C.c_int, C.c_int, C.c_int] + [C.c_int] * 4 + [_P]),
    "wrfb200_unpack_halo_r8": (C.c_int, [_P, C.c_int, C.c_int, C.c_int] + [C.c_int] * 4 + [_P]),
    "wrfb200_standin_advance_uv": (C.c_int, [_P, C.c_int, C.c_float] + [C.c_int] * 4),
    "wrfb200_standin_advance_uv_r8": (C.c_int, [_P, C.c_int, C.c_double] + [C.c_int] * 4),
    "wrfb200_comm_info_bytes": (C.c_int, []),
    "wrfb200_comm_set_wrap": (C.c_int, [_P, C.c_int, C.c_int]),
    "wrfb200_comm_init": (C.c_int, [_P, C.c_int, C.c_int, C.c_int] + [C.c_int] * 4 + [_P]),
    "wrfb200_comm_connect": (C.c_int, [_P, _P, C.c_int]),
    "wrfb200_comm_barrier": (C.c_int, [_P]),
    "wrfb200_comm_push_constants": (C.c_int, [_P]),
    "wrfb200_comm_push_uv": (C.c_int, [_P]),
    "wrfb200_comm_wait_outputs": (C.c_int, [_P]),
    "wrfb200_comm_step": (C.c_int, [_P]),
    "wrfb200_comm_standin_advance_uv": (C.c_int, [_P, C.c_float]),
    "wrfb200_comm_loop": (C.c_int, [_P, C.c_int, C.c_int, C.c_float, C.c_int]),
    "wrfb200_comm_status": (C.c_int, [_P, C.POINTER(C.c_int), C.POINTER(C.c_long)]),
    "wrfb200_comm_init_r8": (C.c_int, [_P, C.c_int, C.c_int, C.c_int] + [C.c_int] * 4 + [_P]),
    "wrfb200_comm_standin_advance_uv_r8": (C.c_int, [_P, C.c_double]),
    "wrfb200_comm_loop_r8": (C.c_int, [_P, C.c_int, C.c_int, C.c_double, C.c_int]),
    "wrfb200_bounds": (C.c_int, [C.c_int] * 13 + [C.POINTER(C.c_int)] * 6),
    "wrfb200_synth_field": (C.c_int, [C.c_int, C.c_uint64, C.POINTER(Domain), C.c_float, _P]),
    "wrfb200_compare": (C.c_int, [_P, _P, C.c_long, C.POINTER(CompareResult)]),
    "wrfb200_compare_r8": (C.c_int, [_P, _P, C.c_long, C.POINTER(CompareResultR8)]),
    "wrfb200_pipe_plan": (C.c_int, [C.POINTER(Domain)] + [C.c_int] * 7 + [C.POINTER(C.c_longlong)]),
    "wrfb200_last_error": (C.c_char_p, []),
    "wrfb200_version": (C.c_int, []),
}

_lib = None


def lib() -> C.CDLL:
    """Load libwrfb200.so (once).  Fails loudly when the CUDA extension has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not found: the CUDA extension is not built. Run "
                "`python -c 'import __graft_entry__ as g; g.build()'` at the repository root. "
                "There is no CPU fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(handle, name)          # AttributeError if the symbol is missing
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(status: int) -> None:
    if status != OK:
        raise WrfB200Error(status, lib().wrfb200_last_error().decode("utf-8", "replace"))
