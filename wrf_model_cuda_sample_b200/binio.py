""".bin dataset reader / writer in the reference's exact wire format, and the golden comparison.

The reference drivers read one raw file per variable from an input directory (argv[1]) and compare against
``*_output.bin`` files in an output directory (argv[2]):  big-endian 4-byte values, stream access, Fortran
(i,k,j) order, no headers (/root/reference/advance_mu_t_driver.f90:38-167 and :357-452,
common.cu:166-327).  A dump from WRF built with -r8 holds 8-byte reals (integers stay 4 bytes): the reader takes the
element size of each real file from its byte length, returns float64 arrays and scalars for such a case, and
refuses a case whose reals mix the two sizes.  File names are the actual-argument names of WRF's solve_em
(advance_mu_t_driver.f90:193-205).  None of those files ship with the reference; with this module anyone
holding the /data2/WRFV3_Input_Output/V3.4.1/dyn_em/advance_mu_t dump can run it through the GPU path and
get the reference's own error report (common.cu:154-161).
"""
from __future__ import annotations

import os
from typing import Dict, Tuple

import numpy as np

from ._lib import FIELDS_1D, FIELDS_2D, FIELDS_3D
from .advance_mu_t import Grid, compare

# dummy-argument name -> file stem (advance_mu_t_driver.f90:91-167, :193-205)
FILE_OF = {
    "ww": "grid_ww", "ww_1": "ww1", "u": "grid_u_2", "u_1": "grid_u_save", "v": "grid_v_2", "v_1": "grid_v_save",
    "t": "grid_t_2", "t_1": "grid_t_save", "t_ave": "t_2save", "ft": "t_tend",
    "mu": "grid_mu_2", "mut": "grid_mut", "muave": "muave", "muts": "grid_muts", "muu": "grid_muu",
    "muv": "grid_muv", "mudf": "grid_mudf", "mu_tend": "mu_tend", "msfuy": "grid_msfuy",
    "msfvx_inv": "grid_msfvx_inv", "msftx": "grid_msftx", "msfty": "grid_msfty",
    "dnw": "grid_dnw", "fnm": "grid_fnm", "fnp": "grid_fnp", "rdnw": "grid_rdnw",
}
DIM_NAMES = ("ids", "ide", "jds", "jde", "kde", "ims", "ime", "jms", "jme", "kms", "kme",
             "its", "ite", "jts", "jte", "kts", "kte")
SCALAR_FILES = ("grid_rdx", "grid_rdy", "dts_rk", "grid_epssm")
FLAG_FILES = {"nested": "config_flags_nested", "periodic_x": "config_flags_periodic_x",
              "specified": "config_flags_specified"}       # advance_mu_t_driver.cu:78-80
# the reference never reads these (INTENT(OUT)): they need not exist in an input directory
OUTPUT_ONLY = ("muave", "muts", "mudf")
GOLDEN = ("ww", "ww_1", "t", "t_ave", "mu", "muave", "muts", "mudf")     # advance_mu_t_driver.f90:224-231


def _read(path: str, dtype: str, count: int) -> np.ndarray:
    a = np.fromfile(path, dtype=dtype)
    if a.size != count:
        raise ValueError(f"{path}: {a.size} values, expected {count}")
    return a


def real_kind(path: str, count: int) -> str:
    """'>f4' or '>f8': the element size of a file of ``count`` reals, from its byte length."""
    nbytes = os.path.getsize(path)
    for kind in (">f4", ">f8"):
        if nbytes == count * np.dtype(kind).itemsize:
            return kind
    raise ValueError(f"{path}: {nbytes} bytes are neither {count} 4-byte nor {count} 8-byte reals")


def read_int(path: str) -> int:
    return int(_read(path, ">i4", 1)[0])


def read_real(path: str):
    """np.float32 from a 4-byte file, np.float64 from an 8-byte one."""
    kind = real_kind(path, 1)
    return np.dtype(kind).newbyteorder("=").type(_read(path, kind, 1)[0])


def read_field(path: str, shape) -> np.ndarray:
    """Raw big-endian stream in Fortran (i,k,j) order -> native float32 (4-byte file) or float64 (8-byte file)
    array in C order [j,k,i]."""
    count = int(np.prod(shape))
    kind = real_kind(path, count)
    a = _read(path, kind, count).astype(np.dtype(kind).newbyteorder("=")).reshape(shape)
    if np.isnan(a).any():                                      # the reference readers flag NaNs, common.cu:39-44
        raise ValueError(f"{path}: contains NaN")
    return np.ascontiguousarray(a)


def write_field(path: str, a: np.ndarray) -> None:
    """float64 arrays as 8-byte reals, anything else as 4-byte reals."""
    if getattr(a, "dtype", None) == np.float64:
        np.ascontiguousarray(a).astype(">f8").tofile(path)
    else:
        np.ascontiguousarray(a, dtype=np.float32).astype(">f4").tofile(path)


def write_int(path: str, v: int) -> None:
    np.array([v], dtype=">i4").tofile(path)


def write_real(path: str, v, kind: str = ">f4") -> None:
    np.array([v], dtype=kind).tofile(path)


def read_case(input_dir: str) -> Tuple[Grid, tuple, Dict[str, np.ndarray]]:
    """(grid, (rdx, rdy, dts, epssm), fields) from a directory of reference-format input files."""
    j = lambda stem: os.path.join(input_dir, stem + ".bin")
    dims = {n: read_int(j(n)) for n in DIM_NAMES}
    flags = {}
    for name, stem in FLAG_FILES.items():
        flags[name] = bool(read_int(j(stem))) if os.path.exists(j(stem)) else (name == "specified")
    g = Grid(**dims, **flags)
    kinds = {}                                   # element size of every real file, to check that they agree

    def real(path, count):
        kinds[path] = real_kind(path, count)
        first = next(iter(kinds.values()))
        if kinds[path] != first:
            raise ValueError(f"{path}: {kinds[path][-1]}-byte reals in a case of {first[-1]}-byte reals "
                             f"({next(iter(kinds))})")
        return path

    scalars = tuple(read_real(real(j(s), 1)) for s in SCALAR_FILES)
    fields = {}
    for name in FIELDS_3D + FIELDS_2D + FIELDS_1D:
        path = j(FILE_OF[name])
        if os.path.exists(path):
            fields[name] = read_field(real(path, int(np.prod(g.shape_of(name)))), g.shape_of(name))
        elif name in OUTPUT_ONLY:
            fields[name] = np.zeros(g.shape_of(name), dtype=scalars[0].dtype)    # the case's precision
        else:
            raise FileNotFoundError(path)
    return g, scalars, fields


def write_case(directory: str, g: Grid, scalars, fields: Dict[str, np.ndarray], suffix: str = "",
               names=None) -> None:
    """Write dims / scalars / flags (when ``suffix`` is empty) and the fields as ``<stem><suffix>.bin``.
    float64 fields make an 8-byte case (scalars included), others a 4-byte one; a mix raises ValueError."""
    os.makedirs(directory, exist_ok=True)
    j = lambda stem: os.path.join(directory, stem + ".bin")
    names = [n for n in (names if names is not None else fields) if n in FILE_OF]
    wide = {n: getattr(fields[n], "dtype", None) == np.float64 for n in names}
    if len(set(wide.values())) > 1:
        raise ValueError("a case holds reals of one size: got float64 fields "
                         f"{[n for n in names if wide[n]]} beside {[n for n in names if not wide[n]]}")
    if not suffix:
        for n in DIM_NAMES:
            write_int(j(n), getattr(g, n))
        write_int(j("kds"), 1)                                # read by the C / CUDA drivers only
        for s, v in zip(SCALAR_FILES, scalars):
            write_real(j(s), v, ">f8" if any(wide.values()) else ">f4")
        for name, stem in FLAG_FILES.items():
            write_int(j(stem), int(getattr(g, name)))
    for name in names:
        write_field(j(FILE_OF[name] + suffix), fields[name])


def compare_with_golden(g: Grid, fields: Dict[str, np.ndarray], golden_dir: str) -> Dict[str, dict]:
    """The reference's final report: every output field against ``<stem>_output.bin`` with its metric set;
    3-D fields and mu over the whole memory extent, muave/muts/mudf over the computed range only
    (advance_mu_t_driver.f90:219-231)."""
    i0, i1, j0, j1 = max(g.its, g.ids + 1), min(g.ite, g.ide - 2), max(g.jts, g.jds + 1), min(g.jte, g.jde - 2)
    report = {}
    for name in GOLDEN:
        path = os.path.join(golden_dir, FILE_OF[name] + "_output.bin")
        if not os.path.exists(path):
            continue
        ref = read_field(path, g.shape_of(name))
        got = fields[name]
        if name in OUTPUT_ONLY:
            J = slice(j0 - g.jms, j1 - g.jms + 1); I = slice(i0 - g.ims, i1 - g.ims + 1)
            ref, got = ref[J, I], got[J, I]
        report[name] = compare(got, ref)
    return report
