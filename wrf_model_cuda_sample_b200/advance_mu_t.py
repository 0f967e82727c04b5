"""Host-side mirror of the reference operator interface, over the C ABI of libwrfb200.so.

``advance_mu_t(...)`` has the reference Fortran subroutine's argument list
(/root/reference/module_small_step_em.f90:7-18; same names, order and meaning; ``config_flags`` is any
object with ``periodic_x / specified / nested`` members, the only ones the routine reads, :97-106).
``Patch`` is the device-resident form that replaces the reference's per-call malloc/copy/free host layer
(/root/reference/advance_mu_t_no_async.cu:35-424).

Arrays are numpy float32 in C order ``[j, k, i]`` / ``[j, i]`` / ``[k]`` -- byte-identical to the Fortran
``(i,k,j)`` / ``(i,j)`` / ``(k)`` layout -- or torch CUDA tensors of the same shape (launched in place).
float64 arrays (WRF built with -r8) take the ``_r8`` entry points and are computed in binary64; one call's
arrays must all have the same precision.
All compute happens in the CUDA library; nothing here falls back to the CPU.
"""
from __future__ import annotations

import contextlib
import ctypes as C
import os
import threading
from dataclasses import dataclass, replace
from types import SimpleNamespace
from typing import Dict, Iterable, Optional, Sequence

import numpy as np

from . import _lib
from ._lib import (FIELD_ID, FIELDS, FIELDS_1D, FIELDS_2D, FIELDS_3D, FORTRAN_ARRAY_ORDER_A,
                   FORTRAN_ARRAY_ORDER_B, Domain, check, lib)

INPUT_FIELDS = ("ww", "ww_1", "u", "u_1", "v", "v_1", "t", "t_1", "ft",
                "mu", "mut", "muu", "muv", "mu_tend", "msfuy", "msfvx_inv", "msftx", "msfty",
                "dnw", "fnm", "fnp", "rdnw")
OUTPUT_FIELDS = ("ww", "t", "t_ave", "mu", "muave", "muts", "mudf")


@dataclass(frozen=True)
class Grid:
    """Index description of one call: domain (d), memory (m) and tile (t) extents, Fortran-numbered."""
    ids: int
    ide: int
    jds: int
    jde: int
    kde: int
    ims: int
    ime: int
    jms: int
    jme: int
    kms: int
    kme: int
    its: int
    ite: int
    jts: int
    jte: int
    kts: int
    kte: int
    periodic_x: bool = False
    specified: bool = True
    nested: bool = False

    @staticmethod
    def from_shape(nx: int, ny: int, nz: int, halo: int = 5, periodic_x: bool = False,
                   specified: bool = True, nested: bool = False) -> "Grid":
        """"AxBxC" = WRF e_we x e_sn x e_vert: ids=jds=1, ide=A, jde=B, kde=C, memory = domain + halo,
        one tile covering the domain (SURVEY.md section 8d, shape convention)."""
        return Grid(1, nx, 1, ny, nz, 1 - halo, nx + halo, 1 - halo, ny + halo, 1, nz,
                    1, nx, 1, ny, 1, nz, periodic_x, specified, nested)

    # ---- derived ----
    @property
    def shape3(self):
        return (self.jme - self.jms + 1, self.kme - self.kms + 1, self.ime - self.ims + 1)

    @property
    def shape2(self):
        return (self.jme - self.jms + 1, self.ime - self.ims + 1)

    @property
    def shape1(self):
        return (self.kme - self.kms + 1,)

    def shape_of(self, field: str):
        return self.shape3 if field in FIELDS_3D else self.shape2 if field in FIELDS_2D else self.shape1

    def bounds(self):
        """(i_start, i_end, j_start, j_end, k_start, k_end) of module_small_step_em.f90:91-106."""
        out = [C.c_int() for _ in range(6)]
        check(lib().wrfb200_bounds(int(self.periodic_x), int(self.specified), int(self.nested),
                                   self.ids, self.ide, self.jds, self.jde,
                                   self.its, self.ite, self.jts, self.jte, self.kts, self.kte,
                                   *[C.byref(o) for o in out]))
        return tuple(o.value for o in out)

    def updated_points(self):
        """(N3, N2): 3-D points and columns one call updates."""
        i0, i1, j0, j1, k0, k1 = self.bounds()
        n2 = max(0, i1 - i0 + 1) * max(0, j1 - j0 + 1)
        return n2 * max(0, k1 - k0 + 1), n2

    def algorithmic_bytes(self) -> int:
        """44 B per updated 3-D point + 52 B per column (SURVEY.md section 8d)."""
        n3, n2 = self.updated_points()
        return 44 * n3 + 52 * n2

    def domain(self) -> Domain:
        return Domain(self.ids, self.ide, self.jds, self.jde, self.kde, self.ims, self.ime, self.jms, self.jme,
                      self.kms, self.kme, int(self.periodic_x), int(self.specified), int(self.nested))

    def flags(self):
        return SimpleNamespace(periodic_x=self.periodic_x, specified=self.specified, nested=self.nested)

    def index_args(self):
        """The 17 trailing integers of the Fortran argument list, in order."""
        return (self.ids, self.ide, self.jds, self.jde, self.kde, self.ims, self.ime, self.jms, self.jme,
                self.kms, self.kme, self.its, self.ite, self.jts, self.jte, self.kts, self.kte)

    def with_tile(self, its, ite, jts, jte) -> "Grid":
        return replace(self, its=its, ite=ite, jts=jts, jte=jte)


def _dtype(a):
    """np.float32 / np.float64 for a numpy array or torch tensor of that precision, else None."""
    if isinstance(a, np.ndarray):
        return a.dtype.type if a.dtype in (np.float32, np.float64) else None
    if hasattr(a, "data_ptr"):
        import torch
        return {torch.float32: np.float32, torch.float64: np.float64}.get(a.dtype)
    return None


def _ptr(a, dtype=np.float32) -> int:
    """Raw address of a numpy array (host) or torch tensor (host or device) of precision ``dtype``."""
    name = np.dtype(dtype).name
    if isinstance(a, np.ndarray):
        if a.dtype != dtype or not a.flags["C_CONTIGUOUS"]:
            raise TypeError(f"fields must be C-contiguous {name} arrays")
        return a.ctypes.data
    if hasattr(a, "data_ptr"):
        if _dtype(a) is not dtype or not a.is_contiguous():
            raise TypeError(f"fields must be contiguous {name} tensors")
        return a.data_ptr()
    raise TypeError(f"unsupported array type {type(a)!r}")


def _precision(arrays) -> type:
    """The one precision (np.float32 or np.float64) shared by every array of a call."""
    kinds = {_dtype(a) for a in arrays}
    if len(kinds) != 1 or None in kinds:
        names = sorted({str(getattr(a, "dtype", type(a).__name__)) for a in arrays})
        raise TypeError("advance_mu_t needs all arrays float32 (default REAL) or all float64 (-r8), "
                        f"got {', '.join(names)}")
    return kinds.pop()


def advance_mu_t(ww, ww_1, u, u_1, v, v_1, mu, mut, muave, muts, muu, muv, mudf, t, t_1, t_ave, ft, mu_tend,
                 rdx, rdy, dts, epssm, dnw, fnm, fnp, rdnw, msfuy, msfvx_inv, msftx, msfty, config_flags,
                 ids, ide, jds, jde, kde, ims, ime, jms, jme, kms, kme, its, ite, jts, jte, kts, kte,
                 nsteps: int = 1) -> None:
    """The reference operator (module_small_step_em.f90:7-18), executed on the GPU.

    Updates ww, mu, muave, muts, mudf, t, t_ave in place.  ``nsteps`` > 1 repeats the step on
    device-resident state with a single upload/download (host arrays only).  All-float32 arrays run the
    binary32 operator, all-float64 arrays the real*8 one (``wrfb200_advance_mu_t_r8``); a mix raises TypeError.
    """
    arrays_a = (ww, ww_1, u, u_1, v, v_1, mu, mut, muave, muts, muu, muv, mudf, t, t_1, t_ave, ft, mu_tend)
    arrays_b = (dnw, fnm, fnp, rdnw, msfuy, msfvx_inv, msftx, msfty)
    dt = _precision(arrays_a + arrays_b)
    args = ([_ptr(a, dt) for a in arrays_a] + [float(rdx), float(rdy), float(dts), float(epssm)]
            + [_ptr(a, dt) for a in arrays_b]
            + [int(bool(config_flags.periodic_x)), int(bool(config_flags.specified)), int(bool(config_flags.nested))]
            + [int(x) for x in (ids, ide, jds, jde, kde, ims, ime, jms, jme, kms, kme, its, ite, jts, jte, kts, kte)])
    sfx = "_r8" if dt is np.float64 else ""
    if nsteps == 1:
        check(getattr(lib(), "wrfb200_advance_mu_t" + sfx)(*args))
    else:
        check(getattr(lib(), "wrfb200_advance_mu_t_loop" + sfx)(*args, int(nsteps)))


def call_with_fields(fields: Dict[str, object], grid: Grid, rdx, rdy, dts, epssm, nsteps: int = 1) -> None:
    """``advance_mu_t`` with the arrays taken from a dict keyed by the Fortran dummy-argument names."""
    a = [fields[n] for n in FORTRAN_ARRAY_ORDER_A]
    b = [fields[n] for n in FORTRAN_ARRAY_ORDER_B]
    advance_mu_t(*a, rdx, rdy, dts, epssm, *b, grid.flags(), *grid.index_args(), nsteps=nsteps)


class Patch:
    """Device-resident state of one patch (one rank): wrfb200_create / upload / step / download.

    ``dtype`` np.float64 (or torch.float64) makes a real*8 patch (wrfb200_create_r8): fields are float64 and the
    step runs in binary64.  Every verb with a precision calls the C verb of the patch's precision (the ``_r8``
    entry points for float64), the fused multi-GPU and halo pack / unpack verbs included."""

    def __init__(self, grid: Grid, device: int = -1, allocate: bool = True, stream: Optional[int] = None,
                 dtype=np.float32):
        self.grid = grid
        self.dtype = _patch_dtype(dtype)
        self._sfx = "_r8" if self.dtype is np.float64 else ""
        self._h = C.c_void_p()
        dom = grid.domain()
        check(getattr(lib(), "wrfb200_create" + self._sfx)(C.byref(self._h), C.byref(dom), device, int(allocate)))
        if stream is not None:
            self.set_stream(stream)

    # ---- life cycle ----
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().wrfb200_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ---- configuration ----
    def set_stream(self, cuda_stream: int):
        check(lib().wrfb200_set_stream(self._h, C.c_void_p(cuda_stream)))

    def _fn(self, name):
        """The C verb of this patch's precision."""
        return getattr(lib(), name + self._sfx)

    def set_scalars(self, rdx, rdy, dts, epssm):
        check(self._fn("wrfb200_set_scalars")(self._h, float(rdx), float(rdy), float(dts), float(epssm)))

    def set_kernel(self, kernel: int):
        check(lib().wrfb200_set_kernel(self._h, int(kernel)))

    def bind(self, field: str, tensor, pitch: Optional[int] = None):
        """Adopt a caller-owned device buffer (e.g. a torch CUDA tensor) for ``field``."""
        if pitch is None:
            pitch = tensor.shape[-1]
        check(self._fn("wrfb200_bind_device")(self._h, FIELD_ID[field], C.c_void_p(_ptr(tensor, self.dtype)),
                                              int(pitch)))

    def device_ptr(self, field: str):
        p, pitch = C.c_void_p(), C.c_long()
        check(self._fn("wrfb200_device_ptr")(self._h, FIELD_ID[field], C.byref(p), C.byref(pitch)))
        return p.value, pitch.value

    # ---- copies (async on the patch stream) ----
    def upload(self, fields: Dict[str, np.ndarray], names: Optional[Iterable[str]] = None):
        for n in (names if names is not None else fields.keys()):
            a = fields[n]
            if tuple(a.shape) != self.grid.shape_of(n):
                raise ValueError(f"{n}: shape {tuple(a.shape)} != {self.grid.shape_of(n)}")
            check(self._fn("wrfb200_upload")(self._h, FIELD_ID[n], C.c_void_p(_ptr(a, self.dtype))))

    def download(self, fields: Dict[str, np.ndarray], names: Iterable[str] = OUTPUT_FIELDS, sync: bool = True):
        for n in names:
            check(self._fn("wrfb200_download")(self._h, FIELD_ID[n], C.c_void_p(_ptr(fields[n], self.dtype))))
        if sync:
            self.sync()

    def download_range(self, field: str, host, i0, i1, k0, k1, j0, j1):
        check(self._fn("wrfb200_download_range")(self._h, FIELD_ID[field], C.c_void_p(_ptr(host, self.dtype)),
                                                 i0, i1, k0, k1, j0, j1))

    def upload_range(self, field: str, host, i0, i1, k0, k1, j0, j1):
        check(self._fn("wrfb200_upload_range")(self._h, FIELD_ID[field], C.c_void_p(_ptr(host, self.dtype)),
                                               i0, i1, k0, k1, j0, j1))

    # ---- resident-state verbs (the three cadences of the acoustic loop) ----
    CONSTANTS = ("ww_1", "u_1", "v_1", "t_1", "ft", "mut", "muu", "muv", "mu_tend",
                 "msfuy", "msfvx_inv", "msftx", "msfty", "dnw", "fnm", "fnp", "rdnw")

    def upload_constants(self, fields: Dict[str, np.ndarray]):
        """Once per RK sub-step: everything advance_mu_t reads and nobody changes inside the acoustic loop."""
        ptrs = [C.c_void_p(_ptr(fields[n], self.dtype)) if n in fields else None for n in self.CONSTANTS]
        check(self._fn("wrfb200_upload_constants")(self._h, *ptrs))

    def upload_state(self, fields: Dict[str, np.ndarray]):
        """Once per RK sub-step: the state the loop starts from (ww, t, mu)."""
        check(self._fn("wrfb200_upload_state")(self._h, *[C.c_void_p(_ptr(fields[n], self.dtype))
                                                          for n in ("ww", "t", "mu")]))

    def set_uv(self, u, v):
        """Every small step: what advance_uv changed."""
        check(self._fn("wrfb200_set_uv")(self._h, C.c_void_p(_ptr(u, self.dtype)), C.c_void_p(_ptr(v, self.dtype))))

    def download_outputs(self, fields: Dict[str, np.ndarray], tile: Optional[Grid] = None, sync: bool = True):
        """Every small step: exactly the cells the routine writes, into the caller's arrays."""
        g = tile or self.grid
        ptrs = [C.c_void_p(_ptr(fields[n], self.dtype)) if n in fields else None for n in OUTPUT_FIELDS]
        check(self._fn("wrfb200_download_outputs")(self._h, g.its, g.ite, g.jts, g.jte, g.kts, g.kte, *ptrs))
        if sync:
            self.sync()

    def last_kernel(self) -> int:
        k = C.c_int()
        check(lib().wrfb200_last_kernel(self._h, C.byref(k)))
        return k.value

    # ---- stepping ----
    def step(self, tile: Optional[Grid] = None):
        g = tile or self.grid
        check(lib().wrfb200_step(self._h, g.its, g.ite, g.jts, g.jte, g.kts, g.kte))

    def step_graph(self, nsteps: int, tile: Optional[Grid] = None):
        g = tile or self.grid
        check(lib().wrfb200_step_graph(self._h, g.its, g.ite, g.jts, g.jte, g.kts, g.kte, int(nsteps)))

    def sync(self):
        check(lib().wrfb200_sync(self._h))

    def launch_count(self) -> int:
        n = C.c_long()
        check(lib().wrfb200_launch_count(self._h, C.byref(n)))
        return n.value

    # ---- halo / stand-in ----
    def _halo_buf(self, device_buf) -> C.c_void_p:
        """Address of a halo buffer: a contiguous CUDA tensor of the patch's dtype."""
        if not (hasattr(device_buf, "is_cuda") and device_buf.is_cuda and _dtype(device_buf) is self.dtype):
            raise TypeError(f"halo buffers of a {np.dtype(self.dtype).name} patch must be CUDA tensors of that dtype, "
                            f"got {getattr(device_buf, 'dtype', type(device_buf).__name__)}")
        return C.c_void_p(_ptr(device_buf, self.dtype))

    def pack_halo(self, field: str, side: int, width: int, ips, ipe, jps, jpe, device_buf):
        check(self._fn("wrfb200_pack_halo")(self._h, FIELD_ID[field], side, width, ips, ipe, jps, jpe,
                                            self._halo_buf(device_buf)))

    def unpack_halo(self, field: str, side: int, width: int, ips, ipe, jps, jpe, device_buf):
        check(self._fn("wrfb200_unpack_halo")(self._h, FIELD_ID[field], side, width, ips, ipe, jps, jpe,
                                              self._halo_buf(device_buf)))

    def standin_advance_uv(self, field: str, c: float, i0, i1, j0, j1):
        check(self._fn("wrfb200_standin_advance_uv")(self._h, FIELD_ID[field], float(c), i0, i1, j0, j1))

    # ---- multi-GPU: halo exchange fused into the kernels over peer-mapped memory (csrc/comm.cu) ----
    def comm_set_wrap(self, wrap_x: bool, wrap_y: bool) -> None:
        """Periodic exchange across the domain edge (WRF's periodic_x / periodic_y); call before comm_init."""
        check(lib().wrfb200_comm_set_wrap(self._h, int(bool(wrap_x)), int(bool(wrap_y))))

    def comm_init(self, px: int, py: int, rank: int, ips, ipe, jps, jpe) -> bytes:
        """-> this rank's opaque info blob; all-gather the blobs in rank order and pass them to comm_connect."""
        n = lib().wrfb200_comm_info_bytes()
        buf = C.create_string_buffer(n)
        check(self._fn("wrfb200_comm_init")(self._h, px, py, rank, ips, ipe, jps, jpe, buf))
        return buf.raw

    def comm_connect(self, infos) -> None:
        blob = b"".join(infos)
        n = lib().wrfb200_comm_info_bytes()
        assert len(blob) % n == 0
        check(lib().wrfb200_comm_connect(self._h, blob, len(blob) // n))

    def comm_barrier(self):
        check(lib().wrfb200_comm_barrier(self._h))

    def comm_push_constants(self):
        check(lib().wrfb200_comm_push_constants(self._h))

    def comm_push_uv(self):
        check(lib().wrfb200_comm_push_uv(self._h))

    def comm_wait_outputs(self):
        check(lib().wrfb200_comm_wait_outputs(self._h))

    def comm_step(self):
        check(lib().wrfb200_comm_step(self._h))

    def comm_standin_advance_uv(self, c: float):
        check(self._fn("wrfb200_comm_standin_advance_uv")(self._h, float(c)))

    def comm_loop(self, nsteps: int, standin: bool = False, c: float = 0.0, graph: bool = True):
        check(self._fn("wrfb200_comm_loop")(self._h, int(nsteps), int(bool(standin)), float(c), int(bool(graph))))

    def comm_status(self):
        """(flag_timeouts, steps_done) after synchronising the stream."""
        t, n = C.c_int(), C.c_long()
        check(lib().wrfb200_comm_status(self._h, C.byref(t), C.byref(n)))
        return t.value, n.value


def _patch_dtype(dtype):
    """np.float32 / np.float64 from a numpy or torch dtype."""
    if dtype in (np.float32, np.float64):
        return np.dtype(dtype).type
    if hasattr(dtype, "is_floating_point"):         # torch.dtype
        import torch
        if dtype in (torch.float32, torch.float64):
            return np.float32 if dtype == torch.float32 else np.float64
    if isinstance(dtype, np.dtype) and dtype.type in (np.float32, np.float64):
        return dtype.type
    raise TypeError(f"Patch dtype must be float32 or float64, got {dtype!r}")


class acoustic_loop:
    """``with acoustic_loop():`` -- host-pointer calls of ``advance_mu_t`` inside the block keep the state
    device-resident: the first call uploads everything, later calls with the same arrays upload only u, v
    (wrfb200_acoustic_loop_begin / _end)."""

    def __enter__(self):
        check(lib().wrfb200_acoustic_loop_begin())
        return self

    def __exit__(self, *exc):
        check(lib().wrfb200_acoustic_loop_end())


_devices_state = threading.local()


def set_default_devices(devices: Optional[Sequence[int]]) -> None:
    """Spread this thread's host-array ``advance_mu_t`` calls over the CUDA devices ``devices`` (j-rows split
    into ``len(devices)`` parts; ids may repeat).  ``None`` or ``[]``: the current device only (the default).
    Device-array calls ignore it (wrfb200_set_default_devices)."""
    ids = [int(d) for d in (devices or ())]
    arr = (C.c_int * max(1, len(ids)))(*ids)
    check(lib().wrfb200_set_default_devices(arr if ids else None, len(ids)))
    _devices_state.devices = ids


@contextlib.contextmanager
def default_devices(devices: Optional[Sequence[int]]):
    """``with default_devices([0, 1]):`` -- ``set_default_devices`` for the block, then the previous list."""
    prev = list(getattr(_devices_state, "devices", []))
    set_default_devices(devices)
    try:
        yield
    finally:
        set_default_devices(prev)


def _env_on(name: str) -> bool:
    try:
        return int(os.environ.get(name, "0")) > 0
    except ValueError:
        return False


_shared_state = {"on": _env_on("WRFB200_SHARED_TILES")}    # the library reads the same variable


def set_shared_tiles(enable: bool) -> None:
    """Process-wide shared-tiles mode (wrfb200_set_shared_tiles): host-array ``advance_mu_t`` calls from any thread
    with the same arrays and memory extents are tiles of one device-resident patch on the device that is current in
    the calling thread now, with acoustic-loop residency kept per tile.  Off frees the shared patches; no call may
    be in flight when it is turned off."""
    check(lib().wrfb200_set_shared_tiles(int(bool(enable))))
    _shared_state["on"] = bool(enable)


@contextlib.contextmanager
def shared_tiles(enable: bool = True):
    """``with shared_tiles():`` -- ``set_shared_tiles`` for the block, then the previous state."""
    prev = _shared_state["on"]
    set_shared_tiles(enable)
    try:
        yield
    finally:
        set_shared_tiles(prev)


def host_split_plan(grid: Grid, n: int):
    """The split of a host-array call of ``grid``'s tile over ``n`` parts: one (first row, last row, first memory
    row, last memory row) per part, Fortran j; a part without rows has first > last.  Needs no GPU."""
    rows4 = (C.c_int * (4 * max(1, int(n))))()
    dom = grid.domain()
    check(lib().wrfb200_host_split_plan(C.byref(dom), grid.its, grid.ite, grid.jts, grid.jte, grid.kts, grid.kte,
                                        int(n), rows4))
    return [tuple(rows4[4 * p:4 * p + 4]) for p in range(int(n))]


def default_last_kernel() -> int:
    """Kernel id the most recent ``advance_mu_t`` call of this thread ran."""
    k = C.c_int()
    check(lib().wrfb200_default_last_kernel(C.byref(k)))
    return k.value


def default_last_transfer() -> int:
    """How the most recent host-array ``advance_mu_t`` call of this thread moved its arrays: ``TRANSFER_DIRECT``
    (every array page-locked, copied directly), ``TRANSFER_MIXED`` (some pageable ones staged through the library's
    pinned bounce buffers) or ``TRANSFER_STAGED`` (all of them).  Raises ``WrfB200Error`` (``ERR_STATE``) before the
    thread's first host-array call."""
    r = C.c_int()
    check(lib().wrfb200_default_last_transfer(C.byref(r)))
    return r.value


def default_last_cache() -> int:
    """What the most recent ``advance_mu_t`` call of this thread (either precision, host arrays or device tensors)
    did with its cache: ``CACHE_REUSED`` (its domain's device state, or device-pointer wrapper, was already there),
    ``CACHE_CREATED`` or ``CACHE_EVICTED`` (created after the least recently used domains were freed).  Raises
    ``WrfB200Error`` (``ERR_STATE``) when no call of this thread has reached its cache yet."""
    r = C.c_int()
    check(lib().wrfb200_default_last_cache(C.byref(r)))
    return r.value


def synth_fields(grid: Grid, seed: int = 20240617, names: Iterable[str] = FIELDS, pinned: bool = False,
                 dx_m: float = 12000.0) -> Dict[str, np.ndarray]:
    """Deterministic atmosphere-like fields for ``grid``'s memory extents (wrfb200_synth_field).
    With ``pinned`` the arrays are views of page-locked torch tensors (kept alive via ``.base``)."""
    dom = grid.domain()
    out = {}
    keep = []
    for n in names:
        shape = grid.shape_of(n)
        if pinned:
            import torch
            tt = torch.empty(shape, dtype=torch.float32, pin_memory=True)
            a = tt.numpy()
            keep.append(tt)
        else:
            a = np.empty(shape, dtype=np.float32)
        check(lib().wrfb200_synth_field(FIELD_ID[n], C.c_uint64(seed), C.byref(dom), float(dx_m),
                                        C.c_void_p(a.ctypes.data)))
        out[n] = a
    if pinned:
        out["__pinned__"] = keep
    return out


def compare(a: np.ndarray, b: np.ndarray) -> dict:
    """The reference's comparison metrics (common.cu:68-164) between two arrays: float32 (or anything else but
    float64, read as float32) through wrfb200_compare, two float64 arrays through wrfb200_compare_r8 in binary64.
    A float64 array against any other dtype raises TypeError rather than narrowing it."""
    r8 = [getattr(x, "dtype", None) == np.float64 for x in (a, b)]
    if any(r8) and not all(r8):
        raise TypeError("compare needs both arrays float64 (binary64 metrics) or neither, got "
                        f"{getattr(a, 'dtype', type(a).__name__)} and {getattr(b, 'dtype', type(b).__name__)}")
    dt, fn, res = ((np.float64, lib().wrfb200_compare_r8, _lib.CompareResultR8()) if all(r8) else
                   (np.float32, lib().wrfb200_compare, _lib.CompareResult()))
    a = np.ascontiguousarray(a, dtype=dt)
    b = np.ascontiguousarray(b, dtype=dt)
    if a.shape != b.shape:
        raise ValueError("shape mismatch")
    check(fn(C.c_void_p(a.ctypes.data), C.c_void_p(b.ctypes.data), a.size, C.byref(res)))
    return {"n": res.n, "n_equal": res.n_equal, "n_different": res.n_different, "max_rel": res.max_rel,
            "max_abs": res.max_abs, "rmse": res.rmse, "max_ulp": res.max_ulp}
