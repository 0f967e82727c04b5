"""2-D (i,j) patch decomposition and the one-cell halo exchange for advance_mu_t, one process per GPU.

The reference's only multi-GPU mechanism is a 1-D j-slab split over three hard-coded devices whose
overlapping rows are re-uploaded from the host on every call, with no GPU-to-GPU traffic at all
(/root/reference/advance_mu_t_no_async.cu:12, :87-162, :276-298).  Here every rank owns a patch
``ips:ipe x jps:jpe`` of the global domain with a halo, calls the operator with ITS tile and the GLOBAL
domain extents -- so the boundary clamps of module_small_step_em.f90:91-106 fire on edge ranks only,
exactly WRF's own patch mechanism -- and the one-cell ring the stencil reads (:143-146, :241-245) moves
between neighbours with ``torch.distributed`` point-to-point operations (NCCL over NVLink on GPUs; gloo in
the CPU tests).  Corners are never read by the routine, so there are at most four neighbours.

What moves when (SURVEY.md section 8e):
  * every acoustic step, BEFORE the step: ``u`` east halo (read at i+1), ``v`` north halo (read at j+1)
  * every acoustic step, AFTER the step (for the caller's next advance_uv): ``mudf``/``mu``/``muts`` halos
  * once per RK sub-step: the constants ``u_1, muu, msfuy`` (east), ``v_1, muv, msfvx_inv`` (north),
    ``t_1`` (all four sides)
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Callable, Dict, List, Optional, Sequence, Tuple

import numpy as np

from ._lib import EAST, NORTH, SOUTH, WEST
from .advance_mu_t import Grid

OPPOSITE = {WEST: EAST, EAST: WEST, SOUTH: NORTH, NORTH: SOUTH}
SIDE_NAME = {WEST: "west", EAST: "east", SOUTH: "south", NORTH: "north"}

# halo sides each field must have filled for one advance_mu_t call
STEP_HALOS: Tuple[Tuple[str, Tuple[int, ...]], ...] = (("u", (EAST,)), ("v", (NORTH,)))
CONSTANT_HALOS: Tuple[Tuple[str, Tuple[int, ...]], ...] = (
    ("u_1", (EAST,)), ("muu", (EAST,)), ("msfuy", (EAST,)),
    ("v_1", (NORTH,)), ("muv", (NORTH,)), ("msfvx_inv", (NORTH,)),
    ("t_1", (WEST, EAST, SOUTH, NORTH)),
)
OUTPUT_HALOS: Tuple[Tuple[str, Tuple[int, ...]], ...] = (
    ("mudf", (WEST, SOUTH)), ("mu", (WEST, SOUTH)), ("muts", (WEST, SOUTH)),
)


def split_range(lo: int, hi: int, parts: int, index: int) -> Tuple[int, int]:
    """WRF-style even split of lo..hi (inclusive) into ``parts`` contiguous chunks."""
    n = hi - lo + 1
    a = lo + (n * index) // parts
    b = lo + (n * (index + 1)) // parts - 1
    return a, b


def choose_process_grid(world: int, nx: int, ny: int) -> Tuple[int, int]:
    """(px, py).  j-slabs (px=1) by default: a j-row halo is contiguous in the (i,k,j) layout and the
    strip that waits for it is one full-width row; fall back to a 2-D grid only if rows run out."""
    if ny // world >= 8:
        return 1, world
    best = (1, world)
    for px in range(1, world + 1):
        if world % px == 0:
            py = world // px
            if ny // py >= 8 and nx // px >= 128:
                best = (px, py)
                break
    return best


@dataclass(frozen=True)
class Decomposition:
    """A px x py process grid over the global domain of ``global_grid``.

    ``wrap_x`` / ``wrap_y`` make the exchange periodic across the domain edge (WRF's periodic_x / periodic_y): the
    neighbours are cyclic, and the edge rank's column ide (row jde), a copy of column ids (row jds), is halo to the
    exchange -- see ``exchange_extents``.  A rank can then be its own neighbour (px = 1 / py = 1) or the same rank
    can sit on both sides of an axis (px = 2 / py = 2)."""
    global_grid: Grid
    px: int
    py: int
    halo: int = 1
    wrap_x: bool = False
    wrap_y: bool = False

    @property
    def world(self) -> int:
        return self.px * self.py

    def coords(self, rank: int) -> Tuple[int, int]:
        return rank % self.px, rank // self.px

    def rank_of(self, pi: int, pj: int) -> Optional[int]:
        if self.wrap_x:
            pi %= self.px
        if self.wrap_y:
            pj %= self.py
        if 0 <= pi < self.px and 0 <= pj < self.py:
            return pj * self.px + pi
        return None

    def neighbour(self, rank: int, side: int) -> Optional[int]:
        pi, pj = self.coords(rank)
        if side == WEST:
            return self.rank_of(pi - 1, pj)
        if side == EAST:
            return self.rank_of(pi + 1, pj)
        if side == SOUTH:
            return self.rank_of(pi, pj - 1)
        return self.rank_of(pi, pj + 1)

    def patch_extents(self, rank: int) -> Tuple[int, int, int, int]:
        g = self.global_grid
        pi, pj = self.coords(rank)
        ips, ipe = split_range(g.ids, g.ide, self.px, pi)
        jps, jpe = split_range(g.jds, g.jde, self.py, pj)
        return ips, ipe, jps, jpe

    def exchange_extents(self, rank: int) -> Tuple[int, int, int, int]:
        """The patch as the halo exchange sees it: on a wrapped axis the edge rank ends at ide-1 (jde-1), and its
        column ide (row jde) is the halo cell that receives the wrap (csrc/comm.cu does the same)."""
        g = self.global_grid
        pi, pj = self.coords(rank)
        ips, ipe, jps, jpe = self.patch_extents(rank)
        if self.wrap_x and pi == self.px - 1:
            ipe = g.ide - 1
        if self.wrap_y and pj == self.py - 1:
            jpe = g.jde - 1
        return ips, ipe, jps, jpe

    def patch_grid(self, rank: int) -> Grid:
        """The rank's call: global domain extents, memory = patch + halo, tile = patch."""
        g = self.global_grid
        ips, ipe, jps, jpe = self.patch_extents(rank)
        h = self.halo
        return Grid(g.ids, g.ide, g.jds, g.jde, g.kde, ips - h, ipe + h, jps - h, jpe + h, g.kms, g.kme,
                    ips, ipe, jps, jpe, g.kts, g.kte, g.periodic_x, g.specified, g.nested)

    def interior_and_boundary_tiles(self, rank: int):
        """Split the rank's tile (its exchange extents) into the part that reads no per-step halo (interior) and
        the strips that do: the last column if there is an east neighbour (u at i+1), the last row if there is a
        north neighbour (v at j+1).  Returns (interior | None, [strips])."""
        ips, ipe, jps, jpe = self.exchange_extents(rank)
        east = self.neighbour(rank, EAST) is not None
        north = self.neighbour(rank, NORTH) is not None
        ie = ipe - 1 if east else ipe
        je = jpe - 1 if north else jpe
        interior = (ips, ie, jps, je) if (ie >= ips and je >= jps) else None
        strips = []
        if north:
            strips.append((ips, ipe, jpe, jpe))
        if east and je >= jps:
            strips.append((ipe, ipe, jps, je))
        return interior, strips


class HaloExchanger:
    """Posts the point-to-point operations of one halo exchange.

    ``pack(field, side, width) -> tensor`` returns a dense buffer holding the ``width`` cells just inside
    the patch edge ``side``; ``recv_buffer(field, side, width) -> tensor`` returns the buffer to receive
    into; ``unpack(field, side, width, tensor)`` stores a received buffer into the halo outside ``side``.
    The exchanger is transport-agnostic: the buffers are CUDA tensors under NCCL and CPU tensors under gloo.
    """

    def __init__(self, decomp: Decomposition, rank: int, pack: Callable, recv_buffer: Callable, unpack: Callable,
                 group=None):
        self.decomp = decomp
        self.rank = rank
        self.pack = pack
        self.recv_buffer = recv_buffer
        self.unpack = unpack
        self.group = group

    def plan(self, halos: Sequence[Tuple[str, Sequence[int]]]):
        """[(kind, field, side, peer)] in an order that is identical on every rank."""
        ops = []
        for field, sides in halos:
            for side in sides:
                # my halo on `side` is filled by the neighbour on that side ...
                src = self.decomp.neighbour(self.rank, side)
                if src is not None:
                    ops.append(("recv", field, side, src))
                # ... and I fill the same halo of the neighbour on the opposite side with my inside edge
                dst = self.decomp.neighbour(self.rank, OPPOSITE[side])
                if dst is not None:
                    ops.append(("send", field, OPPOSITE[side], dst))
        return ops

    def start(self, halos, width: int = 1):
        """Pack and post all sends/receives; returns an opaque token for ``finish``.  A rank that is its own
        neighbour (a wrapped axis with one rank on it) packs and unpacks locally, with no point-to-point op."""
        import torch.distributed as dist
        p2p, recvs = [], []
        for kind, field, side, peer in self.plan(halos):
            if peer == self.rank:
                if kind == "send":                   # my inside edge on `side` is my own halo on the opposite side
                    recvs.append((field, OPPOSITE[side], self.pack(field, side, width)))
            elif kind == "send":
                p2p.append(dist.P2POp(dist.isend, self.pack(field, side, width), peer, self.group))
            else:
                buf = self.recv_buffer(field, side, width)
                recvs.append((field, side, buf))
                p2p.append(dist.P2POp(dist.irecv, buf, peer, self.group))
        works = dist.batch_isend_irecv(p2p) if p2p else []
        return works, recvs, width

    def finish(self, token) -> None:
        works, recvs, width = token
        for w in works:
            w.wait()
        for field, side, buf in recvs:
            self.unpack(field, side, width, buf)

    def exchange(self, halos, width: int = 1) -> None:
        self.finish(self.start(halos, width))


class GpuPatchHalo:
    """pack / recv_buffer / unpack for a device-resident ``Patch`` with preallocated torch buffers of the patch's
    dtype (float64 for a real*8 patch)."""

    def __init__(self, patch, decomp: Decomposition, rank: int, device):
        self.patch = patch
        self.ext = decomp.exchange_extents(rank)
        self.grid = decomp.patch_grid(rank)
        self.device = device
        self._bufs: Dict[Tuple[str, int, str], object] = {}

    def _buf(self, field, side, width, role):
        import torch
        from ._lib import FIELDS_3D
        key = (field, side, role)
        if key not in self._bufs:
            ips, ipe, jps, jpe = self.ext
            nk = self.grid.shape3[1] if field in FIELDS_3D else 1
            n = (width * nk * (jpe - jps + 1)) if side in (WEST, EAST) else ((ipe - ips + 1) * nk * width)
            dtype = torch.float64 if self.patch.dtype is np.float64 else torch.float32
            self._bufs[key] = torch.empty(n, dtype=dtype, device=self.device)
        return self._bufs[key]

    def pack(self, field, side, width):
        buf = self._buf(field, side, width, "send")
        self.patch.pack_halo(field, side, width, *self.ext, buf)
        return buf

    def recv_buffer(self, field, side, width):
        return self._buf(field, side, width, "recv")

    def unpack(self, field, side, width, buf):
        self.patch.unpack_halo(field, side, width, *self.ext, buf)


def connect_fused(patch, decomp: Decomposition, rank: int, allgather: Callable[[bytes], List[bytes]]) -> None:
    """Bootstrap the fused (peer-mapped) halo exchange of csrc/comm.cu for ``patch``.

    ``allgather(blob) -> [blob of rank 0, blob of rank 1, ...]`` is the caller's transport (torch.distributed
    in bench.py; MPI_Allgather in a WRF host; a list when several ranks live in one process).  After this the
    acoustic loop needs no collective library: ``patch.comm_push_constants()`` once per RK sub-step, then
    ``patch.comm_loop(n)`` or ``comm_push_uv(); comm_step()`` per step.  The decomposition's wrap flags are set on
    the patch first."""
    ips, ipe, jps, jpe = decomp.patch_extents(rank)
    patch.comm_set_wrap(decomp.wrap_x, decomp.wrap_y)
    info = patch.comm_init(decomp.px, decomp.py, rank, ips, ipe, jps, jpe)
    patch.comm_connect(allgather(info))


def torch_allgather_bytes(group=None, device=None) -> Callable[[bytes], List[bytes]]:
    """An ``allgather`` for connect_fused over torch.distributed (NCCL needs the bytes on the device)."""
    def gather(blob: bytes) -> List[bytes]:
        import torch
        import torch.distributed as dist
        world = dist.get_world_size(group)
        mine = torch.frombuffer(bytearray(blob), dtype=torch.uint8)
        if device is not None:
            mine = mine.to(device)
        out = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(out, mine, group=group)
        return [bytes(t.cpu().numpy().tobytes()) for t in out]
    return gather
