"""The launch geometry of the TMA kernel (tile columns, remainder strips, 2-row / 1-row block rows), checked on the CPU
through the host-only wrfb200_pipe_plan: every computed column and row is covered exactly once, the shared-memory
budget holds, and the shapes of the BASELINE configs are the ones the profiles were taken with."""
import ctypes as C

import numpy as np
import pytest

import wrf_model_cuda_sample_b200 as wrf
from tests import cases
from wrf_model_cuda_sample_b200._lib import ERR_UNSUPPORTED

TI, STRIP_W, STRIP_ROWS, SLOTS = 128, 16, 2, 2 * 148
KEYS = ("cfg", "tj", "stages", "nbx", "nby2", "nby1", "strip_blocks", "strip_i0", "grid", "smem")
SMEM_SM, SMEM_RESERVE = 227 * 1024, 1024                 # usable shared memory per SM; reserved per resident block
PIPE_MAX_NK = 337


def pipe_smem(tj, stages, nk, tabs=True):
    """Dynamic shared memory of a pipe block (csrc/amt_pipe.cu pipe_smem): ring + stash + level tables + barriers."""
    return (8 * stages * 832 + tj * nk * TI + (4 * nk if tabs else 0)) * 4 + 8 * stages * 8


def plan(g, slots=SLOTS):
    out = (C.c_longlong * 10)()
    d = g.domain()
    rc = wrf.lib().wrfb200_pipe_plan(C.byref(d), g.its, g.ite, g.jts, g.jte, g.kts, g.kte, slots, out)
    assert rc == 0, wrf.lib().wrfb200_last_error()
    return dict(zip(KEYS, list(out)))


def check_cover(g, p):
    i0, i1, j0, j1, k0, k1 = g.bounds()
    mi0, mi1 = i0 - g.ims, i1 - g.ims                     # memory indices, as the kernels see them
    nj = j1 - j0 + 1
    origin = mi0 & ~31
    cols = np.zeros(mi1 + 2 * TI, dtype=int)
    for bx in range(p["nbx"]):                            # tile columns
        lo, hi = origin + bx * TI, origin + bx * TI + TI - 1
        cols[max(lo, mi0):min(hi, mi1) + 1] += 1
    if p["strip_blocks"]:
        assert p["strip_i0"] == origin + p["nbx"] * TI and mi1 - p["strip_i0"] + 1 <= STRIP_W
        cols[p["strip_i0"]:mi1 + 1] += 1
        assert p["strip_blocks"] == -(-nj // STRIP_ROWS)  # strips sweep all computed rows
    assert (cols[mi0:mi1 + 1] == 1).all() and cols[:mi0].sum() == 0 and cols[mi1 + 1:].sum() == 0
    # rows: 2-row block rows first, then 1-row block rows
    assert 2 * p["nby2"] + p["nby1"] >= nj and 2 * (p["nby2"] - 1) + p["nby1"] < nj if p["nby1"] == 0 else \
        2 * p["nby2"] + p["nby1"] == nj
    assert p["grid"] == p["strip_blocks"] + p["nbx"] * (p["nby2"] + p["nby1"])
    # shared memory: at least one block fits an SM, and two whenever the leanest two-block configuration (the level
    # tables in L2) would fit twice
    blocks = SMEM_SM // (p["smem"] + SMEM_RESERVE)
    assert blocks >= 1
    nk = k1 - k0 + 1
    if 2 * (pipe_smem(1, 2, nk, tabs=False) + SMEM_RESERVE) <= SMEM_SM:
        assert blocks >= 2, (nk, p)


def test_baseline_shapes_match_the_profiled_launches():
    g = wrf.Grid.from_shape(1800, 1060, 50, halo=5)
    p = plan(g)
    assert (p["cfg"], p["nbx"], p["nby2"], p["nby1"], p["strip_blocks"], p["grid"]) == (22, 14, 529, 0, 529, 7935)  # profiles/r2_launches_conus3.csv
    p = plan(wrf.Grid.from_shape(1800, 133, 50, halo=5))
    assert p["cfg"] == 22 and p["nbx"] == 14 and p["nby1"] >= 15 and p["grid"] == 1087     # r2_ncu_details_pipe_patch8.txt
    p = plan(wrf.Grid.from_shape(425, 300, 35, halo=5))
    assert (p["cfg"], p["nbx"], p["nby2"], p["nby1"], p["strip_blocks"], p["grid"]) == (22, 4, 149, 0, 0, 596)      # r2_ncu_details_pipe_conus12.txt
    p = plan(wrf.Grid.from_shape(512, 512, 120, halo=5))
    assert p["cfg"] == 62 and p["tj"] == 1 and 2 * (p["smem"] + 1024) <= 227 * 1024          # two blocks per SM for nk = 119
    p = plan(wrf.Grid.from_shape(74, 61, 28, halo=5))
    assert p["nby2"] == 0 and p["nby1"] == 58                                                # less than one wave: all 1-row


@pytest.mark.parametrize("variant", sorted(cases.FLAG_VARIANTS))
def test_every_column_and_row_is_covered_exactly_once(variant):
    rs = np.random.RandomState(hash(variant) % 1000)
    for _ in range(150):
        nx, ny, nz = int(rs.randint(5, 2100)), int(rs.randint(5, 400)), int(rs.randint(2, 471))
        halo = int(rs.randint(1, 8))
        g = cases.grid(nx, ny, nz, halo=halo, variant=variant)
        i0, i1, j0, j1, _, _ = g.bounds()
        if i0 > i1 or j0 > j1:
            continue
        # a random sub-tile, as WRF calls the routine per tile
        if rs.rand() < 0.5:
            its = int(rs.randint(1, nx + 1)); ite = int(rs.randint(its, nx + 1))
            jts = int(rs.randint(1, ny + 1)); jte = int(rs.randint(jts, ny + 1))
            g = g.with_tile(its, ite, jts, jte)
            i0, i1, j0, j1, _, _ = g.bounds()
            if i0 > i1 or j0 > j1:
                continue
        out = (C.c_longlong * 10)()
        d = g.domain()
        rc = wrf.lib().wrfb200_pipe_plan(C.byref(d), g.its, g.ite, g.jts, g.jte, g.kts, g.kte,
                                         int(rs.choice([SLOTS, 2 * 132, 64])), out)
        if nz - 1 > PIPE_MAX_NK:
            assert rc == ERR_UNSUPPORTED, (nx, ny, nz, rc)
            continue
        assert rc == 0, wrf.lib().wrfb200_last_error()
        check_cover(g, dict(zip(KEYS, list(out))))


# The ladder of the pipe kernel's configurations over the level count nk: (cfg at nj >= 2, cfg at nj = 1).
LADDER = {59: (22, 13), 60: (13, 13), 66: (13, 13), 67: (12, 12), 117: (12, 12), 118: (62, 62), 120: (62, 62),
          121: (14, 14), 236: (14, 14), 237: (12, 12), 337: (12, 12)}


def plan_rc(g, slots=SLOTS):
    out = (C.c_longlong * 10)()
    d = g.domain()
    rc = wrf.lib().wrfb200_pipe_plan(C.byref(d), g.its, g.ite, g.jts, g.jte, g.kts, g.kte, slots, out)
    return rc, dict(zip(KEYS, list(out)))


def test_level_ladder_boundaries():
    """Both ends of every configuration, for 2-row-capable tiles and for a single row; refused past nk = 337."""
    for nk, (cfg, cfg_one_row) in LADDER.items():
        for ny, want in ((40, cfg), (4, cfg_one_row)):            # specified: 37 computed rows, or one
            g = cases.grid(300, ny, nk + 1)
            p = plan(g)
            assert p["cfg"] == want, (nk, ny, p)
            # one block per SM from nk = 121 on (the last-resort 12 included), two before
            assert SMEM_SM // (p["smem"] + SMEM_RESERVE) == (1 if nk >= 121 else 2), (nk, p)
            check_cover(g, p)
    for ny in (40, 4):
        rc, _ = plan_rc(cases.grid(300, ny, PIPE_MAX_NK + 2))
        assert rc == ERR_UNSUPPORTED
        msg = wrf.lib().wrfb200_last_error().decode()
        assert "338" in msg and "337" in msg, msg


def test_no_plan_selects_the_two_row_four_stage_configuration():
    """cfg 24 (<2, 4>) would need nk <= 119 and is only considered from nk = 121 on: it must never appear."""
    for ny in (4, 5, 200):                                         # specified: nj = 1, 2, 197
        for nk in range(1, 461):
            rc, p = plan_rc(cases.grid(140, ny, nk + 1))
            if nk > PIPE_MAX_NK:
                assert rc == ERR_UNSUPPORTED, nk
            else:
                assert rc == 0 and p["cfg"] in (22, 13, 12, 62, 14), (nk, ny, p)


def test_plan_rejects_empty_and_unsupported_calls():
    g = cases.grid(3, 3, 4, halo=1, variant="specified")           # empty index sets
    out = (C.c_longlong * 10)()
    d = g.domain()
    assert wrf.lib().wrfb200_pipe_plan(C.byref(d), g.its, g.ite, g.jts, g.jte, g.kts, g.kte, 0, out) == 1
    g = cases.grid(40, 30, 10, halo=2)
    d = g.domain()
    assert wrf.lib().wrfb200_pipe_plan(C.byref(d), g.its, g.ite, g.jts, g.jte, 2, g.kte, 0, out) == 2
    assert wrf.lib().wrfb200_pipe_plan(None, 1, 2, 1, 2, 1, 2, 0, out) == 1
