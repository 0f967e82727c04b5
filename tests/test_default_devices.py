"""The host-array advance_mu_t call split over several devices (wrfb200_set_default_devices): the split plan and
argument checks without a GPU; on the GPU, every split bit-identical to the oracle, in binary32 and binary64, with
ids repeated on one B200 and with distinct devices where the box has them."""
import ctypes as C
import os
from dataclasses import replace

import numpy as np
import pytest

import wrf_model_cuda_sample_b200 as wrf
from wrf_model_cuda_sample_b200 import _lib
from oracle import loader
from tests import cases
from tests.test_r8 import (SCALARS_12KM as SCALARS_12KM_64, SCALARS_3KM as SCALARS_3KM_64, assert_bit_equal64,
                           assert_outside_untouched64, oracle64, oracle_loop64, random_fields64, to64)

RAGGED = [(130, 9, 5, 1), (257, 6, 4, 2), (5, 5, 3, 1), (383, 3, 17, 7), (64, 64, 2, 4)]
REPEATED = [[0, 0], [0, 0, 0], [0] * 5]


def _have_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def _gpu_count():
    import torch
    return torch.cuda.device_count()


# ================================================================ CPU: the split plan and argument checks
def plan_restated(g, n):
    """The split rule in Python: the computed rows cut with j_start + nj*p/n, memory = rows +- 1."""
    i0, i1, j0, j1, k0, k1 = g.bounds()
    nj = 0 if (i0 > i1 or j0 > j1 or k0 > k1) else j1 - j0 + 1
    out = []
    for p in range(n):
        ja, jb = j0 + nj * p // n, j0 + nj * (p + 1) // n - 1
        out.append((ja, jb, ja - 1, jb + 1) if ja <= jb else (ja, jb, ja, jb))
    return out


def test_split_plan_covers_every_row_once():
    rs = np.random.RandomState(7)
    checked = 0
    for _ in range(60):
        nx, ny, nz, halo = int(rs.randint(3, 50)), int(rs.randint(3, 40)), int(rs.randint(2, 12)), int(rs.randint(1, 4))
        for variant in cases.FLAG_VARIANTS:
            whole = cases.grid(nx, ny, nz, halo=halo, variant=variant)
            jts = int(rs.randint(1, ny + 1)); jte = int(rs.randint(jts, ny + 1))
            its = int(rs.randint(1, nx + 1)); ite = int(rs.randint(its, nx + 1))
            for g in (whole, whole.with_tile(its, ite, jts, jte)):
                i0, i1, j0, j1, k0, k1 = g.bounds()
                nonempty = i0 <= i1 and j0 <= j1 and k0 <= k1
                rows = list(range(j0, j1 + 1)) if nonempty else []
                for n in range(1, 10):
                    plan = wrf.host_split_plan(g, n)
                    assert plan == plan_restated(g, n), (g, n)
                    covered = [j for (a, b, _, _) in plan for j in range(a, b + 1)]
                    assert covered == rows, (g, n)                     # each row once, ascending
                    for a, b, ma, mb in plan:
                        if a <= b:
                            assert (ma, mb) == (a - 1, b + 1) and g.jms <= ma and mb <= g.jme
                        else:
                            assert ma > mb
                    if len(rows) < n:
                        assert sum(1 for (a, b, _, _) in plan if a > b) == n - len(rows)
                    checked += 1
    assert checked > 5000


def test_split_plan_examples():
    g = cases.grid(74, 61, 28, halo=5, variant="specified")       # computed rows 2..59
    assert wrf.host_split_plan(g, 1) == [(2, 59, 1, 60)]
    assert wrf.host_split_plan(g, 2) == [(2, 30, 1, 31), (31, 59, 30, 60)]
    small = cases.grid(40, 6, 6, halo=2, variant="open")          # 5 computed rows 1..5, 8 parts
    plan = wrf.host_split_plan(small, 8)
    assert [p for p in plan if p[0] <= p[1]] == [(1, 1, 0, 2), (2, 2, 1, 3), (3, 3, 2, 4), (4, 4, 3, 5), (5, 5, 4, 6)]


def test_split_plan_and_device_list_reject_bad_arguments():
    lib = wrf.lib()
    g = cases.grid(20, 10, 5, halo=1)
    dom = g.domain()
    rows = (C.c_int * (4 * 65))()
    for n in (0, -1, 65):
        assert lib.wrfb200_host_split_plan(C.byref(dom), 1, 20, 1, 10, 1, 5, n, rows) == _lib.ERR_INVALID_ARG
    assert lib.wrfb200_host_split_plan(None, 1, 20, 1, 10, 1, 5, 2, rows) == _lib.ERR_INVALID_ARG
    assert lib.wrfb200_host_split_plan(C.byref(dom), 1, 20, 1, 10, 1, 5, 2, None) == _lib.ERR_INVALID_ARG
    # the computed range needs a ring row inside memory, as for the call itself
    bad = cases.grid(20, 10, 5, halo=1, variant="open").with_tile(1, 20, 0, 10)
    with pytest.raises(wrf.WrfB200Error) as e:
        wrf.host_split_plan(bad, 2)
    assert e.value.status == _lib.ERR_INVALID_ARG and "ring" in str(e.value)
    ids = (C.c_int * 2)(0, 0)
    for n in (-1, 65):
        assert lib.wrfb200_set_default_devices(ids, n) == _lib.ERR_INVALID_ARG
    assert lib.wrfb200_set_default_devices(None, 2) == _lib.ERR_INVALID_ARG
    assert lib.wrfb200_set_default_devices(None, 0) == _lib.OK
    wrf.set_default_devices(None)


@pytest.mark.skipif(_have_gpu(), reason="GPU present: covered by the gpu tests")
def test_device_list_needs_a_gpu():
    with pytest.raises(wrf.WrfB200Error) as e:
        wrf.set_default_devices([0, 0])
    assert e.value.status == _lib.ERR_CUDA and "no CPU fallback" in str(e.value)
    wrf.set_default_devices([])                                  # n = 0 needs no device


# ================================================================ GPU: ids repeated on one device
gpu = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _no_device_list():
    yield
    if _have_gpu():
        wrf.set_default_devices(None)
        wrf.lib().wrfb200_release_cache()


def split_call(fin, g, scalars, devices, nsteps=1):
    got = cases.copy_fields(fin)
    with wrf.default_devices(devices):
        wrf.call_with_fields(got, g, *scalars, nsteps=nsteps)
    return got


@gpu
@pytest.mark.parametrize("devices", REPEATED, ids=lambda d: "x".join(map(str, d)))
@pytest.mark.parametrize("variant", sorted(cases.FLAG_VARIANTS))
def test_split_call_tutorial_domain(variant, devices):
    g = cases.grid(74, 61, 28, halo=5, variant=variant)
    fin = wrf.synth_fields(g)
    want = cases.copy_fields(fin)
    loader.oracle_c(want, g, cases.SCALARS_12KM)
    got = split_call(fin, g, cases.SCALARS_12KM, devices)
    cases.assert_bit_equal(got, want, what=f"{variant}/{devices} ")
    cases.assert_inputs_untouched(got, fin)
    cases.assert_outside_untouched(got, fin, g)


@gpu
@pytest.mark.parametrize("devices", REPEATED, ids=lambda d: "x".join(map(str, d)))
def test_split_call_ragged_and_conus12(devices):
    """Ragged rows and halos, and 425x300x35 (each part of it below the slab pipeline's size in binary32)."""
    shapes = [(s, v) for s in RAGGED for v in ("specified", "periodic_open")] + [((425, 300, 35, 5), "specified")]
    for (nx, ny, nz, halo), variant in shapes:
        g = cases.grid(nx, ny, nz, halo=halo, variant=variant)
        fin = cases.random_fields(g, seed=nx + nz, adversarial=(nz == 4))
        want = cases.copy_fields(fin)
        loader.oracle_c(want, g, cases.SCALARS_3KM, tiles=16)
        got = split_call(fin, g, cases.SCALARS_3KM, devices)
        cases.assert_bit_equal(got, want, what=f"{(nx, ny, nz, halo)}/{variant}/{devices} ")
        cases.assert_inputs_untouched(got, fin)
        cases.assert_outside_untouched(got, fin, g)


@gpu
@pytest.mark.parametrize("devices", REPEATED, ids=lambda d: "x".join(map(str, d)))
@pytest.mark.parametrize("variant", sorted(cases.FLAG_VARIANTS))
def test_split_call_r8_tutorial_domain(variant, devices):
    g = cases.grid(74, 61, 28, halo=5, variant=variant)
    fin = random_fields64(g, seed=2)
    want = oracle64(g, fin, SCALARS_12KM_64)
    got = split_call(fin, g, SCALARS_12KM_64, devices)
    assert_bit_equal64(got, want, what=f"r8 {variant}/{devices} ")
    assert_bit_equal64(got, fin, names=[n for n in wrf.FIELDS if n not in cases.OUTPUTS], what="inputs ")
    assert_outside_untouched64(got, fin, g)


@gpu
@pytest.mark.parametrize("devices", REPEATED, ids=lambda d: "x".join(map(str, d)))
def test_split_call_r8_ragged_and_conus12(devices):
    """binary64; the parts of 425x300x35 are slab-pipelined (staged copies and device re-pitch)."""
    shapes = [(s, v) for s in RAGGED for v in ("specified", "periodic_open")] + [((425, 300, 35, 5), "specified")]
    for (nx, ny, nz, halo), variant in shapes:
        g = cases.grid(nx, ny, nz, halo=halo, variant=variant)
        fin = random_fields64(g, seed=nx + nz, adversarial=(nz == 4))
        want = oracle64(g, fin, SCALARS_3KM_64, tiles=16)
        got = split_call(fin, g, SCALARS_3KM_64, devices)
        assert_bit_equal64(got, want, what=f"r8 {(nx, ny, nz, halo)}/{variant}/{devices} ")
        assert_outside_untouched64(got, fin, g)


@gpu
def test_split_loop_entry_and_sub_tile():
    g = cases.grid(300, 41, 9, halo=3, variant="periodic_specified")
    fin = cases.random_fields(g, seed=5)
    want = cases.oracle_loop(g, fin, cases.SCALARS_12KM, 6)
    got = split_call(fin, g, cases.SCALARS_12KM, [0, 0, 0], nsteps=6)
    cases.assert_bit_equal(got, want, what="loop entry ")
    cases.assert_outside_untouched(got, fin, g)
    tile = g.with_tile(40, 290, 9, 33)
    want_t = cases.copy_fields(fin)
    loader.oracle_c(want_t, tile, cases.SCALARS_12KM)
    got_t = split_call(fin, tile, cases.SCALARS_12KM, [0, 0, 0])
    cases.assert_bit_equal(got_t, want_t, what="sub-tile ")
    cases.assert_outside_untouched(got_t, fin, tile)
    fin64 = random_fields64(g, seed=6)
    want64 = oracle_loop64(g, fin64, SCALARS_12KM_64, 6)
    got64 = split_call(fin64, g, SCALARS_12KM_64, [0, 0, 0], nsteps=6)
    assert_bit_equal64(got64, want64, what="r8 loop entry ")


@gpu
def test_split_acoustic_loop_residency():
    """The residency loop of the single-device test with four parts: first call all inputs, then u, v only; the host
    changes u, v between calls; first-sight pinning on (the whole arrays are registered once)."""
    g = cases.grid(425, 300, 35, halo=5, variant="specified")
    fin = wrf.synth_fields(g, seed=21)
    c, nsteps = 0.25, 4
    want = cases.oracle_loop(g, fin, cases.SCALARS_12KM, nsteps, c=c)
    ubox, vbox = cases.standin_boxes(g, g.ids, g.ide, g.jds, g.jde)
    got = cases.copy_fields(fin)
    wrf.lib().wrfb200_set_host_pinning(1)
    try:
        with wrf.default_devices([0, 0, 0, 0]):
            with wrf.acoustic_loop():
                for s in range(nsteps):
                    wrf.call_with_fields(got, g, *cases.SCALARS_12KM)
                    if s + 1 < nsteps:
                        cases.standin_advance_uv_numpy(got, g, c, ubox, vbox)
        cases.assert_bit_equal(got, want, names=cases.OUTPUTS + ("u", "v"), what="split residency ")
        cases.assert_outside_untouched(got, fin, g)
    finally:
        wrf.lib().wrfb200_set_host_pinning(0)
        wrf.lib().wrfb200_release_cache()


@gpu
def test_more_parts_than_rows():
    g = cases.grid(40, 6, 6, halo=2, variant="open")            # 5 computed rows
    fin = cases.random_fields(g, seed=11)
    want = cases.copy_fields(fin)
    loader.oracle_c(want, g, cases.SCALARS_12KM)
    got = split_call(fin, g, cases.SCALARS_12KM, [0] * 8)
    cases.assert_bit_equal(got, want, what="8 parts, 5 rows ")
    cases.assert_outside_untouched(got, fin, g)


@gpu
def test_list_changes_between_calls():
    g = cases.grid(96, 40, 10, halo=5, variant="specified")
    fin = cases.random_fields(g, seed=13)
    want = cases.copy_fields(fin)
    loader.oracle_c(want, g, cases.SCALARS_12KM)
    for devices in ([0, 0], [0, 0, 0], [], [0], [0, 0]):
        wrf.set_default_devices(devices)
        got = cases.copy_fields(fin)
        wrf.call_with_fields(got, g, *cases.SCALARS_12KM)
        cases.assert_bit_equal(got, want, what=f"list {devices} ")
        wrf.lib().wrfb200_release_cache()


def _threads():
    return len(os.listdir("/proc/self/task"))


@gpu
def test_no_thread_outlives_a_call():
    g = cases.grid(74, 61, 28, halo=5)
    fin = wrf.synth_fields(g)
    got = cases.copy_fields(fin)
    wrf.set_default_devices([0] * 4)
    wrf.call_with_fields(got, g, *cases.SCALARS_12KM)           # warm-up: mirrors, streams, runtime threads
    for nsteps in (1, 1, 3):
        before = _threads()
        wrf.call_with_fields(got, g, *cases.SCALARS_12KM, nsteps=nsteps)
        assert _threads() == before


@gpu
def test_failing_split_call_reports_like_the_single_device_call():
    g = cases.grid(40, 20, 6, halo=1, variant="open")
    fin = cases.random_fields(g, seed=3)
    no_ring = g.with_tile(1, 40, 0, 20)                          # j_start - 1 is outside memory
    kts2 = replace(g, kts=2)                                     # fails inside every part (make_params)
    for bad in (no_ring, kts2):
        statuses = []
        for devices in ([], [0, 0, 0]):
            got = cases.copy_fields(fin)
            wrf.set_default_devices(devices)
            with pytest.raises(wrf.WrfB200Error) as e:
                wrf.call_with_fields(got, bad, *cases.SCALARS_12KM)
            statuses.append(e.value.status)
            if devices and bad is kts2:
                assert "device 0, rows j=" in str(e.value)
        assert statuses[0] == statuses[1], statuses
    want = cases.copy_fields(fin)
    loader.oracle_c(want, g, cases.SCALARS_12KM)
    got = split_call(fin, g, cases.SCALARS_12KM, [0, 0, 0])
    cases.assert_bit_equal(got, want, what="after a failing call ")


# ================================================================ GPU: 1800x1060x50, 6-step loop entry
@pytest.fixture(scope="module")
def conus3():
    g = cases.grid(1800, 1060, 50, halo=5, variant="specified")
    fin = wrf.synth_fields(g)
    want = {n: fin[n].copy() for n in wrf.FIELDS}
    for _ in range(6):
        loader.oracle_c(want, g, cases.SCALARS_3KM, tiles=64)
    return g, fin, want


@pytest.fixture(scope="module")
def conus3_r8():
    g = cases.grid(1800, 1060, 50, halo=5, variant="specified")
    fin = to64(wrf.synth_fields(g))
    want = oracle_loop64(g, fin, SCALARS_3KM_64, 6, tiles=64)
    return g, fin, want


def _full_size(case, devices, r8):
    g, fin, want = case
    got = {n: fin[n].copy() for n in wrf.FIELDS}
    with wrf.default_devices(devices):
        wrf.call_with_fields(got, g, *(SCALARS_3KM_64 if r8 else cases.SCALARS_3KM), nsteps=6)
    if r8:
        assert_bit_equal64(got, want, what=f"conus3 r8 {devices} ")
        assert_outside_untouched64(got, fin, g)
    else:
        cases.assert_bit_equal(got, want, what=f"conus3 {devices} ")
        cases.assert_outside_untouched(got, fin, g)
    wrf.lib().wrfb200_release_cache()


@gpu
def test_full_size_four_parts_on_one_device(conus3):
    _full_size(conus3, [0, 0, 0, 0], r8=False)


DISTINCT = [pytest.param(n, id=f"{n}gpus") for n in (2, 4, 8)]


@gpu
@pytest.mark.parametrize("r8", [False, True], ids=["f32", "r8"])
@pytest.mark.parametrize("n", DISTINCT)
def test_full_size_distinct_devices(request, n, r8):
    if _gpu_count() < n:                                         # before the fixture builds its 6-step reference
        pytest.skip(f"{_gpu_count()} GPU(s) on this box, {n} needed")
    _full_size(request.getfixturevalue("conus3_r8" if r8 else "conus3"), list(range(n)), r8=r8)
