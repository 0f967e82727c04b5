"""Host-array calls on pageable arrays: the staged route, which copies them through the library's pinned bounce buffers
with its own host threads instead of handing pageable memory to the driver.  Every result is compared with the oracle
bit for bit, and the caller's inputs and every cell outside the written range must keep their bytes.  Page-locked
arrays keep the direct route; wrfb200_default_last_transfer reports which route a call took."""
import ctypes as C
import os
import threading
import time
import warnings

import numpy as np
import pytest

import wrf_model_cuda_sample_b200 as wrf
from wrf_model_cuda_sample_b200 import _lib
from oracle import loader
from tests import cases
from tests.test_r8 import SCALARS_12KM as SCALARS_12KM_64
from tests.test_r8 import assert_bit_equal64, assert_outside_untouched64, oracle64, random_fields64
from tests.test_shared_tiles import tiles_from_threads, tiling

gpu = pytest.mark.gpu

# (nx, ny, nz, halo).  74x61x28: the tutorial domain, one slab.  97x53x17 at halo 3: ragged.  425x300x35: 16 slabs
# on a padded mirror (landed in the device staging buffer and re-pitched).  1020x1100x4 at halo 2: 1024-wide rows,
# an unpadded mirror (2-D copies out of the bounce buffer), and 2-D fields larger than one bounce buffer.
SHAPES = [(74, 61, 28, 5), (97, 53, 17, 3), (425, 300, 35, 5), (1020, 1100, 4, 2)]


def _have_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def _threads():
    return len(os.listdir("/proc/self/task"))


@pytest.fixture(autouse=True)
def _release_afterwards():
    yield
    if _have_gpu():
        wrf.set_default_devices(None)
        wrf.lib().wrfb200_release_cache()


def _route():
    return wrf.default_last_transfer()


def _single_call(g, fin, scalars, what):
    want = cases.copy_fields(fin)
    loader.oracle_c(want, g, scalars, tiles=64)
    got = cases.copy_fields(fin)
    wrf.call_with_fields(got, g, *scalars)
    assert _route() == wrf.TRANSFER_STAGED, what
    cases.assert_bit_equal(got, want, what=what)
    cases.assert_inputs_untouched(got, fin)
    cases.assert_outside_untouched(got, fin, g)


# ================================================================ CPU
def test_python_api_is_exported():
    assert callable(wrf.default_last_transfer) and "default_last_transfer" in wrf.__all__
    assert (wrf.TRANSFER_DIRECT, wrf.TRANSFER_MIXED, wrf.TRANSFER_STAGED) == (0, 1, 2)


def test_no_host_array_call_yet_is_a_state_error():
    """Thread-local: a thread that has made no host-array call has no route to report."""
    out = {}

    def body():
        r = C.c_int(-7)
        out["rc"] = wrf.lib().wrfb200_default_last_transfer(C.byref(r))
        out["route"] = r.value
        out["msg"] = wrf.lib().wrfb200_last_error()

    t = threading.Thread(target=body)
    t.start()
    t.join()
    assert out["rc"] == _lib.ERR_STATE and out["route"] == -7 and b"no host-array call" in out["msg"]
    assert wrf.lib().wrfb200_default_last_transfer(None) == _lib.ERR_INVALID_ARG


# ================================================================ GPU: single calls
@gpu
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_single_call_pageable(shape):
    nx, ny, nz, halo = shape
    g = cases.grid(nx, ny, nz, halo=halo)
    _single_call(g, wrf.synth_fields(g, seed=nx + ny), cases.SCALARS_12KM, f"pageable {shape} ")


@gpu
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_single_call_pageable_r8(shape):
    nx, ny, nz, halo = shape
    g = cases.grid(nx, ny, nz, halo=halo)
    fin = random_fields64(g, seed=nx + nz)
    want = oracle64(g, fin, SCALARS_12KM_64, tiles=64)
    got = cases.copy_fields(fin)
    wrf.call_with_fields(got, g, *SCALARS_12KM_64)
    assert _route() == wrf.TRANSFER_STAGED
    assert_bit_equal64(got, want, what=f"pageable r8 {shape} ")
    for n in wrf.INPUT_FIELDS:
        if n not in cases.OUTPUTS:
            assert np.array_equal(got[n].view(np.uint64), fin[n].view(np.uint64)), n
    assert_outside_untouched64(got, fin, g)


@gpu
@pytest.mark.parametrize("variant", sorted(cases.FLAG_VARIANTS))
def test_single_call_pageable_flag_variants(variant):
    g = cases.grid(74, 61, 28, halo=5, variant=variant)
    _single_call(g, cases.random_fields(g, seed=5), cases.SCALARS_12KM, f"pageable {variant} ")


@gpu
def test_single_call_pageable_full_size():
    """1800x1060x50, the size whose pageable call the staged route exists for."""
    g = cases.grid(1800, 1060, 50, halo=5)
    _single_call(g, wrf.synth_fields(g), cases.SCALARS_3KM, "pageable 1800x1060x50 ")


@gpu
def test_loop_entry_pageable():
    g = cases.grid(425, 300, 35, halo=5)
    fin = wrf.synth_fields(g, seed=8)
    want = cases.oracle_loop(g, fin, cases.SCALARS_12KM, 6)
    got = cases.copy_fields(fin)
    wrf.call_with_fields(got, g, *cases.SCALARS_12KM, nsteps=6)
    assert _route() == wrf.TRANSFER_STAGED
    cases.assert_bit_equal(got, want, what="pageable _loop ")
    cases.assert_inputs_untouched(got, fin)
    cases.assert_outside_untouched(got, fin, g)


# ================================================================ GPU: acoustic-loop residency
@gpu
def test_acoustic_loop_residency_pageable():
    """u, v change on the host between calls (the stand-in advance_uv).  Two loop constants changed on the host after
    the priming call must be ignored: resident calls upload u and v only."""
    g = cases.grid(425, 300, 35, halo=5)
    fin = wrf.synth_fields(g, seed=21)
    c, nsteps = 0.25, 4
    want = cases.oracle_loop(g, fin, cases.SCALARS_12KM, nsteps, c=c)
    ubox, vbox = cases.standin_boxes(g, g.ids, g.ide, g.jds, g.jde)
    got = cases.copy_fields(fin)
    with wrf.acoustic_loop():
        for s in range(nsteps):
            wrf.call_with_fields(got, g, *cases.SCALARS_12KM)
            assert _route() == wrf.TRANSFER_STAGED
            if s == 0:
                got["ft"][...] = np.float32(1.0e3)
                got["mut"][...] = np.float32(5.0e4)
            if s + 1 < nsteps:
                cases.standin_advance_uv_numpy(got, g, c, ubox, vbox)
    cases.assert_bit_equal(got, want, names=cases.OUTPUTS + ("u", "v"), what="pageable residency ")
    cases.assert_outside_untouched(got, fin, g)


# ================================================================ GPU: mixed and pinned calls
@gpu
def test_mixed_and_pinned_calls_keep_the_direct_route():
    g = cases.grid(425, 300, 35, halo=5)
    pinned = wrf.synth_fields(g, seed=3, pinned=True)
    keep = pinned.pop("__pinned__")
    fin = cases.copy_fields(pinned)
    want = cases.copy_fields(fin)
    loader.oracle_c(want, g, cases.SCALARS_12KM, tiles=64)
    for n in wrf.FIELDS:                       # restore the pinned arrays' inputs between the calls below
        pinned[n][...] = fin[n]
    wrf.call_with_fields(pinned, g, *cases.SCALARS_12KM)
    assert _route() == wrf.TRANSFER_DIRECT
    cases.assert_bit_equal(pinned, want, what="pinned ")
    cases.assert_outside_untouched(pinned, fin, g)
    # some of each kind: outputs, 3-D, 2-D and 1-D inputs on both routes
    for n in wrf.FIELDS:
        pinned[n][...] = fin[n]
    mixed = {n: (pinned[n] if i % 2 else fin[n].copy()) for i, n in enumerate(wrf.FIELDS)}
    wrf.call_with_fields(mixed, g, *cases.SCALARS_12KM)
    assert _route() == wrf.TRANSFER_MIXED
    cases.assert_bit_equal(mixed, want, what="mixed ")
    cases.assert_inputs_untouched(mixed, fin)
    cases.assert_outside_untouched(mixed, fin, g)
    del keep


# ================================================================ GPU: split calls and shared tiles
@gpu
def test_split_call_pageable():
    g = cases.grid(425, 300, 35, halo=5)
    fin = cases.random_fields(g, seed=30)
    want = cases.copy_fields(fin)
    loader.oracle_c(want, g, cases.SCALARS_12KM, tiles=64)
    got = cases.copy_fields(fin)
    with wrf.default_devices([0, 0]):
        wrf.call_with_fields(got, g, *cases.SCALARS_12KM)
        assert _route() == wrf.TRANSFER_STAGED
    cases.assert_bit_equal(got, want, what="pageable split ")
    cases.assert_inputs_untouched(got, fin)
    cases.assert_outside_untouched(got, fin, g)


@gpu
@pytest.mark.parametrize("tiles", [(4, 1), (1, 4), (2, 2)])
def test_shared_tiles_pageable(tiles):
    g = cases.grid(425, 300, 35, halo=5)
    fin = cases.random_fields(g, seed=31)
    want = cases.copy_fields(fin)
    loader.oracle_c(want, g, cases.SCALARS_12KM, tiles=64)
    got = cases.copy_fields(fin)
    try:
        with wrf.shared_tiles():
            tiles_from_threads(got, g, tiling(g, *tiles), cases.SCALARS_12KM)
    finally:
        wrf.set_shared_tiles(False)
    cases.assert_bit_equal(got, want, what=f"pageable shared tiles {tiles} ")
    cases.assert_inputs_untouched(got, fin)
    cases.assert_outside_untouched(got, fin, g)


# ================================================================ GPU: return semantics
@gpu
def test_caller_may_reuse_its_arrays_when_the_call_returns():
    g = cases.grid(425, 300, 35, halo=5)
    fin = wrf.synth_fields(g, seed=40)
    want = cases.copy_fields(fin)
    loader.oracle_c(want, g, cases.SCALARS_12KM, tiles=64)
    got = cases.copy_fields(fin)
    wrf.call_with_fields(got, g, *cases.SCALARS_12KM)
    for n in wrf.FIELDS:
        if n not in cases.OUTPUTS:
            got[n][...] = np.float32(-9.0)
    time.sleep(0.2)                             # nothing of the call may still be writing
    cases.assert_bit_equal(got, want, what="outputs after the inputs were overwritten ")
    cases.assert_outside_untouched(got, fin, g)


@gpu
def test_refused_call_leaves_the_arrays_untouched():
    g = cases.grid(40, 20, 6, halo=1, variant="open")
    fin = cases.random_fields(g, seed=3)
    got = cases.copy_fields(fin)
    with pytest.raises(wrf.WrfB200Error) as e:
        wrf.call_with_fields(got, g.with_tile(1, 40, 0, 20), *cases.SCALARS_12KM)   # j_start - 1 outside memory
    assert e.value.status == _lib.ERR_INVALID_ARG and "ring" in str(e.value)
    for n in wrf.FIELDS:
        assert np.array_equal(cases.bits(got[n]), cases.bits(fin[n])), n
    want = cases.copy_fields(fin)
    loader.oracle_c(want, g, cases.SCALARS_12KM)
    wrf.call_with_fields(got, g, *cases.SCALARS_12KM)
    assert _route() == wrf.TRANSFER_STAGED
    cases.assert_bit_equal(got, want, what="after a refused call ")


# ================================================================ GPU: the worker pool
@gpu
def test_release_cache_joins_the_workers():
    g = cases.grid(425, 300, 35, halo=5)
    fin = wrf.synth_fields(g, seed=50)
    want = cases.copy_fields(fin)
    loader.oracle_c(want, g, cases.SCALARS_12KM, tiles=64)
    pinned = wrf.synth_fields(g, seed=50, pinned=True)
    keep = pinned.pop("__pinned__")
    wrf.lib().wrfb200_release_cache()
    wrf.call_with_fields(pinned, g, *cases.SCALARS_12KM)          # the runtime's own threads, no pool
    assert _route() == wrf.TRANSFER_DIRECT
    wrf.lib().wrfb200_release_cache()
    base = _threads()
    pool = min(16, len(os.sched_getaffinity(0)))
    for _ in range(2):
        got = cases.copy_fields(fin)
        wrf.call_with_fields(got, g, *cases.SCALARS_12KM)
        assert _route() == wrf.TRANSFER_STAGED
        assert _threads() >= base + pool
        cases.assert_bit_equal(got, want, what="pageable, pool (re)started ")
        wrf.lib().wrfb200_release_cache()
        assert _threads() == base
    del keep


@gpu
def test_forked_child_forgets_the_pool():
    """A child forked after a staged call has none of the parent's workers and no usable CUDA context: it only
    releases the cache and exits, without waiting for workers it does not have."""
    g = cases.grid(425, 300, 35, halo=5)
    fin = wrf.synth_fields(g, seed=60)
    want = cases.copy_fields(fin)
    loader.oracle_c(want, g, cases.SCALARS_12KM, tiles=64)
    got = cases.copy_fields(fin)
    wrf.call_with_fields(got, g, *cases.SCALARS_12KM)
    assert _route() == wrf.TRANSFER_STAGED
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", DeprecationWarning)      # fork() of a multi-threaded process
        pid = os.fork()
    if pid == 0:
        rc = 1
        try:
            rc = wrf.lib().wrfb200_release_cache()
        finally:
            os._exit(0 if rc == 0 else 1)
    deadline = time.monotonic() + 60
    status = None
    while time.monotonic() < deadline:
        done, st = os.waitpid(pid, os.WNOHANG)
        if done == pid:
            status = st
            break
        time.sleep(0.05)
    if status is None:
        os.kill(pid, 9)
        os.waitpid(pid, 0)
        pytest.fail("the forked child did not exit within 60 s")
    assert os.WIFEXITED(status) and os.WEXITSTATUS(status) == 0
    got = cases.copy_fields(fin)
    wrf.call_with_fields(got, g, *cases.SCALARS_12KM)
    assert _route() == wrf.TRANSFER_STAGED
    cases.assert_bit_equal(got, want, what="parent after the fork ")
