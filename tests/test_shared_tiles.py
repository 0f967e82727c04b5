"""Shared-tiles mode (wrfb200_set_shared_tiles): the host-array calls of WRF's OpenMP tile loop, made from several
threads, share one device-resident patch.  Without a GPU: the entry points, their errors and the C harness's usage.
On the GPU: tiles from concurrent threads bit-identical to the oracle in binary32 and binary64, per-tile residency
whichever thread calls, one mirror set instead of one per thread, the patch device, the errors and the mode off."""
import os
import subprocess
import threading

import numpy as np
import pytest

import wrf_model_cuda_sample_b200 as wrf
from wrf_model_cuda_sample_b200 import _lib
from oracle import loader
from tests import cases
from tests.test_r8 import (SCALARS_12KM as SCALARS_12KM_64, SCALARS_3KM as SCALARS_3KM_64, assert_bit_equal64,
                           assert_outside_untouched64, oracle64, oracle_loop64, random_fields64)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu


def _have_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def _gpu_count():
    import torch
    return torch.cuda.device_count()


@pytest.fixture(autouse=True)
def _mode_off_afterwards():
    yield
    if _have_gpu():
        wrf.set_shared_tiles(False)
        wrf.set_default_devices(None)
        wrf.lib().wrfb200_release_cache()


# ================================================================ helpers
def cuts(lo, hi, n):
    """lo..hi cut into n contiguous ranges (ragged when n does not divide the length)."""
    m = hi - lo + 1
    edges = [lo + m * p // n for p in range(n + 1)]
    return [(edges[p], edges[p + 1] - 1) for p in range(n)]


def tiling(g, ni, nj):
    """ni x nj WRF tiles (its, ite, jts, jte) covering the domain ids..ide x jds..jde."""
    return [(a, b, c, d) for (c, d) in cuts(g.jds, g.jde, nj) for (a, b) in cuts(g.ids, g.ide, ni)]


def run_threads(n, body):
    """body(t) in n threads started together; the first exception of any thread is raised here."""
    errors = [None] * n

    def run(t):
        try:
            body(t)
        except BaseException as e:                               # noqa: BLE001 -- re-raised in the caller
            errors[t] = e

    threads = [threading.Thread(target=run, args=(t,)) for t in range(n)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    for e in errors:
        if e is not None:
            raise e


def tiles_from_threads(fields, g, tiles, scalars, nsteps=1):
    """One call per tile, tile t from thread t, the calls released together by a barrier so that they overlap."""
    barrier = threading.Barrier(len(tiles))

    def body(t):
        barrier.wait()
        wrf.call_with_fields(fields, g.with_tile(*tiles[t]), *scalars, nsteps=nsteps)

    run_threads(len(tiles), body)


# ================================================================ CPU: entry points and argument checks
def test_python_api_is_exported():
    assert callable(wrf.set_shared_tiles) and callable(wrf.shared_tiles)
    assert "set_shared_tiles" in wrf.__all__ and "shared_tiles" in wrf.__all__


def test_turning_the_mode_off_needs_no_gpu():
    assert wrf.lib().wrfb200_set_shared_tiles(0) == _lib.OK
    wrf.set_shared_tiles(False)


@pytest.mark.skipif(_have_gpu(), reason="GPU present: covered by the gpu tests")
def test_enabling_needs_a_gpu():
    with pytest.raises(wrf.WrfB200Error) as e:
        wrf.set_shared_tiles(True)
    assert e.value.status == _lib.ERR_CUDA and "no CPU fallback" in str(e.value)
    with pytest.raises(wrf.WrfB200Error):
        with wrf.shared_tiles():
            pass


def test_tiling_helper_covers_the_domain_once():
    g = cases.grid(74, 61, 28)
    for ni, nj in ((4, 1), (1, 4), (2, 2)):
        seen = np.zeros((g.jde + 1, g.ide + 1), dtype=int)
        for its, ite, jts, jte in tiling(g, ni, nj):
            seen[jts:jte + 1, its:ite + 1] += 1
        assert (seen[1:, 1:] == 1).all()
    assert {b - a + 1 for a, b in cuts(1, 74, 4)} == {18, 19}             # ragged


def _build_tiles_harness(tmp_path):
    exe = str(tmp_path / "c_tiles_harness")
    libdir = os.path.join(ROOT, "wrf_model_cuda_sample_b200")
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    subprocess.run([cc, "-O1", "-ffp-contract=off", os.path.join(ROOT, "tests", "c_tiles_harness.c"),
                    "-I", os.path.join(ROOT, "include"), "-L", libdir, "-lwrfb200", f"-Wl,-rpath,{libdir}",
                    "-lpthread", "-o", exe], check=True)
    return exe


def test_tiles_harness_builds_and_checks_usage(tmp_path):
    r = subprocess.run([_build_tiles_harness(tmp_path)], capture_output=True, text=True)
    assert r.returncode == 2 and "usage" in r.stderr


@pytest.mark.skipif(_have_gpu(), reason="GPU present")
def test_tiles_harness_fails_loudly_without_gpu(tmp_path):
    r = subprocess.run([_build_tiles_harness(tmp_path), str(tmp_path)], capture_output=True, text=True)
    assert r.returncode == 3 and "no CPU fallback" in r.stderr


# ================================================================ GPU: 1. bit-exact tiles from concurrent threads
SIZES = [(74, 61, 28), (425, 300, 35)]
TILINGS = [(4, 1), (1, 4), (2, 2)]


@gpu
@pytest.mark.parametrize("variant", sorted(cases.FLAG_VARIANTS))
def test_concurrent_tiles_bit_exact(variant):
    for nx, ny, nz in SIZES:
        g = cases.grid(nx, ny, nz, halo=5, variant=variant)
        fin = cases.random_fields(g, seed=nx + nz)
        want = cases.copy_fields(fin)
        loader.oracle_c(want, g, cases.SCALARS_12KM)
        for ni, nj in TILINGS:
            got = cases.copy_fields(fin)
            with wrf.shared_tiles():
                tiles_from_threads(got, g, tiling(g, ni, nj), cases.SCALARS_12KM)
            what = f"{(nx, ny, nz)}/{variant}/{ni}x{nj} "
            cases.assert_bit_equal(got, want, what=what)
            cases.assert_inputs_untouched(got, fin)
            cases.assert_outside_untouched(got, fin, g)


@gpu
@pytest.mark.parametrize("variant", sorted(cases.FLAG_VARIANTS))
def test_concurrent_tiles_bit_exact_r8(variant):
    for nx, ny, nz in SIZES:
        g = cases.grid(nx, ny, nz, halo=5, variant=variant)
        fin = random_fields64(g, seed=nx + nz)
        want = oracle64(g, fin, SCALARS_12KM_64)
        for ni, nj in TILINGS:
            got = cases.copy_fields(fin)
            with wrf.shared_tiles():
                tiles_from_threads(got, g, tiling(g, ni, nj), SCALARS_12KM_64)
            what = f"r8 {(nx, ny, nz)}/{variant}/{ni}x{nj} "
            assert_bit_equal64(got, want, what=what)
            assert_bit_equal64(got, fin, names=[n for n in wrf.FIELDS if n not in cases.OUTPUTS], what=what + "inputs ")
            assert_outside_untouched64(got, fin, g)


@gpu
def test_loop_entry_per_tile():
    """wrfb200_advance_mu_t_loop per tile: nsteps on the tile's device-resident state, u, v fixed."""
    g = cases.grid(300, 41, 9, halo=3, variant="periodic_specified")
    fin = cases.random_fields(g, seed=5)
    want = cases.oracle_loop(g, fin, cases.SCALARS_12KM, 6)
    got = cases.copy_fields(fin)
    with wrf.shared_tiles():
        tiles_from_threads(got, g, tiling(g, 2, 2), cases.SCALARS_12KM, nsteps=6)
    cases.assert_bit_equal(got, want, what="loop entry ")
    cases.assert_outside_untouched(got, fin, g)


# ================================================================ GPU: 2. residency across threads
def _residency_loop(g, fin, scalars, tiles, nsteps, c, poke=None):
    """nsteps inside acoustic_loop, tile (t + step) % n from thread t, the stand-in advance_uv on the host arrays
    between steps (while the threads wait).  poke(fields) runs once after the priming step."""
    got = cases.copy_fields(fin)
    ubox, vbox = cases.standin_boxes(g, g.ids, g.ide, g.jds, g.jde)
    n = len(tiles)
    start, done = threading.Barrier(n + 1), threading.Barrier(n + 1)

    errors = []

    def body(t):
        for step in range(nsteps):
            start.wait()
            errors.append(_catch(lambda: wrf.call_with_fields(got, g.with_tile(*tiles[(t + step) % n]), *scalars)))
            done.wait()                                          # every thread takes part in every step

    threads = [threading.Thread(target=body, args=(t,)) for t in range(n)]
    with wrf.shared_tiles():
        with wrf.acoustic_loop():
            for th in threads:
                th.start()
            for step in range(nsteps):
                start.wait()
                done.wait()
                if step + 1 < nsteps:
                    cases.standin_advance_uv_numpy(got, g, c, ubox, vbox)
                if step == 0 and poke is not None:
                    poke(got)
            for th in threads:
                th.join()
    for e in errors:
        if e is not None:
            raise e
    return got


def _catch(fn, *args):
    try:
        fn(*args)
        return None
    except BaseException as e:                                   # noqa: BLE001 -- re-raised by the caller
        return e


def _poke_ft(f):
    f["ft"] += f["ft"].dtype.type(1.0)                         # a loop constant: resident calls must not re-read it


@gpu
@pytest.mark.parametrize("poke", [False, True], ids=["plain", "ft_changed_after_priming"])
def test_residency_across_threads(poke):
    g = cases.grid(425, 300, 35, halo=5, variant="specified")  # slab-pipelined tiles (staged copies, re-pitch)
    fin = wrf.synth_fields(g, seed=21)
    c, nsteps = 0.25, 6
    want = cases.oracle_loop(g, fin, cases.SCALARS_12KM, nsteps, c=c)
    got = _residency_loop(g, fin, cases.SCALARS_12KM, tiling(g, 2, 2), nsteps, c, poke=_poke_ft if poke else None)
    cases.assert_bit_equal(got, want, names=cases.OUTPUTS + ("u", "v"), what="shared residency ")
    cases.assert_outside_untouched(got, fin, g)


@gpu
@pytest.mark.parametrize("poke", [False, True], ids=["plain", "ft_changed_after_priming"])
def test_residency_across_threads_r8(poke):
    g = cases.grid(200, 150, 20, halo=5, variant="open")
    fin = random_fields64(g, seed=8)
    c, nsteps = 0.25, 6
    want = oracle_loop64(g, fin, SCALARS_3KM_64, nsteps, c=c)
    got = _residency_loop(g, fin, SCALARS_3KM_64, tiling(g, 1, 4), nsteps, c, poke=_poke_ft if poke else None)
    assert_bit_equal64(got, want, names=cases.OUTPUTS + ("u", "v"), what="r8 shared residency ")
    assert_outside_untouched64(got, fin, g)


@gpu
def test_a_tile_the_loop_has_not_seen_gets_a_full_upload():
    """Within one loop the tiling changes after the first step: every tile of the new tiling is new to the loop and
    must read the current host state (including the changed ft), not a stale device copy."""
    g = cases.grid(200, 96, 12, halo=5, variant="specified")
    fin = cases.random_fields(g, seed=31)
    got = cases.copy_fields(fin)
    with wrf.shared_tiles(), wrf.acoustic_loop():
        tiles_from_threads(got, g, tiling(g, 2, 2), cases.SCALARS_12KM)
        got["ft"] += np.float32(1.0)
        mid = cases.copy_fields(got)
        tiles_from_threads(got, g, tiling(g, 4, 1), cases.SCALARS_12KM)
    loader.oracle_c(mid, g, cases.SCALARS_12KM)
    cases.assert_bit_equal(got, mid, what="new tiling ")


# ================================================================ GPU: 3. one mirror set
def _mirror_bytes(g, esize=4):
    idim, jdim, kdim = g.ime - g.ims + 1, g.jme - g.jms + 1, g.kme - g.kms + 1
    pitch = -(-idim * esize // 128) * 128 // esize
    return esize * (len(wrf.FIELDS_3D) * pitch * kdim * jdim + len(wrf.FIELDS_2D) * pitch * jdim
                    + len(wrf.FIELDS_1D) * kdim)


def _device_bytes_taken(fields, g, tiles, scalars, shared, device=0):
    """Device memory taken once every thread has made its tile's call (the threads still alive), then released."""
    import torch
    torch.cuda.synchronize(device)
    free0 = torch.cuda.mem_get_info(device)[0]
    n = len(tiles)
    primed, measured = threading.Barrier(n + 1), threading.Barrier(n + 1)

    def body(t):
        try:
            wrf.call_with_fields(fields, g.with_tile(*tiles[t]), *scalars)
        finally:
            primed.wait()
            measured.wait()
            wrf.lib().wrfb200_release_cache()                    # this thread's own caches, before it ends

    errors = []
    threads = [threading.Thread(target=lambda t=t: errors.append(_catch(body, t))) for t in range(n)]
    if shared:
        wrf.set_shared_tiles(True)
    for th in threads:
        th.start()
    primed.wait()
    taken = free0 - torch.cuda.mem_get_info(device)[0]
    measured.wait()
    for th in threads:
        th.join()
    wrf.set_shared_tiles(False)
    for e in errors:
        if e is not None:
            raise e
    return taken


@gpu
def test_one_mirror_set_for_eight_threads():
    g = cases.grid(1800, 1060, 50, halo=5, variant="specified")
    fin = wrf.synth_fields(g)
    want = cases.copy_fields(fin)
    loader.oracle_c(want, g, cases.SCALARS_3KM, tiles=64)
    tiles = tiling(g, 1, 8)
    mirrors = _mirror_bytes(g)
    got = cases.copy_fields(fin)
    shared = _device_bytes_taken(got, g, tiles, cases.SCALARS_3KM, shared=True)
    cases.assert_bit_equal(got, want, what="8 shared tiles ")
    got = cases.copy_fields(fin)
    per_thread = _device_bytes_taken(got, g, tiles, cases.SCALARS_3KM, shared=False)
    cases.assert_bit_equal(got, want, what="8 per-thread tiles ")
    assert shared < 1.5 * mirrors, (shared, mirrors)
    assert per_thread > 6 * mirrors, (per_thread, mirrors)           # today's behaviour: one set per thread


# ================================================================ GPU: 4. the patch device
@gpu
def test_patch_device_is_the_enabling_threads_device():
    import torch
    if _gpu_count() < 2:
        pytest.skip(f"{_gpu_count()} GPU(s) on this box, 2 needed")
    g = cases.grid(425, 300, 35, halo=5, variant="specified")
    fin = cases.random_fields(g, seed=3)
    want = cases.copy_fields(fin)
    loader.oracle_c(want, g, cases.SCALARS_12KM)
    got = cases.copy_fields(fin)
    tiles = tiling(g, 2, 2)
    prev = torch.cuda.current_device()
    torch.cuda.set_device(1)
    try:
        wrf.set_shared_tiles(True)                                   # patch device 1
    finally:
        torch.cuda.set_device(prev)
    free = [torch.cuda.mem_get_info(d)[0] for d in (0, 1)]
    barrier = threading.Barrier(len(tiles))
    seen = {}

    def body(t):
        torch.cuda.set_device(0)
        barrier.wait()
        wrf.call_with_fields(got, g.with_tile(*tiles[t]), *cases.SCALARS_12KM)
        seen[t] = torch.cuda.current_device()

    run_threads(len(tiles), body)
    taken = [free[d] - torch.cuda.mem_get_info(d)[0] for d in (0, 1)]
    assert seen == {t: 0 for t in range(len(tiles))}, seen          # each thread's device is unchanged
    assert taken[1] >= _mirror_bytes(g), taken                      # the mirrors live on device 1 ...
    assert taken[0] < _mirror_bytes(g) // 2, taken                  # ... and not on device 0
    cases.assert_bit_equal(got, want, what="patch device 1 ")


# ================================================================ GPU: 5. errors, and the mode off
@gpu
def test_device_list_other_than_the_patch_device_is_unsupported():
    g = cases.grid(96, 40, 10, halo=5, variant="specified")
    fin = cases.random_fields(g, seed=13)
    want = cases.copy_fields(fin)
    loader.oracle_c(want, g, cases.SCALARS_12KM)
    wrf.set_shared_tiles(True)
    statuses = {}

    def body(t):
        got = cases.copy_fields(fin)
        with wrf.default_devices([0, 0] if t == 0 else [0]):
            try:
                wrf.call_with_fields(got, g, *cases.SCALARS_12KM)
                statuses[t] = _lib.OK
                cases.assert_bit_equal(got, want, what="list [0] ")      # the patch device alone is allowed
            except wrf.WrfB200Error as e:
                statuses[t] = (e.status, "patch device" in str(e))

    run_threads(2, body)
    assert statuses == {0: (_lib.ERR_UNSUPPORTED, True), 1: _lib.OK}, statuses
    if _gpu_count() >= 2:
        got = cases.copy_fields(fin)
        with wrf.default_devices([1]):
            with pytest.raises(wrf.WrfB200Error) as e:
                wrf.call_with_fields(got, g, *cases.SCALARS_12KM)
        assert e.value.status == _lib.ERR_UNSUPPORTED


@gpu
def test_mode_off_behaves_as_before():
    """After set_shared_tiles(False) each thread gets its own mirrors again, and a device list splits the call."""
    g = cases.grid(425, 300, 35, halo=5, variant="specified")
    fin = cases.random_fields(g, seed=17)
    want = cases.copy_fields(fin)
    loader.oracle_c(want, g, cases.SCALARS_12KM)
    tiles = tiling(g, 1, 2)
    mirrors = _mirror_bytes(g)
    got = cases.copy_fields(fin)
    shared = _device_bytes_taken(got, g, tiles, cases.SCALARS_12KM, shared=True)
    cases.assert_bit_equal(got, want, what="on ")
    got = cases.copy_fields(fin)
    off = _device_bytes_taken(got, g, tiles, cases.SCALARS_12KM, shared=False)
    cases.assert_bit_equal(got, want, what="off ")
    assert shared < 1.5 * mirrors and off >= 2 * mirrors, (shared, off, mirrors)
    got = cases.copy_fields(fin)
    with wrf.default_devices([0, 0]):
        wrf.call_with_fields(got, g, *cases.SCALARS_12KM)
    cases.assert_bit_equal(got, want, what="split, mode off ")


@gpu
def test_set_shared_tiles_restores_and_release_frees():
    g = cases.grid(74, 61, 28)
    fin = wrf.synth_fields(g)
    want = cases.copy_fields(fin)
    loader.oracle_c(want, g, cases.SCALARS_12KM)
    with wrf.shared_tiles():
        with wrf.shared_tiles(False):
            got = cases.copy_fields(fin)
            wrf.call_with_fields(got, g, *cases.SCALARS_12KM)         # per-thread path
            cases.assert_bit_equal(got, want, what="inner off ")
        got = cases.copy_fields(fin)
        tiles_from_threads(got, g, tiling(g, 2, 2), cases.SCALARS_12KM)
        cases.assert_bit_equal(got, want, what="restored on ")
        wrf.lib().wrfb200_release_cache()                             # frees the shared patch; the next call rebuilds
        got = cases.copy_fields(fin)
        tiles_from_threads(got, g, tiling(g, 2, 2), cases.SCALARS_12KM)
        cases.assert_bit_equal(got, want, what="after release ")


# ================================================================ GPU: 6. from C, as WRF calls it
@gpu
def test_tiles_harness_matches_oracle(tmp_path):
    out = tmp_path / "out"
    out.mkdir()
    r = subprocess.run([_build_tiles_harness(tmp_path), str(out)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    g = cases.grid(150, 110, 16, halo=5, variant="specified")
    want = cases.oracle_loop(g, wrf.synth_fields(g, seed=99), cases.SCALARS_3KM, 6, c=0.25)
    got = {n: np.fromfile(out / f"field{wrf.FIELD_ID[n]}.bin", dtype=np.float32).reshape(g.shape_of(n))
           for n in cases.OUTPUTS + ("u", "v")}
    cases.assert_bit_equal(got, want, names=cases.OUTPUTS + ("u", "v"), what="C tiles harness ")
