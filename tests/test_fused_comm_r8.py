"""The fused multi-GPU path (csrc/comm.cu) on real*8 patches: wrfb200_comm_init_r8 / wrfb200_comm_loop_r8 and the
fused double2 tile kernel (amt_tile_kernel_r8<TJ, true>).  As in tests/test_fused_comm.py the ranks are handles of ONE
process on device 0, so the flag protocol, the peer stores and the kernels are those of the multi-process runs
(tests/c_comm_harness_r8.c, tools/multi_gpu_check.py --dtype float64).
Bar: every rank's patch BIT-IDENTICAL to the binary64 checker loop over the whole domain, halos poisoned beforehand;
inputs are float64 with low mantissa bits a float cannot hold."""
import ctypes as C
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

import wrf_model_cuda_sample_b200 as wrf
from wrf_model_cuda_sample_b200 import _lib, parallel
from tests import cases, r8_checkers

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F64 = np.float64
C_UV = 0.25
SCALARS = (1.0 / 3000.0, 1.0 / 3000.0, 3.0, 0.1)          # doubles, as the C harness passes them
gpu = pytest.mark.gpu


def widen64(f):
    """x * (1 + 2^-40) in binary64: the float32 synthetic field with its low mantissa bits filled."""
    return {n: a.astype(F64) * (1.0 + 2.0 ** -40) for n, a in f.items() if isinstance(a, np.ndarray)}


def checker_loop64(G, whole, nsteps, c=None, tiles=0):
    """nsteps of the binary64 C checker over the whole domain, with the stand-in advance_uv between steps."""
    f = cases.copy_fields(whole)
    ubox, vbox = cases.standin_boxes(G, G.ids, G.ide, G.jds, G.jde)
    for s in range(nsteps):
        r8_checkers.oracle_c_r8(f, G, SCALARS, tiles=tiles)
        if c is not None and s + 1 < nsteps:
            cases.standin_advance_uv_numpy(f, G, c, ubox, vbox)
    return f


def run_ranks64(G, px, py, nsteps, standin=True, graph=True, seed=99, halo=3, stepwise=False, repeats=1):
    decomp = parallel.Decomposition(G, px, py, halo=halo)
    whole = widen64(wrf.synth_fields(G, seed=seed))
    ranks = []
    for r in range(px * py):
        pg = decomp.patch_grid(r)
        f = cases.carve_patch(whole, G, pg)
        cases.poison_neighbour_halos(f, decomp, r, pg, (parallel.CONSTANT_HALOS, parallel.STEP_HALOS, parallel.OUTPUT_HALOS))
        p = wrf.Patch(pg, device=0, dtype=F64)
        p.set_scalars(*SCALARS)
        p.upload(f)
        ranks.append((p, pg, f))
    try:
        infos = [p.comm_init(px, py, r, *decomp.patch_extents(r)) for r, (p, _, _) in enumerate(ranks)]
        for p, _, _ in ranks:
            p.comm_connect(infos)
        for p, _, _ in ranks:
            p.comm_push_constants()
        for _ in range(repeats):
            if stepwise:
                for s in range(nsteps):
                    for p, _, _ in ranks:
                        p.comm_push_uv()
                        p.comm_step()
                        if standin and s + 1 < nsteps:
                            p.comm_standin_advance_uv(C_UV)
            else:
                for p, _, _ in ranks:
                    p.comm_loop(nsteps, standin=standin, c=C_UV, graph=graph)
        for r, (p, pg, f) in enumerate(ranks):
            timeouts, steps = p.comm_status()
            assert timeouts == 0, f"rank {r}: {timeouts} halo waits timed out"
            assert steps == nsteps * repeats
            p.download(f, names=cases.OUTPUTS + ("u", "v"))
    finally:
        for p, _, _ in ranks:
            p.close()
    return decomp, whole, ranks


def assert_ranks_match(decomp, G, ranks, want, what, names=cases.OUTPUTS + ("u", "v")):
    for r, (_, pg, f) in enumerate(ranks):
        bad = cases.patch_mismatches(f, want, G, pg, decomp.patch_extents(r), names=names)
        assert not bad, f"{what} rank {r}: {bad}"


# ================================================================ CPU: argument checks before any device work
def test_new_r8_entry_points_reject_a_null_handle():
    lib = wrf.lib()
    info = C.create_string_buffer(lib.wrfb200_comm_info_bytes())
    calls = {
        "wrfb200_comm_init_r8": lambda: lib.wrfb200_comm_init_r8(None, 1, 1, 0, 1, 8, 1, 8, info),
        "wrfb200_comm_loop_r8": lambda: lib.wrfb200_comm_loop_r8(None, 3, 1, 0.25, 1),
        "wrfb200_comm_standin_advance_uv_r8": lambda: lib.wrfb200_comm_standin_advance_uv_r8(None, 0.25),
        "wrfb200_standin_advance_uv_r8": lambda: lib.wrfb200_standin_advance_uv_r8(None, 2, 0.25, 1, 8, 1, 8),
        "wrfb200_upload_constants_r8": lambda: lib.wrfb200_upload_constants_r8(None, *([None] * 17)),
        "wrfb200_upload_state_r8": lambda: lib.wrfb200_upload_state_r8(None, None, None, None),
        "wrfb200_set_uv_r8": lambda: lib.wrfb200_set_uv_r8(None, None, None),
        "wrfb200_download_outputs_r8": lambda: lib.wrfb200_download_outputs_r8(None, 1, 8, 1, 8, 1, 4, *([None] * 7)),
    }
    for name, call in calls.items():
        assert call() == _lib.ERR_INVALID_ARG, name
        assert b"null" in lib.wrfb200_last_error(), name


# ================================================================ GPU: ranks sharing device 0
@gpu
@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("px,py,shape", [
    (1, 2, (300, 160, 20)),       # nk = 19: two-row tiles
    (2, 1, (300, 160, 20)),       # patches 150 wide, the east one starting at the odd ips = 151
    (2, 2, (300, 160, 20)),
    (1, 4, (300, 160, 20)),
    (1, 2, (200, 64, 70)),        # nk = 69: one-row tiles
    (2, 2, (200, 64, 70)),        # one-row tiles with an east neighbour: east-column waits, east_blocks = nby
])
def test_fused_r8_matches_binary64_checker_loop(px, py, shape, graph):
    G = cases.grid(*shape, halo=5, variant="specified")
    nsteps = 4
    decomp, whole, ranks = run_ranks64(G, px, py, nsteps, graph=graph)
    want = checker_loop64(G, whole, nsteps, c=C_UV)
    assert_ranks_match(decomp, G, ranks, want, f"{px}x{py} {shape} graph={graph}")


@gpu
@pytest.mark.parametrize("variant", ["open", "periodic_specified"])
def test_fused_r8_flag_variants_stepwise(variant):
    """Edge clamps on the boundary ranks only, driven step by step through the untyped C verbs and the _r8 stand-in."""
    G = cases.grid(280, 90, 12, halo=4, variant=variant)
    nsteps = 3
    decomp, whole, ranks = run_ranks64(G, 2, 2, nsteps, stepwise=True, seed=7, halo=2)
    want = checker_loop64(G, whole, nsteps, c=C_UV)
    assert_ranks_match(decomp, G, ranks, want, variant)


@gpu
def test_fused_r8_loop_replays_keep_epochs_consistent():
    G = cases.grid(260, 64, 10, halo=5, variant="specified")
    decomp, whole, ranks = run_ranks64(G, 1, 2, 3, standin=False, graph=True, repeats=5)
    want = checker_loop64(G, whole, 15)
    assert_ranks_match(decomp, G, ranks, want, "5 replays", names=cases.OUTPUTS)


@gpu
def test_resident_bundle_r8_round_trip():
    """Usage (B) of the resident module in an -r8 build: constants and state once, then per step set_uv_r8, step and
    download_outputs_r8 into the caller's arrays, with the caller's advance_uv (the stand-in) between steps."""
    g = cases.grid(140, 50, 12, halo=4, variant="periodic_specified")
    fin = widen64(wrf.synth_fields(g, seed=8))
    nsteps = 4
    want = checker_loop64(g, fin, nsteps, c=C_UV)
    host = cases.copy_fields(fin)
    ubox, vbox = cases.standin_boxes(g, g.ids, g.ide, g.jds, g.jde)
    with wrf.Patch(g, device=0, dtype=F64) as p:
        p.set_scalars(*SCALARS)
        p.upload_constants(host)
        p.upload_state(host)
        for s in range(nsteps):
            p.set_uv(host["u"], host["v"])
            p.step()
            p.download_outputs(host)
            if s + 1 < nsteps:
                cases.standin_advance_uv_numpy(host, g, C_UV, ubox, vbox)
    for n in wrf.FIELDS:
        assert np.array_equal(host[n].view(np.uint64), want[n].view(np.uint64)), n
    # what the routine does not write keeps the caller's bytes
    i0, i1, j0, j1, k0, k1 = g.bounds()
    for n in cases.OUTPUTS:
        a, b = host[n].view(np.uint64).copy(), fin[n].view(np.uint64).copy()
        if a.ndim == 3:
            a[j0 - g.jms:j1 - g.jms + 1, k0 - g.kms:k1 - g.kms + 1, i0 - g.ims:i1 - g.ims + 1] = 0
            b[j0 - g.jms:j1 - g.jms + 1, k0 - g.kms:k1 - g.kms + 1, i0 - g.ims:i1 - g.ims + 1] = 0
        else:
            a[j0 - g.jms:j1 - g.jms + 1, i0 - g.ims:i1 - g.ims + 1] = 0
            b[j0 - g.jms:j1 - g.jms + 1, i0 - g.ims:i1 - g.ims + 1] = 0
        assert np.array_equal(a, b), f"{n}: cells outside the computed range were written"


@gpu
def test_r8_comm_rejections_carry_status_and_message():
    lib = wrf.lib()
    G = cases.grid(64, 32, 6, halo=2)
    decomp = parallel.Decomposition(G, 1, 2, halo=2)
    info = C.create_string_buffer(lib.wrfb200_comm_info_bytes())

    def err():
        return lib.wrfb200_last_error().decode()

    # ranks of mixed precision: a binary32 blob given to a real*8 rank at connect, and the other way round
    with wrf.Patch(decomp.patch_grid(0), device=0, dtype=F64) as p8, wrf.Patch(decomp.patch_grid(1), device=0) as p4:
        infos = [p8.comm_init(1, 2, 0, *decomp.patch_extents(0)), p4.comm_init(1, 2, 1, *decomp.patch_extents(1))]
        for p in (p8, p4):
            with pytest.raises(wrf.WrfB200Error) as e:
                p.comm_connect(infos)
            assert e.value.status == _lib.ERR_INVALID_ARG and "mixed precision" in str(e.value)
        # the typed verbs of the other precision
        assert lib.wrfb200_comm_loop(p8._h, 2, 0, 0.0, 1) == _lib.ERR_UNSUPPORTED and "binary32 only" in err()
        assert lib.wrfb200_comm_standin_advance_uv(p8._h, 0.25) == _lib.ERR_UNSUPPORTED and "binary32 only" in err()
        assert lib.wrfb200_comm_loop_r8(p4._h, 2, 0, 0.0, 1) == _lib.ERR_STATE and "real*4" in err()
        # comm_init_r8 on a binary32 handle
        assert lib.wrfb200_comm_init_r8(p4._h, 1, 1, 0, 1, 64, 1, 32, info) == _lib.ERR_STATE and "real*4" in err()
    # an untyped verb on a real*8 handle without comm_init_r8
    with wrf.Patch(G, device=0, dtype=F64) as p8:
        assert lib.wrfb200_comm_step(p8._h) == _lib.ERR_UNSUPPORTED and "binary32 only" in err()
        assert lib.wrfb200_comm_status(p8._h, None, None) == _lib.ERR_UNSUPPORTED
    # more levels than the double2 tile kernel holds: refused at init, not at the first step
    deep = cases.grid(16, 8, 230, halo=2)
    with wrf.Patch(deep, device=0, dtype=F64) as p8:
        with pytest.raises(wrf.WrfB200Error) as e:
            p8.comm_init(1, 1, 0, 1, 16, 1, 8)
        assert e.value.status == _lib.ERR_UNSUPPORTED and "220" in str(e.value)
    # caller-owned buffers cannot be exported to the neighbours
    with wrf.Patch(G, device=0, allocate=False, dtype=F64) as p8:
        with pytest.raises(wrf.WrfB200Error) as e:
            p8.comm_init(1, 1, 0, 1, 64, 1, 32)
        assert e.value.status == _lib.ERR_STATE and "handle-owned" in str(e.value)


def _build_harness(tmp_path):
    exe = str(tmp_path / "c_comm_harness_r8")
    libdir = os.path.join(ROOT, "wrf_model_cuda_sample_b200")
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    subprocess.run([cc, "-O1", os.path.join(ROOT, "tests", "c_comm_harness_r8.c"), "-I", os.path.join(ROOT, "include"),
                    "-L", libdir, "-lwrfb200", f"-Wl,-rpath,{libdir}", "-o", exe], check=True)
    return exe


def test_comm_harness_r8_builds_and_rejects_bad_usage(tmp_path):
    r = subprocess.run([_build_harness(tmp_path)], capture_output=True, text=True)
    assert r.returncode == 2 and "usage" in r.stderr


@gpu
@pytest.mark.parametrize("px,py", [(1, 2), (2, 2)])
def test_comm_harness_r8_processes_match_checker(tmp_path, px, py):
    """One PROCESS per rank (fork), CUDA IPC between them, all ranks on one device when the box has fewer GPUs."""
    import torch
    exe = _build_harness(tmp_path)
    nx, ny, nz, nsteps = 200, 96, 14, 3
    out = tmp_path / "out"
    out.mkdir()
    env = dict(os.environ, WRFB200_FLAG_TIMEOUT_MS="20000")
    r = subprocess.run([exe, str(px), str(py), str(nx), str(ny), str(nz), str(nsteps),
                        str(max(1, torch.cuda.device_count())), str(out)],
                       capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    G = cases.grid(nx, ny, nz, halo=5, variant="specified")
    want = checker_loop64(G, widen64(wrf.synth_fields(G, seed=99)), nsteps, c=C_UV)
    decomp = parallel.Decomposition(G, px, py, halo=3)
    for rank in range(px * py):
        pg = decomp.patch_grid(rank)
        f = {n: np.fromfile(out / f"rank{rank}_field{wrf.FIELD_ID[n]}.bin", dtype=F64).reshape(pg.shape_of(n))
             for n in cases.OUTPUTS + ("u", "v")}
        bad = cases.patch_mismatches(f, want, G, pg, decomp.patch_extents(rank))
        assert not bad, f"rank {rank}: {bad}"


def _ngpu():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@gpu
@pytest.mark.parametrize("nproc,pgrid", [(2, "1x2"), (4, "2x2"), (8, "1x8")])
def test_torchrun_r8_full_grid_bit_identical(nproc, pgrid):
    """One process per GPU on the full 1800x1060x50 grid (tools/multi_gpu_check.py --dtype float64)."""
    if _ngpu() < nproc:
        pytest.skip(f"needs {nproc} GPUs")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
           "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(ROOT, "tools", "multi_gpu_check.py"), "--pgrid", pgrid, "--shape", "1800x1060x50",
           "--dtype", "float64"]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "BIT-IDENTICAL" in r.stdout and "timed out" not in r.stdout
