#!/usr/bin/env python
"""bench.py -- advance_mu_t grid-points/s on N B200s of one node (BASELINE.json's metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload conus3|conus12|weak2048|deep120|tiny]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...      # the reference's own CPU C code on the host cores
    python bench.py ... --dump-outputs DIR    # also write the last timed step's output fields to DIR/<name>.npy

A "step" is one pass of the hot path over the workload: for the default workload (conus3, the
CONUS-3km-class 1800x1060x50 grid BASELINE.json's target is quoted on) that is the device-resident
6-acoustic-step loop of one RK3 sub-step, i.e. six advance_mu_t calls over the whole grid.  With N > 1 the
grid is split into 2-D (i,j) patches, one rank per GPU (strong scaling), and every small step exchanges the
one-cell halo: u / v edges pushed into the neighbours' memory before the call, mu / muts / mudf edges pushed
by the advance_mu_t kernel itself -- peer-mapped NVLink stores fused into the kernels (csrc/comm.cu), the
whole loop replayed from one CUDA graph per rank.  Before timing, every N > 1 run checks the very same C-ABI
loop (with the advance_uv stand-in that makes the exchange load-bearing, halos poisoned) bit for bit against
the single-domain oracle on a small grid and prints the outcome under "parity".
Prints ONE JSON line (rank 0).  Every number is measured in this run; nothing is cached.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

# name -> (nx, ny, nz, small steps per bench step, dx [m], dts [s], scaling, description)
WORKLOADS = {
    "conus3": (1800, 1060, 50, 6, 3000.0, 3.0, "strong",
               "CONUS 3 km-class grid 1800x1060x50, device-resident 6-acoustic-step loop"),
    "conus12": (425, 300, 35, 1, 12000.0, 12.0, "strong", "CONUS 12 km-class grid 425x300x35, single small step"),
    "weak2048": (2048, 2048, 80, 6, 3000.0, 3.0, "weak", "2048x2048x80 per-GPU tile, 6-acoustic-step loop"),
    "deep120": (512, 512, 120, 6, 3000.0, 3.0, "strong", "deep-column 512x512x120, 6-acoustic-step loop"),
    "tiny": (74, 61, 28, 1, 12000.0, 12.0, "strong", "driver-equivalent tiny domain 74x61x28"),
    "patch8": (1800, 133, 50, 6, 3000.0, 3.0, "strong", "one rank's j-slab of conus3 at 8 GPUs (tuning aid)"),
    "patch4": (1800, 265, 50, 6, 3000.0, 3.0, "strong", "one rank's j-slab of conus3 at 4 GPUs (tuning aid)"),
}
HALO = 5
EPSSM = 0.1
METRIC = "advance_mu_t grid-points/s"
UNIT = "grid-points/s"
C_UV = 0.25                     # coefficient of the advance_uv stand-in
KERNEL_NAMES = {0: "auto", 1: "amt_column_kernel", 2: "amt_tile_kernel", 3: "amt_pipe_kernel"}
OUTPUTS = ("ww", "t", "t_ave", "mu", "muave", "muts", "mudf")     # what advance_mu_t hands back to its caller
DUMP_BYTES = 64_000_000          # all files of one --dump-outputs run, .npy headers included
NPY_HEADER_BYTES = 4096         # room kept per file; numpy writes 128 bytes for these arrays
DUMP_SEED = 20240617


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def scalars_of(dx, dts):
    return (np.float32(1.0 / dx), np.float32(1.0 / dx), np.float32(dts), np.float32(EPSSM))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                 "-i", str(self.gpu)], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        try:
            for line in open(self.path):
                c = [x.strip() for x in line.split(",")]
                if len(c) < 9:
                    continue
                try:
                    sm.append(float(c[1])); smax.append(float(c[2])); power.append(float(c[3]))
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        finally:
            try:
                os.unlink(self.path)
            except OSError:
                pass
        if not sm:
            return None
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(smax), "power_w_max": max(power),
                "samples": len(sm), "reasons": sorted(reasons)}


def dump_outputs(out_dir, fields, prefix="", share=1):
    """Write the output fields to out_dir/<prefix><name>.npy as float32, so that two builds run with the same
    arguments can be compared value for value.  All files of a run (`share` writers) stay within DUMP_BYTES: a
    field larger than its part is replaced by a stratified sample of its flattened [j,k,i] values, one value from
    each of `cap` equal runs at offsets drawn with a fixed seed, so the same positions are sampled in every run."""
    os.makedirs(out_dir, exist_ok=True)
    cap = (DUMP_BYTES // (len(OUTPUTS) * share) - NPY_HEADER_BYTES) // 4
    for name in OUTPUTS:
        a = np.ascontiguousarray(fields[name], dtype=np.float32)
        if a.size > cap:
            run = a.size // cap
            idx = np.arange(cap, dtype=np.int64) * run + np.random.default_rng(DUMP_SEED).integers(0, run, cap)
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, prefix + name + ".npy"), a)


def global_grid(workload, n_gpus):
    """(Grid, scalars, small steps per bench step, dx).  Grid is index arithmetic only (no library call)."""
    from wrf_model_cuda_sample_b200.advance_mu_t import Grid
    nx, ny, nz, nsmall, dx, dts, scaling, desc = WORKLOADS[workload]
    if scaling == "weak" and n_gpus > 1:
        ny = ny * n_gpus          # j-slabs: the per-GPU tile stays the named nx x ny
    g = Grid.from_shape(nx, ny, nz, halo=HALO, periodic_x=False, specified=True, nested=False)
    return g, scalars_of(dx, dts), nsmall, dx


# -------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the reference's own C (oracle/_ref) on the host cores
# -------------------------------------------------------------------------------------------------
def use_all_host_threads():
    cores = os.cpu_count() or 1
    # torchrun exports OMP_NUM_THREADS=1 to its children, which would silently turn this into a
    # single-thread measurement
    os.environ["OMP_NUM_THREADS"] = str(cores)
    try:
        ctypes.CDLL("libgomp.so.1").omp_set_num_threads(cores)
    except OSError:
        pass
    return cores


def cpu_reference_run(g, scalars, fields, steps, warmup):
    """Times ONE advance_mu_t small step of the reference C over the full grid per step (a bounded sample of
    the workload step), j-tiled over all host threads as WRF tiles it (advance_mu_t_driver.f90:175-205).
    `fields`: dict of numpy arrays; the seven output arrays are modified in place.  -> dict."""
    from oracle import loader, synth_np
    cores = use_all_host_threads()
    if loader.have_ref():
        fn, kind, what = loader.reference_c, "reference", "reference advance_mu_t.c (unmodified, gcc -O3 -ffp-contract=off)"
    else:
        fn, kind, what = loader.oracle_c, "port", "oracle/advance_mu_t_oracle.c (gcc -O3 -ffp-contract=off)"
    n3, n2 = synth_np.updated_points(g)
    tiles = max(1, cores * 4)
    times = []
    for s in range(warmup + steps):
        t0 = time.perf_counter()
        fn(fields, g, scalars, tiles=tiles)
        dt = time.perf_counter() - t0
        if s >= warmup:
            times.append(dt)
    total = sum(times)
    return {"value": n3 * len(times) / total, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": f"{len(times)} x one small step over {g.ide}x{g.jde}x{g.kde} ({n3} points), {what}, "
                      f"OpenMP over {tiles} j-tiles on {cores} threads",
            "ms_per_small_step": 1e3 * total / len(times)}


def run_reference_arm(args):
    """The reference's own CPU implementation on this box's host cores.  Nothing of the product is on this
    path: inputs come from oracle/synth_np.py (numpy port of the generator), compute is oracle/_ref."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import synth_np
    g, scalars, nsmall, dx = global_grid(args.workload, 1)
    steps = args.steps                         # each step is one small step over the full grid
    warmup = max(1, args.warmup)
    fields = synth_np.synth_fields(g)
    r = cpu_reference_run(g, scalars, fields, steps, warmup)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, fields)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": r["ms_per_small_step"],
        "higher_is_better": True, "scaling": WORKLOADS[args.workload][6], "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.workload}: {WORKLOADS[args.workload][7]}",
                   "grid": f"{g.ide}x{g.jde}x{g.kde}", "small_steps_per_step": 1,
                   "note": "each timed step is ONE small step over the full grid (a bounded sample of the "
                           "%d-small-step workload step); ms_per_step is the timed value" % nsmall},
        "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# -------------------------------------------------------------------------------------------------
# our arm: helpers
# -------------------------------------------------------------------------------------------------
def fused_parity_preflight(decomp_px, decomp_py, rank, world, local_rank, dev, allgather, nsmall):
    """The multi-GPU loop that is about to be timed -- the same C-ABI calls, the same kernels, the same CUDA-graph
    path -- on a small grid where the single-domain oracle is cheap: halos poisoned, advance_uv stand-in between
    steps so that every exchanged cell is load-bearing.  Returns the parity record (all ranks agree on it)."""
    import torch
    import torch.distributed as dist
    import wrf_model_cuda_sample_b200 as wrf
    from wrf_model_cuda_sample_b200 import parallel
    from tests import cases                          # the checker lives with the tests (oracle loop, patch compare)
    nx, ny, nz = max(320, 40 * decomp_px), max(192, 12 * decomp_py), 20
    G = cases.grid(nx, ny, nz, halo=HALO, variant="specified")
    decomp = parallel.Decomposition(G, decomp_px, decomp_py, halo=3)
    pg, ext = decomp.patch_grid(rank), decomp.patch_extents(rank)
    whole = wrf.synth_fields(G, seed=99)
    bad = 0
    timeouts = 0
    checks = []
    for standin, nsteps in ((True, 4), (False, nsmall)):
        f = cases.carve_patch(whole, G, pg)
        cases.poison_neighbour_halos(f, decomp, rank, pg,
                                     (parallel.CONSTANT_HALOS, parallel.STEP_HALOS, parallel.OUTPUT_HALOS))
        with wrf.Patch(pg, device=local_rank) as p:
            p.set_stream(torch.cuda.current_stream().cuda_stream)
            p.set_scalars(*cases.SCALARS_3KM)
            p.upload(f)
            parallel.connect_fused(p, decomp, rank, allgather)
            p.comm_push_constants()
            p.comm_loop(nsteps, standin=standin, c=C_UV, graph=True)
            to, done = p.comm_status()
            timeouts += to + (0 if done == nsteps else 1)
            p.download(f, names=cases.OUTPUTS + ("u", "v"))
            dist.barrier()                            # nobody unmaps a neighbour that is still storing into it
        want = cases.oracle_loop(G, whole, cases.SCALARS_3KM, nsteps, c=C_UV if standin else None)
        bad += sum(cases.patch_mismatches(f, want, G, pg, ext).values())
        checks.append(f"{nsteps} steps {'with' if standin else 'without'} the advance_uv stand-in")
    t = torch.tensor([bad, timeouts], device=dev, dtype=torch.int64)
    dist.all_reduce(t)
    return {"nranks": world, "pgrid": f"{decomp_px}x{decomp_py}", "grid": f"{nx}x{ny}x{nz}",
            "mismatches": int(t[0].item()), "halo_wait_timeouts": int(t[1].item()),
            "checked": "every rank's patch (ww, t, t_ave, mu, muave, muts, mudf, u, v) bit for bit against the "
                       "single-domain oracle loop; " + "; ".join(checks),
            "path": "wrfb200_comm_connect / comm_push_constants / comm_loop (CUDA graph) -- the calls timed below"}


def fill_patch_slabwise(patch, pg, dx, slab_rows=256, seed=20240617):
    """Fill a large device-resident patch without holding all of its fields on the host: generate j-slabs of
    the (counter-based, decomposition-independent) synthetic fields and upload each into its rows."""
    import wrf_model_cuda_sample_b200 as wrf
    from wrf_model_cuda_sample_b200._lib import check
    from wrf_model_cuda_sample_b200.advance_mu_t import Grid
    ja = pg.jms
    while ja <= pg.jme:
        jb = min(pg.jme, ja + slab_rows - 1)
        sg = Grid(pg.ids, pg.ide, pg.jds, pg.jde, pg.kde, pg.ims, pg.ime, ja, jb, pg.kms, pg.kme,
                  pg.its, pg.ite, max(ja, pg.jts), min(jb, pg.jte), pg.kts, pg.kte,
                  pg.periodic_x, pg.specified, pg.nested)
        names = wrf.FIELDS_3D + wrf.FIELDS_2D + (wrf.FIELDS_1D if ja == pg.jms else ())
        f = wrf.synth_fields(sg, seed=seed, names=names, dx_m=dx)
        for n in names:
            a = f[n]
            if n in wrf.FIELDS_1D:
                patch.upload({n: a}, names=(n,))
                continue
            # wrfb200_upload_range addresses a DENSE array with the patch's full extents: hand it the address
            # that array would have, only rows ja..jb of it are ever read
            row = a[0].size
            base = a.ctypes.data - (ja - pg.jms) * row * 4
            check(wrf.lib().wrfb200_upload_range(
                patch._h, wrf.FIELD_ID[n], ctypes.c_void_p(base), pg.ims, pg.ime, pg.kms, pg.kme, ja, jb))
        patch.sync()
        ja = jb + 1


def time_loop(step, steps, warmup, main, barrier, flush=None):
    """CUDA-event time of `steps` calls of step() on stream `main` (ms, this rank)."""
    import torch
    for _ in range(warmup):
        step()
    barrier()
    if flush is None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(main)
        for _ in range(steps):
            step()
        e1.record(main)
        barrier()
        return e0.elapsed_time(e1)
    total = 0.0
    for _ in range(steps):
        flush.fill_(1)                                     # evict the previous step's lines from L2
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(main)
        step()
        e1.record(main)
        barrier()
        total += e0.elapsed_time(e1)
    return total


def max_over_ranks(x, dev, world):
    if world == 1:
        return x
    import torch
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def measure_extra_workload(name, world, rank, local_rank, dev, main, barrier, allgather, kernel, steps=10, warmup=3):
    """Device-timed value of another BASELINE.json config (same method as the headline), -> dict."""
    import torch
    import torch.distributed as dist
    import wrf_model_cuda_sample_b200 as wrf
    from wrf_model_cuda_sample_b200 import parallel
    g, scalars, nsmall, dx = global_grid(name, world)
    px, py = (1, world)
    decomp = parallel.Decomposition(g, px, py, halo=HALO)
    pg = decomp.patch_grid(rank)
    peak, _ = peaks()
    patch = wrf.Patch(pg, device=local_rank)
    try:
        patch.set_stream(main.cuda_stream)
        patch.set_scalars(*scalars)
        patch.set_kernel(kernel)
        if pg.shape3[0] * pg.shape3[1] * pg.shape3[2] > 200_000_000:
            fill_patch_slabwise(patch, pg, dx)
        else:
            patch.upload(wrf.synth_fields(pg, dx_m=dx))
            patch.sync()
        flush = None
        if pg.algorithmic_bytes() < 512 * 1024 * 1024:
            flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
        if world == 1:
            def step():
                patch.step_graph(nsmall)
        else:
            parallel.connect_fused(patch, decomp, rank, allgather)
            patch.comm_push_constants()

            def step():
                patch.comm_loop(nsmall, standin=False, graph=True)
        ms = max_over_ranks(time_loop(step, steps, warmup, main, barrier, flush), dev, world)
        timeouts = patch.comm_status()[0] if world > 1 else 0
        n3_global, _ = g.updated_points()
        kernel_ms = ms / (steps * nsmall)
        achieved = pg.algorithmic_bytes() / (kernel_ms * 1e-3) / 1e9
        out = {"value": n3_global * nsmall * steps / (ms * 1e-3), "unit": UNIT, "grid": f"{g.ide}x{g.jde}x{g.kde}",
               "scaling": WORKLOADS[name][6], "small_steps_per_step": nsmall, "steps": steps,
               "avg_launch_ms": kernel_ms, "frac": achieved / peak, "achieved_gbs": achieved,
               "kernel": KERNEL_NAMES[patch.last_kernel()],
               "l2": "flushed before every timed step" if flush is not None else "inputs larger than L2"}
        if world > 1:
            out["decomposition"] = f"{px}x{py}"
            out["halo_wait_timeouts"] = timeouts
            dist.barrier()
        return out
    finally:
        patch.close()


def measure_device_pointer_call(nx, ny, nz, scalars, dx, dev, main, barrier, reps=10):
    """wrfb200_advance_mu_t with DEVICE pointers to the caller's dense Fortran-layout arrays (no mirrors, no copies):
    halo 6 -> rows of 1812 floats (16-byte multiples): the TMA kernel runs in place; halo 5 -> 1810 floats: rows
    cannot be TMA / float4 addressed and the any-layout column kernel runs."""
    import torch
    import wrf_model_cuda_sample_b200 as wrf
    peak, _ = peaks()
    out = {}
    for halo in (6, 5):
        g = wrf.Grid.from_shape(nx, ny, nz, halo=halo, periodic_x=False, specified=True, nested=False)
        host = wrf.synth_fields(g, dx_m=dx)
        d = {n: torch.from_numpy(host[n]).to(dev) for n in wrf.FIELDS}
        del host
        wrf.lib().wrfb200_set_default_stream(ctypes.c_void_p(main.cuda_stream))
        for _ in range(3):
            wrf.call_with_fields(d, g, *scalars)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(main)
        for _ in range(reps):
            wrf.call_with_fields(d, g, *scalars)
        e1.record(main)
        barrier()
        ms = e0.elapsed_time(e1) / reps
        n3, _ = g.updated_points()
        out["halo%d_rows_of_%d_floats" % (halo, g.shape3[2])] = {
            "kernel": KERNEL_NAMES[wrf.default_last_kernel()], "ms_per_call": ms, "value": n3 / (ms * 1e-3),
            "frac": g.algorithmic_bytes() / (ms * 1e-3) / 1e9 / peak}
        wrf.lib().wrfb200_set_default_stream(None)
        del d
        torch.cuda.empty_cache()
    return out


def e2e_measurements(fields, pg, scalars, nsmall, kernel, world, dev, barrier, e2e_steps, n3_global, with_pageable):
    """The same metric end to end through the reference-facing 48-argument C-ABI call with HOST arrays; host<->device
    copies inside the timed region.  Headline = the per-small-step drop-in pattern of a host-resident model."""
    import torch
    import wrf_model_cuda_sample_b200 as wrf
    lib = wrf.lib()
    n3_local, n2_local = pg.updated_points()
    b3 = fields["u"].nbytes
    in_all = sum(fields[n].nbytes for n in ("ww_1", "u", "u_1", "v", "v_1", "t", "t_1", "ft", "mu", "mut", "muu",
                                            "muv", "mu_tend", "msfuy", "msfvx_inv", "msftx", "msfty",
                                            "dnw", "fnm", "fnp", "rdnw"))
    in_all += fields["ww"].nbytes // pg.shape3[1]          # ww: level 1 only
    # 3-D inputs travel as whole rows js-1..je+1 (dense host rows); count what is copied
    in_uv = 2 * b3
    out_b = 4 * (3 * n3_local + 4 * n2_local)
    lib.wrfb200_set_default_kernel(kernel)

    def timed(fn, reps):
        fn()                                                # warm-up: allocates the cached mirrors etc.
        barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        return max_over_ranks(time.perf_counter() - t0, dev, world) / reps

    def loop_resident(f):
        with wrf.acoustic_loop():                           # first call: everything up; then only u, v
            for _ in range(nsmall):
                wrf.call_with_fields(f, pg, *scalars)

    out = {}
    dt = timed(lambda: loop_resident(fields), e2e_steps)
    head = {"value": n3_global * nsmall / dt, "unit": UNIT,
            "h2d_bytes_per_step": int(in_all + (nsmall - 1) * in_uv), "d2h_bytes_per_step": int(nsmall * out_b),
            "ms_per_step": 1e3 * dt, "steps": e2e_steps,
            "api": "wrfb200_acoustic_loop_begin; %d x wrfb200_advance_mu_t(pinned host arrays) -- first call uploads all "
                   "inputs, later calls only u,v; every call downloads the 7 outputs and syncs; wrfb200_acoustic_loop_end"
                   % nsmall}
    variants = {}
    dt = timed(lambda: wrf.call_with_fields(fields, pg, *scalars, nsteps=nsmall), e2e_steps)
    variants["loop_entry_pinned"] = {
        "value": n3_global * nsmall / dt, "ms": 1e3 * dt, "h2d_bytes": int(in_all), "d2h_bytes": int(out_b),
        "api": "wrfb200_advance_mu_t_loop(nsteps=%d): one upload, %d launches, one download (u,v held fixed)" % (nsmall, nsmall)}
    dt = timed(lambda: wrf.call_with_fields(fields, pg, *scalars), e2e_steps)
    variants["single_call_pinned"] = {
        "value": n3_global / dt, "ms": 1e3 * dt, "h2d_bytes": int(in_all), "d2h_bytes": int(out_b),
        "api": "wrfb200_advance_mu_t, one small step per call, everything re-uploaded (the reference's call pattern)"}

    def resident_step():
        wrf.call_with_fields(fields, pg, *scalars)
    with wrf.acoustic_loop():
        wrf.call_with_fields(fields, pg, *scalars)          # primes the mirrors
        dt = timed(resident_step, e2e_steps)
    variants["resident_step_pinned"] = {
        "value": n3_global / dt, "ms": 1e3 * dt, "h2d_bytes": int(in_uv), "d2h_bytes": int(out_b),
        "api": "wrfb200_advance_mu_t inside an acoustic loop after its first call: u,v up, 7 outputs down"}
    if with_pageable:
        pageable = {k: np.array(v, copy=True) for k, v in fields.items()}
        dt = timed(lambda: wrf.call_with_fields(pageable, pg, *scalars), max(1, e2e_steps // 2))
        variants["single_call_pageable"] = {"value": n3_global / dt, "ms": 1e3 * dt,
                                            "api": "as single_call_pinned with ordinary (pageable) numpy arrays"}
        lib.wrfb200_set_host_pinning(1)
        t0 = time.perf_counter()
        wrf.call_with_fields(pageable, pg, *scalars)
        first = time.perf_counter() - t0
        dt = timed(lambda: wrf.call_with_fields(pageable, pg, *scalars), max(1, e2e_steps // 2))
        variants["single_call_pageable_first_sight_pinning"] = {
            "value": n3_global / dt, "ms": 1e3 * dt, "first_call_ms": 1e3 * first,
            "api": "wrfb200_set_host_pinning(1): arrays cudaHostRegister'ed the first time they are seen"}
        with wrf.acoustic_loop():
            wrf.call_with_fields(pageable, pg, *scalars)
            dt = timed(lambda: wrf.call_with_fields(pageable, pg, *scalars), max(1, e2e_steps // 2))
        variants["resident_step_pageable_first_sight_pinning"] = {"value": n3_global / dt, "ms": 1e3 * dt}
        lib.wrfb200_set_host_pinning(0)
        del pageable
    lib.wrfb200_release_cache()
    return head, variants


# -------------------------------------------------------------------------------------------------
# our arm
# -------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    import wrf_model_cuda_sample_b200 as wrf
    from wrf_model_cuda_sample_b200 import parallel

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly ONE JSON line: native libraries (NCCL prints its version banner to stdout)
    # are pointed at stderr for the whole run, the line itself is written to the saved descriptor.
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus or world == 1 and args.gpus == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"

    g, scalars, nsmall, dx = global_grid(args.workload, world)
    if args.pgrid:
        px, py = (int(x) for x in args.pgrid.lower().split("x"))
    else:
        px, py = parallel.choose_process_grid(world, g.ide, g.jde)
    assert px * py == world
    decomp = parallel.Decomposition(g, px, py, halo=HALO)
    pg = decomp.patch_grid(rank)
    kernel = {"auto": wrf.KERNEL_AUTO, "pipe": wrf.KERNEL_PIPE, "tile": wrf.KERNEL_TILE, "column": wrf.KERNEL_COLUMN}[args.kernel]
    allgather = parallel.torch_allgather_bytes(device=dev) if world > 1 else (lambda blob: [blob])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    main = torch.cuda.Stream(device=dev)                       # a real stream: capturable, and what events time
    torch.cuda.set_stream(main)

    # ---- N > 1: parity of the multi-GPU loop, through the calls that are timed below ----
    parity = None
    if world > 1:
        parity = fused_parity_preflight(px, py, rank, world, local_rank, dev, allgather, nsmall)

    # ---- inputs: pinned host arrays (also the e2e source), uploaded once for the resident loop ----
    host = wrf.synth_fields(pg, pinned=True, dx_m=dx)
    pinned_keep = host.pop("__pinned__")
    patch = wrf.Patch(pg, device=local_rank)
    patch.set_stream(main.cuda_stream)
    patch.set_scalars(*scalars)
    patch.set_kernel(kernel)
    patch.upload(host)
    patch.sync()

    n3_local, n2_local = pg.updated_points()
    n3_global, n2_global = g.updated_points()
    bytes_local = pg.algorithmic_bytes()

    # ---- one bench step ----
    if world == 1:
        def step():
            patch.step_graph(nsmall)
        exec_mode = "cuda graph (wrfb200_step_graph)"
        exchange = None
    else:
        parallel.connect_fused(patch, decomp, rank, allgather)
        patch.comm_push_constants()                            # once per RK sub-step
        graph = not args.no_graph

        def step():
            patch.comm_loop(nsmall, standin=False, graph=graph)
        exec_mode = ("cuda graph" if graph else "eager launches") + \
            " (wrfb200_comm_loop: per small step a u/v halo push kernel + ONE advance_mu_t launch over the patch)"
        exchange = ("fused: u west column / v south row stored into the neighbours' halos by the push kernel, mu/muts/mudf "
                    "edges by the advance_mu_t kernel itself; peer-mapped memory (CUDA IPC over NVLink), release/acquire "
                    "epoch flags; edge blocks wait, interior blocks run; no NCCL call in the loop")

    flush = None
    if args.workload in ("conus12", "tiny"):
        flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = patch.launch_count()
    elapsed_ms = time_loop(step, args.steps, 0, main, barrier, flush)
    launches = patch.launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    l2_note = ("inputs larger than L2 (%.2f GB touched per small step vs 126 MB L2)" % (bytes_local / 1e9)
               if flush is None else "L2 flushed (256 MB write) before every timed step")
    halo_timeouts = patch.comm_status()[0] if world > 1 else 0
    if args.dump_outputs:                                      # the state the last timed step left on the device
        out = {n: np.empty(pg.shape_of(n), dtype=np.float32) for n in OUTPUTS}
        patch.download(out, names=OUTPUTS)
        dump_outputs(args.dump_outputs, out, prefix=f"rank{rank}_" if world > 1 else "", share=world)
        del out

    elapsed_ms = max_over_ranks(elapsed_ms, dev, world)
    ms_per_step = elapsed_ms / args.steps
    value = n3_global * nsmall * args.steps / (elapsed_ms * 1e-3)

    # ---- roofline of the dominant kernel (advance_mu_t over this rank's patch) ----
    peak, peak_src = peaks()
    kernel_ms = elapsed_ms / (args.steps * nsmall)             # average duration of one full-patch pass, live
    achieved = bytes_local / (kernel_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": bytes_local,
                "kernel": KERNEL_NAMES[patch.last_kernel()],
                "avg_launch_ms": kernel_ms,
                "frac_of_nominal_8TBs": achieved / 8000.0}
    if world > 1:
        roofline["note"] = ("per-rank patch; avg_launch_ms is one small step of the rank (halo push + advance_mu_t, "
                            "max over ranks); no ncu traffic capture at N > 1")
    prof = os.path.join(ROOT, "profiles", "traffic.json")
    if world == 1 and os.path.exists(prof):
        try:
            tr = json.load(open(prof)).get(args.workload)
            if tr:
                roofline["traffic"] = tr["dram_bytes_per_launch"]
                roofline["traffic_source"] = tr.get("source")
        except Exception:
            pass

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": WORKLOADS[args.workload][6],
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.workload}: {WORKLOADS[args.workload][7]}",
                   "grid": f"{g.ide}x{g.jde}x{g.kde}", "small_steps_per_step": nsmall,
                   "points_per_small_step": n3_global, "flags": "specified=T periodic_x=F nested=F",
                   "decomposition": f"{px}x{py} (i x j) patches, halo {HALO}",
                   "kernel": args.kernel, "l2": l2_note, "launch": exec_mode},
        "roofline": roofline, "gpu_launches": launches,
    }
    try:                                                        # the launch the TMA kernel makes for this rank's patch
        plan = (ctypes.c_longlong * 10)()
        dom = pg.domain()
        if kernel in (wrf.KERNEL_AUTO, wrf.KERNEL_PIPE) and wrf.lib().wrfb200_pipe_plan(
                ctypes.byref(dom), pg.its, pg.ite, pg.jts, pg.jte, pg.kts, pg.kte, 0, plan) == 0:
            line["config"]["launch_shape"] = (
                "grid %d = %d remainder-strip blocks + %d tile columns x (%d block rows of 2-row tiles + %d of 1-row tiles), "
                "TJ*10+STAGES %d, %d B dynamic shared memory" % (plan[8], plan[6], plan[3], plan[4], plan[5], plan[0], plan[9]))
    except Exception:
        pass
    if exchange:
        line["config"]["halo_exchange"] = exchange
        line["halo_wait_timeouts"] = halo_timeouts
    if parity is not None:
        line["parity"] = parity
    if clocks:
        line["clocks"] = clocks

    # ---- the load-bearing loop: the same steps with the advance_uv stand-in between them (all N) ----
    if not args.no_extras:
        if world == 1:
            parallel.connect_fused(patch, decomp, rank, allgather)       # 1x1 grid: no neighbours, same code path
            patch.comm_push_constants()
        ms = max_over_ranks(time_loop(lambda: patch.comm_loop(nsmall, standin=True, c=C_UV, graph=True),
                                      min(args.steps, 10), 2, main, barrier, flush), dev, world)
        k = min(args.steps, 10)
        line["standin_loop"] = {
            "value": n3_global * nsmall * k / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / k,
            "what": "the same loop with the deterministic advance_uv stand-in between steps (u, v rewritten every step, "
                    "so every exchanged halo cell changes): +2 elementwise kernels per step that are not part of advance_mu_t"}
        if world > 1:
            line["standin_loop"]["halo_wait_timeouts"] = patch.comm_status()[0]

    # ---- end to end through the reference-facing C-ABI call with HOST buffers (rank-local patch) ----
    if not args.no_e2e:
        e2e_steps = max(1, min(args.steps, args.e2e_steps))
        head, variants = e2e_measurements(host, pg, scalars, nsmall, kernel, world, dev, barrier, e2e_steps, n3_global,
                                          with_pageable=(world == 1 and not args.no_extras))
        line["e2e"] = head
        line["e2e_variants"] = variants

    # ---- the other BASELINE.json configs, same method (N = 1: conus12, deep120, weak2048; N > 1: weak2048) ----
    if not args.no_extras and args.workload == "conus3":
        barrier()                                               # nobody unmaps a neighbour that is still in its loop
        patch.close()
        patch = None
        extras = {}
        names = ("conus12", "deep120", "weak2048") if world == 1 else ("weak2048",)
        for name in names:
            try:
                extras[name] = measure_extra_workload(name, world, rank, local_rank, dev, main, barrier, allgather, kernel)
            except Exception as e:                              # reported, never fatal
                extras[name] = {"unavailable": f"{type(e).__name__}: {e}"[:200]}
        line["workloads"] = extras

    # ---- device-pointer drop-in: the caller's OWN dense device arrays, launched in place (N = 1) ----
    if world == 1 and not args.no_extras and args.workload == "conus3":
        try:
            line["device_pointer_call"] = measure_device_pointer_call(g.ide, g.jde, g.kde, scalars, dx, dev, main, barrier)
        except Exception as e:                                  # reported, never fatal
            line["device_pointer_call"] = {"unavailable": f"{type(e).__name__}: {e}"[:200]}

    # ---- CPU baseline beside it (rank 0, N=1 only) ----
    if world == 1 and not args.no_cpu:
        cpu_fields = {k: (v.copy() if k in ("ww", "t", "t_ave", "mu", "muave", "muts", "mudf") else v) for k, v in host.items()}
        r = cpu_reference_run(g, scalars, cpu_fields, steps=10, warmup=2)     # ~1 s wall = 10-30 core-seconds of CPU work
        line["cpu_baseline"] = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}
        del cpu_fields

    # ---- the repo's own CUDA-C kernel, recompiled for sm_100a, kernel-only like the reference's timer ----
    if world == 1 and not args.no_ref_cuda:
        try:
            line["ref_cuda_kernel"] = time_reference_cuda_kernel(g, scalars, host, dev)
        except Exception as e:                                  # reported, never fatal
            line["ref_cuda_kernel"] = {"unavailable": str(e)[:200]}

    if rank == 0:
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if patch is not None:
        if world > 1:
            torch.cuda.synchronize()
            dist.barrier()                                      # nobody unmaps a neighbour that is still in its loop
        patch.close()
    del pinned_keep
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def time_reference_cuda_kernel(g, scalars, host, dev, reps=5):
    """The reference's advance_mu_t_kernel (unmodified TU, -arch=sm_100a -fmad=false) on the same inputs,
    launch geometry of advance_mu_t_no_async.cu:54-55, scratch arrays in global memory."""
    import torch
    import wrf_model_cuda_sample_b200 as wrf
    from oracle import loader
    if not loader.have_ref_cuda():
        raise RuntimeError("oracle/_ref/libref_cuda_kernel.so not built")
    d = {n: torch.from_numpy(host[n]).to(dev) for n in wrf.FIELDS}
    scratch = {"wdtn": torch.empty_like(d["u"]), "dvdxi": torch.empty_like(d["u"]), "dmdt": torch.empty_like(d["mu"])}
    ptrs = {n: d[n].data_ptr() for n in d}
    sptr = {n: scratch[n].data_ptr() for n in scratch}
    stream = torch.cuda.current_stream().cuda_stream
    for _ in range(2):
        loader.reference_cuda_kernel(ptrs, sptr, g, scalars, stream)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        loader.reference_cuda_kernel(ptrs, sptr, g, scalars, stream)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    n3, _ = g.updated_points()
    return {"value": n3 / (ms * 1e-3), "unit": UNIT, "ms_per_small_step": ms,
            "what": "reference advance_mu_t_kernel.cu, unmodified, nvcc -O3 -arch=sm_100a -fmad=false, "
                    "<<<(idim/64+1, jdim), 64>>>, kernel-only"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=("ours", "reference"), default="ours")
    ap.add_argument("--workload", choices=sorted(WORKLOADS), default="conus3")
    ap.add_argument("--kernel", choices=("auto", "pipe", "tile", "column"), default="auto")
    ap.add_argument("--pgrid", default="", help="process grid PXxPY (default: j-slabs 1xN)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="N>1: launch the loop eagerly instead of replaying a CUDA graph")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-ref-cuda", action="store_true")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the stand-in loop, the other BASELINE configs and the pageable e2e variants")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the output fields of the last one to DIR/<name>.npy "
                         "(float32, at most 64 MB in all: larger fields are sampled at fixed seeded positions)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if os.environ.get("BENCH_HANG_DUMP"):                       # debugging aid: dump all stacks after N seconds
        import faulthandler
        faulthandler.dump_traceback_later(int(os.environ["BENCH_HANG_DUMP"]), exit=True)
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
