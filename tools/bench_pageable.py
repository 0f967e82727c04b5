"""Time the host-array advance_mu_t call on ordinary pageable arrays (the staged route) against the same call on
page-locked arrays (the direct route).

    python tools/bench_pageable.py --out profiles/pageable.json [--devices 0,1]

On 1800x1060x50, in binary32 and in real*8, it times in one run, alternating the modes over --rounds rounds:
  (a) one call on pageable numpy arrays (every array staged through the library's pinned bounce buffers);
  (b) the same call on torch-pinned copies of the same arrays (every array copied directly);
  (c) the 6-call acoustic loop with residency on the pageable arrays (bench.py's `e2e` pattern);
  (d) one resident step on the pageable arrays (u, v up, the 7 outputs down);
  (e) one pageable cudaMemcpyAsync of a 387 MB array handed to the driver: the rate of the route the staged one
      replaces.
Each call ends with the host synchronised, so a host clock around it is the call's time; the median over the rounds
is reported.  With --devices naming more than one device, (a) is also timed with the call split over them
(wrfb200_set_default_devices).  The outputs of (a) and (b) are compared bit for bit.  The card's name and power
limit, the host's CPU count and affinity, the worker pool's size (the threads the first staged call started), the
pinned bounce bytes each cache holds and the route wrfb200_default_last_transfer reported are read in the same run.
The JSON goes only to --out.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import wrf_model_cuda_sample_b200 as wrf  # noqa: E402

NSMALL = 6
ROUTES = {wrf.TRANSFER_DIRECT: "direct", wrf.TRANSFER_MIXED: "mixed", wrf.TRANSFER_STAGED: "staged"}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    rows = [[c.strip() for c in line.split(",")] for line in q.stdout.strip().splitlines() if line.strip()]
    return [{"index": int(r[0]), "name": r[1], "power_limit": r[2]} for r in rows]


def threads():
    return len(os.listdir("/proc/self/task"))


def bounce_bytes(g, esize):
    """The pinned bounce bytes one cache holds for a whole-patch call of g (run_host_compat_body): five buffers of one
    slab of a 3-D field, four of the same rows of a 2-D one."""
    i0, i1, j0, j1, k0, k1 = g.bounds()
    nj = j1 - j0 + 1
    idim, jdim, kdim = g.ime - g.ims + 1, g.jme - g.jms + 1, g.kme - g.kms + 1
    nslab = 1
    if idim * kdim * jdim * esize >= 16 << 20 and nj >= 32:
        nslab = min(nj // 16, 16)
    rows = nj // nslab + 3
    return 5 * rows * kdim * idim * esize + 4 * rows * idim * esize


def pinned_copy(fields):
    import torch
    keep, out = [], {}
    for k, v in fields.items():
        t = torch.empty(v.shape, dtype=torch.float32 if v.dtype == np.float32 else torch.float64, pin_memory=True)
        a = t.numpy()
        np.copyto(a, v)
        keep.append(t)
        out[k] = a
    return out, keep


def driver_pageable_rate(nbytes, reps):
    """GB/s of one pageable host->device cudaMemcpyAsync of nbytes, synchronised."""
    import torch
    src = torch.from_numpy(np.ones(nbytes // 4, dtype=np.float32))
    dst = torch.empty(src.shape, dtype=src.dtype, device="cuda")
    dst.copy_(src, non_blocking=True)
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts)


def run_precision(dtype, g, scalars, devs, rounds, reps, pool_seen):
    lib = wrf.lib()
    n3 = g.updated_points()[0]
    pristine = {k: v.astype(dtype) for k, v in wrf.synth_fields(g).items()}
    pageable = {k: v.copy() for k, v in pristine.items()}
    pinned, keep = pinned_copy(pristine)
    esize = np.dtype(dtype).itemsize
    raw_bytes = pristine["u"].nbytes if dtype == np.float32 else pristine["u"].nbytes // 2   # 387 MB either way

    def call(f, nsteps=1):
        wrf.call_with_fields(f, g, *scalars, nsteps=nsteps)

    def residency_loop():
        with wrf.acoustic_loop():
            for _ in range(NSMALL):
                call(pageable)

    def resident_step():
        with wrf.acoustic_loop():
            call(pageable)                                   # primes the mirrors (untimed below)
            t0 = time.perf_counter()
            for _ in range(reps):
                call(pageable)
            return (time.perf_counter() - t0) / reps

    def timed(fn):
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        return (time.perf_counter() - t0) / reps

    # the pool's size: the threads the first staged call of the process starts, with the runtime already up
    routes = {}
    call(pinned)
    routes["b_single_call_pinned"] = ROUTES[wrf.default_last_transfer()]
    if pool_seen is None:
        lib.wrfb200_release_cache()
        call(pinned)
        before = threads()
        call(pageable)
        pool_seen = threads() - before
    else:
        call(pageable)
    routes["a_single_call_pageable"] = ROUTES[wrf.default_last_transfer()]

    modes = {
        "a_single_call_pageable": lambda: timed(lambda: call(pageable)),
        "b_single_call_pinned": lambda: timed(lambda: call(pinned)),
        "c_residency_loop_6_pageable": lambda: timed(residency_loop),
        "d_resident_step_pageable": resident_step,
        "e_driver_pageable_memcpy_387MB": lambda: driver_pageable_rate(raw_bytes, reps),
    }
    if len(devs) > 1:
        def split():
            wrf.set_default_devices(devs)
            try:
                call(pageable)                               # warm-up of the parts' mirrors
                return timed(lambda: call(pageable))
            finally:
                wrf.set_default_devices(None)
        modes["a_single_call_pageable_devices_" + ",".join(map(str, devs))] = split
    samples = {m: [] for m in modes}
    for m, fn in modes.items():
        fn()                                                 # warm-up
    for r in range(rounds):
        order = list(modes) if r % 2 == 0 else list(modes)[::-1]
        for m in order:
            samples[m].append(modes[m]())

    # (a) against (b), bit for bit, from the same inputs
    for f in (pageable, pinned):
        for k in f:
            np.copyto(f[k], pristine[k])
    call(pageable)
    call(pinned)
    view = np.uint32 if esize == 4 else np.uint64
    mismatches = int(sum(np.count_nonzero(pageable[n].view(view) != pinned[n].view(view)) for n in wrf.OUTPUT_FIELDS))
    lib.wrfb200_release_cache()
    del keep

    steps = {m: (NSMALL if m.startswith("c_") else 1) for m in modes}
    rows = {}
    for m, v in samples.items():
        med = statistics.median(v)
        row = {"ms_median": round(1e3 * med, 2), "ms_all": [round(1e3 * x, 2) for x in v]}
        if m.startswith("e_"):
            row["bytes"] = int(raw_bytes)
            row["gb_per_s"] = round(raw_bytes / med / 1e9, 2)
        else:
            row["gpts_per_s"] = round(n3 * steps[m] / med / 1e9, 3)
        rows[m] = row
    return {"ms": rows, "routes": routes, "pinned_bounce_bytes_per_cache": bounce_bytes(g, esize),
            "outputs_a_vs_b_mismatches": mismatches}, pool_seen


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True, help="JSON summary file")
    ap.add_argument("--devices", default="0", help="comma-separated CUDA device ids for the split call, e.g. 0,1")
    ap.add_argument("--shape", default="1800,1060,50", help="e_we,e_sn,e_vert")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=3, help="timed repetitions of each mode per round")
    ap.add_argument("--precisions", default="r4,r8", help="r4 (binary32), r8 (real*8) or both")
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures on the GPU only")
    ngpu = torch.cuda.device_count()
    devs = [int(x) for x in args.devices.split(",")]
    bad = [d for d in devs if not 0 <= d < ngpu]
    if bad:
        raise SystemExit(f"devices {bad} not on this box ({ngpu} GPUs)")
    torch.cuda.set_device(devs[0])
    nx, ny, nz = (int(x) for x in args.shape.split(","))
    g = wrf.Grid.from_shape(nx, ny, nz, halo=5)
    scalars32 = (np.float32(1.0 / 3000.0), np.float32(1.0 / 3000.0), np.float32(3.0), np.float32(0.1))
    results, pool_seen = {}, None
    for p in args.precisions.split(","):
        dtype = {"r4": np.float32, "r8": np.float64}[p]
        scalars = tuple(dtype(x) for x in scalars32)
        results["binary32" if p == "r4" else "real*8"], pool_seen = run_precision(
            dtype, g, scalars, devs, args.rounds, args.reps, pool_seen)

    gpus = gpu_info()
    summary = {
        "tool": "tools/bench_pageable.py",
        "shape": [nx, ny, nz], "halo": 5,
        "rounds": args.rounds, "reps_per_round": args.reps,
        "gpu_count": ngpu, "gpus": gpus, "devices": devs,
        "host_nproc": os.cpu_count(), "host_affinity": len(os.sched_getaffinity(0)),
        "pool_threads_started_by_first_staged_call": pool_seen,
        "results": results,
    }
    with open(args.out, "w") as fh:
        json.dump(summary, fh, indent=1)
    print(f"{gpus[0]['name'] if gpus else '?'} x{ngpu}, power limit {gpus[0]['power_limit'] if gpus else '?'}; "
          f"nproc {os.cpu_count()}, affinity {len(os.sched_getaffinity(0))}, pool {pool_seen}; {nx}x{ny}x{nz}, "
          f"median of {args.rounds} rounds x {args.reps}")
    for prec, r in results.items():
        print(f"[{prec}] routes {r['routes']}, bounce {r['pinned_bounce_bytes_per_cache'] / 2**20:.1f} MiB per cache, "
              f"(a) vs (b) mismatches {r['outputs_a_vs_b_mismatches']}")
        for m, row in r["ms"].items():
            extra = f"{row['gb_per_s']} GB/s" if "gb_per_s" in row else f"{row['gpts_per_s']} Gpt/s"
            print(f"  {m:>44} {row['ms_median']:9.1f} ms  {extra}")


if __name__ == "__main__":
    main()
