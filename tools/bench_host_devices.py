"""Time the host-array advance_mu_t call split over several GPUs of one box (wrfb200_set_default_devices).

    python tools/bench_host_devices.py --devices 0,1,2,3,4,5,6,7 --out profiles/host_devices.json

On 1800x1060x50 (binary32, ordinary numpy arrays page-locked by the library, wrfb200_set_host_pinning(1)) it
times, for the device lists [d0], [d0,d1], [d0..d3], [d0..d7] (as far as --devices reaches) and [d0,d0]:
  (a) one call that re-uploads everything (the reference's call pattern);
  (b) the 6-call acoustic loop with residency (first call all inputs, then u, v only: bench.py's `e2e`);
  (c) one resident step (u, v up, the 7 outputs down);
  (d) the _loop entry with nsteps = 6 (one upload, 6 steps, one download).
Each call ends with the host synchronised, so a host clock around it is the call's time.  The lists are
alternated over --rounds rounds and the median is reported.  Every list's outputs of (a) and (d) are compared bit
for bit with those of [d0].  The host->device rate of the library-pinned arrays is measured on every device, to
show that the registration is portable.  GPU name, power limit, GPU count and host CPU count are read in the same
run.  The JSON goes only to --out.
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

SCALARS = (np.float32(1.0 / 3000.0), np.float32(1.0 / 3000.0), np.float32(3.0), np.float32(0.1))
NSMALL = 6


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    rows = [[c.strip() for c in line.split(",")] for line in q.stdout.strip().splitlines() if line.strip()]
    return [{"index": int(r[0]), "name": r[1], "power_limit": r[2]} for r in rows]


def device_lists(devs):
    lists = [devs[:n] for n in (1, 2, 4, 8) if n <= len(devs)]
    return lists + [[devs[0], devs[0]]]


def h2d_rate(a, device, reps=3):
    """GB/s of a host->device copy of the numpy array `a` (as the library left it: registered or not)."""
    import torch
    src = torch.from_numpy(a)
    with torch.cuda.device(device):
        dst = torch.empty(src.shape, dtype=src.dtype, device=f"cuda:{device}")
        best = 0.0
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            dst.copy_(src, non_blocking=True)
            e1.record()
            e1.synchronize()
            best = max(best, a.nbytes / (e0.elapsed_time(e1) * 1e-3) / 1e9)
        pinned = bool(src.is_pinned())
        del dst
    return best, pinned


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--devices", default="0", help="comma-separated CUDA device ids, e.g. 0,1,2,3")
    ap.add_argument("--out", required=True, help="JSON summary file")
    ap.add_argument("--shape", default="1800,1060,50", help="e_we,e_sn,e_vert")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3, help="timed repetitions of each mode per round")
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures on the GPU only")
    ngpu = torch.cuda.device_count()
    devs = [int(x) for x in args.devices.split(",")]
    bad = [d for d in devs if not 0 <= d < ngpu]
    if bad:
        raise SystemExit(f"devices {bad} not on this box ({ngpu} GPUs)")
    nx, ny, nz = (int(x) for x in args.shape.split(","))
    g = wrf.Grid.from_shape(nx, ny, nz, halo=5)
    n3 = g.updated_points()[0]
    pristine = wrf.synth_fields(g)
    fields = {k: v.copy() for k, v in pristine.items()}
    lib = wrf.lib()
    lib.wrfb200_set_host_pinning(1)                         # the library registers the arrays (portable)
    lists = device_lists(devs)
    key = lambda dl: ",".join(map(str, dl))                  # noqa: E731

    def timed(fn, reps):
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        return (time.perf_counter() - t0) / reps

    def residency_loop():
        with wrf.acoustic_loop():
            for _ in range(NSMALL):
                wrf.call_with_fields(fields, g, *SCALARS)

    modes = {
        "a_single_call": lambda: wrf.call_with_fields(fields, g, *SCALARS),
        "b_residency_loop_6": residency_loop,
        "d_loop_entry_6": lambda: wrf.call_with_fields(fields, g, *SCALARS, nsteps=NSMALL),
    }
    samples = {key(dl): {m: [] for m in list(modes) + ["c_resident_step"]} for dl in lists}
    for r in range(args.rounds):
        for dl in (lists if r % 2 == 0 else lists[::-1]):
            wrf.set_default_devices(dl)
            for m, fn in modes.items():
                fn()                                        # warm-up: mirrors, lanes, registration
                samples[key(dl)][m].append(timed(fn, args.reps))
            with wrf.acoustic_loop():
                wrf.call_with_fields(fields, g, *SCALARS)   # primes the mirrors
                samples[key(dl)]["c_resident_step"].append(
                    timed(lambda: wrf.call_with_fields(fields, g, *SCALARS), args.reps))

    # bit-for-bit against the first list, from the same inputs
    outputs = {}
    mismatches = {}
    for dl in lists:
        wrf.set_default_devices(dl)
        res = {}
        for m in ("a_single_call", "d_loop_entry_6"):
            for k in fields:
                np.copyto(fields[k], pristine[k])
            modes[m]()
            res[m] = {n: fields[n].copy() for n in wrf.OUTPUT_FIELDS}
        if not outputs:
            outputs = res
        mismatches[key(dl)] = {m: int(sum(np.count_nonzero(res[m][n].view(np.uint32) != outputs[m][n].view(np.uint32))
                                          for n in wrf.OUTPUT_FIELDS)) for m in res}
        del res

    # host->device rate of the arrays the library registered, per device
    wrf.set_default_devices(None)
    h2d = {}
    for d in sorted(set(devs)):
        rate, pinned = h2d_rate(fields["u"], d)
        h2d[str(d)] = {"gb_per_s": round(rate, 2), "seen_as_pinned": pinned, "bytes": int(fields["u"].nbytes)}
    lib.wrfb200_set_host_pinning(0)
    lib.wrfb200_release_cache()

    steps = {"a_single_call": 1, "b_residency_loop_6": NSMALL, "c_resident_step": 1, "d_loop_entry_6": NSMALL}
    table = {}
    base = {m: statistics.median(v) for m, v in samples[key(lists[0])].items()}
    for dl in lists:
        row = {}
        for m, v in samples[key(dl)].items():
            med = statistics.median(v)
            row[m] = {"ms_median": round(1e3 * med, 2), "ms_all": [round(1e3 * x, 2) for x in v],
                      "gpts_per_s": round(n3 * steps[m] / med / 1e9, 3), "speedup_vs_first": round(base[m] / med, 3)}
        table[key(dl)] = row
    gpus = gpu_info()
    summary = {
        "tool": "tools/bench_host_devices.py",
        "shape": [nx, ny, nz], "halo": 5, "precision": "binary32",
        "host_arrays": "numpy, page-locked by the library (wrfb200_set_host_pinning(1), cudaHostRegisterPortable)",
        "rounds": args.rounds, "reps_per_round": args.reps,
        "gpu_count": ngpu, "gpus": gpus, "host_cpus": os.cpu_count(),
        "host_cpus_usable": len(os.sched_getaffinity(0)),
        "device_lists": [key(dl) for dl in lists],
        "ms": table,
        "mismatches_vs_first_list": mismatches,
        "h2d_library_pinned": h2d,
    }
    with open(args.out, "w") as fh:
        json.dump(summary, fh, indent=1)
    print(f"{gpus[0]['name'] if gpus else '?'} x{ngpu}, power limit {gpus[0]['power_limit'] if gpus else '?'}, "
          f"{os.cpu_count()} host CPUs; {nx}x{ny}x{nz}, median of {args.rounds} rounds x {args.reps}")
    print(f"{'devices':>16} {'(a) ms':>9} {'(b) ms':>9} {'(c) ms':>9} {'(d) ms':>9}  mismatches")
    for dl in lists:
        r = table[key(dl)]
        print(f"{key(dl):>16} " + " ".join(f"{r[m]['ms_median']:9.1f}" for m in
                                         ("a_single_call", "b_residency_loop_6", "c_resident_step", "d_loop_entry_6"))
              + f"  {mismatches[key(dl)]}")
    print("h2d GB/s of library-pinned arrays:", {d: v["gb_per_s"] for d, v in h2d.items()})


if __name__ == "__main__":
    main()
