"""Time the host-array advance_mu_t call as WRF's OpenMP builds make it -- one call per j-tile from a pool of
threads -- with the per-thread caches (the default) and with shared-tiles mode (wrfb200_set_shared_tiles).

    python tools/bench_omp_tiles.py --out profiles/omp_tiles.json

On 1800x1060x50 (binary32, host arrays in page-locked torch memory), for 1, 4, 8 and 16 threads each calling its
own j-tile (the patch's rows cut evenly, as WRF's tile loop does), it measures, per mode:
  (a) the 6-call acoustic loop: wrfb200_acoustic_loop_begin / _end on the main thread, six steps, each step every
      thread's tile call and a join (residency holds on the worker threads in shared mode only);
  (b) one call per tile that uploads everything (no loop);
  (c) the device memory taken once every thread has made its first call (cudaMemGetInfo, threads still alive).
Threads persist across the timed calls, as an OpenMP pool does.  The two modes alternate over --rounds rounds and
the median is reported.  The outputs of one full call from the same inputs are compared bit for bit between the
modes.  GPU name and power limit are read in the same run.  The JSON goes only to --out.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import wrf_model_cuda_sample_b200 as wrf  # noqa: E402

SCALARS = (np.float32(1.0 / 3000.0), np.float32(1.0 / 3000.0), np.float32(3.0), np.float32(0.1))
NSMALL = 6
MODES = ("per_thread", "shared")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    rows = [[c.strip() for c in line.split(",")] for line in q.stdout.strip().splitlines() if line.strip()]
    return [{"index": int(r[0]), "name": r[1], "power_limit": r[2]} for r in rows]


class Pool:
    """n persistent threads; run(job) calls job(t) in every thread t and returns when all are done."""

    def __init__(self, n):
        self.n = n
        self.job = None
        self.errors = []
        self.start, self.done = threading.Barrier(n + 1), threading.Barrier(n + 1)
        self.threads = [threading.Thread(target=self._work, args=(t,)) for t in range(n)]
        for th in self.threads:
            th.start()

    def _work(self, t):
        while True:
            self.start.wait()
            job = self.job
            if job is None:
                wrf.lib().wrfb200_release_cache()           # this thread's own caches, before it ends
                self.done.wait()
                return
            try:
                job(t)
            except BaseException as e:                       # noqa: BLE001 -- reported by run()
                self.errors.append(e)
            self.done.wait()

    def run(self, job):
        self.job = job
        self.start.wait()
        self.done.wait()
        if self.errors:
            raise self.errors[0]

    def close(self):
        self.job = None
        self.start.wait()
        self.done.wait()
        for th in self.threads:
            th.join()


def j_tiles(g, n):
    m = g.jde - g.jds + 1
    edges = [g.jds + m * p // n for p in range(n + 1)]
    return [g.with_tile(g.ids, g.ide, edges[p], edges[p + 1] - 1) for p in range(n)]


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True, help="JSON summary file")
    ap.add_argument("--shape", default="1800,1060,50", help="e_we,e_sn,e_vert")
    ap.add_argument("--threads", default="1,4,8,16")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3, help="timed repetitions of (a) and (b) per round")
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures on the GPU only")
    torch.cuda.set_device(0)
    nx, ny, nz = (int(x) for x in args.shape.split(","))
    g = wrf.Grid.from_shape(nx, ny, nz, halo=5)
    n3 = g.updated_points()[0]
    counts = [int(x) for x in args.threads.split(",")]
    fields = wrf.synth_fields(g, pinned=True)
    pristine = {k: v.copy() for k, v in fields.items() if isinstance(v, np.ndarray)}
    arrays = {k: v for k, v in fields.items() if isinstance(v, np.ndarray)}

    def full_call(tiles):
        return lambda t: wrf.call_with_fields(arrays, tiles[t], *SCALARS)

    def timed(fn, reps):
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        return (time.perf_counter() - t0) / reps

    samples = {n: {m: {"a_loop_6": [], "b_full_call": [], "c_device_bytes": []} for m in MODES} for n in counts}
    reference, mismatches = None, {}
    for r in range(args.rounds):
        for n in counts:
            tiles = j_tiles(g, n)
            for mode in (MODES if r % 2 == 0 else MODES[::-1]):
                wrf.lib().wrfb200_release_cache()
                torch.cuda.synchronize()
                free0 = torch.cuda.mem_get_info()[0]
                wrf.set_shared_tiles(mode == "shared")
                pool = Pool(n)
                try:
                    if r == 0:                              # outputs of one full call from the pristine inputs
                        for k in arrays:
                            np.copyto(arrays[k], pristine[k])
                    pool.run(full_call(tiles))              # also the warm-up: mirrors, lanes, staging
                    samples[n][mode]["c_device_bytes"].append(free0 - torch.cuda.mem_get_info()[0])
                    if r == 0:
                        out = {k: arrays[k].copy() for k in wrf.OUTPUT_FIELDS}
                        if reference is None:
                            reference = out
                        mismatches[f"{n}/{mode}"] = int(sum(np.count_nonzero(out[k].view(np.uint32) !=
                                                                             reference[k].view(np.uint32))
                                                            for k in wrf.OUTPUT_FIELDS))
                        del out

                    def loop6():
                        with wrf.acoustic_loop():
                            for _ in range(NSMALL):
                                pool.run(full_call(tiles))

                    loop6()                                 # warm-up of the resident path
                    samples[n][mode]["a_loop_6"].append(timed(loop6, args.reps))
                    samples[n][mode]["b_full_call"].append(timed(lambda: pool.run(full_call(tiles)), args.reps))
                finally:
                    pool.close()
                    wrf.set_shared_tiles(False)
    wrf.lib().wrfb200_release_cache()

    table = {}
    for n in counts:
        row = {}
        for mode in MODES:
            s = samples[n][mode]
            a, b = statistics.median(s["a_loop_6"]), statistics.median(s["b_full_call"])
            row[mode] = {"a_loop_6_ms": round(1e3 * a, 1), "a_loop_6_ms_all": [round(1e3 * x, 1) for x in s["a_loop_6"]],
                         "a_gpts_per_s": round(n3 * NSMALL / a / 1e9, 3),
                         "b_full_call_ms": round(1e3 * b, 1),
                         "b_full_call_ms_all": [round(1e3 * x, 1) for x in s["b_full_call"]],
                         "c_device_gb": round(max(s["c_device_bytes"]) / 1e9, 2)}
        table[str(n)] = row
    gpus = gpu_info()
    summary = {
        "tool": "tools/bench_omp_tiles.py",
        "shape": [nx, ny, nz], "halo": 5, "precision": "binary32",
        "host_arrays": "page-locked torch tensors (synth_fields(pinned=True))",
        "tiles": "j-tiles, one per thread, the domain's rows cut evenly",
        "rounds": args.rounds, "reps_per_round": args.reps,
        "gpu": gpus[0] if gpus else None, "gpu_count": torch.cuda.device_count(), "host_cpus": os.cpu_count(),
        "threads": counts, "results": table,
        "output_mismatches_vs_first_run": mismatches,
    }
    with open(args.out, "w") as fh:
        json.dump(summary, fh, indent=1)
    print(f"{gpus[0]['name'] if gpus else '?'}, power limit {gpus[0]['power_limit'] if gpus else '?'}; "
          f"{nx}x{ny}x{nz} binary32, pinned host arrays, median of {args.rounds} rounds x {args.reps}")
    print(f"{'threads':>7} {'mode':>10} {'(a) loop ms':>12} {'(b) call ms':>12} {'(c) GB':>8}")
    for n in counts:
        for mode in MODES:
            x = table[str(n)][mode]
            print(f"{n:>7} {mode:>10} {x['a_loop_6_ms']:12.1f} {x['b_full_call_ms']:12.1f} {x['c_device_gb']:8.2f}")
    print("output mismatches:", mismatches)


if __name__ == "__main__":
    main()
