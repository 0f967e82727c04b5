"""Time a nested run's host-array advance_mu_t calls with the domain caches (parent and nest keep their device state)
against the same calls when every domain switch frees the cache first.

    python tools/bench_nests.py --out profiles/nests.json [--rounds 5] [--cycles 3] [--precisions r4,r8]

One parent time step of a WRF-like sequence, on pageable numpy arrays: the parent (1800x1060x50, `specified`) runs
one acoustic loop of 6 calls with residency (wrfb200_acoustic_loop_begin / _end), then the nest (901x601x50, `nested`)
runs three such loops (parent_time_step_ratio 3).  A cycle is that parent step; each timed sequence is --cycles of
them.  Two variants, alternated over --rounds rounds in one run:
  kept:     the calls as they are: a switch back to a domain finds its mirrors (one untimed call of each domain
            before the sequence re-creates what a preceding "released" sequence freed);
  released: before every switch of domain, the thread's host-array caches are freed -- mirrors, staging and
            bounce buffers, lanes and events, and nothing else (not the staged route's host threads, not the
            device-pointer wrappers) -- so that each switch frees and rebuilds exactly what a cache of one memory
            shape did.  The tool frees them by changing the thread's device list (wrfb200_set_default_devices to
            the current device and back), which releases those caches and leaves the calls on the single-device
            path.
Each call ends with the host synchronised, so a host clock around it is the call's time.  Reported per variant: the
sequence time, and the time of each call after a switch (the first call of the parent's loop, the first call of the
nest's first loop), medians over the rounds, with what wrfb200_default_last_cache said about those calls.  The card's
name and power limit are read in the same run.  The JSON goes only to --out.
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

NSMALL = 6              # acoustic steps per loop
RATIO = 3               # nest steps per parent step
VARIANTS = ("kept", "released")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    rows = [[c.strip() for c in line.split(",")] for line in q.stdout.strip().splitlines() if line.strip()]
    return [{"index": int(r[0]), "name": r[1], "power_limit": r[2]} for r in rows]


def release_host_caches(device):
    """Free this thread's host-array caches only: a change of the device list releases them."""
    wrf.set_default_devices([device])
    wrf.set_default_devices(None)


def run_precision(dtype, parent, nest, cycles, rounds):
    import torch
    lib = wrf.lib()
    device = torch.cuda.current_device()
    scalars = tuple(dtype(x) for x in (1.0 / 3000.0, 1.0 / 3000.0, 3.0, 0.1))
    fields = {"parent": {k: v.astype(dtype) for k, v in wrf.synth_fields(parent, seed=1).items()},
              "nest": {k: v.astype(dtype) for k, v in wrf.synth_fields(nest, seed=2).items()}}
    grids = {"parent": parent, "nest": nest}

    def loop(name, release):
        """One acoustic loop of the domain; returns the first call's time and cache state."""
        if release:
            release_host_caches(device)
        first = state = None
        with wrf.acoustic_loop():
            for s in range(NSMALL):
                t0 = time.perf_counter()
                wrf.call_with_fields(fields[name], grids[name], *scalars)
                if s == 0:
                    first, state = time.perf_counter() - t0, wrf.default_last_cache()
        return first, state

    def sequence(variant):
        release = variant == "released"
        if not release:
            for name in ("nest", "parent"):                  # untimed: a "released" sequence before freed both
                wrf.call_with_fields(fields[name], grids[name], *scalars)
        after_switch = {"parent": [], "nest": []}
        states = {"parent": set(), "nest": set()}
        t0 = time.perf_counter()
        for _ in range(cycles):
            t, s = loop("parent", release)
            after_switch["parent"].append(t)
            states["parent"].add(s)
            for r in range(RATIO):
                t, s = loop("nest", release and r == 0)        # one switch into the nest per parent step
                if r == 0:
                    after_switch["nest"].append(t)
                    states["nest"].add(s)
        return time.perf_counter() - t0, after_switch, states

    for v in VARIANTS:
        sequence(v)                                          # warm-up: both domains' mirrors, the pool, the modules
    samples = {v: {"sequence": [], "parent": [], "nest": [], "states": {"parent": set(), "nest": set()}}
               for v in VARIANTS}
    for r in range(rounds):
        for v in (VARIANTS if r % 2 == 0 else VARIANTS[::-1]):
            total, after, states = sequence(v)
            samples[v]["sequence"].append(total)
            for d in ("parent", "nest"):
                samples[v][d] += after[d]
                samples[v]["states"][d] |= states[d]
    lib.wrfb200_release_cache()

    def row(xs):
        return {"ms_median": round(1e3 * statistics.median(xs), 2), "ms_all": [round(1e3 * x, 2) for x in xs]}

    out = {}
    for v in VARIANTS:
        s = samples[v]
        out[v] = {"sequence": row(s["sequence"]),
                  "first_call_after_switch": {d: row(s[d]) for d in ("parent", "nest")},
                  "cache_states_after_switch": {d: sorted(s["states"][d]) for d in ("parent", "nest")}}
    k, rel = out["kept"]["sequence"]["ms_median"], out["released"]["sequence"]["ms_median"]
    out["released_minus_kept_ms_per_parent_step"] = round((rel - k) / cycles, 2)
    spread = [1e3 * x for x in samples["kept"]["sequence"]]
    out["kept_sequence_spread_ms"] = round(max(spread) - min(spread), 2)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True, help="JSON summary file")
    ap.add_argument("--parent", default="1800,1060,50", help="e_we,e_sn,e_vert of the parent (specified)")
    ap.add_argument("--nest", default="901,601,50", help="e_we,e_sn,e_vert of the nest (nested)")
    ap.add_argument("--cycles", type=int, default=3, help="parent time steps per timed sequence")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--precisions", default="r4", help="r4 (binary32), r8 (real*8) or both")
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures on the GPU only")
    px, py, pz = (int(x) for x in args.parent.split(","))
    nx, ny, nz = (int(x) for x in args.nest.split(","))
    parent = wrf.Grid.from_shape(px, py, pz, halo=5, specified=True)
    nest = wrf.Grid.from_shape(nx, ny, nz, halo=5, specified=False, nested=True)
    results = {}
    for p in args.precisions.split(","):
        dtype = {"r4": np.float32, "r8": np.float64}[p]
        results["binary32" if p == "r4" else "real*8"] = run_precision(dtype, parent, nest, args.cycles, args.rounds)

    gpus = gpu_info()
    summary = {
        "tool": "tools/bench_nests.py",
        "parent": [px, py, pz], "nest": [nx, ny, nz], "halo": 5,
        "calls_per_loop": NSMALL, "nest_loops_per_parent_step": RATIO,
        "cycles_per_sequence": args.cycles, "rounds": args.rounds,
        "gpus": gpus, "host_nproc": os.cpu_count(), "host_affinity": len(os.sched_getaffinity(0)),
        "results": results,
    }
    with open(args.out, "w") as fh:
        json.dump(summary, fh, indent=1)
    print(f"{gpus[0]['name'] if gpus else '?'}, power limit {gpus[0]['power_limit'] if gpus else '?'}; parent "
          f"{px}x{py}x{pz}, nest {nx}x{ny}x{nz}; {args.cycles} parent steps per sequence, median of {args.rounds}")
    for prec, r in results.items():
        print(f"[{prec}] released - kept: {r['released_minus_kept_ms_per_parent_step']} ms per parent step "
              f"(kept sequences spread {r['kept_sequence_spread_ms']} ms)")
        for v in VARIANTS:
            a = r[v]
            print(f"  {v:>8}: sequence {a['sequence']['ms_median']:9.1f} ms; first call after a switch: parent "
                  f"{a['first_call_after_switch']['parent']['ms_median']:7.1f} ms, nest "
                  f"{a['first_call_after_switch']['nest']['ms_median']:7.1f} ms; states "
                  f"{a['cache_states_after_switch']}")


if __name__ == "__main__":
    main()
