"""Measure the real*8 advance_mu_t kernels on one GPU and check what they computed.

    python tools/bench_r8.py [--out FILE] [--reps R] [--launches N]

In one run: the device name and power limit; the device-to-device copy peak (a >= 2 GB cudaMemcpyAsync, read +
write bytes); then for 1800x1060x50, 425x300x35 and 512x512x120 the r8 tile kernel, the r8 column kernel and the
binary32 AUTO kernel, timed with CUDA events over N back-to-back launches, alternated R times; the r8 end-to-end
time of a 6-step host-pointer loop under wrfb200_acoustic_loop_begin/end with pinned arrays; and a check of
every timed r8 kernel's output against the binary64 C checker (mismatches must be 0).  One JSON line per size is
printed; with --out the summary JSON is also written to FILE.  Needs a GPU; there is no CPU fallback.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import wrf_model_cuda_sample_b200 as wrf  # noqa: E402
from tests import r8_checkers  # noqa: E402

SIZES = [(1800, 1060, 50), (425, 300, 35), (512, 512, 120)]
SCALARS = (1.0 / 3000.0, 1.0 / 3000.0, 3.0, 0.1)        # 3 km spacing; exact in float32 and float64 alike
L2_BYTES = 126 * 2 ** 20


def device_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = r.stdout.strip().splitlines()[torch.cuda.current_device()] if r.returncode == 0 else ""
    return {"name": torch.cuda.get_device_name(), "nvidia_smi": line}


def copy_peak(gbytes=4.0, reps=20):
    """Device-to-device copy rate (read + write bytes per second) of one cudaMemcpyAsync of gbytes/2 each way."""
    n = int(gbytes * 2 ** 30 / 2) // 4
    a = torch.empty(n, dtype=torch.float32, device="cuda")
    b = torch.empty_like(a)
    a.fill_(1.0)
    for _ in range(3):
        b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    del a, b
    return {"bytes_per_copy": 2 * n * 4, "ms": ms, "GBps": 2 * n * 4 / ms / 1e6}


def patch(g, fields, dtype, kernel):
    p = wrf.Patch(g, dtype=dtype)
    p.set_scalars(*SCALARS)
    p.set_kernel(kernel)
    p.upload(fields)
    p.sync()
    return p


def time_arms(arms, launches, reps):
    """CUDA-event time per launch of each arm, the arms alternated `reps` times; median over reps."""
    for p in arms.values():                  # warm-up: module load, smem opt-in
        for _ in range(3):
            p.step()
    torch.cuda.synchronize()
    ms = {k: [] for k in arms}
    for _ in range(reps):
        for k, p in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(launches):
                p.step()
            e1.record()
            torch.cuda.synchronize()
            ms[k].append(e0.elapsed_time(e1) / launches)
    return {k: float(np.median(v)) for k, v in ms.items()}, ms


def mismatches(g, f64, kernel):
    """One fresh step of `kernel` on a real*8 patch against the binary64 C checker: number of differing values."""
    outs = {n: f64[n].copy() for n in wrf.OUTPUT_FIELDS}
    with wrf.Patch(g, dtype=np.float64) as p:
        p.set_scalars(*SCALARS)
        p.set_kernel(kernel)
        p.upload(f64)
        p.step()
        p.download(outs)
        ran = p.last_kernel()
    want = dict(f64)
    for n in wrf.OUTPUT_FIELDS:
        want[n] = f64[n].copy()
    r8_checkers.oracle_c_r8(want, g, SCALARS, tiles=64)
    bad = sum(int(np.count_nonzero(outs[n].view(np.uint64) != want[n].view(np.uint64))) for n in wrf.OUTPUT_FIELDS)
    return bad, ran


def e2e_host_loop(g, f32, nsteps=6):
    """Wall time of nsteps host-pointer r8 calls under acoustic-loop residency, arrays page-locked up front."""
    keep, f = [], {}
    for n, a in f32.items():
        t = torch.empty(a.shape, dtype=torch.float64, pin_memory=True)
        t.numpy()[...] = a
        keep.append(t)
        f[n] = t.numpy()
    wrf.call_with_fields(f, g, *SCALARS)              # warm-up: mirrors, modules
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    with wrf.acoustic_loop():
        for _ in range(nsteps):
            wrf.call_with_fields(f, g, *SCALARS)      # returns after its outputs are in the host arrays
    dt = time.perf_counter() - t0
    wrf.lib().wrfb200_release_cache()
    return {"nsteps": nsteps, "total_ms": dt * 1e3, "ms_per_step": dt * 1e3 / nsteps, "pinned": True}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the summary JSON to this file")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--launches", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_r8: no CUDA device (this library has no CPU fallback)")
    torch.cuda.set_device(0)
    info = device_info()
    peak = copy_peak()
    print(json.dumps({"device": info, "copy_peak": peak}), flush=True)
    rows = []
    for nx, ny, nz in SIZES:
        g = wrf.Grid.from_shape(nx, ny, nz, halo=5)
        f32 = wrf.synth_fields(g)
        f64 = {n: a.astype(np.float64) for n, a in f32.items()}
        n3, n2 = g.updated_points()
        b8, b4 = 88 * n3 + 104 * n2, 44 * n3 + 52 * n2
        arms = {"r8_tile": patch(g, f64, np.float64, wrf.KERNEL_TILE),
                "r8_column": patch(g, f64, np.float64, wrf.KERNEL_COLUMN),
                "f32_auto": patch(g, f32, np.float32, wrf.KERNEL_AUTO)}
        med, samples = time_arms(arms, args.launches, args.reps)
        kern = {k: p.last_kernel() for k, p in arms.items()}
        for p in arms.values():
            p.close()
        row = {"size": f"{nx}x{ny}x{nz}", "N3": n3, "N2": n2,
               "working_set_vs_L2": round(b8 / L2_BYTES, 1), "launches": args.launches, "reps": args.reps}
        for k, ms in med.items():
            b = b4 if k == "f32_auto" else b8
            row[k] = {"ms": round(ms, 4), "Gpt_s": round(n3 / ms / 1e6, 2), "alg_bytes": b,
                      "GBps": round(b / ms / 1e6, 1), "frac_copy_peak": round(b / ms / 1e6 / peak["GBps"], 3),
                      "kernel_id": kern[k], "samples_ms": [round(x, 4) for x in samples[k]]}
        row["r8_auto_over_column"] = round(med["r8_column"] / med["r8_tile"], 2)
        for k, kernel in (("r8_tile", wrf.KERNEL_TILE), ("r8_column", wrf.KERNEL_COLUMN), ("r8_auto", wrf.KERNEL_AUTO)):
            bad, ran = mismatches(g, f64, kernel)
            row.setdefault("mismatches", {})[k] = bad
            if k == "r8_auto":
                row["r8_auto_kernel_id"] = ran
        if (nx, ny, nz) == SIZES[0]:
            row["e2e_host_loop_r8"] = e2e_host_loop(g, f32)
        del f32, f64
        rows.append(row)
        print(json.dumps(row), flush=True)
    summary = {"device": info, "copy_peak": peak, "sizes": rows,
               "all_mismatches_zero": all(v == 0 for r in rows for v in r["mismatches"].values())}
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(summary, fh, indent=1)
    print("mismatches: %d" % sum(v for r in rows for v in r["mismatches"].values()), flush=True)


if __name__ == "__main__":
    main()
