"""A/B two builds of the library on one GPU: alternate bench.py runs of each and print, per workload, the median
and range of avg_launch_ms (one advance_mu_t pass over the grid) and the ratio of the medians.

    python tools/ab_bench.py --a wrf_model_cuda_sample_b200/libwrfb200_parent.so --b wrf_model_cuda_sample_b200/libwrfb200.so \
        --reps 4 -- --no-e2e --no-cpu --no-ref-cuda --steps 50

Arguments after `--` go to every bench.py run unchanged; the library of a run is chosen with WRFB200_LIB.  The runs
alternate A, B, A, B, ... so that a drift of the machine's state hits both builds alike.  Ranges of the two builds
that do not overlap are flagged.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def launch_times(line):
    """workload -> avg_launch_ms of one bench.py JSON line (the headline workload and the `workloads` extras)."""
    out = {line["config"]["workload"].split(":")[0]: line["roofline"]["avg_launch_ms"]}
    for name, w in (line.get("workloads") or {}).items():
        if "avg_launch_ms" in w:
            out[name] = w["avg_launch_ms"]
    return out


def run(lib, bench_args):
    env = dict(os.environ, WRFB200_LIB=os.path.abspath(lib))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + bench_args, env=env,
                       capture_output=True, text=True)
    for l in reversed(r.stdout.splitlines()):
        if l.startswith("{"):
            return json.loads(l)
    raise RuntimeError(f"bench.py with {lib}: no JSON line (exit {r.returncode}): {r.stderr[-500:]}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--a", required=True, help="library A (baseline)")
    ap.add_argument("--b", required=True, help="library B (candidate)")
    ap.add_argument("--reps", type=int, default=4)
    ap.add_argument("bench_args", nargs=argparse.REMAINDER)
    args = ap.parse_args()
    bench_args = [a for a in args.bench_args if a != "--"]
    times = {"A": {}, "B": {}}
    for rep in range(args.reps):
        for tag, lib in (("A", args.a), ("B", args.b)):
            t = launch_times(run(lib, bench_args))
            for w, ms in t.items():
                times[tag].setdefault(w, []).append(ms)
            print(f"rep {rep} {tag}: " + "  ".join(f"{w} {ms:.4f}" for w, ms in t.items()), flush=True)
    print(f"A = {args.a}\nB = {args.b}\nbench.py {' '.join(bench_args)}; {args.reps} runs each, avg_launch_ms")
    for w in times["A"]:
        a, b = times["A"][w], times["B"].get(w, [])
        if not b:
            continue
        ma, mb = statistics.median(a), statistics.median(b)
        apart = max(b) < min(a) or max(a) < min(b)
        print(f"{w:10s} A {ma:.4f} [{min(a):.4f}, {max(a):.4f}]  B {mb:.4f} [{min(b):.4f}, {max(b):.4f}]  "
              f"B/A {mb / ma:.4f}{'  (ranges apart)' if apart else ''}")


if __name__ == "__main__":
    main()
