"""Command-line twin of the reference drivers (advance_mu_t_driver.{f90,c,cu}): read the reference-format
.bin inputs from argv[1], run advance_mu_t on the GPU through the C ABI, time it, and -- if argv[2] holds
``*_output.bin`` goldens -- print the reference's error report.  A case of 8-byte reals (a dump of WRF built with
-r8) runs the real*8 operator, writes 8-byte outputs and is reported with the binary64 metrics.

    python -m wrf_model_cuda_sample_b200.cli INPUT_DIR [GOLDEN_DIR] [--write OUT_DIR] [--steps N]
"""
from __future__ import annotations

import argparse
import sys
import time

from . import binio
from .advance_mu_t import call_with_fields


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("input_dir")
    ap.add_argument("golden_dir", nargs="?")
    ap.add_argument("--write", metavar="OUT_DIR", help="write the outputs as <name>_output.bin")
    ap.add_argument("--steps", type=int, default=1)
    args = ap.parse_args(argv)

    g, scalars, fields = binio.read_case(args.input_dir)
    t0 = time.perf_counter()
    call_with_fields(fields, g, *scalars, nsteps=args.steps)          # host arrays: upload, step(s), download, sync
    ms = 1e3 * (time.perf_counter() - t0)
    n3, _ = g.updated_points()
    print(f"advance_mu_t GPU time (incl. H2D/D2H) is\t{ms:.3f} ms\t({n3} points, {args.steps} step(s))")
    if args.write:
        binio.write_case(args.write, g, scalars, fields, suffix="_output", names=binio.GOLDEN)
    worst = 0
    if args.golden_dir:
        for name, r in binio.compare_with_golden(g, fields, args.golden_dir).items():
            print(f"\n# of equal values: {r['n_equal']}, # of non-equal values: {r['n_different']}")
            print(f"max relative error: {r['max_rel']:e}\tmax absolute error: {r['max_abs']:e}\t{binio.FILE_OF[name]}_output.bin")
            print(f"max ulp = {r['max_ulp']}\t\t\t\trmse = {r['rmse']:e}")
            worst = max(worst, r["max_ulp"])
        print(f"\nworst max-ulp over all fields: {worst}")
    return 0 if worst <= 2 else 1


if __name__ == "__main__":
    sys.exit(main())
