"""Time what periodic wrap costs the fused multi-GPU acoustic loop (launch with torchrun, one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \\
        tools/bench_wrap.py [--shape 1800x1060x50] [--pgrids 1x8,2x4] [--replays 20] [--rounds 5] [--out FILE]

Without torchrun it runs as one rank (1x1, where a wrapped rank is its own neighbour on every wrapped side).
For every process grid of --pgrids that has N ranks, one binary32 patch per wrap (none / x / y / xy) on a
periodic_x domain with specified = nested = 0, each connected with wrfb200_comm_set_wrap, its constants pushed and
its 6-step wrfb200_comm_loop captured and warmed up; then `rounds` rounds that each time the four wraps in turn,
`replays` graph replays apiece between CUDA events, the maximum over ranks.  The four are alternated in one run so
that drift of the shared machine falls on all of them alike.  Prints one JSON line (and writes it to FILE) with the
card name and power limit beside the median times.  Needs GPUs; there is no CPU fallback.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import wrf_model_cuda_sample_b200 as wrf  # noqa: E402
from wrf_model_cuda_sample_b200 import parallel  # noqa: E402
from tests import cases  # noqa: E402

NSMALL = 6                                       # acoustic steps per RK sub-step
WRAPS = {"none": (False, False), "x": (True, False), "y": (False, True), "xy": (True, True)}


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = r.stdout.strip().splitlines()[torch.cuda.current_device()] if r.returncode == 0 else ""
    return {"name": torch.cuda.get_device_name(), "nvidia_smi_name_power_limit": line.strip()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shape", default="1800x1060x50")
    ap.add_argument("--pgrids", default="1x8,2x4")
    ap.add_argument("--replays", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_wrap: no CUDA device")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    allgather = parallel.torch_allgather_bytes(device=dev) if world > 1 else (lambda blob: [blob])
    barrier = dist.barrier if world > 1 else (lambda: None)
    nx, ny, nz = (int(x) for x in args.shape.lower().split("x"))
    G = cases.grid(nx, ny, nz, halo=5, variant="periodic_open")
    whole = wrf.synth_fields(G, seed=99)
    stream = torch.cuda.Stream(device=dev)          # the patches' stream: the events below are recorded on it
    result = {"bench": "bench_wrap", "shape": args.shape, "steps_per_loop": NSMALL, "replays": args.replays,
              "rounds": args.rounds, "world": world, "card": card(), "grids": {}}
    pgrids = [tuple(int(v) for v in g.lower().split("x")) for g in args.pgrids.split(",")]
    if world == 1:
        pgrids = [(1, 1)]
    for px, py in pgrids:
        if px * py != world:
            continue
        patches = {}
        try:
            for name, (wx, wy) in WRAPS.items():
                decomp = parallel.Decomposition(G, px, py, halo=3, wrap_x=wx, wrap_y=wy)
                pg = decomp.patch_grid(rank)
                p = wrf.Patch(pg, device=local)
                patches[name] = p
                p.set_stream(stream.cuda_stream)
                p.set_scalars(*cases.SCALARS_3KM)
                p.upload(cases.carve_patch(whole, G, pg))
                parallel.connect_fused(p, decomp, rank, allgather)
                p.comm_push_constants()
                for _ in range(args.warmup):
                    p.comm_loop(NSMALL, graph=True)
                torch.cuda.synchronize()
                barrier()
            times = {name: [] for name in WRAPS}
            for _ in range(args.rounds):
                for name, p in patches.items():
                    barrier()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    for _ in range(args.replays):
                        p.comm_loop(NSMALL, graph=True)
                    e1.record(stream)
                    e1.synchronize()
                    ms = torch.tensor([e0.elapsed_time(e1) / args.replays], device=dev, dtype=torch.float64)
                    if world > 1:
                        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
                    times[name].append(ms.item())
            timeouts = sum(p.comm_status()[0] for p in patches.values())
            barrier()                                  # nobody unmaps a neighbour that is still storing into it
        finally:
            for p in patches.values():
                p.close()
        med = {name: statistics.median(v) for name, v in times.items()}
        result["grids"][f"{px}x{py}"] = {
            "loop_ms_median": med,
            "loop_ms_all": times,
            "wrap_cost_vs_none_pct": {n: 100.0 * (med[n] / med["none"] - 1.0) for n in WRAPS if n != "none"},
            "flag_timeouts_rank0": timeouts,
        }
    if rank == 0:
        line = json.dumps(result)
        print(line, flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as fh:
                fh.write(line + "\n")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
