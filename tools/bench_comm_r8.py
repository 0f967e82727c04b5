"""Time the fused multi-GPU acoustic loop on real*8 patches (launch with torchrun, one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \\
        tools/bench_comm_r8.py [--shape 1800x1060x50] [--replays 20] [--warmup 3] [--out FILE]

In one run:
  * the card name, its power limit and the host CPU count;
  * a parity pre-flight on a small grid (200x96x14, 1xN j-slabs, halos poisoned, 3 steps with the stand-in
    advance_uv): every rank compared bit for bit with the binary64 checker loop; the mismatch count is printed;
  * on the full grid in binary64, 1xN j-slabs: wrfb200_comm_push_constants, then the 6-step wrfb200_comm_loop_r8
    replayed from its CUDA graph, CUDA events over `replays` replays after `warmup`, the maximum over ranks;
  * on rank 0, two N = 1 references on the full grid, alternated: the single-GPU r8 tile kernel
    (wrfb200_step_graph(6), AUTO) and a 1x1 fused loop (the fused kernel with no neighbours), which isolates the
    cost of the coherent u / v loads and the flag logic.
The summary goes to FILE (default profiles/r5_comm_r8_n{N}.json).  Needs GPUs; there is no CPU fallback.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import wrf_model_cuda_sample_b200 as wrf  # noqa: E402
from wrf_model_cuda_sample_b200 import parallel  # noqa: E402
from tests import cases, r8_checkers  # noqa: E402

SCALARS = (1.0 / 3000.0, 1.0 / 3000.0, 3.0, 0.1)
NSMALL = 6                                       # acoustic steps per RK sub-step
C_UV = 0.25


def widen64(f):
    return {n: a.astype(np.float64) * (1.0 + 2.0 ** -40) for n, a in f.items() if isinstance(a, np.ndarray)}


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = r.stdout.strip().splitlines()[torch.cuda.current_device()] if r.returncode == 0 else ""
    return {"name": torch.cuda.get_device_name(), "nvidia_smi_name_power_limit": line.strip(),
            "host_cpus": os.cpu_count()}


def preflight(world, rank, dev, allgather):
    """Mismatching values of this rank's patch against the binary64 checker loop, plus flag time-outs."""
    G = cases.grid(200, 96, 14, halo=5, variant="specified")
    decomp = parallel.Decomposition(G, 1, world, halo=3)
    whole = widen64(wrf.synth_fields(G, seed=99))
    pg = decomp.patch_grid(rank)
    f = cases.carve_patch(whole, G, pg)
    cases.poison_neighbour_halos(f, decomp, rank, pg, (parallel.CONSTANT_HALOS, parallel.STEP_HALOS, parallel.OUTPUT_HALOS))
    with wrf.Patch(pg, device=dev.index, dtype=np.float64) as p:
        p.set_stream(torch.cuda.current_stream().cuda_stream)
        p.set_scalars(*SCALARS)
        p.upload(f)
        parallel.connect_fused(p, decomp, rank, allgather)
        p.comm_push_constants()
        p.comm_loop(3, standin=True, c=C_UV, graph=True)
        timeouts, _ = p.comm_status()
        p.download(f, names=cases.OUTPUTS + ("u", "v"))
        dist.barrier()                                   # nobody unmaps a neighbour that is still storing into it
    want = cases.copy_fields(whole)
    ubox, vbox = cases.standin_boxes(G, G.ids, G.ide, G.jds, G.jde)
    for s in range(3):
        r8_checkers.oracle_c_r8(want, G, SCALARS)
        if s < 2:
            cases.standin_advance_uv_numpy(want, G, C_UV, ubox, vbox)
    return sum(cases.patch_mismatches(f, want, G, pg, decomp.patch_extents(rank)).values()), timeouts


def time_replays(fn, replays, warmup, barrier):
    """CUDA-event ms per call of fn() over `replays` calls on the current stream, after `warmup` calls."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(replays):
        fn()
    e1.record()
    e1.synchronize()
    barrier()
    return e0.elapsed_time(e1) / replays


def references(G, dev, replays, warmup, rounds=5):
    """Rank 0 alone, on the full grid: the plain r8 tile kernel and the 1x1 fused loop, alternated `rounds` times."""
    fields = widen64(wrf.synth_fields(G, seed=99))
    stream = torch.cuda.current_stream().cuda_stream
    plain = wrf.Patch(G, device=dev.index, dtype=np.float64)
    fused = wrf.Patch(G, device=dev.index, dtype=np.float64)
    try:
        for p in (plain, fused):
            p.set_stream(stream)
            p.set_scalars(*SCALARS)
            p.upload(fields)
        fused.comm_connect([fused.comm_init(1, 1, 0, G.ids, G.ide, G.jds, G.jde)])
        fused.comm_push_constants()
        arms = {"plain_tile_step_graph6": lambda: plain.step_graph(NSMALL),
                "fused_1x1_comm_loop6": lambda: fused.comm_loop(NSMALL, standin=False, graph=True)}
        ms = {k: [] for k in arms}
        for _ in range(rounds):
            for k, fn in arms.items():
                ms[k].append(time_replays(fn, replays, warmup, lambda: None))
        plain_kernel = plain.last_kernel()
        timeouts, _ = fused.comm_status()
    finally:
        plain.close()
        fused.close()
    assert plain_kernel == wrf.KERNEL_TILE, plain_kernel
    return {k: {"median_ms": statistics.median(v), "all_ms": v} for k, v in ms.items()}, timeouts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shape", default="1800x1060x50")
    ap.add_argument("--replays", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # a stream of its own: on the legacy default stream (handle 0) the patches would create private streams that
    # the timing events recorded here do not follow
    torch.cuda.set_stream(torch.cuda.Stream(device=dev))
    dist.init_process_group("nccl", device_id=dev)
    allgather = parallel.torch_allgather_bytes(device=dev)
    barrier = dist.barrier

    info = card()
    mism, pre_timeouts = preflight(world, rank, dev, allgather)
    t = torch.tensor([mism, pre_timeouts], device=dev, dtype=torch.int64)
    dist.all_reduce(t)
    if rank == 0:
        print(f"bench_comm_r8: {info['nvidia_smi_name_power_limit']}, {info['host_cpus']} host CPUs; pre-flight 1x{world} "
              f"on 200x96x14 (binary64, poisoned halos): {int(t[0])} mismatches, {int(t[1])} flag time-outs", flush=True)

    nx, ny, nz = (int(x) for x in args.shape.lower().split("x"))
    G = cases.grid(nx, ny, nz, halo=5, variant="specified")
    refs, ref_timeouts = (references(G, dev, args.replays, args.warmup) if rank == 0 else (None, 0))
    barrier()

    decomp = parallel.Decomposition(G, 1, world, halo=5)
    pg = decomp.patch_grid(rank)
    f = widen64(wrf.synth_fields(pg, seed=99))          # counter-based: the same cells as the global field
    with wrf.Patch(pg, device=local, dtype=np.float64) as p:
        p.set_stream(torch.cuda.current_stream().cuda_stream)
        p.set_scalars(*SCALARS)
        p.upload(f)
        p.sync()
        parallel.connect_fused(p, decomp, rank, allgather)
        p.comm_push_constants()
        ms = time_replays(lambda: p.comm_loop(NSMALL, standin=False, graph=True), args.replays, args.warmup, barrier)
        timeouts, steps = p.comm_status()
        barrier()
    per_rank = [torch.zeros(2, dtype=torch.float64, device=dev) for _ in range(world)]
    dist.all_gather(per_rank, torch.tensor([ms, timeouts], dtype=torch.float64, device=dev))
    if rank == 0:
        ranks_ms = [float(x[0]) for x in per_rank]
        worst = max(ranks_ms)
        plain = refs["plain_tile_step_graph6"]["median_ms"]
        fused1 = refs["fused_1x1_comm_loop6"]["median_ms"]
        out = {
            "what": f"6-step wrfb200_comm_loop_r8 (CUDA graph replay) on {nx}x{ny}x{nz} binary64, 1x{world} j-slabs, "
                    f"max over ranks of CUDA-event ms per loop over {args.replays} replays after {args.warmup}",
            "card": info, "world": world, "pgrid": f"1x{world}", "shape": [nx, ny, nz],
            "preflight": {"grid": "200x96x14", "steps": 3, "mismatches": int(t[0]), "flag_timeouts": int(t[1])},
            "comm_loop_r8_ms_per_rank": ranks_ms, "comm_loop_r8_ms_max": worst,
            "flag_timeouts": int(sum(float(x[1]) for x in per_rank)) + ref_timeouts,
            "n1_references": refs,
            "fused_1x1_over_plain": fused1 / plain,
            "strong_scaling_efficiency_vs_plain": plain / (world * worst),
        }
        path = args.out or os.path.join(ROOT, "profiles", f"r5_comm_r8_n{world}.json")
        os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
        with open(path, "w") as fp:
            json.dump(out, fp, indent=1)
        print(json.dumps({k: out[k] for k in ("world", "comm_loop_r8_ms_max", "fused_1x1_over_plain",
                                              "strong_scaling_efficiency_vs_plain", "flag_timeouts")}), flush=True)
        print(f"plain r8 tile step_graph(6): {plain:.3f} ms; 1x1 fused loop: {fused1:.3f} ms; "
              f"1x{world} fused loop: {worst:.3f} ms -> {path}", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
