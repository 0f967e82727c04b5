"""Multi-GPU parity check (launch with torchrun, one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        tools/multi_gpu_check.py [--pgrid PXxPY] [--shape NXxNYxNZ] [--steps S] [--mode fused|nccl]
        [--dtype float32|float64] [--wrap none|x|y|xy]

Every rank runs the CUDA path on its patch (tile = patch, domain = global) and applies the advance_uv stand-in
between steps.  --mode fused (default): the one-cell ring moves by peer-mapped stores fused into the kernels
(csrc/comm.cu; torch.distributed only all-gathers the bootstrap blobs).  --mode nccl: pack / NCCL send-recv /
unpack through HaloExchanger, overlapped with the interior tile (the round-1 path).  Each rank then checks its
patch BIT FOR BIT against the single-domain oracle loop.  --dtype float64: real*8 patches on float64 inputs with
full 53-bit mantissas (fused: wrfb200_comm_init_r8 / wrfb200_comm_loop_r8; nccl: wrfb200_pack_halo_r8 /
_unpack_halo_r8 around float64 NCCL send-recv), checked against the binary64 checker loop (tests/r8_checkers.py).
--wrap x|y|xy: the exchange wraps across the domain edge (Decomposition(wrap_x=, wrap_y=); the --variant must allow
it, e.g. periodic_open), and the reference is the periodic oracle loop of tests/test_periodic_wrap.py.
Exit code 0 = every rank identical.
"""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import wrf_model_cuda_sample_b200 as wrf  # noqa: E402
from wrf_model_cuda_sample_b200 import parallel  # noqa: E402
from tests import cases, r8_checkers  # noqa: E402
from tests.test_periodic_wrap import periodic_oracle_loop, periodic_standin_boxes, poison_wrapped_halos  # noqa: E402

SCALARS_3KM_R8 = (1.0 / 3000.0, 1.0 / 3000.0, 3.0, 0.1)


def widen64(f):
    """float32 fields -> float64 with low mantissa bits a float cannot hold (x * (1 + 2^-40), one rounding)."""
    return {n: a.astype(np.float64) * (1.0 + 2.0 ** -40) for n, a in f.items() if isinstance(a, np.ndarray)}


def checker_loop64(G, whole, scalars, nsteps, c):
    """The binary64 checker over the whole domain, with the stand-in advance_uv between steps."""
    f = cases.copy_fields(whole)
    ubox, vbox = cases.standin_boxes(G, G.ids, G.ide, G.jds, G.jde)
    for s in range(nsteps):
        r8_checkers.oracle_c_r8(f, G, scalars, tiles=64)
        if s + 1 < nsteps:
            cases.standin_advance_uv_numpy(f, G, c, ubox, vbox)
    return f


def run_fused(patch, decomp, rank, dev, steps, c_uv, graph):
    parallel.connect_fused(patch, decomp, rank, parallel.torch_allgather_bytes(device=dev))
    patch.comm_push_constants()
    patch.comm_loop(steps, standin=True, c=c_uv, graph=graph)
    timeouts, steps_done = patch.comm_status()
    assert steps_done == steps, (steps_done, steps)
    return timeouts


def run_nccl(patch, decomp, rank, dev, pg, ext, G, steps, c_uv, main_stream, wrap_x=False, wrap_y=False):
    comm = torch.cuda.Stream(device=dev)
    halo = parallel.GpuPatchHalo(patch, decomp, rank, dev)
    ex = parallel.HaloExchanger(decomp, rank, halo.pack, halo.recv_buffer, halo.unpack)
    ex.exchange(parallel.CONSTANT_HALOS)
    interior, strips = decomp.interior_and_boundary_tiles(rank)
    ubox, vbox = periodic_standin_boxes(G, ext, wrap_x, wrap_y)
    for s in range(steps):
        comm.wait_stream(main_stream)
        with torch.cuda.stream(comm):
            patch.set_stream(comm.cuda_stream)
            ex.finish(ex.start(parallel.STEP_HALOS))
            for t in strips:                     # halo-dependent strips right behind the unpack, same stream
                patch.step(pg.with_tile(*t))
        patch.set_stream(main_stream.cuda_stream)
        if interior:
            patch.step(pg.with_tile(*interior))  # concurrent with exchange + strips
        main_stream.wait_stream(comm)
        ex.exchange(parallel.OUTPUT_HALOS)
        if s + 1 < steps:
            patch.standin_advance_uv("u", c_uv, *ubox)
            patch.standin_advance_uv("v", c_uv, *vbox)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pgrid", default="")
    ap.add_argument("--shape", default="300x160x20")
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--variant", default="specified")
    ap.add_argument("--mode", choices=("fused", "nccl"), default="fused")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--dtype", choices=("float32", "float64"), default="float32")
    ap.add_argument("--wrap", choices=("none", "x", "y", "xy"), default="none")
    args = ap.parse_args()
    r8 = args.dtype == "float64"
    wrap_x, wrap_y = "x" in args.wrap, "y" in args.wrap
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    nx, ny, nz = (int(x) for x in args.shape.lower().split("x"))
    G = cases.grid(nx, ny, nz, halo=5, variant=args.variant)
    px, py = (int(x) for x in args.pgrid.lower().split("x")) if args.pgrid else parallel.choose_process_grid(world, nx, ny)
    assert px * py == world
    decomp = parallel.Decomposition(G, px, py, halo=3, wrap_x=wrap_x, wrap_y=wrap_y)
    pg, ext = decomp.patch_grid(rank), decomp.exchange_extents(rank)
    c_uv = 0.25

    whole = wrf.synth_fields(G, seed=99)
    if r8:
        whole = widen64(whole)
    scalars = SCALARS_3KM_R8 if r8 else cases.SCALARS_3KM
    f = cases.carve_patch(whole, G, pg)
    # poison every halo that a neighbour must fill, so a missing exchange cannot go unnoticed
    poison_wrapped_halos(f, decomp, rank, pg, (parallel.CONSTANT_HALOS, parallel.STEP_HALOS, parallel.OUTPUT_HALOS))

    main_stream = torch.cuda.current_stream()
    with wrf.Patch(pg, device=local, dtype=np.float64 if r8 else np.float32) as patch:
        patch.set_stream(main_stream.cuda_stream)
        patch.set_scalars(*scalars)
        patch.upload(f)
        if args.mode == "fused":
            timeouts = run_fused(patch, decomp, rank, dev, args.steps, c_uv, not args.no_graph)
        else:
            timeouts = run_nccl(patch, decomp, rank, dev, pg, ext, G, args.steps, c_uv, main_stream, wrap_x, wrap_y)
        patch.download(f, names=cases.OUTPUTS + ("u", "v"))
        dist.barrier()                               # nobody unmaps a neighbour that is still storing into it

    if wrap_x or wrap_y:
        step = (lambda f_, g_, s_: r8_checkers.oracle_c_r8(f_, g_, s_, tiles=64)) if r8 else None
        want = periodic_oracle_loop(G, whole, scalars, args.steps, wrap_x, wrap_y, c=c_uv, step=step)
    elif r8:
        want = checker_loop64(G, whole, scalars, args.steps, c_uv)
    else:
        want = cases.oracle_loop(G, whole, cases.SCALARS_3KM, args.steps, c=c_uv)
    mism = cases.patch_mismatches(f, want, G, pg, ext)
    for n, nb in mism.items():
        print(f"rank {rank}: field {n}: {nb} values differ", flush=True)
    if timeouts:
        print(f"rank {rank}: {timeouts} halo waits timed out", flush=True)
    bad = sum(mism.values()) + timeouts
    t = torch.tensor([bad], device=dev, dtype=torch.int64)
    dist.all_reduce(t)
    if rank == 0:
        ref = "binary64 checker" if r8 else "oracle"
        mode = f"{args.mode}, float64" if r8 else args.mode
        mode += "" if args.wrap == "none" else f", wrap {args.wrap}"
        print(f"multi_gpu_check [{mode}] {px}x{py} on {nx}x{ny}x{nz}, {args.steps} steps: "
              f"{f'BIT-IDENTICAL to the single-domain {ref}' if t.item() == 0 else str(t.item()) + ' MISMATCHES'}", flush=True)
    dist.destroy_process_group()
    sys.exit(0 if t.item() == 0 else 1)


if __name__ == "__main__":
    main()
