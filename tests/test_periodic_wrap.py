"""Periodic lateral boundaries in the multi-GPU path: the halo exchange wraps across the domain edge
(wrfb200_comm_set_wrap, Decomposition(wrap_x=, wrap_y=)).

The reference is a PERIODIC ORACLE LOOP: the single-domain oracle with exactly the copies WRF makes to refresh the
ring of a periodic domain, and which the exchange performs (WRAP_COPIES).  It is checked on its own first: a periodic
loop is translation-equivariant, so rolling the inputs by s cells rolls every output by s bit for bit -- which holds
only if no cell the routine reads past the domain edge is missing from the table.  Then the decomposed runs must equal
it bit for bit: over gloo with the oracle as each rank's compute (CPU), and through the fused exchange of csrc/comm.cu
with ranks as handles of one process on device 0 (GPU), halos and the wrapped column ide / row jde poisoned."""
import os
import tempfile

import numpy as np
import pytest

import wrf_model_cuda_sample_b200 as wrf
from wrf_model_cuda_sample_b200 import EAST, NORTH, SOUTH, WEST, parallel
from tests import cases
from tests.test_parallel_gloo import NumpyPatchHalo, _free_port

C_UV = 0.25
WRAPS = {"x": (True, False), "y": (False, True), "xy": (True, True)}

# (when, axis, direction, fields): "fwd" f[ide] <- f[ids] (the staggered end takes the first column),
# "back" f[ids-1] <- f[ide-1]; the same with jds / jde in j.  Over the rows (columns) that are pushed: jds..jde, or
# jds..jde-1 when j wraps too (ids..ide / ids..ide-1 for the j copies).
WRAP_COPIES = (
    ("once", "x", "fwd", ("u_1", "muu", "msfuy", "t_1")),
    ("once", "x", "back", ("t_1",)),
    ("once", "y", "fwd", ("v_1", "muv", "msfvx_inv", "t_1")),
    ("once", "y", "back", ("t_1",)),
    ("before", "x", "fwd", ("u",)),
    ("before", "y", "fwd", ("v",)),
    ("after", "x", "back", ("mu", "muts", "mudf")),
    ("after", "y", "back", ("mu", "muts", "mudf")),
)


def wrap_copy(f, G, when, wrap_x, wrap_y):
    for w, axis, direction, names in WRAP_COPIES:
        if w != when or not (wrap_x if axis == "x" else wrap_y):
            continue
        for n in names:
            a = f[n]
            if axis == "x":
                J = slice(G.jds - G.jms, (G.jde - 1 if wrap_y else G.jde) - G.jms + 1)
                dst, src = (G.ide, G.ids) if direction == "fwd" else (G.ids - 1, G.ide - 1)
                a[J, ..., dst - G.ims] = a[J, ..., src - G.ims]
            else:
                I = slice(G.ids - G.ims, (G.ide - 1 if wrap_x else G.ide) - G.ims + 1)
                dst, src = (G.jde, G.jds) if direction == "fwd" else (G.jds - 1, G.jde - 1)
                a[dst - G.jms, ..., I] = a[src - G.jms, ..., I]


def periodic_standin_boxes(G, ext, wrap_x, wrap_y):
    """cases.standin_boxes, but u from i_start (v from j_start) on a wrapped axis: mudf at i-1 is the ring."""
    ips, ipe, jps, jpe = ext
    (ui0, ui1, uj0, uj1), (vi0, vi1, vj0, vj1) = cases.standin_boxes(G, ips, ipe, jps, jpe)
    gi0, _, gj0, _, _, _ = G.with_tile(G.ids, G.ide, G.jds, G.jde).bounds()
    if wrap_x:
        ui0 = max(ips, gi0)
    if wrap_y:
        vj0 = max(jps, gj0)
    return (ui0, ui1, uj0, uj1), (vi0, vi1, vj0, vj1)


def periodic_oracle_loop(G, fin, scalars, nsteps, wrap_x, wrap_y, c=None, step=None):
    """nsteps of the oracle on the whole domain with the ring refreshed as the wrapped exchange refreshes it."""
    from oracle import loader
    step = step or loader.oracle_c
    f = cases.copy_fields(fin)
    ubox, vbox = periodic_standin_boxes(G, (G.ids, G.ide, G.jds, G.jde), wrap_x, wrap_y)
    wrap_copy(f, G, "once", wrap_x, wrap_y)
    for s in range(nsteps):
        wrap_copy(f, G, "before", wrap_x, wrap_y)
        step(f, G, scalars)
        wrap_copy(f, G, "after", wrap_x, wrap_y)
        if c is not None and s + 1 < nsteps:
            cases.standin_advance_uv_numpy(f, G, c, ubox, vbox)
    return f


def poison_wrapped_halos(f, decomp, rank, pg, halo_sets):
    """cases.poison_neighbour_halos over the exchange extents: on a wrapped edge column ide / row jde is halo too."""
    ips, ipe, jps, jpe = decomp.exchange_extents(rank)
    for halos in halo_sets:
        for field, sides in halos:
            a = f[field]
            for side in sides:
                if decomp.neighbour(rank, side) is None:
                    continue
                if side == EAST: a[..., ipe + 1 - pg.ims:] = cases.POISON
                if side == WEST: a[..., :ips - pg.ims] = cases.POISON
                if side == NORTH: a[jpe + 1 - pg.jms:] = cases.POISON
                if side == SOUTH: a[:jps - pg.jms] = cases.POISON


ALL_HALOS = (parallel.CONSTANT_HALOS, parallel.STEP_HALOS, parallel.OUTPUT_HALOS)


# ------------------------------------------------------------------------------------------------ CPU
def _roll(f, G, axis, s):
    """Roll every field's periodic cells (ids..ide-1 or jds..jde-1) by s; the ring is left for the copies to fill."""
    out = cases.copy_fields(f)
    for n in wrf.FIELDS_3D + wrf.FIELDS_2D:
        a = out[n]
        if axis == "x":
            P = slice(G.ids - G.ims, G.ide - G.ims)
            a[..., P] = np.roll(a[..., P], s, axis=-1)
        else:
            P = slice(G.jds - G.jms, G.jde - G.jms)
            a[P] = np.roll(a[P], s, axis=0)
    return out


@pytest.mark.parametrize("variant,wrap,axis", [("periodic_open", "x", "x"), ("periodic_open", "y", "y"),
                                               ("periodic_open", "xy", "x"), ("periodic_open", "xy", "y"),
                                               ("periodic_specified", "x", "x"), ("open", "y", "y")])
def test_periodic_oracle_is_translation_equivariant(variant, wrap, axis):
    G = cases.grid(29, 23, 7, halo=3, variant=variant)
    wrap_x, wrap_y = WRAPS[wrap]
    fin = cases.random_fields(G, seed=5)
    s = 5
    base = periodic_oracle_loop(G, fin, cases.SCALARS_3KM, 3, wrap_x, wrap_y, c=C_UV)
    moved = periodic_oracle_loop(G, _roll(fin, G, axis, s), cases.SCALARS_3KM, 3, wrap_x, wrap_y, c=C_UV)
    want = _roll(base, G, axis, s)
    i1 = G.ide - 1 if axis == "x" else G.ide           # compare the periodic cells of the rolled axis
    j1 = G.jde - 1 if axis == "y" else G.jde
    J = slice(G.jds - G.jms, j1 - G.jms + 1); I = slice(G.ids - G.ims, i1 - G.ims + 1)
    for n in cases.OUTPUTS + ("u", "v"):
        assert np.array_equal(cases.bits(moved[n][J, ..., I]), cases.bits(want[n][J, ..., I])), \
            f"{variant} wrap {wrap}, roll in {axis}: {n} is not rolled with the inputs"
    # and the roll is not vacuous: the outputs did change
    assert not np.array_equal(cases.bits(moved["mu"][J, I]), cases.bits(base["mu"][J, I]))


def test_decomposition_wrap_geometry():
    G = cases.grid(1800, 1060, 50, variant="periodic_open")
    d = parallel.Decomposition(G, 1, 8, halo=5, wrap_x=True)
    for r in range(8):
        assert d.neighbour(r, WEST) == r and d.neighbour(r, EAST) == r          # j-slabs: own east / west neighbour
        ips, ipe, jps, jpe = d.exchange_extents(r)
        assert (ips, ipe) == (1, 1799) and (jps, jpe) == d.patch_extents(r)[2:]
    assert d.neighbour(0, SOUTH) is None and d.neighbour(7, NORTH) is None
    d = parallel.Decomposition(G, 2, 4, halo=5, wrap_x=True, wrap_y=True)
    assert d.neighbour(0, WEST) == 1 and d.neighbour(0, EAST) == 1              # doubled east / west neighbour
    assert d.neighbour(0, SOUTH) == 6 and d.neighbour(6, NORTH) == 0
    assert d.exchange_extents(7) == (901, 1799, 796, 1059)
    assert d.exchange_extents(0) == d.patch_extents(0)
    d = parallel.Decomposition(G, 1, 1, wrap_x=True, wrap_y=True)
    assert all(d.neighbour(0, s) == 0 for s in (WEST, EAST, SOUTH, NORTH))
    assert parallel.Decomposition(G, 3, 1).neighbour(0, WEST) is None          # wrap stays opt-in


@pytest.mark.parametrize("px,py", [(1, 1), (2, 1), (1, 2), (2, 2), (3, 1), (2, 4)])
def test_wrapped_exchange_plans_match(px, py):
    """Every receive has exactly one matching send on the peer, in the same order -- self and doubled peers too."""
    G = cases.grid(400, 300, 6, variant="periodic_open")
    d = parallel.Decomposition(G, px, py, wrap_x=True, wrap_y=True)
    for halos in ALL_HALOS:
        plans = {r: parallel.HaloExchanger(d, r, None, None, None).plan(halos) for r in range(d.world)}
        for r, plan in plans.items():
            for peer in range(d.world):
                mine = [(f, s) for kind, f, s, p in plan if kind == "recv" and p == peer]
                theirs = [(f, parallel.OPPOSITE[s]) for kind, f, s, p in plans[peer] if kind == "send" and p == r]
                assert mine == theirs


def _gloo_worker(rank, world, px, py, wrap, port, outdir, shape, variant):
    import torch.distributed as dist
    from oracle import loader
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        wrap_x, wrap_y = WRAPS[wrap]
        G = cases.grid(*shape, halo=5, variant=variant)
        decomp = parallel.Decomposition(G, px, py, halo=2, wrap_x=wrap_x, wrap_y=wrap_y)
        pg, ext = decomp.patch_grid(rank), decomp.exchange_extents(rank)
        f = cases.carve_patch(wrf.synth_fields(G, seed=77), G, pg)
        halo = NumpyPatchHalo(f, pg, ext)
        ex = parallel.HaloExchanger(decomp, rank, halo.pack, halo.recv_buffer, halo.unpack)
        poison_wrapped_halos(f, decomp, rank, pg, ALL_HALOS)
        ex.exchange(parallel.CONSTANT_HALOS)
        ubox, vbox = periodic_standin_boxes(G, ext, wrap_x, wrap_y)
        for s in range(3):
            ex.exchange(parallel.STEP_HALOS)
            loader.oracle_c(f, pg, cases.SCALARS_3KM)
            ex.exchange(parallel.OUTPUT_HALOS)
            if s + 1 < 3:
                cases.standin_advance_uv_numpy(f, pg, C_UV, ubox, vbox)
        ips, ipe, jps, jpe = ext
        Jp = slice(jps - pg.jms, jpe - pg.jms + 1); Ip = slice(ips - pg.ims, ipe - pg.ims + 1)
        out = {n: f[n][Jp, ..., Ip] for n in cases.OUTPUTS + ("u", "v")}
        np.savez(os.path.join(outdir, f"rank{rank}.npz"), ext=np.array(ext), **out)
        dist.barrier()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("px,py,wrap,variant", [(1, 2, "x", "periodic_specified"), (2, 1, "y", "open"),
                                                 (2, 2, "xy", "periodic_open"), (1, 4, "xy", "periodic_open")])
def test_gloo_wrapped_loop_equals_periodic_oracle(px, py, wrap, variant):
    import torch.multiprocessing as mp
    shape = (61, 43, 9)
    world = px * py
    with tempfile.TemporaryDirectory() as outdir:
        mp.spawn(_gloo_worker, args=(world, px, py, wrap, _free_port(), outdir, shape, variant), nprocs=world,
                 join=True)
        G = cases.grid(*shape, halo=5, variant=variant)
        want = periodic_oracle_loop(G, wrf.synth_fields(G, seed=77), cases.SCALARS_3KM, 3, *WRAPS[wrap], c=C_UV)
        for r in range(world):
            z = np.load(os.path.join(outdir, f"rank{r}.npz"))
            ips, ipe, jps, jpe = (int(x) for x in z["ext"])
            J = slice(jps - G.jms, jpe - G.jms + 1); I = slice(ips - G.ims, ipe - G.ims + 1)
            for n in cases.OUTPUTS + ("u", "v"):
                assert np.array_equal(cases.bits(z[n]), cases.bits(want[n][J, ..., I])), f"rank {r} field {n} differs"


# ------------------------------------------------------------------------------------------------ GPU
SCALARS_R8 = (1.0 / 3000.0, 1.0 / 3000.0, 3.0, 0.1)


def run_wrapped_ranks(G, px, py, wrap, nsteps, graph=True, stepwise=False, standin=True, repeats=1, r8=False,
                      seed=99, halo=3):
    """Ranks as handles of one process on device 0 (as tests/test_fused_comm.py), exchange wrapped."""
    wrap_x, wrap_y = WRAPS[wrap]
    decomp = parallel.Decomposition(G, px, py, halo=halo, wrap_x=wrap_x, wrap_y=wrap_y)
    whole = wrf.synth_fields(G, seed=seed)
    if r8:
        whole = {n: a.astype(np.float64) * (1.0 + 2.0 ** -40) for n, a in whole.items()}
    ranks = []
    try:
        for r in range(px * py):
            pg = decomp.patch_grid(r)
            f = cases.carve_patch(whole, G, pg)
            poison_wrapped_halos(f, decomp, r, pg, ALL_HALOS)
            p = wrf.Patch(pg, device=0, dtype=np.float64 if r8 else np.float32)
            ranks.append((p, pg, f))
            p.set_scalars(*(SCALARS_R8 if r8 else cases.SCALARS_3KM))
            p.upload(f)
        infos = []
        for r, (p, _, _) in enumerate(ranks):
            p.comm_set_wrap(wrap_x, wrap_y)
            infos.append(p.comm_init(px, py, r, *decomp.patch_extents(r)))
        for p, _, _ in ranks:
            p.comm_connect(infos)
        for p, _, _ in ranks:
            p.comm_push_constants()
        for _ in range(repeats):
            if stepwise:
                for s in range(nsteps):
                    for p, _, _ in ranks:
                        p.comm_push_uv()
                        p.comm_step()
                        if standin and s + 1 < nsteps:
                            p.comm_standin_advance_uv(C_UV)
            else:
                for p, _, _ in ranks:
                    p.comm_loop(nsteps, standin=standin, c=C_UV, graph=graph)
        for r, (p, pg, f) in enumerate(ranks):
            timeouts, steps = p.comm_status()
            assert timeouts == 0, f"rank {r}: {timeouts} halo waits timed out"
            assert steps == nsteps * repeats
            p.download(f, names=cases.OUTPUTS + ("u", "v"))
    finally:
        for p, _, _ in ranks:
            p.close()
    return decomp, whole, ranks


def _check(decomp, want, G, ranks, what, names=cases.OUTPUTS + ("u", "v")):
    for r, (_, pg, f) in enumerate(ranks):
        bad = cases.patch_mismatches(f, want, G, pg, decomp.exchange_extents(r), names=names)
        assert not bad, f"{what} rank {r}: {bad}"


WRAP_CASES = [("periodic_open", "x"), ("periodic_open", "y"), ("periodic_open", "xy"), ("periodic_specified", "x")]


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("variant,wrap", WRAP_CASES)
@pytest.mark.parametrize("px,py", [(1, 1), (1, 2), (2, 1), (2, 2), (1, 4), (3, 1)])
def test_fused_wrapped_exchange_matches_periodic_oracle(px, py, variant, wrap, graph):
    G = cases.grid(390, 120, 12, halo=5, variant=variant)
    decomp, whole, ranks = run_wrapped_ranks(G, px, py, wrap, 4, graph=graph)
    want = periodic_oracle_loop(G, whole, cases.SCALARS_3KM, 4, *WRAPS[wrap], c=C_UV)
    _check(decomp, want, G, ranks, f"{px}x{py} {variant} wrap {wrap}")


@pytest.mark.gpu
@pytest.mark.parametrize("stepwise", [False, True])
@pytest.mark.parametrize("px,py", [(1, 2), (2, 2), (1, 1)])
def test_fused_wrapped_exchange_r8(px, py, stepwise):
    from tests import r8_checkers
    G = cases.grid(280, 96, 12, halo=4, variant="periodic_open")
    decomp, whole, ranks = run_wrapped_ranks(G, px, py, "xy", 3, stepwise=stepwise, r8=True, seed=7)
    want = periodic_oracle_loop(G, whole, SCALARS_R8, 3, True, True, c=C_UV,
                                step=lambda f, g, s: r8_checkers.oracle_c_r8(f, g, s, tiles=32))
    _check(decomp, want, G, ranks, f"real*8 {px}x{py}")


@pytest.mark.gpu
def test_fused_wrapped_replays_keep_epochs_consistent():
    G = cases.grid(260, 64, 10, halo=5, variant="periodic_open")
    decomp, whole, ranks = run_wrapped_ranks(G, 2, 2, "xy", 3, standin=False, repeats=5)
    want = periodic_oracle_loop(G, whole, cases.SCALARS_3KM, 15, True, True)
    _check(decomp, want, G, ranks, "5 replays", names=cases.OUTPUTS)


@pytest.mark.gpu
def test_wrap_argument_errors():
    with wrf.Patch(cases.grid(64, 32, 6, halo=2, variant="specified"), device=0) as p:
        p.comm_set_wrap(True, False)
        with pytest.raises(wrf.WrfB200Error, match="periodic_x"):
            p.comm_init(1, 1, 0, 1, 64, 1, 32)
    with wrf.Patch(cases.grid(64, 32, 6, halo=2, variant="periodic_specified"), device=0) as p:
        p.comm_set_wrap(False, True)
        with pytest.raises(wrf.WrfB200Error, match="specified"):
            p.comm_init(1, 1, 0, 1, 64, 1, 32)
    G = cases.grid(300, 64, 6, halo=2, variant="periodic_open")
    d = parallel.Decomposition(G, 1, 2, halo=2)
    with wrf.Patch(d.patch_grid(0), device=0) as a, wrf.Patch(d.patch_grid(1), device=0) as b:
        a.comm_set_wrap(True, False)                                  # rank 1 keeps the default: no wrap
        infos = [a.comm_init(1, 2, 0, *d.patch_extents(0)), b.comm_init(1, 2, 1, *d.patch_extents(1))]
        with pytest.raises(wrf.WrfB200Error, match="wrap"):
            a.comm_connect(infos)
        with pytest.raises(wrf.WrfB200Error, match="wrap"):
            b.comm_connect(infos)
