"""The level-count ladder: every kernel configuration the level count nk can select, run on the GPU against the oracle.

Each kernel keeps all nk levels of its columns in shared memory, so nk picks the template instance and launch shape
that run (DESIGN.md section 4, "Level ladder and limits").  The pipe kernel's ladder is not written down here: it is
read from the host-only launch plan (wrfb200_pipe_plan) at import, and both ends of every configuration it finds are
tested, plus the first level count the plan refuses.  A later change to the ladder keeps this file covering every
configuration.  Bar: every output BIT-IDENTICAL to the oracle (binary32) or the binary64 checker (real*8)."""
import functools

import numpy as np
import pytest

import wrf_model_cuda_sample_b200 as wrf
from wrf_model_cuda_sample_b200 import parallel
from wrf_model_cuda_sample_b200._lib import ERR_UNSUPPORTED
from oracle import loader
from tests import cases
from tests.test_fused_comm import run_ranks, C_UV
from tests.test_launch_plan import plan_rc, SMEM_SM, SMEM_RESERVE
from tests.test_r8 import assert_bit_equal64, assert_outside_untouched64, oracle64, random_fields64

pytestmark = pytest.mark.gpu

SCALARS = cases.SCALARS_3KM
ROWS = 23                                   # computed rows of the ladder grids: odd, so TJ=2 leaves a half-filled tile
MAX_NK_SCAN = 460
PIPE, TILE, COLUMN, AUTO = wrf.KERNEL_PIPE, wrf.KERNEL_TILE, wrf.KERNEL_COLUMN, wrf.KERNEL_AUTO
TILE_MAX, COLUMN_MAX, TILE_R8_MAX, COLUMN_R8_MAX = 223, 454, 220, 227


def _sm_count():
    """SMs of device 0, as the launcher's resident_slots reads them.  Without a device (collection on a CPU-only
    machine, where the tests of this file are deselected) the B200's 148 keeps the module importable."""
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count if torch.cuda.is_available() else 148


SMS = _sm_count()
SLOTS = 2 * SMS                             # two resident blocks per SM


def ladder_grid(nx, nk, variant="specified", rows=ROWS):
    ny = rows + (3 if variant == "specified" else 1)            # specified computes rows 2 .. ny-2, periodic_open 1 .. ny-1
    return cases.grid(nx, ny, nk + 1, halo=5, variant=variant)


def blocks_per_sm(pl):
    return SMEM_SM // (pl["smem"] + SMEM_RESERVE)


def config(pl):
    """A configuration's name: the plan's cfg, and 'last' for the one-block last-resort form of cfg 12."""
    return f"{pl['cfg']}" + ("last" if pl["cfg"] == 12 and blocks_per_sm(pl) == 1 else "")


def scan_ladder():
    """{configuration: (smallest nk, largest nk)} over nk = 1 .. MAX_NK_SCAN, and the first nk the plan refuses."""
    ends, refused = {}, None
    for nk in range(1, MAX_NK_SCAN + 1):
        rc, pl = plan_rc(ladder_grid(270, nk), SLOTS)
        if rc != 0:
            assert rc == ERR_UNSUPPORTED, (nk, rc)
            refused = refused or nk
            continue
        assert refused is None, f"the plan accepts nk={nk} after refusing nk={refused}"
        c = config(pl)
        lo, hi = ends.get(c, (nk, nk))
        ends[c] = (min(lo, nk), max(hi, nk))
    return ends, refused


LADDER, PIPE_REFUSED = scan_ladder()
PIPE_MAX = PIPE_REFUSED - 1

# (label, nk): both ends of every configuration, the first refused nk, and the tile / column kernels' boundaries
LEVEL_CASES = sorted({(f"cfg{c}-{end}", nk) for c, (lo, hi) in LADDER.items() for end, nk in (("lo", lo), ("hi", hi))}
                     | {("pipe-refused", PIPE_REFUSED)}
                     | {("tile-tj2-hi", 56), ("tile-tj1-lo", 57), ("tile-hi", TILE_MAX)}
                     | {("column-static-hi", 96), ("column-optin-lo", 97), ("column-hi", COLUMN_MAX)},
                     key=lambda c: (c[1], c[0]))


def kernels_for(nk):
    """(requested, expected to run) for every kernel that holds nk levels, and AUTO."""
    ks = [(PIPE, PIPE)] if nk <= PIPE_MAX else []
    ks += [(TILE, TILE)] if nk <= TILE_MAX else []
    ks += [(COLUMN, COLUMN), (AUTO, PIPE if nk <= PIPE_MAX else COLUMN)]
    return ks


def oracle_case(g, seed, adversarial=False):
    fin = cases.random_fields(g, seed=seed, adversarial=True) if adversarial else wrf.synth_fields(g, seed=seed)
    want = cases.copy_fields(fin)
    loader.oracle_c(want, g, SCALARS, tiles=8)
    return fin, want


def run(g, fin, kernel, dtype=np.float32):
    out = cases.copy_fields(fin)
    with wrf.Patch(g, dtype=dtype) as p:
        p.set_scalars(*SCALARS)
        p.set_kernel(kernel)
        p.upload(out)
        p.step()
        p.download(out, names=wrf.FIELDS)
        return out, p.last_kernel()


def assert_plan(g, nk, nx, label):
    """The launch the case is meant to exercise: its configuration, TJ, remainder strips and one-row tail."""
    rc, pl = plan_rc(g, SLOTS)
    if nk > PIPE_MAX:
        assert rc == ERR_UNSUPPORTED, (label, rc)
        return
    assert rc == 0
    if label.startswith("cfg"):
        assert config(pl) == label[3:].split("-")[0], (label, pl)
    assert pl["tj"] == (2 if pl["cfg"] == 22 else 1), pl
    assert (pl["strip_blocks"] > 0) == (nx == 266), pl             # 266: the last tile column folds into strips
    # one-row tiles: all of them at TJ=1; at cfg 22 these grids are less than a wave, which the mixed kernel runs as
    # one-row tiles only (test_cfg22_plain_and_mixed_forms runs its two-row tiles)
    assert pl["nby1"] > 0 and (pl["nby2"] == 0 or pl["cfg"] != 22), pl


def assert_all_kernels_match(g, fin, want, nk, what):
    for kernel, expect in kernels_for(nk):
        got, ran = run(g, fin, kernel)
        w = f"{what} kernel {kernel}: "
        assert ran == expect, w + f"ran kernel {ran}"
        cases.assert_bit_equal(got, want, what=w)
        cases.assert_inputs_untouched(got, fin)
        cases.assert_outside_untouched(got, fin, g)


@pytest.mark.parametrize("variant", ["specified", "periodic_open"])
@pytest.mark.parametrize("nx", [266, 270])
@pytest.mark.parametrize("label,nk", LEVEL_CASES, ids=[f"{lab}-nk{nk}" for lab, nk in LEVEL_CASES])
def test_ladder_matches_oracle(label, nk, nx, variant):
    g = ladder_grid(nx, nk, variant)
    assert_plan(g, nk, nx, label)
    for adversarial in ((False, True) if nk <= 4 else (False,)):
        fin, want = oracle_case(g, nk, adversarial)
        assert_all_kernels_match(g, fin, want, nk, f"{label} nk={nk} {nx} {variant}{' adversarial' if adversarial else ''}")


@pytest.mark.parametrize("variant", ["specified", "periodic_open"])
@pytest.mark.parametrize("nx", [266, 270])
@pytest.mark.parametrize("nk", [1, 66])
def test_one_row_patch(nk, nx, variant):
    """nj = 1: no two-row tile can be formed, so the pipe kernel runs cfg 13 for every nk up to 66."""
    g = ladder_grid(nx, nk, variant, rows=1)
    rc, pl = plan_rc(g, SLOTS)
    assert rc == 0 and pl["cfg"] == 13 and pl["nby2"] == 0 and pl["nby1"] == 1, pl
    assert (pl["strip_blocks"] > 0) == (nx == 266), pl
    for adversarial in ((False, True) if nk <= 4 else (False,)):
        fin, want = oracle_case(g, nk, adversarial)
        assert_all_kernels_match(g, fin, want, nk, f"one row nk={nk} {nx} {variant}{' adversarial' if adversarial else ''}")


def test_ladder_covers_every_configuration():
    assert set(LADDER) == {"22", "13", "12", "62", "14", "12last"}, LADDER
    assert PIPE_MAX < COLUMN_MAX


def cfg22_form(pl):
    """'plain': two-row tiles only; 'mixed': two-row tiles followed by a one-row tail."""
    if pl["rc"] != 0 or pl["cfg"] != 22 or pl["nby2"] == 0:
        return None
    return "mixed" if pl["nby1"] > 0 else "plain"


@pytest.mark.parametrize("variant", ["specified", "periodic_open"])
@pytest.mark.parametrize("nx", [266, 270])
@pytest.mark.parametrize("end", ["lo", "hi"])
@pytest.mark.parametrize("form", ["plain", "mixed"])
def test_cfg22_plain_and_mixed_forms(form, end, nx, variant):
    """cfg 22 at both ends of its range, with the two-row tile body running: as one launch of two-row tiles, and as
    two-row tiles followed by one-row tiles.  The grid is the smallest with an odd row count (so the last two-row
    tile is half filled) whose plan has that form."""
    nk = LADDER["22"][0 if end == "lo" else 1]

    def plan_of(rows):
        rc, pl = plan_rc(ladder_grid(nx, nk, variant, rows=rows), SLOTS)
        return dict(pl, rc=rc)

    rows = next(r for r in range(ROWS, 2000, 2) if cfg22_form(plan_of(r)) == form)
    g = ladder_grid(nx, nk, variant, rows=rows)
    pl = plan_of(rows)
    assert pl["tj"] == 2 and (pl["strip_blocks"] > 0) == (nx == 266), pl
    _, _, j0, j1, _, _ = g.bounds()
    assert (j1 - j0 + 1) % 2 == 1
    fin, want = oracle_case(g, rows)
    for kernel in (PIPE, AUTO):
        got, ran = run(g, fin, kernel)
        what = f"cfg 22 {form} nk={nk} {nx} {variant} ({rows} rows, plan {pl}) kernel {kernel}: "
        assert ran == PIPE, what
        cases.assert_bit_equal(got, want, what=what)
        cases.assert_inputs_untouched(got, fin)
        cases.assert_outside_untouched(got, fin, g)


# ---------------------------------------------------------------- real*8
R8_CASES = [(55, TILE), (56, TILE), (TILE_R8_MAX, TILE), (TILE_R8_MAX + 1, COLUMN), (COLUMN_R8_MAX, COLUMN)]


@pytest.mark.parametrize("variant", ["specified", "periodic_open"])
@pytest.mark.parametrize("nx", [266, 270])
@pytest.mark.parametrize("nk,auto_runs", R8_CASES, ids=[f"nk{nk}" for nk, _ in R8_CASES])
def test_r8_ladder_matches_binary64_checker(nk, auto_runs, nx, variant):
    """Tile TJ=2 up to nk 55, TJ=1 up to 220; AUTO runs the column kernel from 221 to its limit, 227."""
    g = ladder_grid(nx, nk, variant)
    fin = random_fields64(g, seed=nk)
    want = oracle64(g, fin, SCALARS)
    kernels = [(AUTO, auto_runs), (COLUMN, COLUMN)] + ([(TILE, TILE)] if nk <= TILE_R8_MAX else [])
    for kernel, expect in kernels:
        got, ran = run(g, fin, kernel, dtype=np.float64)
        assert ran == expect, (nk, kernel, ran)
        assert_bit_equal64(got, want, what=f"real*8 nk={nk} {nx} {variant} kernel {kernel}: ")
        assert_outside_untouched64(got, fin, g)


# ---------------------------------------------------------------- multi-step and host-array paths
@pytest.mark.parametrize("nk,cfg", [(150, "14"), (300, "12last")])
def test_resident_graph_loop_with_standin(nk, cfg):
    g = ladder_grid(266, nk)
    rc, pl = plan_rc(g, SLOTS)
    assert rc == 0 and config(pl) == cfg and pl["strip_blocks"] > 0, pl
    fin = wrf.synth_fields(g, seed=nk)
    want = cases.oracle_loop(g, fin, SCALARS, 6, c=C_UV)
    i0, i1, j0, j1, _, _ = g.bounds()
    got = cases.copy_fields(fin)
    with wrf.Patch(g) as p:
        p.set_scalars(*SCALARS)
        p.upload(got)
        for s in range(6):
            p.step_graph(1)
            if s < 5:
                p.standin_advance_uv("u", C_UV, i0 + 1, i1, j0, j1)
                p.standin_advance_uv("v", C_UV, i0, i1, j0 + 1, j1)
        p.download(got, names=wrf.FIELDS)
        assert p.last_kernel() == PIPE
    cases.assert_bit_equal(got, want, names=cases.OUTPUTS + ("u", "v"), what=f"6-step graph loop nk={nk}: ")
    cases.assert_outside_untouched(got, fin, g)


def test_host_array_slab_pipeline_at_cfg14():
    """The host-array entry at a size whose 3-D fields exceed 16 MB (the j-slab pipeline), three steps."""
    g = cases.grid(260, 120, 151, halo=5, variant="specified")
    assert 4 * np.prod(g.shape3) > 16 << 20
    rc, pl = plan_rc(g, SLOTS)
    assert rc == 0 and config(pl) == "14", pl
    fin = wrf.synth_fields(g, seed=151)
    want = cases.oracle_loop(g, fin, SCALARS, 3)
    got = cases.copy_fields(fin)
    try:
        wrf.call_with_fields(got, g, *SCALARS, nsteps=3)
        assert wrf.default_last_kernel() == PIPE
    finally:
        wrf.lib().wrfb200_release_cache()
    cases.assert_bit_equal(got, want, what="host-array nk=150: ")
    cases.assert_inputs_untouched(got, fin)
    cases.assert_outside_untouched(got, fin, g)


# ---------------------------------------------------------------- fused binary32 exchange at one-row configurations
FUSED_CONFIGS = ["13", "12", "62", "14", "12last"]


@functools.lru_cache(maxsize=1)
def fused_oracle(nk):
    G = cases.grid(266, 46, nk + 1, halo=5, variant="specified")
    return cases.oracle_loop(G, wrf.synth_fields(G, seed=99), SCALARS, 4, c=C_UV)


@pytest.mark.parametrize("mode", ["graph", "stepwise"])
@pytest.mark.parametrize("px,py", [(1, 2), (2, 1), (2, 2)])
@pytest.mark.parametrize("cfg", FUSED_CONFIGS)
def test_fused_exchange_at_one_row_configurations(cfg, px, py, mode):
    nk = LADDER[cfg][0]
    G = cases.grid(266, 46, nk + 1, halo=5, variant="specified")
    decomp = parallel.Decomposition(G, px, py, halo=3)
    plans = [plan_rc(decomp.patch_grid(r), SLOTS) for r in range(px * py)]
    for rc, pl in plans:
        assert rc == 0 and config(pl) == cfg and pl["tj"] == 1 and pl["strip_blocks"] > 0, pl
    # All ranks share one GPU: their blocks together must fit one wave, or a block waiting on a halo flag could
    # keep the producer of that flag from ever being scheduled.
    blocks = sum(pl["grid"] for _, pl in plans)
    assert blocks <= (SMS if blocks_per_sm(plans[0][1]) == 1 else SLOTS), (blocks, SMS)
    want = fused_oracle(nk)
    decomp, whole, ranks = run_ranks(G, px, py, 4, standin=True, graph=(mode == "graph"),
                                     stepwise=(mode == "stepwise"), scalars=SCALARS)
    for r, (_, pg, f) in enumerate(ranks):
        bad = cases.patch_mismatches(f, want, G, pg, decomp.patch_extents(r))
        assert not bad, f"cfg {cfg} nk={nk} {px}x{py} {mode} rank {r}: {bad}"


# ---------------------------------------------------------------- refusals: no launch happens
def small_patch(nk, dtype=np.float32):
    g = cases.grid(40, 7, nk + 1, halo=2)
    p = wrf.Patch(g, dtype=dtype)
    p.set_scalars(*SCALARS)
    fin = random_fields64(g, seed=1) if dtype == np.float64 else cases.random_fields(g, seed=1)
    p.upload(fin)
    return p


def assert_refused(fn, nk, limit):
    with pytest.raises(wrf.WrfB200Error) as e:
        fn()
    msg = str(e.value)
    assert e.value.status == ERR_UNSUPPORTED, msg
    assert f"nk={nk}" in msg and f"at most {limit} levels" in msg, msg


@pytest.mark.parametrize("kernel,nk,limit,dtype", [
    (PIPE, PIPE_REFUSED, PIPE_MAX, np.float32),
    (TILE, TILE_MAX + 1, TILE_MAX, np.float32),
    (COLUMN, COLUMN_MAX + 1, COLUMN_MAX, np.float32),
    (AUTO, COLUMN_MAX + 1, COLUMN_MAX, np.float32),
    (TILE, COLUMN_R8_MAX + 1, TILE_R8_MAX, np.float64),
    (COLUMN, COLUMN_R8_MAX + 1, COLUMN_R8_MAX, np.float64),
    (AUTO, COLUMN_R8_MAX + 1, COLUMN_R8_MAX, np.float64),
], ids=["pipe", "tile", "column", "auto", "r8-tile", "r8-column", "r8-auto"])
def test_level_counts_past_a_kernels_limit_are_refused(kernel, nk, limit, dtype):
    with small_patch(nk, dtype) as p:
        p.set_kernel(kernel)
        assert_refused(p.step, nk, limit)
        assert p.launch_count() == 0


def test_comm_init_refuses_a_patch_the_pipe_kernel_cannot_hold():
    with small_patch(PIPE_REFUSED) as p:
        assert_refused(lambda: p.comm_init(1, 1, 0, 1, 40, 1, 7), PIPE_REFUSED, PIPE_MAX)
        assert p.launch_count() == 0
