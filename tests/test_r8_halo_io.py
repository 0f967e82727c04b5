"""Real*8 halo pack / unpack (wrfb200_pack_halo_r8 / _unpack_halo_r8), the binary64 error report
(wrfb200_compare_r8) and 8-byte .bin cases (binio, cli).

The multi-rank test moves the packed edges itself -- pack, a device-to-device copy, unpack -- as a host with its own
transport (MPI, NCCL) does, with the ranks as handles of one process on device 0.  Bar: every rank's patch
BIT-IDENTICAL to the binary64 checker loop, halos poisoned beforehand; inputs are float64 with low mantissa bits a
float cannot hold."""
import ctypes as C
import os

import numpy as np
import pytest

import wrf_model_cuda_sample_b200 as wrf
from wrf_model_cuda_sample_b200 import _lib, binio, parallel
from tests import cases, r8_checkers
from tests.test_fused_comm_r8 import C_UV, SCALARS, checker_loop64, widen64

F64 = np.float64
gpu = pytest.mark.gpu


# ================================================================ CPU: wrf.compare / wrfb200_compare_r8
def test_compare_rejects_mixed_precision():
    a32, a64 = np.ones(4, dtype=np.float32), np.ones(4, dtype=F64)
    for a, b in ((a32, a64), (a64, a32), (a64, [1.0] * 4)):
        with pytest.raises(TypeError):
            wrf.compare(a, b)


def test_compare_r8_metrics_follow_reference_definitions():
    a = np.array([1.0, -2.0, 0.0, 3.0, 5.0], dtype=F64)
    b = np.array([1.0, -2.0, 0.5, np.nextafter(3.0, 4.0), 4.0], dtype=F64)
    r = wrf.compare(a, b)
    assert r["n"] == 5 and r["n_equal"] == 2 and r["n_different"] == 3
    assert r["max_abs"] == 1.0
    assert r["max_rel"] == 0.5                              # zero on one side -> max(|a|,|b|) (common.cu:117-120)
    assert r["max_ulp"] == int(np.float64(0.5).view(np.int64))          # 0.0 vs 0.5
    assert r["rmse"] == np.sqrt((0.5 ** 2 + (np.nextafter(3.0, 4.0) - 3.0) ** 2 + 1.0) / 5)
    assert wrf.compare(a[4:], b[4:])["max_ulp"] == int(np.float64(5.0).view(np.int64)) - int(np.float64(4.0).view(np.int64))
    # one binary64 ulp, below float32 resolution: the float32 report cannot see it, the binary64 one must
    x, y = np.array([1.0], dtype=F64), np.array([np.nextafter(1.0, 2.0)], dtype=F64)
    assert wrf.compare(x.astype(np.float32), y.astype(np.float32))["n_different"] == 0
    r = wrf.compare(x, y)
    assert r["n_different"] == 1 and r["max_ulp"] == 1 and r["max_abs"] == 2.0 ** -52
    # ulp distance across zero: -x and +x are 2*magnitude-bits apart (common.cu:51-66)
    tiny = np.float64(5e-324)
    assert wrf.compare(np.array([tiny]), np.array([-tiny]))["max_ulp"] == 2
    assert wrf.compare(np.array([-0.0]), np.array([0.0]))["max_ulp"] == 0
    # only opposite-signed values near the infinities exceed a long: saturated
    assert wrf.compare(np.array([np.inf]), np.array([-np.inf]))["max_ulp"] == 2 ** 63 - 1
    with pytest.raises(wrf.WrfB200Error) as e:
        wrf.compare(np.array([1.0, np.nan]), np.array([1.0, 1.0]))
    assert e.value.status == _lib.ERR_INVALID_ARG and "NaN" in str(e.value)


def test_r8_halo_verbs_reject_a_null_handle():
    lib = wrf.lib()
    buf = (C.c_double * 8)()
    for name in ("wrfb200_pack_halo_r8", "wrfb200_unpack_halo_r8"):
        assert getattr(lib, name)(None, 2, wrf.WEST, 1, 1, 8, 1, 8, buf) == _lib.ERR_INVALID_ARG, name
        assert b"null" in lib.wrfb200_last_error(), name
    assert lib.wrfb200_compare_r8(None, None, 1, None) == _lib.ERR_INVALID_ARG


# ================================================================ CPU: 8-byte .bin cases
def _case64(tmp_path, variant="specified"):
    g = cases.grid(30, 22, 8, halo=3, variant=variant)
    f = widen64(cases.random_fields(g, seed=42))
    inp = str(tmp_path / "in")
    binio.write_case(inp, g, SCALARS, f)
    return g, f, inp


def test_8byte_case_round_trips_bit_for_bit(tmp_path):
    g, f, inp = _case64(tmp_path, "periodic_specified")
    raw = open(os.path.join(inp, "grid_u_2.bin"), "rb").read()
    assert len(raw) == 8 * f["u"].size
    assert np.frombuffer(raw, dtype=">f8").reshape(g.shape3)[3, 1, 2] == f["u"][3, 1, 2]
    assert os.path.getsize(os.path.join(inp, "dts_rk.bin")) == 8
    assert os.path.getsize(os.path.join(inp, "ime.bin")) == 4              # integers stay 4 bytes
    g2, scalars, f2 = binio.read_case(inp)
    assert g2 == g
    assert all(type(s) is np.float64 and s == want for s, want in zip(scalars, SCALARS))
    for n in wrf.FIELDS:
        assert f2[n].dtype == F64 and np.array_equal(f2[n].view(np.uint64), f[n].view(np.uint64)), n


def test_8byte_case_without_output_only_fields_reads_them_as_float64_zeros(tmp_path):
    g, f, inp = _case64(tmp_path)
    os.remove(os.path.join(inp, "muave.bin"))
    _, _, f2 = binio.read_case(inp)
    assert f2["muave"].dtype == F64 and not f2["muave"].any()


def test_case_mixing_4_and_8_byte_reals_is_rejected(tmp_path):
    g, f, inp = _case64(tmp_path)
    path = os.path.join(inp, "grid_t_2.bin")
    binio.write_field(path, f["t"].astype(np.float32))
    with pytest.raises(ValueError, match="grid_t_2.bin"):
        binio.read_case(inp)
    # a 4-byte scalar in an 8-byte case: named too
    binio.write_field(path, f["t"])
    binio.write_real(os.path.join(inp, "grid_epssm.bin"), 0.1)
    with pytest.raises(ValueError, match="grid_epssm.bin: 4-byte"):
        binio.read_case(inp)
    # a file whose length fits neither size
    with open(os.path.join(inp, "grid_epssm.bin"), "wb") as fh:
        fh.write(b"\0" * 6)
    with pytest.raises(ValueError, match="grid_epssm.bin"):
        binio.read_case(inp)
    # and the writer refuses to make such a case
    mixed = dict(f, t=f["t"].astype(np.float32))
    with pytest.raises(ValueError):
        binio.write_case(str(tmp_path / "mixed"), g, SCALARS, mixed)


def test_4byte_case_bytes_are_unchanged(tmp_path):
    """Every file of a float32 case holds exactly the big-endian bytes of its values (what the writer always wrote)."""
    g = cases.grid(30, 22, 8, halo=3, variant="periodic_specified")
    f = cases.random_fields(g, seed=3)
    d = str(tmp_path / "in")
    binio.write_case(d, g, cases.SCALARS_12KM, f)
    want = {binio.FILE_OF[n]: np.asarray(f[n], dtype=">f4").tobytes() for n in wrf.FIELDS}
    want.update({s: np.array([v], dtype=">f4").tobytes() for s, v in zip(binio.SCALAR_FILES, cases.SCALARS_12KM)})
    want.update({n: np.array([getattr(g, n)], dtype=">i4").tobytes() for n in binio.DIM_NAMES})
    want.update({stem: np.array([int(getattr(g, n))], dtype=">i4").tobytes() for n, stem in binio.FLAG_FILES.items()})
    want["kds"] = np.array([1], dtype=">i4").tobytes()
    assert sorted(os.listdir(d)) == sorted(k + ".bin" for k in want)
    for stem, b in want.items():
        assert open(os.path.join(d, stem + ".bin"), "rb").read() == b, stem
    g2, scalars, f2 = binio.read_case(d)
    assert all(type(s) is np.float32 for s in scalars) and all(f2[n].dtype == np.float32 for n in wrf.FIELDS)


# ================================================================ GPU: the verbs on one patch
def _box(g, side, width, inside, ext):
    """(J, I) slices of the halo box of the memory arrays, as the C layer defines it (halo.cu, halo_box)."""
    ips, ipe, jps, jpe = ext
    if side in (wrf.WEST, wrf.EAST):
        i0 = (ips if inside else ips - width) if side == wrf.WEST else (ipe - width + 1 if inside else ipe + 1)
        i1, j0, j1 = i0 + width - 1, jps, jpe
    else:
        j0 = (jps if inside else jps - width) if side == wrf.SOUTH else (jpe - width + 1 if inside else jpe + 1)
        j1, i0, i1 = j0 + width - 1, ips, ipe
    return slice(j0 - g.jms, j1 - g.jms + 1), slice(i0 - g.ims, i1 - g.ims + 1)


def _sub(a, J, I):
    return a[J, :, I] if a.ndim == 3 else a[J, I]


@gpu
@pytest.mark.parametrize("field", ["u", "mu"])
def test_pack_unpack_r8_round_trip(field):
    import torch
    g = cases.grid(40, 30, 7, halo=3)
    ext = (g.ids, g.ide, g.jds, g.jde)
    fin = widen64(wrf.synth_fields(g, seed=11))
    with wrf.Patch(g, device=0, dtype=F64) as p:
        p.upload(fin)
        for side in (wrf.WEST, wrf.EAST, wrf.SOUTH, wrf.NORTH):
            for width in (1, 2):
                J, I = _box(g, side, width, True, ext)
                inside = _sub(fin[field], J, I)
                buf = torch.full((inside.size,), 7.0, dtype=torch.float64, device="cuda:0")
                n0 = p.launch_count()
                p.pack_halo(field, side, width, *ext, buf)
                p.sync()
                got = buf.cpu().numpy()
                assert np.array_equal(got.view(np.uint64), np.ascontiguousarray(inside).ravel().view(np.uint64)), \
                    (side, width)
                # unpack values that are in no field into the halo just outside the same edge
                Jo, Io = _box(g, side, width, False, ext)
                new = (np.arange(inside.size, dtype=F64) + 0.5) * (1.0 + 2.0 ** -45)
                src = torch.from_numpy(new).to("cuda:0")
                p.unpack_halo(field, side, width, *ext, src)
                assert p.launch_count() == n0 + 2
                after = {n: np.empty_like(a) for n, a in fin.items()}
                p.download(after, names=wrf.FIELDS)
                want = cases.copy_fields(fin)
                _sub(want[field], Jo, Io)[...] = new.reshape(_sub(want[field], Jo, Io).shape)
                for n in wrf.FIELDS:
                    assert np.array_equal(after[n].view(np.uint64), want[n].view(np.uint64)), (n, side, width)
                p.upload(fin, names=[field])


@gpu
def test_r8_halo_verbs_reject_bad_arguments():
    import torch
    lib = wrf.lib()
    g = cases.grid(40, 20, 6, halo=2)
    ext = (g.ids, g.ide, g.jds, g.jde)

    def err():
        return lib.wrfb200_last_error().decode()

    buf = torch.zeros(4096, dtype=torch.float64, device="cuda:0")
    b = C.c_void_p(buf.data_ptr())
    u, dnw = wrf.FIELD_ID["u"], wrf.FIELD_ID["dnw"]
    with wrf.Patch(g, device=0, dtype=F64) as p8, wrf.Patch(g, device=0) as p4:
        for fn in (lib.wrfb200_pack_halo_r8, lib.wrfb200_unpack_halo_r8):
            assert fn(p8._h, u, 7, 1, *ext, b) == _lib.ERR_INVALID_ARG and "bad side" in err()
            assert fn(p8._h, u, wrf.WEST, 0, *ext, b) == _lib.ERR_INVALID_ARG and "width" in err()
            assert fn(p8._h, u, wrf.WEST, 45, *ext, b) == _lib.ERR_INVALID_ARG and "outside memory" in err()
            assert fn(p8._h, dnw, wrf.WEST, 1, *ext, b) == _lib.ERR_INVALID_ARG and "no horizontal halo" in err()
            assert fn(p8._h, u, wrf.WEST, 1, *ext, None) == _lib.ERR_INVALID_ARG and "null" in err()
            # a real*4 handle
            assert fn(p4._h, u, wrf.WEST, 1, *ext, b) == _lib.ERR_STATE and "real*4" in err()
        assert p8.launch_count() == 0 and p4.launch_count() == 0
        # Patch checks the buffer before the library sees it
        for bad in (torch.zeros(64, dtype=torch.float32, device="cuda:0"), np.zeros(64, dtype=F64),
                    torch.zeros(64, dtype=torch.float64)):
            with pytest.raises(TypeError):
                p8.pack_halo("u", wrf.WEST, 1, *ext, bad)
            with pytest.raises(TypeError):
                p8.unpack_halo("u", wrf.WEST, 1, *ext, bad)
        with pytest.raises(TypeError):
            p4.pack_halo("u", wrf.WEST, 1, *ext, buf)
    # a field without a device buffer
    with wrf.Patch(g, device=0, allocate=False, dtype=F64) as p8:
        assert lib.wrfb200_pack_halo_r8(p8._h, u, wrf.WEST, 1, *ext, b) == _lib.ERR_STATE and "no device buffer" in err()


# ================================================================ GPU: ranks exchanging through the caller's transport
def _exchange(halos, decomp, hs):
    """Fill every rank's halos of ``halos``: the neighbour packs its inside edge, a device-to-device copy moves it,
    this rank unpacks it (what a host does around MPI_Sendrecv)."""
    for r, h in enumerate(hs):
        for field, sides in halos:
            for side in sides:
                src = decomp.neighbour(r, side)
                if src is None:
                    continue
                sent = hs[src].pack(field, parallel.OPPOSITE[side], 1)
                recv = h.recv_buffer(field, side, 1)
                recv.copy_(sent)
                h.unpack(field, side, 1, recv)


@gpu
@pytest.mark.parametrize("px,py", [(1, 2), (2, 1), (2, 2)])
def test_pack_transport_unpack_r8_ranks_match_binary64_checker_loop(px, py):
    import torch
    G = cases.grid(200, 96, 14, halo=5, variant="specified")
    nsteps = 4
    decomp = parallel.Decomposition(G, px, py, halo=3)
    whole = widen64(wrf.synth_fields(G, seed=99))
    ranks = []
    try:
        for r in range(px * py):
            pg = decomp.patch_grid(r)
            f = cases.carve_patch(whole, G, pg)
            cases.poison_neighbour_halos(f, decomp, r, pg,
                                         (parallel.CONSTANT_HALOS, parallel.STEP_HALOS, parallel.OUTPUT_HALOS))
            p = wrf.Patch(pg, device=0, dtype=F64)
            p.set_scalars(*SCALARS)
            p.upload(f)
            ranks.append((p, pg, f, parallel.GpuPatchHalo(p, decomp, r, torch.device("cuda", 0))))
        hs = [h for _, _, _, h in ranks]
        _exchange(parallel.CONSTANT_HALOS, decomp, hs)
        for s in range(nsteps):
            _exchange(parallel.STEP_HALOS, decomp, hs)
            for p, pg, _, _ in ranks:
                p.step(pg)
            _exchange(parallel.OUTPUT_HALOS, decomp, hs)
            if s + 1 < nsteps:
                for r, (p, _, _, _) in enumerate(ranks):
                    ubox, vbox = cases.standin_boxes(G, *decomp.patch_extents(r))
                    p.standin_advance_uv("u", C_UV, *ubox)
                    p.standin_advance_uv("v", C_UV, *vbox)
        for p, _, f, h in ranks:
            assert all(b.dtype == torch.float64 for b in h._bufs.values())
            p.download(f, names=cases.OUTPUTS + ("u", "v"))
    finally:
        for p, _, _, _ in ranks:
            p.close()
    want = checker_loop64(G, whole, nsteps, c=C_UV)
    for r, (_, pg, f, _) in enumerate(ranks):
        bad = cases.patch_mismatches(f, want, G, pg, decomp.patch_extents(r))
        assert not bad, f"{px}x{py} rank {r}: {bad}"


# ================================================================ GPU: the CLI on an 8-byte case
@gpu
def test_cli_runs_8byte_case_through_the_r8_operator(tmp_path, capsys):
    from wrf_model_cuda_sample_b200 import cli
    g = cases.grid(30, 22, 8, halo=3)
    f = widen64(wrf.synth_fields(g, seed=4))
    inp, gold, out = str(tmp_path / "in"), str(tmp_path / "gold"), str(tmp_path / "out")
    binio.write_case(inp, g, SCALARS, f)
    want = cases.copy_fields(f)
    r8_checkers.oracle_c_r8(want, g, SCALARS)
    binio.write_case(gold, g, SCALARS, want, suffix="_output", names=binio.GOLDEN)
    assert cli.main([inp, gold, "--write", out]) == 0
    text = capsys.readouterr().out
    assert "worst max-ulp over all fields: 0" in text and "# of non-equal values: 0" in text
    for n in binio.GOLDEN:
        path = os.path.join(out, binio.FILE_OF[n] + "_output.bin")
        assert os.path.getsize(path) == 8 * want[n].size, n
        got = binio.read_field(path, g.shape_of(n))
        assert got.dtype == F64 and np.array_equal(got.view(np.uint64), want[n].view(np.uint64)), n
    # the binary64 report sees a one-ulp change that a float32 one would not
    t = want["t"].copy()
    t.flat[5] = np.nextafter(t.flat[5], np.inf)
    binio.write_field(os.path.join(gold, "grid_t_2_output.bin"), t)
    assert cli.main([inp, gold]) == 0
    assert "# of non-equal values: 1" in capsys.readouterr().out
