"""C-ABI checks that need no GPU: the library loads, exports every symbol include/wrfb200.h declares,
its host-side utilities work, and compute entry points fail LOUDLY (no CPU fallback) without a device."""
import ctypes as C
import os
import re
import threading

import numpy as np
import pytest

import wrf_model_cuda_sample_b200 as wrf
from wrf_model_cuda_sample_b200 import _lib
from tests import cases

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _have_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def _header_functions():
    text = open(os.path.join(ROOT, "include", "wrfb200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(wrfb200_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = wrf.lib()
    declared = _header_functions()
    assert len(declared) >= 25
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/wrfb200.h but not exported"
    assert sorted(_lib.PROTOTYPES) == declared, "ctypes prototypes out of sync with the header"
    assert lib.wrfb200_version() == 100


def test_field_enum_matches_header():
    text = open(os.path.join(ROOT, "include", "wrfb200.h")).read()
    body = text[text.index("typedef enum wrfb200_field"):text.index("} wrfb200_field;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = re.findall(r"WRFB200_([A-Z0-9_]+)\s*(?:=\s*0)?\s*,", body)
    assert [n.lower() for n in names if n != "NUM_FIELDS"] == list(wrf.FIELDS)


def test_bounds_match_oracle():
    from oracle import oracle_np
    rs = np.random.RandomState(0)
    for _ in range(200):
        ids, jds = 1, 1
        ide, jde = int(rs.randint(4, 60)), int(rs.randint(4, 60))
        its = int(rs.randint(1, ide)); ite = int(rs.randint(its, ide + 1))
        jts = int(rs.randint(1, jde)); jte = int(rs.randint(jts, jde + 1))
        px, sp, ne = (bool(x) for x in rs.randint(0, 2, 3))
        g = wrf.Grid(ids, ide, jds, jde, 9, -1, ide + 2, -1, jde + 2, 1, 9, its, ite, jts, jte, 1, 9, px, sp, ne)
        assert g.bounds() == oracle_np.bounds(px, sp, ne, ids, ide, jds, jde, its, ite, jts, jte, 1, 9)


def test_compare_metrics_follow_reference_definitions():
    a = np.array([1.0, -2.0, 0.0, 3.0, 5.0], dtype=np.float32)
    b = np.array([1.0, -2.0, 0.5, np.nextafter(np.float32(3.0), np.float32(4.0)), 4.0], dtype=np.float32)
    r = wrf.compare(a, b)
    assert r["n"] == 5 and r["n_equal"] == 2 and r["n_different"] == 3
    assert r["max_abs"] == pytest.approx(1.0)
    assert r["max_rel"] == pytest.approx(0.5)              # zero on one side -> max(|a|,|b|) (common.cu:117-120)
    assert r["max_ulp"] == int(np.float32(0.5).view(np.int32))        # 0.0 vs 0.5
    assert wrf.compare(a[3:], b[3:])["max_ulp"] == int(np.float32(5.0).view(np.int32)) - int(np.float32(4.0).view(np.int32))
    assert wrf.compare(a[3:4], b[3:4])["max_ulp"] == 1
    # ulp distance across zero: -x and +x are 2*magnitude-bits apart (common.cu:51-66)
    tiny = np.float32(1e-45)
    assert wrf.compare(np.array([tiny]), np.array([-tiny]))["max_ulp"] == 2
    with pytest.raises(wrf.WrfB200Error):
        wrf.compare(np.array([np.nan], dtype=np.float32), np.array([1.0], dtype=np.float32))


def test_synthetic_fields_are_decomposition_independent():
    """Counter-based generator: a patch's values equal the same cells of the global field."""
    g = cases.grid(48, 36, 10, halo=3, variant="specified")
    whole = wrf.synth_fields(g, seed=1234)
    # a patch covering global i 20..40, j 10..30 with its own 2-wide halo
    p = wrf.Grid(g.ids, g.ide, g.jds, g.jde, g.kde, 18, 42, 8, 32, 1, g.kme, 20, 40, 10, 30, 1, g.kte,
                 g.periodic_x, g.specified, g.nested)
    part = wrf.synth_fields(p, seed=1234)
    for n in wrf.FIELDS_3D:
        sub = whole[n][p.jms - g.jms:p.jme - g.jms + 1, :, p.ims - g.ims:p.ime - g.ims + 1]
        assert np.array_equal(cases.bits(part[n]), cases.bits(sub)), n
    for n in wrf.FIELDS_2D:
        sub = whole[n][p.jms - g.jms:p.jme - g.jms + 1, p.ims - g.ims:p.ime - g.ims + 1]
        assert np.array_equal(cases.bits(part[n]), cases.bits(sub)), n
    for n in wrf.FIELDS_1D:
        assert np.array_equal(cases.bits(part[n]), cases.bits(whole[n])), n
    other = wrf.synth_fields(g, seed=99, names=("u",))
    assert not np.array_equal(other["u"], whole["u"])


def test_synthetic_fields_are_atmosphere_like():
    g = cases.grid(60, 50, 20, halo=2)
    f = wrf.synth_fields(g)
    assert 9.0e4 <= f["mut"].min() and f["mut"].max() <= 9.8e4
    for n in ("msftx", "msfty", "msfuy"):
        assert 0.85 <= f[n].min() and f[n].max() <= 1.15
    assert np.all(f["dnw"][: g.kde - 1] < 0)
    assert np.allclose(f["rdnw"][: g.kde - 1] * f["dnw"][: g.kde - 1], 1.0, rtol=1e-6)
    assert np.allclose((f["fnm"] + f["fnp"])[1: g.kde - 1], 1.0, rtol=1e-6)
    assert np.all(f["ww"][:, 0, :] == 0) and np.all(f["ww_1"][:, 0, :] == 0)
    assert np.all(np.diff(f["t_1"].mean(axis=(0, 2))) > 0)


def test_unsupported_calls_are_rejected_with_a_message():
    lib = wrf.lib()
    dom = wrf.Grid.from_shape(8, 8, 4).domain()
    dom.kms = 2                                           # level 1 is addressed literally
    h = C.c_void_p()
    rc = lib.wrfb200_create(C.byref(h), C.byref(dom), -1, 0)
    assert rc == _lib.ERR_UNSUPPORTED and b"kms" in lib.wrfb200_last_error()
    assert lib.wrfb200_set_kernel(None, 1) == _lib.ERR_INVALID_ARG


@pytest.mark.skipif(_have_gpu(), reason="GPU present: covered by the gpu tests")
def test_compute_fails_loudly_without_a_gpu():
    """No CPU fallback: with no device the operator returns WRFB200_ERR_CUDA and says why."""
    g = cases.grid(10, 8, 5, halo=1)
    f = cases.random_fields(g, seed=1)
    before = cases.copy_fields(f)
    with pytest.raises(wrf.WrfB200Error) as e:
        wrf.call_with_fields(f, g, *cases.SCALARS_12KM)
    assert e.value.status == _lib.ERR_CUDA and "no CPU fallback" in str(e.value)
    for n in f:
        assert np.array_equal(cases.bits(f[n]), cases.bits(before[n]))
    with pytest.raises(wrf.WrfB200Error):
        wrf.Patch(g)


def test_product_package_never_touches_the_oracle():
    """The shipped package must not import, load or mention anything under oracle/."""
    pkg = os.path.join(ROOT, "wrf_model_cuda_sample_b200")
    for dirpath, _, files in os.walk(pkg):
        for fn in files:
            if fn.endswith((".py", ".cu", ".h", ".cpp")):
                text = open(os.path.join(dirpath, fn)).read()
                assert "oracle" not in text.lower(), f"{fn} refers to the oracle"


def _check_sass():
    import subprocess
    r = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True)
    assert r.returncode == 0
    assert "UTMALDG" in r.stdout, "the product kernel must stage its operands with TMA"
    assert "FMUL2" in r.stdout
    assert "FFMA2" not in r.stdout, "a packed multiply-add contraction slipped in"


def test_no_packed_fma_contraction_in_sass():
    """ptxas (CUDA 12.9) fuses mul.rn.f32x2 + add.rn.f32x2 into FFMA2 even under --fmad false, which would
    break bit-exactness.  The kernels avoid every packed add of a packed product; prove it on the built
    library: no FFMA2 anywhere in its SASS."""
    import shutil
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not available")
    _check_sass()


@pytest.mark.gpu
def test_no_packed_fma_contraction_in_sass_on_the_gpu_box():
    """The same check in the GPU lane, where it may not be skipped: the library that just produced the parity
    results is the one whose SASS is inspected (the image ships cuobjdump with the CUDA toolkit)."""
    import shutil
    assert shutil.which("cuobjdump") is not None, "cuobjdump missing on the GPU box: cannot prove the absence of FFMA2"
    _check_sass()


def test_null_pointer_is_rejected_before_anything_runs():
    """Argument validation needs no device: a NULL field pointer is WRFB200_ERR_INVALID_ARG with a message."""
    lib = wrf.lib()
    g = cases.grid(10, 8, 5, halo=1)
    f = cases.random_fields(g, seed=1)
    ptrs = [f[n].ctypes.data for n in _lib.FORTRAN_ARRAY_ORDER_A]
    ptrs[3] = None                                             # u_1
    args = (ptrs + [1e-4, 1e-4, 12.0, 0.1] + [f[n].ctypes.data for n in _lib.FORTRAN_ARRAY_ORDER_B]
            + [0, 1, 0] + list(g.index_args()))
    assert lib.wrfb200_advance_mu_t(*args) == _lib.ERR_INVALID_ARG
    assert b"null pointer" in lib.wrfb200_last_error()
    assert lib.wrfb200_advance_mu_t_loop(*(args + [0])) == _lib.ERR_INVALID_ARG     # nsteps < 1


def test_fortran_interfaces_bind_exported_symbols():
    """Every BIND(C, NAME=...) of the two Fortran modules (source only: no Fortran compiler in the image) names a
    symbol the built library exports and the header declares."""
    lib = wrf.lib()
    declared = set(_header_functions())
    fdir = os.path.join(ROOT, "wrf_model_cuda_sample_b200", "fortran")
    seen = set()
    for fn in ("module_small_step_em.F90", "module_small_step_em_resident.F90"):
        text = open(os.path.join(fdir, fn)).read()
        for name in re.findall(r'BIND\(C,\s*NAME="([a-z0-9_]+)"\)', text):
            assert name in declared, f"{fn}: {name} is not declared in include/wrfb200.h"
            assert hasattr(lib, name), f"{fn}: {name} is not exported"
            seen.add(name)
    for must in ("wrfb200_advance_mu_t", "wrfb200_acoustic_loop_begin", "wrfb200_set_uv", "wrfb200_download_outputs",
                 "wrfb200_comm_init", "wrfb200_comm_connect", "wrfb200_comm_loop"):
        assert must in seen


def test_comm_and_residency_entry_points_fail_cleanly_without_state():
    lib = wrf.lib()
    assert lib.wrfb200_comm_info_bytes() == 2048
    assert lib.wrfb200_comm_step(None) == _lib.ERR_INVALID_ARG
    assert lib.wrfb200_comm_connect(None, None, 0) == _lib.ERR_INVALID_ARG
    assert lib.wrfb200_acoustic_loop_begin() == 0 and lib.wrfb200_acoustic_loop_end() == 0
    # the last kernel is per thread: ask from one that has made no call, whatever ran earlier in this process
    k, rc = C.c_int(-1), []
    t = threading.Thread(target=lambda: rc.append(lib.wrfb200_default_last_kernel(C.byref(k))))
    t.start()
    t.join()
    assert rc == [0] and k.value == 0
