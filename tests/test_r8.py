"""real*8 advance_mu_t (WRF built with -r8): the binary64 checkers, the _r8 C ABI and the double kernels.

CPU tests pin the two binary64 checkers (tests/r8_checkers.py: the oracle's C and numpy restatements evaluated
in double) to each other bit for bit and
check everything the library decides before device work.  GPU tests (-m gpu) compare every real*8 kernel and
entry point with the C checker bit for bit (integer compare of the float64 bit patterns)."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import wrf_model_cuda_sample_b200 as wrf
from wrf_model_cuda_sample_b200 import _lib
from oracle import loader
from tests import cases, r8_checkers

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F64 = np.float64
SCALARS_12KM = tuple(F64(x) for x in cases.SCALARS_12KM)
SCALARS_3KM = tuple(F64(x) for x in cases.SCALARS_3KM)
KERNELS = {"tile": wrf.KERNEL_TILE, "column": wrf.KERNEL_COLUMN, "auto": wrf.KERNEL_AUTO}
RAGGED = [(130, 9, 5, 1), (257, 6, 4, 2), (5, 5, 3, 1), (383, 3, 17, 7), (64, 64, 2, 4)]


# ---------------------------------------------------------------- float64 inputs and comparisons
def random_fields64(g, seed, adversarial=False):
    """float64 inputs with full 53-bit mantissas: the float32 case generator's magnitudes, each value
    perturbed by a random relative 1e-7 so that no input is a float32 value."""
    f32 = cases.random_fields(g, seed, adversarial=adversarial)
    rs = np.random.RandomState(seed + 1)
    f = {}
    for n, a in f32.items():
        f[n] = a.astype(F64) * (1.0 + rs.uniform(-1e-7, 1e-7, size=a.shape))
    if not adversarial:
        f["rdnw"] = 1.0 / f["dnw"]
        f["fnp"] = 1.0 - f["fnm"]
    return f


def to64(f):
    return {k: v.astype(F64) for k, v in f.items() if isinstance(v, np.ndarray)}


def bits64(a):
    return np.ascontiguousarray(a).view(np.uint64)


def assert_bit_equal64(got, want, names=cases.OUTPUTS, what=""):
    for n in names:
        assert got[n].dtype == F64 and want[n].dtype == F64, n
        g_, w_ = bits64(got[n]), bits64(want[n])
        same = (g_ == w_) | (np.isnan(got[n]) & np.isnan(want[n]))
        if not same.all():
            bad = np.argwhere(~same)
            first = tuple(bad[0])
            raise AssertionError(f"{what}{n}: {len(bad)} of {g_.size} values differ; first at [j,k,i]={first}: "
                                 f"got {got[n][first]!r} want {want[n][first]!r}")


def assert_outside_untouched64(after, before, g):
    i0, i1, j0, j1, k0, k1 = g.bounds()
    for n in cases.OUTPUTS:
        a, b = bits64(after[n]).copy(), bits64(before[n]).copy()
        if a.ndim == 3:
            a[j0 - g.jms:j1 - g.jms + 1, k0 - g.kms:k1 - g.kms + 1, i0 - g.ims:i1 - g.ims + 1] = 0
            b[j0 - g.jms:j1 - g.jms + 1, k0 - g.kms:k1 - g.kms + 1, i0 - g.ims:i1 - g.ims + 1] = 0
        else:
            a[j0 - g.jms:j1 - g.jms + 1, i0 - g.ims:i1 - g.ims + 1] = 0
            b[j0 - g.jms:j1 - g.jms + 1, i0 - g.ims:i1 - g.ims + 1] = 0
        assert np.array_equal(a, b), f"{n}: cells outside the computed range were written"


def oracle64(g, fin, scalars, tiles=0):
    want = cases.copy_fields(fin)
    r8_checkers.oracle_c_r8(want, g, scalars, tiles=tiles)
    return want


def oracle_loop64(g, fin, scalars, nsteps, c=None, tiles=0):
    """nsteps of the binary64 C checker, with the stand-in advance_uv between steps."""
    f = cases.copy_fields(fin)
    ubox, vbox = cases.standin_boxes(g, g.ids, g.ide, g.jds, g.jde)
    for s in range(nsteps):
        r8_checkers.oracle_c_r8(f, g, scalars, tiles=tiles)
        if c is not None and s + 1 < nsteps:
            cases.standin_advance_uv_numpy(f, g, c, ubox, vbox)   # 0.25 is exact: float64 result
    return f


def run_patch64(g, fin, scalars, kernel, nsteps=1, graph=False, tiles=None):
    out = cases.copy_fields(fin)
    with wrf.Patch(g, dtype=np.float64) as p:
        p.set_scalars(*scalars)
        p.set_kernel(kernel)
        p.upload(out)
        if tiles is not None:
            for t in tiles:
                p.step(g.with_tile(*t))
        elif graph:
            p.step_graph(nsteps)
        else:
            for _ in range(nsteps):
                p.step()
        p.download(out, names=wrf.FIELDS)
        ran = p.last_kernel()
    return out, ran


def _have_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


# ================================================================ CPU: the binary64 checkers
@pytest.mark.parametrize("variant", sorted(cases.FLAG_VARIANTS))
def test_c_and_numpy_checkers_agree_r8(variant):
    g = cases.grid(37, 23, 11, halo=2, variant=variant)
    for adversarial in (False, True):
        fin = random_fields64(g, seed=11, adversarial=adversarial)
        a, b = cases.copy_fields(fin), cases.copy_fields(fin)
        r8_checkers.oracle_c_r8(a, g, SCALARS_12KM)
        r8_checkers.oracle_numpy_r8(b, g, SCALARS_12KM)
        assert_bit_equal64(a, b, what=f"{variant}/adversarial={adversarial} ")
        assert_outside_untouched64(a, fin, g)


@pytest.mark.parametrize("shape", RAGGED + [(40, 12, 120, 5)])
def test_c_and_numpy_checkers_agree_r8_ragged_and_deep(shape):
    nx, ny, nz, halo = shape
    g = cases.grid(nx, ny, nz, halo=halo, variant="periodic_open")
    fin = random_fields64(g, seed=nx + nz, adversarial=(nz == 4))
    a, b = cases.copy_fields(fin), cases.copy_fields(fin)
    r8_checkers.oracle_c_r8(a, g, SCALARS_3KM)
    r8_checkers.oracle_numpy_r8(b, g, SCALARS_3KM)
    assert_bit_equal64(a, b, what=f"{shape} ")


def test_r8_is_the_same_formula_evaluated_in_double():
    """On float32-representable inputs the binary64 result agrees with the binary32 checker to float32 accuracy,
    but is not the float32 result widened: the arithmetic really is double."""
    g = cases.grid(60, 30, 20, halo=3, variant="specified")
    f32 = cases.random_fields(g, seed=12)
    want32 = cases.copy_fields(f32)
    loader.oracle_c(want32, g, cases.SCALARS_12KM)
    got64 = to64(f32)
    r8_checkers.oracle_c_r8(got64, g, SCALARS_12KM)
    i0, i1, j0, j1, k0, k1 = g.bounds()
    J, I = slice(j0 - g.jms, j1 - g.jms + 1), slice(i0 - g.ims, i1 - g.ims + 1)
    K = slice(k0 - g.kms, k1 - g.kms + 1)
    for n in cases.OUTPUTS:
        a = got64[n][J, K, I] if got64[n].ndim == 3 else got64[n][J, I]
        b = want32[n][J, K, I] if want32[n].ndim == 3 else want32[n][J, I]
        scale = float(np.max(np.abs(a)))
        assert np.allclose(a, b.astype(F64), rtol=1e-5, atol=1e-5 * scale), n
        if n != "t_ave":                            # t_ave is a copy of the input t
            assert np.any(a != b.astype(F64)), f"{n}: the double result equals the widened float result"


def test_c_checker_r8_exports_only_suffixed_names():
    """The binary64 build of the oracle's C file carries _r8 names only, so it can never be mistaken for (or
    loaded in place of) the binary32 oracle."""
    lib = r8_checkers.c_library()
    assert hasattr(lib, "oracle_advance_mu_t_r8") and hasattr(lib, "oracle_advance_mu_t_tiled_r8")
    assert not hasattr(lib, "oracle_advance_mu_t") and not hasattr(lib, "oracle_advance_mu_t_tiled")


# ================================================================ CPU: validation before any device work
def test_mixed_precision_arrays_raise_type_error():
    g = cases.grid(10, 8, 5, halo=1)
    f = cases.random_fields(g, seed=1)
    f["u"] = f["u"].astype(F64)
    with pytest.raises(TypeError, match=r"all arrays float32 \(default REAL\) or all float64"):
        wrf.call_with_fields(f, g, *cases.SCALARS_12KM)
    f = to64(cases.random_fields(g, seed=1))
    f["dnw"] = f["dnw"].astype(np.float32)
    with pytest.raises(TypeError, match="float64"):
        wrf.call_with_fields(f, g, *SCALARS_12KM)
    with pytest.raises(TypeError):
        wrf.Patch(g, dtype=np.float16)


def _r8_args(f, g, scalars):
    a = [f[n].ctypes.data for n in _lib.FORTRAN_ARRAY_ORDER_A]
    b = [f[n].ctypes.data for n in _lib.FORTRAN_ARRAY_ORDER_B]
    return a + [float(x) for x in scalars] + b + [int(g.periodic_x), int(g.specified), int(g.nested)] + \
        list(g.index_args())


def test_r8_null_pointer_and_bad_nsteps_are_rejected_before_anything_runs():
    lib = wrf.lib()
    g = cases.grid(10, 8, 5, halo=1)
    f = to64(cases.random_fields(g, seed=1))
    args = _r8_args(f, g, SCALARS_12KM)
    args[_lib.FORTRAN_ARRAY_ORDER_A.index("v_1")] = None
    assert lib.wrfb200_advance_mu_t_r8(*args) == _lib.ERR_INVALID_ARG
    assert b"null pointer" in lib.wrfb200_last_error()
    assert lib.wrfb200_advance_mu_t_loop_r8(*(_r8_args(f, g, SCALARS_12KM) + [0])) == _lib.ERR_INVALID_ARG


@pytest.mark.skipif(_have_gpu(), reason="GPU present")
def test_r8_entry_has_no_cpu_fallback():
    g = cases.grid(10, 8, 5, halo=1)
    f = to64(cases.random_fields(g, seed=1))
    before = cases.copy_fields(f)
    with pytest.raises(wrf.WrfB200Error) as e:
        wrf.call_with_fields(f, g, *SCALARS_12KM)
    assert e.value.status == _lib.ERR_CUDA and "no CPU fallback" in str(e.value)
    for n in f:
        assert np.array_equal(bits64(f[n]), bits64(before[n]))
    with pytest.raises(wrf.WrfB200Error) as e:
        wrf.Patch(g, dtype=np.float64)
    assert e.value.status == _lib.ERR_CUDA


# ================================================================ CPU: what the compiler made
def _sass_functions(path):
    out = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    funcs, name = {}, None
    for ln in out.splitlines():
        m = re.search(r"Function : (\S+)", ln)
        if m:
            name = m.group(1)
            funcs[name] = []
        elif name and re.match(r"\s+/\*[0-9a-f]{4}\*/", ln):
            funcs[name].append(" ".join(re.sub(r"/\*[0-9a-f]{4,}\*/", "", ln).split()))
    return funcs


def _r8_kernels(funcs):
    return {n: v for n, v in funcs.items() if "amt_tile_kernel_r8" in n or "amt_column_kernel_r8" in n}


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not available")
def test_r8_kernels_present_and_no_packed_fma():
    funcs = _sass_functions(_lib.LIB_PATH)
    r8 = _r8_kernels(funcs)
    names = sorted(r8)
    assert any("amt_tile_kernel_r8ILi1E" in n for n in names), names
    assert any("amt_tile_kernel_r8ILi2E" in n for n in names), names
    assert any("amt_column_kernel_r8" in n for n in names), names
    for n, ins in funcs.items():
        assert not any(i.startswith("FFMA2") for i in ins), f"{n}: packed FMA"
    for n, ins in r8.items():
        assert any(i.split()[0].startswith("DADD") for i in ins), f"{n}: no binary64 arithmetic"


@pytest.mark.skipif(shutil.which("cuobjdump") is None or shutil.which("nvcc") is None, reason="CUDA toolkit absent")
def test_r8_kernels_contract_nothing(tmp_path):
    """The only DFMA in a real*8 kernel is inside IEEE __ddiv_rn (whose correctly rounded sequence is made of
    them).  Proof: compiled with contraction allowed (-fmad=true) the kernels are instruction for instruction the
    ones in the library (built -fmad=false), so no multiply-add of the formula itself was fused."""
    csrc = os.path.join(ROOT, "wrf_model_cuda_sample_b200", "csrc")
    built = _r8_kernels(_sass_functions(_lib.LIB_PATH))
    for tu in ("amt_tile_r8.cu", "amt_column.cu"):
        cubin = str(tmp_path / (tu + ".cubin"))
        subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-fmad=true",
                        "-lineinfo", "-cubin", "-o", cubin, os.path.join(csrc, tu)], check=True)
        fmad = _r8_kernels(_sass_functions(cubin))
        assert fmad, tu
        for n, ins in fmad.items():
            assert built[n] == ins, f"{n}: -fmad=true changes the code"


# ================================================================ GPU: every kernel against the binary64 checker
gpu = pytest.mark.gpu


@pytest.fixture
def _reset_default_kernel():
    yield
    wrf.lib().wrfb200_set_default_kernel(wrf.KERNEL_AUTO)


@gpu
@pytest.mark.parametrize("kernel", ["auto", "tile", "column"])
@pytest.mark.parametrize("variant", sorted(cases.FLAG_VARIANTS))
def test_r8_tutorial_domain_all_flag_variants(variant, kernel):
    g = cases.grid(74, 61, 28, halo=5, variant=variant)
    fin = random_fields64(g, seed=2)
    want = oracle64(g, fin, SCALARS_12KM)
    got, ran = run_patch64(g, fin, SCALARS_12KM, KERNELS[kernel])
    assert_bit_equal64(got, want, what=f"{variant}/{kernel} ")
    assert_bit_equal64(got, fin, names=[n for n in wrf.FIELDS if n not in cases.OUTPUTS], what="inputs ")
    assert_outside_untouched64(got, fin, g)
    assert ran == (wrf.KERNEL_TILE if kernel == "auto" else KERNELS[kernel])


@gpu
@pytest.mark.parametrize("kernel", ["auto", "tile", "column"])
@pytest.mark.parametrize("shape", RAGGED)
def test_r8_ragged_shapes(shape, kernel):
    nx, ny, nz, halo = shape
    for variant in ("specified", "periodic_open"):
        g = cases.grid(nx, ny, nz, halo=halo, variant=variant)
        fin = random_fields64(g, seed=nx + nz, adversarial=(nz == 4))
        want = oracle64(g, fin, SCALARS_3KM)
        got, _ = run_patch64(g, fin, SCALARS_3KM, KERNELS[kernel])
        assert_bit_equal64(got, want, what=f"{shape}/{variant}/{kernel} ")
        assert_outside_untouched64(got, fin, g)


@gpu
@pytest.mark.parametrize("kernel", ["auto", "tile", "column"])
def test_r8_deep_column_nz120(kernel):
    g = cases.grid(200, 96, 120, halo=5, variant="periodic_specified")
    fin = to64(wrf.synth_fields(g, seed=4))
    want = oracle64(g, fin, SCALARS_3KM, tiles=8)
    got, ran = run_patch64(g, fin, SCALARS_3KM, KERNELS[kernel])
    assert_bit_equal64(got, want, what=f"nz120/{kernel} ")
    assert ran == (wrf.KERNEL_TILE if kernel == "auto" else KERNELS[kernel])


@gpu
@pytest.mark.parametrize("kernel", ["tile", "column"])
def test_r8_sub_tile_calls_compose(kernel):
    g = cases.grid(300, 41, 9, halo=3, variant="specified")
    fin = random_fields64(g, seed=5)
    want = oracle64(g, fin, SCALARS_12KM)
    tiles = [(i0, i1, j0, j1) for (i0, i1) in ((1, 130), (131, 131), (132, 300))
             for (j0, j1) in ((1, 1), (2, 20), (21, 41))]
    got, _ = run_patch64(g, fin, SCALARS_12KM, KERNELS[kernel], tiles=tiles)
    assert_bit_equal64(got, want, what=f"tiles/{kernel} ")


@gpu
def test_r8_graph_equals_steps_equals_loop_entry():
    g = cases.grid(140, 50, 12, halo=4, variant="periodic_specified")
    fin = random_fields64(g, seed=8)
    want = oracle_loop64(g, fin, SCALARS_12KM, 6)
    plain, _ = run_patch64(g, fin, SCALARS_12KM, wrf.KERNEL_AUTO, nsteps=6)
    graph, _ = run_patch64(g, fin, SCALARS_12KM, wrf.KERNEL_AUTO, nsteps=6, graph=True)
    assert_bit_equal64(plain, want, what="plain ")
    assert_bit_equal64(graph, want, what="graph ")
    loop = cases.copy_fields(fin)
    wrf.call_with_fields(loop, g, *SCALARS_12KM, nsteps=6)              # wrfb200_advance_mu_t_loop_r8
    assert_bit_equal64(loop, want, what="loop entry ")
    assert_outside_untouched64(loop, fin, g)
    wrf.lib().wrfb200_release_cache()


@gpu
def test_r8_set_scalars_invalidates_the_graph():
    g = cases.grid(96, 40, 10, halo=5, variant="specified")
    fin = random_fields64(g, seed=13)
    other = (SCALARS_12KM[0], SCALARS_12KM[1], F64(7.0), SCALARS_12KM[3])
    want = oracle_loop64(g, fin, SCALARS_12KM, 3)
    want = oracle_loop64(g, want, other, 3)
    got = cases.copy_fields(fin)
    with wrf.Patch(g, dtype=np.float64) as p:
        p.set_scalars(*SCALARS_12KM)
        p.upload(got)
        p.step_graph(3)
        p.set_scalars(*other)
        p.step_graph(3)                                                   # same nsteps: must not replay dts=12
        p.download(got)
    assert_bit_equal64(got, want, what="set_scalars_r8 between graphs ")


@gpu
def test_r8_host_pointer_residency_loop():
    """acoustic_loop_begin/end with float64 host arrays, pinning on, u and v changed on the host between calls."""
    g = cases.grid(425, 300, 35, halo=5, variant="specified")
    fin = random_fields64(g, seed=21)
    c, nsteps = 0.25, 4
    want = oracle_loop64(g, fin, SCALARS_12KM, nsteps, c=c, tiles=64)
    ubox, vbox = cases.standin_boxes(g, g.ids, g.ide, g.jds, g.jde)
    got = cases.copy_fields(fin)
    wrf.lib().wrfb200_set_host_pinning(1)
    try:
        with wrf.acoustic_loop():
            for s in range(nsteps):
                wrf.call_with_fields(got, g, *SCALARS_12KM)
                assert wrf.default_last_kernel() == wrf.KERNEL_TILE
                if s + 1 < nsteps:
                    cases.standin_advance_uv_numpy(got, g, c, ubox, vbox)
        assert_bit_equal64(got, want, names=cases.OUTPUTS + ("u", "v"), what="r8 residency ")
        assert_outside_untouched64(got, fin, g)
    finally:
        wrf.lib().wrfb200_set_host_pinning(0)
        wrf.lib().wrfb200_release_cache()


@gpu
@pytest.mark.parametrize("nx,halo,kernel", [(100, 2, wrf.KERNEL_TILE), (100, 5, wrf.KERNEL_TILE),
                                            (101, 2, wrf.KERNEL_COLUMN)])
def test_r8_device_pointer_call_in_place(nx, halo, kernel, _reset_default_kernel):
    """Dense caller layout: rows of an even number of doubles (WRF's halo-5 layout among them) run the tile kernel
    in place; an odd row length cannot be addressed by 16-byte pairs and takes the column kernel."""
    import torch
    g = cases.grid(nx, 40, 10, halo=halo, variant="specified")
    fin = random_fields64(g, seed=9)
    want = oracle64(g, fin, SCALARS_12KM)
    dev = {n: torch.from_numpy(fin[n]).cuda() for n in wrf.FIELDS}
    wrf.call_with_fields(dev, g, *SCALARS_12KM)
    torch.cuda.synchronize()
    assert wrf.default_last_kernel() == kernel
    got = {n: dev[n].cpu().numpy() for n in wrf.FIELDS}
    assert_bit_equal64(got, want, what=f"device nx={nx} halo={halo} ")
    assert_outside_untouched64(got, fin, g)
    # a forced kernel the layout cannot take fails with a message instead of falling back
    if kernel == wrf.KERNEL_COLUMN:
        wrf.lib().wrfb200_set_default_kernel(wrf.KERNEL_TILE)
        with pytest.raises(wrf.WrfB200Error) as e:
            wrf.call_with_fields(dev, g, *SCALARS_12KM)
        assert e.value.status == _lib.ERR_UNSUPPORTED and "even" in str(e.value)


@gpu
def test_r8_bound_torch_buffers():
    import torch
    g = cases.grid(96, 33, 8, halo=4, variant="open")
    fin = random_fields64(g, seed=10)
    want = oracle64(g, fin, SCALARS_12KM)
    dev = {n: torch.from_numpy(fin[n]).cuda() for n in wrf.FIELDS}
    with wrf.Patch(g, allocate=False, dtype=torch.float64) as p:
        for n in wrf.FIELDS:
            p.bind(n, dev[n])
        assert p.device_ptr("u") == (dev["u"].data_ptr(), g.shape3[-1])
        p.set_scalars(*SCALARS_12KM)
        p.set_stream(torch.cuda.current_stream().cuda_stream)
        p.step()
        p.sync()
        assert p.last_kernel() == wrf.KERNEL_TILE
    got = {n: dev[n].cpu().numpy() for n in wrf.FIELDS}
    assert_bit_equal64(got, want)


@gpu
@pytest.mark.parametrize("kernel", ["tile", "column"])
def test_r8_extreme_operands(kernel):
    g = cases.grid(140, 12, 9, halo=3, variant="open")
    f = random_fields64(g, seed=31)
    rs = np.random.RandomState(5)
    pick = lambda a, frac: rs.uniform(size=a.shape) < frac
    f["u_1"][pick(f["u_1"], 0.2)] = 0.0
    f["u_1"][pick(f["u_1"], 0.1)] = 1e-310                         # binary64 denormal
    f["u_1"][pick(f["u_1"], 0.05)] = 3e290
    f["muu"][pick(f["muu"], 0.1)] = 1e-300
    f["msfuy"][pick(f["msfuy"], 0.1)] = 2.0 ** -900
    f["msfuy"][pick(f["msfuy"], 0.1)] = 1.9999999999999998
    f["msfty"][pick(f["msfty"], 0.2)] = 2.0 ** 600
    f["dnw"][2] = 0.0
    f["dnw"][4] = 1e-315
    with np.errstate(all="ignore"):
        want = oracle64(g, f, SCALARS_3KM)
    got, _ = run_patch64(g, f, SCALARS_3KM, KERNELS[kernel])
    assert_bit_equal64(got, want, what=f"extreme/{kernel} ")


@gpu
def test_r8_precision_of_verbs_and_out_of_scope_verbs():
    lib = wrf.lib()
    g = cases.grid(40, 20, 6, halo=2)
    f32 = cases.random_fields(g, seed=3)
    f64 = to64(f32)
    with wrf.Patch(g, dtype=np.float64) as p8, wrf.Patch(g) as p4:
        h8, h4 = p8._h, p4._h
        d = C.c_void_p()
        pitch = C.c_long()
        # a float verb on a real*8 handle and an r8 verb on a float handle: WRFB200_ERR_STATE naming the precision
        for rc in (lib.wrfb200_set_scalars(h8, 1.0, 1.0, 1.0, 0.1),
                   lib.wrfb200_upload(h8, 0, f32["ww"].ctypes.data),
                   lib.wrfb200_download_range(h8, 0, f32["ww"].ctypes.data, 1, 2, 1, 2, 1, 2),
                   lib.wrfb200_device_ptr(h8, 0, C.byref(d), C.byref(pitch))):
            assert rc == _lib.ERR_STATE and b"real*8" in lib.wrfb200_last_error()
        for rc in (lib.wrfb200_set_scalars_r8(h4, 1.0, 1.0, 1.0, 0.1),
                   lib.wrfb200_upload_r8(h4, 0, f64["ww"].ctypes.data),
                   lib.wrfb200_upload_range_r8(h4, 0, f64["ww"].ctypes.data, 1, 2, 1, 2, 1, 2),
                   lib.wrfb200_bind_device_r8(h4, 0, d, 50)):
            assert rc == _lib.ERR_STATE and b"real*4" in lib.wrfb200_last_error()
        # binary32-only verbs on a real*8 handle: WRFB200_ERR_UNSUPPORTED
        buf = C.c_void_p(p8.device_ptr("ww")[0])
        info = C.create_string_buffer(lib.wrfb200_comm_info_bytes())
        for rc in (lib.wrfb200_comm_init(h8, 1, 1, 0, 1, 40, 1, 20, info),
                   lib.wrfb200_comm_step(h8),
                   lib.wrfb200_pack_halo(h8, 0, wrf.WEST, 1, 1, 40, 1, 20, buf),
                   lib.wrfb200_unpack_halo(h8, 0, wrf.WEST, 1, 1, 40, 1, 20, buf),
                   lib.wrfb200_standin_advance_uv(h8, wrf.FIELD_ID["u"], 0.25, 2, 39, 1, 19),
                   lib.wrfb200_upload_state(h8, None, None, None),
                   lib.wrfb200_set_uv(h8, None, None),
                   lib.wrfb200_upload_constants(h8, *([None] * 17)),
                   lib.wrfb200_download_outputs(h8, 1, 40, 1, 20, 1, 6, *([None] * 7))):
            assert rc == _lib.ERR_UNSUPPORTED and b"binary32 only" in lib.wrfb200_last_error()
        # the pipe kernel is binary32 only
        p8.upload(f64)
        p8.set_scalars(*SCALARS_12KM)
        p8.set_kernel(wrf.KERNEL_PIPE)
        with pytest.raises(wrf.WrfB200Error) as e:
            p8.step()
        assert e.value.status == _lib.ERR_UNSUPPORTED and "binary32" in str(e.value)
        assert p8.launch_count() == 0
    # bad index sets on the r8 entry: the same preconditions as binary32
    bad = g.with_tile(1, 40, 1, 20)
    bad = wrf.Grid(*(bad.index_args()[:15] + (2, bad.kte)), periodic_x=False, specified=True, nested=False)
    with pytest.raises(wrf.WrfB200Error) as e:
        wrf.call_with_fields(cases.copy_fields(f64), bad, *SCALARS_12KM)
    assert e.value.status == _lib.ERR_UNSUPPORTED
    wrf.lib().wrfb200_release_cache()


@gpu
def test_r8_conus12_full_size_bit_exact():
    """425x300x35, one step, every kernel against the binary64 checker on all host cores."""
    g = cases.grid(425, 300, 35, halo=5, variant="specified")
    fin = to64(wrf.synth_fields(g))
    want = oracle64(g, fin, SCALARS_12KM, tiles=64)
    for kernel in ("tile", "column"):
        got, _ = run_patch64(g, fin, SCALARS_12KM, KERNELS[kernel])
        assert_bit_equal64(got, want, what=f"conus12/{kernel} ")
        assert_outside_untouched64(got, fin, g)


@gpu
def test_r8_conus3_full_size_bit_exact():
    """1800x1060x50 (0.78 GB per 3-D field in double): AUTO (the tile kernel) and the column kernel, the whole
    grid of every output compared bit for bit."""
    g = cases.grid(1800, 1060, 50, halo=5, variant="specified")
    fin = to64(wrf.synth_fields(g))
    want = oracle64(g, fin, SCALARS_3KM, tiles=64)
    for kernel in ("auto", "column"):
        got = cases.copy_fields(fin)
        with wrf.Patch(g, dtype=np.float64) as p:
            p.set_scalars(*SCALARS_3KM)
            p.set_kernel(KERNELS[kernel])
            p.upload(got)
            p.step()
            p.download(got)
            assert p.last_kernel() == (wrf.KERNEL_TILE if kernel == "auto" else wrf.KERNEL_COLUMN)
        assert_bit_equal64(got, want, what=f"conus3/{kernel} ")
        del got


# ================================================================ C harness: the Fortran -r8 calling convention
def _build_harness(tmp_path):
    exe = str(tmp_path / "c_abi_harness_r8")
    libdir = os.path.join(ROOT, "wrf_model_cuda_sample_b200")
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    subprocess.run([cc, "-O1", os.path.join(ROOT, "tests", "c_abi_harness_r8.c"), "-I", os.path.join(ROOT, "include"),
                    "-L", libdir, "-lwrfb200", f"-Wl,-rpath,{libdir}", "-o", exe], check=True)
    return exe


def _fnv1a(a):
    h = 1469598103934665603
    for b in a.tobytes():
        h = ((h ^ b) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    return f"{h:016x}"


@pytest.mark.skipif(_have_gpu(), reason="GPU present")
def test_r8_harness_fails_loudly_without_gpu(tmp_path):
    r = subprocess.run([_build_harness(tmp_path)], capture_output=True, text=True)
    assert r.returncode == 3 and "no CPU fallback" in r.stderr


@gpu
def test_r8_harness_matches_checker(tmp_path):
    r = subprocess.run([_build_harness(tmp_path)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = dict(line.split()[1::2] for line in r.stdout.strip().splitlines())
    g = wrf.Grid(1, 40, 1, 30, 12, -2, 43, -2, 33, 1, 12, 1, 40, 1, 30, 1, 12, False, True, False)
    f = to64(wrf.synth_fields(g))
    for n in wrf.FIELDS:                     # the harness's widening: x * (1 + 2^-40) fills the low mantissa bits
        f[n] = f[n] * (1.0 + 2.0 ** -40)
    r8_checkers.oracle_c_r8(f, g, (1.0 / 12000.0, 1.0 / 12000.0, 12.0, 0.1))
    for name in cases.OUTPUTS:
        assert got[str(wrf.FIELD_ID[name])] == _fnv1a(f[name]), name
