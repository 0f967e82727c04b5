"""The oracle is pinned before it is trusted (not gpu):
  1. against the committed golden vectors = outputs of the reference's own advance_mu_t.c (tests/golden/),
  2. against that reference C executed live when oracle/_ref is built (`make -C oracle REF=<reference checkout>`),
  3. C restatement == numpy restatement, single call == j-tiled calls,
  4. in/out contract: inputs untouched, cells outside the index sets untouched, empty tiles legal.
"""
import numpy as np
import pytest

from oracle import loader
from tests import cases
from tests.golden import make_golden

needs_ref = pytest.mark.skipif(not loader.have_ref(), reason="oracle/_ref not built (needs REF=<reference checkout>)")


@pytest.mark.parametrize("name", sorted(make_golden.CASES))
def test_oracle_c_matches_golden(name):
    g, scalars, fin, want = make_golden.load(name)
    got = cases.copy_fields(fin)
    loader.oracle_c(got, g, scalars)
    cases.assert_bit_equal(got, want, what=name + " ")
    cases.assert_inputs_untouched(got, fin)
    cases.assert_outside_untouched(got, fin, g)


@pytest.mark.parametrize("name", sorted(make_golden.CASES))
def test_oracle_numpy_matches_golden(name):
    g, scalars, fin, want = make_golden.load(name)
    got = cases.copy_fields(fin)
    loader.oracle_numpy(got, g, scalars)
    cases.assert_bit_equal(got, want, what=name + " ")
    cases.assert_outside_untouched(got, fin, g)


@needs_ref
@pytest.mark.parametrize("variant", sorted(cases.FLAG_VARIANTS))
@pytest.mark.parametrize("shape", [(74, 61, 28, 5), (20, 16, 10, 1), (45, 7, 120, 2), (6, 5, 3, 1)])
def test_oracle_c_matches_live_reference(shape, variant):
    nx, ny, nz, halo = shape
    g = cases.grid(nx, ny, nz, halo=halo, variant=variant)
    fin = cases.random_fields(g, seed=nx * 1000 + nz)
    want, got = cases.copy_fields(fin), cases.copy_fields(fin)
    loader.reference_c(want, g, cases.SCALARS_12KM)
    loader.oracle_c(got, g, cases.SCALARS_12KM)
    cases.assert_bit_equal(got, want, what=f"{shape} {variant} ")
    cases.assert_inputs_untouched(got, fin)


@needs_ref
def test_oracle_c_matches_live_reference_on_synthetic_fields():
    import wrf_model_cuda_sample_b200 as wrf
    g = cases.grid(74, 61, 28, halo=5, variant="specified")      # the driver-equivalent tiny domain
    fin = wrf.synth_fields(g)
    want, got = cases.copy_fields(fin), cases.copy_fields(fin)
    loader.reference_c(want, g, cases.SCALARS_12KM)
    loader.oracle_c(got, g, cases.SCALARS_12KM)
    cases.assert_bit_equal(got, want)
    n3, n2 = g.updated_points()
    assert wrf.compare(got["t"], fin["t"])["n_different"] > 0.99 * n3   # the step really changed t


@needs_ref
def test_reference_tiled_equals_single_call():
    g = cases.grid(50, 40, 12, halo=2, variant="specified")
    fin = cases.random_fields(g, seed=7)
    a, b = cases.copy_fields(fin), cases.copy_fields(fin)
    loader.reference_c(a, g, cases.SCALARS_3KM)
    loader.reference_c(b, g, cases.SCALARS_3KM, tiles=7)
    cases.assert_bit_equal(b, a)


@pytest.mark.parametrize("tiles", [1, 3, 16, 1000])
def test_oracle_tiled_equals_single_call(tiles):
    g = cases.grid(31, 16, 9, halo=1, variant="periodic_specified")
    fin = cases.random_fields(g, seed=11)
    a, b = cases.copy_fields(fin), cases.copy_fields(fin)
    loader.oracle_c(a, g, cases.SCALARS_12KM)
    loader.oracle_c(b, g, cases.SCALARS_12KM, tiles=tiles)
    cases.assert_bit_equal(b, a)


@pytest.mark.parametrize("variant", sorted(cases.FLAG_VARIANTS))
def test_oracle_numpy_equals_c(variant):
    g = cases.grid(23, 17, 15, halo=2, variant=variant)
    fin = cases.random_fields(g, seed=23, adversarial=(variant == "open"))
    a, b = cases.copy_fields(fin), cases.copy_fields(fin)
    loader.oracle_c(a, g, cases.SCALARS_3KM)
    loader.oracle_numpy(b, g, cases.SCALARS_3KM)
    cases.assert_bit_equal(b, a)


def test_sub_tile_calls_compose():
    """Calling the routine per (i,j) tile, as WRF does, equals one call over the union."""
    g = cases.grid(40, 30, 8, halo=3, variant="specified")
    fin = cases.random_fields(g, seed=5)
    whole, parts = cases.copy_fields(fin), cases.copy_fields(fin)
    loader.oracle_c(whole, g, cases.SCALARS_12KM)
    for (i0, i1) in ((1, 13), (14, 14), (15, 40)):
        for (j0, j1) in ((1, 1), (2, 17), (18, 30)):
            loader.oracle_c(parts, g.with_tile(i0, i1, j0, j1), cases.SCALARS_12KM)
    cases.assert_bit_equal(parts, whole)


def test_empty_index_sets_are_legal_and_write_nothing():
    g = cases.grid(3, 3, 4, halo=1, variant="specified")      # i_start=2 > i_end=1
    fin = cases.random_fields(g, seed=3)
    got = cases.copy_fields(fin)
    loader.oracle_c(got, g, cases.SCALARS_12KM)
    for n in fin:
        assert np.array_equal(cases.bits(got[n]), cases.bits(fin[n]))


def test_index_sets_table():
    """The three rows of the bounds table (module_small_step_em.f90:91-106)."""
    from oracle import oracle_np
    args = dict(ids=1, ide=50, jds=1, jde=40, its=1, ite=50, jts=1, jte=40, kts=1, kte=20)
    assert oracle_np.bounds(False, True, False, **args) == (2, 48, 2, 38, 1, 19)
    assert oracle_np.bounds(True, True, False, **args) == (1, 49, 2, 38, 1, 19)
    assert oracle_np.bounds(False, False, False, **args) == (1, 49, 1, 39, 1, 19)
    assert oracle_np.bounds(False, False, True, **args) == (2, 48, 2, 38, 1, 19)
    assert oracle_np.bounds(True, False, True, **args) == (1, 49, 2, 38, 1, 19)
    inner = dict(ids=1, ide=50, jds=1, jde=40, its=10, ite=20, jts=5, jte=9, kts=1, kte=20)
    assert oracle_np.bounds(False, True, False, **inner) == (10, 20, 5, 9, 1, 19)


def test_numpy_input_generator_matches_the_c_generator():
    """oracle/synth_np.py builds the reference arm's inputs without loading the product library; it must
    produce the same fields as wrfb200_synth_field (same workload on both arms)."""
    import numpy as np
    import wrf_model_cuda_sample_b200 as wrf
    from oracle import synth_np
    for g in (wrf.Grid.from_shape(130, 50, 12, halo=5), wrf.Grid.from_shape(37, 21, 9, halo=2, periodic_x=True)):
        a = wrf.synth_fields(g, seed=7)
        b = synth_np.synth_fields(g, seed=7)
        for n in wrf.FIELDS:
            x, y = a[n].view(np.uint32), b[n].view(np.uint32)
            # libm's sin/cos may differ from numpy's in the last ulp of a double, which almost never
            # survives the rounding to float32
            assert np.count_nonzero(x != y) <= x.size // 100000, n
            assert np.allclose(a[n], b[n], rtol=1e-6, atol=0)
        assert synth_np.bounds(g) == g.bounds()
        assert synth_np.updated_points(g) == g.updated_points()
