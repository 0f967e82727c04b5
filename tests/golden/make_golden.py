"""Generate (or --check) the golden vectors in tests/golden/.

The reference ships no golden data (its .bin dumps live in an un-shipped /data2 directory,
advance_mu_t_driver.f90:36), so the vectors are OUTPUTS OF THE REFERENCE ITSELF: its advance_mu_t.c,
unmodified, compiled in place by oracle/Makefile into oracle/_ref/libref_advance_mu_t.so, executed on seeded
numpy inputs.  The reference sources are not part of this repository; these files are.

    python tests/golden/make_golden.py          # regenerate (needs oracle/_ref: make -C oracle REF=<reference checkout>)
    python tests/golden/make_golden.py --check  # verify the committed files against a fresh run
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from oracle import loader  # noqa: E402
from tests import cases  # noqa: E402

# name -> (nx, ny, nz, halo, variant, seed, adversarial, tile or None, scalars)
CASES = {
    "g20x16x10_specified": (20, 16, 10, 2, "specified", 101, False, None, cases.SCALARS_12KM),
    "g20x16x10_periodic_specified": (20, 16, 10, 2, "periodic_specified", 102, False, None, cases.SCALARS_12KM),
    "g20x16x10_open": (20, 16, 10, 2, "open", 103, False, None, cases.SCALARS_12KM),
    "g20x16x10_nested": (20, 16, 10, 2, "nested", 104, False, None, cases.SCALARS_3KM),
    "g37x11x7_adversarial": (37, 11, 7, 1, "specified", 105, True, None, cases.SCALARS_12KM),
    "g33x19x13_tile": (33, 19, 13, 3, "specified", 106, False, (9, 27, 4, 15), cases.SCALARS_3KM),
    "g9x8x31_deep": (9, 8, 31, 1, "periodic_specified", 107, False, None, cases.SCALARS_3KM),
}


def build(name):
    nx, ny, nz, halo, variant, seed, adv, tile, scalars = CASES[name]
    g = cases.grid(nx, ny, nz, halo=halo, variant=variant)
    if tile is not None:
        g = g.with_tile(*tile)
    fin = cases.random_fields(g, seed, adversarial=adv)
    fout = cases.copy_fields(fin)
    loader.reference_c(fout, g, scalars)
    return g, scalars, fin, fout


def path(name):
    return os.path.join(cases.GOLDEN_DIR, name + ".npz")


def save(name):
    g, scalars, fin, fout = build(name)
    payload = {"in_" + k: v for k, v in fin.items()}
    payload.update({"out_" + k: fout[k] for k in cases.OUTPUTS})
    payload["index_args"] = np.array(g.index_args(), dtype=np.int32)
    payload["flags"] = np.array([g.periodic_x, g.specified, g.nested], dtype=np.int32)
    payload["scalars"] = np.array(scalars, dtype=np.float32)
    np.savez_compressed(path(name), **payload)


def load(name):
    """-> (grid, scalars, inputs, reference outputs) from the committed file."""
    z = np.load(path(name))
    ia = [int(x) for x in z["index_args"]]
    fl = [bool(x) for x in z["flags"]]
    from wrf_model_cuda_sample_b200 import Grid
    g = Grid(*ia, periodic_x=fl[0], specified=fl[1], nested=fl[2])
    fin = {k[3:]: z[k] for k in z.files if k.startswith("in_")}
    fout = {k[4:]: z[k] for k in z.files if k.startswith("out_")}
    return g, tuple(np.float32(x) for x in z["scalars"]), fin, fout


if __name__ == "__main__":
    if "--check" in sys.argv:
        for name in CASES:
            g, scalars, fin, fout = build(name)
            g2, s2, fin2, fout2 = load(name)
            assert g == g2 and all(a == b for a, b in zip(scalars, s2))
            for k in fin:
                assert np.array_equal(cases.bits(fin[k]), cases.bits(fin2[k])), (name, k)
            cases.assert_bit_equal(fout2, fout, what=name + " ")
        print("golden vectors match a fresh run of the reference C")
    else:
        for name in CASES:
            save(name)
            print("wrote", path(name), os.path.getsize(path(name)), "bytes")
