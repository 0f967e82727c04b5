"""Domain caches: host-array and device-pointer calls keep the device state of several domains per thread, so a nested
run that alternates parent and nest stops rebuilding its cache at every switch.  Without a GPU: the new query, its
constants and its errors.  On the GPU: every result bit-identical to the oracle with the cells outside the written
range untouched, for domains called alternately in binary32 and real*8, on pageable and page-locked arrays, through
both entry points, split over devices and with device pointers; acoustic-loop residency kept per domain; the bound on
the number of domains; and wrfb200_release_cache handing the memory back."""
import ctypes as C
import os
import re
import threading

import numpy as np
import pytest

import wrf_model_cuda_sample_b200 as wrf
from wrf_model_cuda_sample_b200 import _lib
from oracle import loader
from tests import cases
from tests.test_r8 import (SCALARS_12KM as SCALARS_12KM_64, assert_bit_equal64, assert_outside_untouched64, oracle64,
                           oracle_loop64, random_fields64)
from tests.test_shared_tiles import _mirror_bytes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu

MAX_DOMAINS = 8          # domains a thread keeps per precision (include/wrfb200.h, "Domain caches")

# A parent, a nest, and a nest with vertical refinement (another kde): three memory shapes.  The parent's padded
# mirror is slab-pipelined (staging buffer and re-pitch); the nests take one slab.
PARENT = cases.grid(425, 300, 35, halo=5, variant="specified")
NEST = cases.grid(301, 241, 35, halo=5, variant="nested")
NEST_DEEP = cases.grid(181, 151, 44, halo=5, variant="nested")
DOMAINS = {"parent": PARENT, "nest": NEST, "nest_deep": NEST_DEEP}
# A B A B A, then the deeper nest joins: only a domain's first call creates anything
SEQUENCE = ["parent", "nest", "parent", "nest", "parent", "nest_deep", "nest", "nest_deep", "parent"]


def _have_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


@pytest.fixture(autouse=True)
def _release_around():
    """Each test starts from empty caches (earlier modules may have left domains behind) and leaves none."""
    if _have_gpu():
        wrf.lib().wrfb200_release_cache()
    yield
    if _have_gpu():
        wrf.set_default_devices(None)
        wrf.lib().wrfb200_release_cache()


def _expected_states(sequence):
    seen, out = set(), []
    for d in sequence:
        out.append(wrf.CACHE_REUSED if d in seen else wrf.CACHE_CREATED)
        seen.add(d)
    return out


# ================================================================ CPU
def test_python_api_is_exported():
    assert callable(wrf.default_last_cache) and "default_last_cache" in wrf.__all__
    for n in ("CACHE_REUSED", "CACHE_CREATED", "CACHE_EVICTED"):
        assert n in wrf.__all__


def test_cache_constants_match_header():
    text = open(os.path.join(ROOT, "include", "wrfb200.h")).read()
    body = text[text.index("typedef enum wrfb200_cache"):text.index("} wrfb200_cache;")]
    values = dict((k, int(v)) for k, v in re.findall(r"WRFB200_(CACHE_[A-Z]+)\s*=\s*(\d+)", body))
    assert values == {"CACHE_REUSED": wrf.CACHE_REUSED, "CACHE_CREATED": wrf.CACHE_CREATED,
                      "CACHE_EVICTED": wrf.CACHE_EVICTED}
    assert (wrf.CACHE_REUSED, wrf.CACHE_CREATED, wrf.CACHE_EVICTED) == (0, 1, 2)


def test_bounce_allocation_count_needs_no_gpu():
    n = C.c_long(-1)
    assert wrf.lib().wrfb200_bounce_allocations(C.byref(n)) == _lib.OK and n.value >= 0
    assert wrf.lib().wrfb200_bounce_allocations(None) == _lib.ERR_INVALID_ARG


def test_no_call_yet_is_a_state_error():
    """Thread-local: a thread that has made no call has no cache decision to report."""
    out = {}

    def body():
        r = C.c_int(-7)
        out["rc"] = wrf.lib().wrfb200_default_last_cache(C.byref(r))
        out["state"] = r.value
        out["msg"] = wrf.lib().wrfb200_last_error()

    t = threading.Thread(target=body)
    t.start()
    t.join()
    assert out["rc"] == _lib.ERR_STATE and out["state"] == -7 and b"no advance_mu_t call" in out["msg"]
    assert wrf.lib().wrfb200_default_last_cache(None) == _lib.ERR_INVALID_ARG


# ================================================================ GPU helpers
_FIELDS = {}


def _inputs(name, r8):
    """The domain's inputs (made once per module run)."""
    key = (name, r8)
    if key not in _FIELDS:
        g = DOMAINS[name]
        seed = g.ide + g.kde
        _FIELDS[key] = random_fields64(g, seed=seed) if r8 else wrf.synth_fields(g, seed=seed)
    return _FIELDS[key]


def _want(g, fin, r8, nsteps):
    if r8:
        return oracle64(g, fin, SCALARS_12KM_64) if nsteps == 1 else oracle_loop64(g, fin, SCALARS_12KM_64, nsteps)
    if nsteps == 1:
        want = cases.copy_fields(fin)
        loader.oracle_c(want, g, cases.SCALARS_12KM)
        return want
    return cases.oracle_loop(g, fin, cases.SCALARS_12KM, nsteps)


def _pinned_like(fin):
    """Page-locked copies of fin (views of pinned torch tensors, kept alive in the returned list)."""
    import torch
    keep, out = [], {}
    for n, a in fin.items():
        t = torch.empty(a.shape, dtype=torch.float64 if a.dtype == np.float64 else torch.float32, pin_memory=True)
        keep.append(t)
        out[n] = t.numpy()
        out[n][...] = a
    return out, keep


def _check(got, want, fin, g, r8, what):
    if r8:
        assert_bit_equal64(got, want, what=what)
        assert_outside_untouched64(got, fin, g)
    else:
        cases.assert_bit_equal(got, want, what=what)
        cases.assert_outside_untouched(got, fin, g)


# ================================================================ GPU: alternating domains
@gpu
@pytest.mark.parametrize("nsteps", [1, 3], ids=["advance_mu_t", "loop"])
@pytest.mark.parametrize("memory", ["pageable", "pinned"])
@pytest.mark.parametrize("r8", [False, True], ids=["binary32", "real8"])
def test_alternating_domains(r8, memory, nsteps):
    scalars = SCALARS_12KM_64 if r8 else cases.SCALARS_12KM
    want = {d: _want(DOMAINS[d], _inputs(d, r8), r8, nsteps) for d in DOMAINS}
    pinned, keep = {}, []
    if memory == "pinned":
        for d in DOMAINS:
            pinned[d], k = _pinned_like(_inputs(d, r8))
            keep += k
    states = []
    for x, d in enumerate(SEQUENCE):
        g, fin = DOMAINS[d], _inputs(d, r8)
        if memory == "pinned":
            got = pinned[d]                          # the same page-locked arrays at every call of the domain
            for n in wrf.FIELDS:
                got[n][...] = fin[n]
        else:
            got = cases.copy_fields(fin)             # new arrays, new addresses, at every call
        wrf.call_with_fields(got, g, *scalars, nsteps=nsteps)
        states.append(wrf.default_last_cache())
        assert wrf.default_last_transfer() == (wrf.TRANSFER_DIRECT if memory == "pinned" else wrf.TRANSFER_STAGED)
        _check(got, want[d], fin, g, r8, f"call {x} ({d}) ")
    assert states == _expected_states(SEQUENCE), states
    del keep


# ================================================================ GPU: residency per domain
def _loop(got, g, scalars, nsteps, c):
    """One acoustic loop of the domain: ft (a loop constant) changed on the host after the priming call, which the
    loop's later calls must ignore and the next loop's first call must pick up; u, v changed between steps."""
    ubox, vbox = cases.standin_boxes(g, g.ids, g.ide, g.jds, g.jde)
    with wrf.acoustic_loop():
        for s in range(nsteps):
            wrf.call_with_fields(got, g, *scalars)
            if s == 0:
                got["ft"] += got["ft"].dtype.type(1.0)
            if s + 1 < nsteps:
                cases.standin_advance_uv_numpy(got, g, c, ubox, vbox)


@gpu
@pytest.mark.parametrize("r8", [False, True], ids=["binary32", "real8"])
def test_residency_per_domain(r8):
    """begin, parent loop, end; begin, nest loop, end; begin, parent loop, end: the nest's loop between the parent's
    two loops must not let the parent's second loop skip its first full upload."""
    scalars = SCALARS_12KM_64 if r8 else cases.SCALARS_12KM
    c, nsteps = 0.25, 4
    state = {d: cases.copy_fields(_inputs(d, r8)) for d in ("parent", "nest")}
    for x, d in enumerate(["parent", "nest", "parent", "nest"]):
        g, got = DOMAINS[d], state[d]
        start = cases.copy_fields(got)               # the host state the loop starts from, poked ft included
        if r8:
            want = oracle_loop64(g, start, scalars, nsteps, c=c)
        else:
            want = cases.oracle_loop(g, start, scalars, nsteps, c=c)
        _loop(got, g, scalars, nsteps, c)
        names = cases.OUTPUTS + ("u", "v")
        if r8:
            assert_bit_equal64(got, want, names=names, what=f"loop {x} ({d}) ")
            assert_outside_untouched64(got, start, g)
        else:
            cases.assert_bit_equal(got, want, names=names, what=f"loop {x} ({d}) ")
            cases.assert_outside_untouched(got, start, g)


# ================================================================ GPU: split calls
@gpu
def test_split_call_alternating_domains():
    sequence = ["parent", "nest", "parent", "nest"]
    want = {d: _want(DOMAINS[d], _inputs(d, False), False, 1) for d in ("parent", "nest")}
    states = []
    with wrf.default_devices([0, 0]):
        for x, d in enumerate(sequence):
            g, fin = DOMAINS[d], _inputs(d, False)
            got = cases.copy_fields(fin)
            wrf.call_with_fields(got, g, *cases.SCALARS_12KM)
            states.append(wrf.default_last_cache())
            _check(got, want[d], fin, g, False, f"split call {x} ({d}) ")
    assert states == _expected_states(sequence), states


def _bounce_allocations():
    n = C.c_long(-1)
    assert wrf.lib().wrfb200_bounce_allocations(C.byref(n)) == _lib.OK
    return n.value


def _bounce_sizes(g, esize=4):
    """(upload buffer bytes, 2-D buffer bytes) a whole-domain call of g asks for (the slab rule of
    run_host_compat_body)."""
    i0, i1, j0, j1, k0, k1 = g.bounds()
    nj = j1 - j0 + 1
    idim, jdim, kdim = g.ime - g.ims + 1, g.jme - g.jms + 1, g.kme - g.kms + 1
    nslab = min(nj // 16, 16) if idim * kdim * jdim * esize >= 16 << 20 and nj >= 32 else 1
    rows = nj // nslab + 3
    return rows * kdim * idim * esize, rows * idim * esize


@gpu
def test_bounce_buffers_are_not_reallocated_across_switches():
    """Two domains, each needing more of one of the two bounce sizes (the deeper nest: larger 3-D slabs, narrower
    rows).  The buffers grow to both maxima once; switching back and forth then allocates no pinned memory."""
    wide, deep = PARENT, cases.grid(401, 281, 60, halo=5, variant="nested")
    (w3, w2), (d3, d2) = _bounce_sizes(wide), _bounce_sizes(deep)
    assert w2 > d2 and d3 > w3, "the premise: each domain dominates one size"
    grids = {"wide": wide, "deep": deep}
    fins = {"wide": _inputs("parent", False), "deep": cases.random_fields(deep, seed=11)}
    wants = {d: _want(grids[d], fins[d], False, 1) for d in grids}
    sequence = ["wide", "deep", "wide", "deep", "wide", "deep"]
    for x, d in enumerate(sequence):
        if x == 2:
            grown = _bounce_allocations()
        got = cases.copy_fields(fins[d])
        wrf.call_with_fields(got, grids[d], *cases.SCALARS_12KM)
        assert wrf.default_last_transfer() == wrf.TRANSFER_STAGED
        _check(got, wants[d], fins[d], grids[d], False, f"call {x} ({d}) ")
    assert _bounce_allocations() == grown


def _split_alternation(devices):
    """A whole domain and a thin one (one computed row: only the last part of the list has rows) in turn, split over
    `devices`; returns the bounce allocations made after the first two calls."""
    thin = cases.grid(40, 4, 8, halo=3)
    grids = {"parent": PARENT, "thin": thin}
    fins = {"parent": _inputs("parent", False), "thin": cases.random_fields(thin, seed=12)}
    wants = {d: _want(grids[d], fins[d], False, 1) for d in grids}
    plan = wrf.host_split_plan(thin, len(devices))
    assert [r[0] <= r[1] for r in plan] == [False] * (len(devices) - 1) + [True]
    sequence = ["parent", "thin", "parent", "thin", "parent"]
    states = []
    with wrf.default_devices(devices):
        for x, d in enumerate(sequence):
            if x == 2:
                before = _bounce_allocations()
            got = cases.copy_fields(fins[d])
            wrf.call_with_fields(got, grids[d], *cases.SCALARS_12KM)
            states.append(wrf.default_last_cache())
            _check(got, wants[d], fins[d], grids[d], False, f"split over {devices}, call {x} ({d}) ")
    assert states == _expected_states(sequence), states
    return _bounce_allocations() - before


@gpu
def test_split_call_with_unused_parts():
    """Parts without rows are skipped, and each part keeps its own cache all the same."""
    assert _split_alternation([0, 0]) == 0


@gpu
def test_split_call_with_unused_parts_keeps_each_cache_on_its_device():
    """The thin domain runs on the second device only.  Its part must use that device's cache: the first part's
    cache (device 0) would have to move its lanes and reallocate its bounce buffers at every switch."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip(f"{torch.cuda.device_count()} GPU(s) on this box, 2 needed")
    assert _split_alternation([0, 1]) == 0


# ================================================================ GPU: device pointers
@gpu
def test_device_pointer_calls_alternating_domains():
    import torch
    sequence = ["parent", "nest", "parent", "nest", "parent"]
    want = {d: _want(DOMAINS[d], _inputs(d, False), False, 1) for d in ("parent", "nest")}
    dev = {d: {n: torch.from_numpy(_inputs(d, False)[n]).cuda() for n in wrf.FIELDS} for d in ("parent", "nest")}
    states = []
    for x, d in enumerate(sequence):
        g, fin = DOMAINS[d], _inputs(d, False)
        for n in wrf.FIELDS:
            dev[d][n].copy_(torch.from_numpy(fin[n]))
        wrf.call_with_fields(dev[d], g, *cases.SCALARS_12KM)
        states.append(wrf.default_last_cache())
        torch.cuda.synchronize()
        got = {n: dev[d][n].cpu().numpy() for n in wrf.FIELDS}
        _check(got, want[d], fin, g, False, f"device call {x} ({d}) ")
    assert states == _expected_states(sequence), states


# ================================================================ GPU: the bound on the number of domains
@gpu
def test_one_domain_more_than_the_limit():
    """MAX_DOMAINS + 1 domains in a cycle: the least recently used one is freed for the newest and re-created when
    its turn comes; the most recent MAX_DOMAINS stay."""
    grids = [cases.grid(40 + 4 * d, 30 + d, 8 + d, halo=3, variant="specified") for d in range(MAX_DOMAINS + 1)]
    fins = [cases.random_fields(g, seed=70 + d) for d, g in enumerate(grids)]
    wants = []
    for g, fin in zip(grids, fins):
        w = cases.copy_fields(fin)
        loader.oracle_c(w, g, cases.SCALARS_12KM)
        wants.append(w)
    n = MAX_DOMAINS
    # first pass: n created, the (n+1)th evicts domain 0; then domain n and 1 are still there, 0 and 2 are not
    sequence = list(range(n + 1)) + [n, 1, 0, 2]
    expected = [wrf.CACHE_CREATED] * n + [wrf.CACHE_EVICTED] + [wrf.CACHE_REUSED, wrf.CACHE_REUSED,
                                                                 wrf.CACHE_EVICTED, wrf.CACHE_EVICTED]
    states = []
    for x, d in enumerate(sequence):
        got = cases.copy_fields(fins[d])
        wrf.call_with_fields(got, grids[d], *cases.SCALARS_12KM)
        states.append(wrf.default_last_cache())
        _check(got, wants[d], fins[d], grids[d], False, f"call {x} (domain {d}) ")
    assert states == expected, states


# ================================================================ GPU: release
@gpu
def test_release_cache_frees_every_domain():
    import torch
    grids = [cases.grid(1000, 800, 40, halo=5), cases.grid(800, 700, 40, halo=5, variant="nested"),
             cases.grid(600, 500, 60, halo=5, variant="nested")]
    mirrors = sum(_mirror_bytes(g) for g in grids)
    for g in grids:
        fin = wrf.synth_fields(g, seed=g.ide)
        wrf.call_with_fields(fin, g, *cases.SCALARS_12KM)
        assert wrf.default_last_cache() == wrf.CACHE_CREATED
    for g in grids:                                  # all three retained
        wrf.call_with_fields(wrf.synth_fields(g, seed=g.ide), g, *cases.SCALARS_12KM)
        assert wrf.default_last_cache() == wrf.CACHE_REUSED
    torch.cuda.synchronize()
    before = torch.cuda.mem_get_info()[0]
    assert wrf.lib().wrfb200_release_cache() == _lib.OK
    after = torch.cuda.mem_get_info()[0]
    assert after - before >= mirrors, (after - before, mirrors)
    g = grids[0]
    wrf.call_with_fields(wrf.synth_fields(g, seed=g.ide), g, *cases.SCALARS_12KM)
    assert wrf.default_last_cache() == wrf.CACHE_CREATED
