"""The epoch-flag protocol model of tests/test_flag_protocol_model.py on periodic (torus) process grids: the
exchange of csrc/comm.cu with wrap_x and wrap_y.  Neighbours are cyclic, so a rank can be its own neighbour (px = 1 /
py = 1) or have the same neighbour on both sides of an axis (px = 2 / py = 2).

A self side has no flag: its u / v edge is copied by a push kernel that runs before the step, and its outputs are
stores into the rank's own ring, read by later kernels only -- stream order serves it, so no flag wait ever depends
on a block of the same launch.  The model must stay safe (no halo read before its value arrives, none overwritten
before it is read) and live (no deadlock) under random interleavings and, for two ranks, under every interleaving."""
import random

import pytest

import tests.test_flag_protocol_model as fpm

W, E, S, N = fpm.W, fpm.E, fpm.S, fpm.N
BACK = {E: W, N: S}


def torus(px, py, nsteps, standin):
    ranks = [fpm.Rank(r, px, py) for r in range(px * py)]
    for rk in ranks:
        pi, pj = rk.pi, rk.pj
        rk.nbr = {W: pj * px + (pi - 1) % px, E: pj * px + (pi + 1) % px,
                  S: ((pj - 1) % py) * px + pi, N: ((pj + 1) % py) * px + pi}
        rk.self = {s: rk.nbr[s] == rk.r for s in rk.nbr}
        for n in range(1, nsteps + 1):
            if standin and n > 1:
                rk.kernels.append([("standin", n)])
            # push_kernel: the u west edge (to a neighbour or to myself) and, on a self south side, the v south edge
            rk.kernels.append([("push", n)])
            groups = [("interior", n), ("east_col", n), ("north_row", n)]
            if not rk.self[S]:
                groups.append(("south_row", n))      # fused v push into the south neighbour
            rk.kernels.append(groups)
    return ranks


def enabled(ranks, rk, ev, guard_wrapped_push=True):
    kind, n = ev
    if kind == "interior":
        return True
    if kind == "standin":
        return all(rk.out_from[s] >= n - 1 for s in (W, S) if not rk.self[s])
    if kind == "push":
        if rk.self[W] or (not guard_wrapped_push and rk.pi == 0):
            return True
        return rk.out_from[W] >= n - 1
    if kind == "south_row":
        return rk.out_from[S] >= n - 1
    if kind == "east_col":
        return rk.self[E] or rk.uv_from[E] >= n
    if kind == "north_row":
        return rk.self[N] or rk.uv_from[N] >= n
    raise AssertionError(kind)


def execute(ranks, rk, ev):
    kind, n = ev
    if kind == "standin":
        for s in (W, S):
            assert rk.out_halo[s] == n - 1, f"rank {rk.r}: stand-in of step {n} read mudf halo of step {rk.out_halo[s]}"
    elif kind == "push":
        w = ranks[rk.nbr[W]]
        assert w.uv_halo[E] == n - 1, f"u halo of rank {w.r} overwritten out of order"
        w.uv_halo[E] = n
        if not rk.self[W]:
            w.uv_from[E] = n
        if rk.self[S]:
            assert rk.uv_halo[N] == n - 1
            rk.uv_halo[N] = n
    elif kind == "south_row":
        s = ranks[rk.nbr[S]]
        assert s.uv_halo[N] == n - 1, f"v halo of rank {s.r} overwritten out of order"
        s.uv_halo[N] = n
        s.uv_from[N] = n
    elif kind in ("east_col", "north_row"):
        side = E if kind == "east_col" else N
        assert rk.uv_halo[side] == n, f"rank {rk.r}: step {n} read the {side} halo of step {rk.uv_halo[side]}"
        nb = ranks[rk.nbr[side]]
        assert nb.out_halo[BACK[side]] == n - 1
        nb.out_halo[BACK[side]] = n
        if not rk.self[side]:
            nb.out_from[BACK[side]] = n


def frontier(ranks, guard=True):
    return [(rk, ev) for rk in ranks if rk.pos < len(rk.kernels)
            for ev in rk.kernels[rk.pos] if enabled(ranks, rk, ev, guard)]


def step(ranks, rk, ev):
    execute(ranks, rk, ev)
    rk.kernels[rk.pos].remove(ev)
    if not rk.kernels[rk.pos]:
        rk.pos += 1


def state(ranks):
    return tuple((rk.pos, tuple(sorted(rk.kernels[rk.pos])) if rk.pos < len(rk.kernels) else (),
                  tuple(sorted(rk.uv_from.items())), tuple(sorted(rk.out_from.items())),
                  tuple(sorted(rk.uv_halo.items())), tuple(sorted(rk.out_halo.items()))) for rk in ranks)


TORI = [(1, 1), (1, 2), (2, 1), (2, 2), (1, 3), (3, 1), (2, 4)]


@pytest.mark.parametrize("px,py", TORI)
@pytest.mark.parametrize("standin", [False, True])
def test_torus_random_interleavings_are_safe_and_live(px, py, standin):
    rng = random.Random(1000 * px + 10 * py + standin)
    for _ in range(150):
        ranks = torus(px, py, nsteps=5, standin=standin)
        favourite = rng.randrange(px * py) if rng.random() < 0.5 else None
        while not fpm.finished(ranks):
            f = frontier(ranks)
            assert f, "deadlock: no block group can make progress"
            fav = [x for x in f if x[0].r == favourite]
            rk, ev = rng.choice(fav) if fav and rng.random() < 0.8 else rng.choice(f)
            step(ranks, rk, ev)


@pytest.mark.parametrize("px,py", [(1, 2), (2, 1)])
def test_two_rank_torus_exhaustively(px, py):
    """Every reachable state of two ranks over three steps with the stand-in: every transition safe, no dead end."""
    import copy
    seen = set()
    todo = [torus(px, py, nsteps=3, standin=True)]
    while todo:
        ranks = todo.pop()
        key = state(ranks)
        if key in seen:
            continue
        seen.add(key)
        if fpm.finished(ranks):
            continue
        f = frontier(ranks)
        assert f, "deadlock"
        for idx in range(len(f)):
            clone = copy.deepcopy(ranks)
            g = frontier(clone)
            step(clone, g[idx][0], g[idx][1])
            todo.append(clone)
    assert len(seen) > 100


def test_the_model_catches_a_missing_guard_on_a_wrapped_edge():
    """Drop the write-after-read wait of the u push that crosses the domain edge and some schedule must fail."""
    rng = random.Random(7)
    failed = False
    for _ in range(300):
        ranks = torus(3, 1, nsteps=4, standin=False)
        try:
            while not fpm.finished(ranks):
                f = frontier(ranks, guard=False)
                if not f:
                    failed = True
                    break
                rk, ev = rng.choice(f)
                step(ranks, rk, ev)
        except AssertionError:
            failed = True
        if failed:
            break
    assert failed, "the model did not notice a missing write-after-read guard on the wrapped edge"
