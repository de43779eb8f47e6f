"""The schedule of the unsplit tensor-core candidate pass (tc::sched_bound, the function every CTA evaluates at kernel
start), checked on the CPU through the library's debug export: for every item count in (grid, 8 grid] the pieces cover
each (item, reference tile) exactly once, a tail waits only on a lower ticket whose head ends (in model cost) before the
tail starts, and no CTA's modelled cost exceeds the even share T by more than one tile."""
import ctypes as C

import numpy as np
import pytest

from nabo_b200 import _lib, build


@pytest.fixture(scope="module")
def L():
    build.build()
    lib = _lib.lib()
    lib.nabo_dbg_tc_sched_bounds.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int)]
    lib.nabo_dbg_tc_sched_bounds.restype = C.c_int
    lib.nabo_dbg_tc_sweep_cost.argtypes = [C.c_int, C.c_int]
    lib.nabo_dbg_tc_sweep_cost.restype = C.c_double
    return lib


def pieces(bounds, c, n_rtiles):
    """The pieces ticket c runs, in order, as (kind, item, j0, j1) - the enumeration of work_piece<false>."""
    (i0, x0), (i1, x1) = bounds[c], bounds[c + 1]
    out = []
    if x1 > 0:
        out.append(("head", i1, 0, x1))
    first = i0 + 1 if x0 > 0 else i0
    out += [("whole", i, 0, n_rtiles) for i in range(first, i1)]
    if x0 > 0:
        out.append(("tail", i0, x0, n_rtiles))
    return out


@pytest.mark.parametrize("grid", [148, 20])
@pytest.mark.parametrize("n_rtiles,kprime", [(782, 39), (782, 9), (32, 39), (100, 76), (9766, 38)])
def test_schedule_covers_orders_and_balances(L, grid, n_rtiles, kprime):
    F = np.array([L.nabo_dbg_tc_sweep_cost(x, kprime) for x in range(n_rtiles + 1)])
    assert np.all(np.diff(F) >= 1.0)
    C_item = F[n_rtiles]
    one_tile = F[1]                                        # the most expensive tile: the first of a cold sweep
    buf = (C.c_int * (2 * (8 * grid + 1)))()
    for n_items in range(grid + 1, 8 * grid + 1):
        L.nabo_dbg_tc_sched_bounds(n_items, n_rtiles, grid, kprime, buf)
        bounds = [(buf[2 * b], buf[2 * b + 1]) for b in range(grid + 1)]
        assert bounds[0] == (0, 0) and bounds[grid] == (n_items, 0)
        assert all(0 <= x < n_rtiles for _, x in bounds)
        assert all(bounds[b] < bounds[b + 1] for b in range(grid))
        covered = [[] for _ in range(n_items)]
        head_of = {}
        T = n_items * C_item / grid
        for c in range(grid):
            ps = pieces(bounds, c, n_rtiles)
            t = 0.0
            for kind, item, j0, j1 in ps:
                covered[item].append((j0, j1))
                if kind == "head":
                    assert ps[0][0] == "head"
                    head_of[item] = (c, F[j1])                  # ticket, model time at which the head ends
                if kind == "tail":
                    assert ps[-1][0] == "tail"
                    hc, h_end = head_of[item]                   # KeyError: the head is not on a lower ticket
                    assert hc == c - 1
                    assert h_end <= t, (n_items, c, h_end, t)
                t += F[j1] - F[j0]
            assert t <= T + one_tile, (n_items, c, t, T)
            assert t >= T - one_tile, (n_items, c, t, T)
        for item, iv in enumerate(covered):
            iv.sort()
            assert iv[0][0] == 0 and iv[-1][1] == n_rtiles, (n_items, item, iv)
            assert all(iv[i][1] == iv[i + 1][0] for i in range(len(iv) - 1)), (n_items, item, iv)


@pytest.mark.parametrize("grid", [148, 7])
def test_one_item_per_cta_when_items_do_not_outnumber_ctas(L, grid):
    """grid = n_items (the launch never has more CTAs than items): every CTA sweeps exactly its own item; with a whole
    number of waves every CTA sweeps the same number of whole items."""
    buf = (C.c_int * (2 * (grid + 1)))()
    L.nabo_dbg_tc_sched_bounds(grid, 782, grid, 39, buf)
    assert [(buf[2 * b], buf[2 * b + 1]) for b in range(grid + 1)] == [(b, 0) for b in range(grid + 1)]
    for m in (2, 4):
        L.nabo_dbg_tc_sched_bounds(m * grid, 782, grid, 39, buf)
        assert [(buf[2 * b], buf[2 * b + 1]) for b in range(grid + 1)] == [(m * b, 0) for b in range(grid + 1)]
