"""CPU checks of the 256-key tensor-core plan (k + drop_first from 89 to 128): the public candidate pass keeps its
K' <= 96 width for every k, and the balanced-cut schedule (tc::sched_bound) still covers every (item, reference tile)
exactly once, with each tail on the ticket right after its head, at the new plan's K' of 111 and 160."""
import ctypes as C

import pytest

from nabo_b200 import _lib, build


@pytest.fixture(scope="module")
def L():
    build.build()
    lib = _lib.lib()
    lib.nabo_dbg_tc_sched_bounds.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int)]
    lib.nabo_dbg_tc_sched_bounds.restype = C.c_int
    return lib


def test_candidates_width_unchanged(L):
    for drop_first in (0, 1):
        for k in range(1, 129):
            ksel = k + drop_first
            assert L.nabo_knn_candidates_width(k, drop_first) == min(ksel + max(ksel // 4, 8), 96), (k, drop_first)


@pytest.mark.parametrize("grid", [148, 20])
@pytest.mark.parametrize("n_rtiles,kprime", [(782, 111), (782, 160), (32, 160), (2344, 135)])
def test_schedule_covers_every_tile_once_at_large_kprime(L, grid, n_rtiles, kprime):
    buf = (C.c_int * (2 * (8 * grid + 1)))()
    for n_items in range(grid + 1, 8 * grid + 1):
        L.nabo_dbg_tc_sched_bounds(n_items, n_rtiles, grid, kprime, buf)
        bounds = [(buf[2 * b], buf[2 * b + 1]) for b in range(grid + 1)]
        assert bounds[0] == (0, 0) and bounds[grid] == (n_items, 0)
        covered = [[] for _ in range(n_items)]
        head_ticket = {}
        for c in range(grid):
            (i0, x0), (i1, x1) = bounds[c], bounds[c + 1]
            if x1 > 0:                                              # head: first piece of ticket c
                covered[i1].append((0, x1))
                head_ticket[i1] = c
            first = i0 + 1 if x0 > 0 else i0
            for i in range(first, i1):                              # whole items
                covered[i].append((0, n_rtiles))
            if x0 > 0:                                              # tail: resumes the head of ticket c - 1
                assert head_ticket[i0] == c - 1, (n_items, c)
                covered[i0].append((x0, n_rtiles))
        for item, iv in enumerate(covered):
            iv.sort()
            assert iv[0][0] == 0 and iv[-1][1] == n_rtiles, (n_items, item, iv)
            assert all(iv[i][1] == iv[i + 1][0] for i in range(len(iv) - 1)), (n_items, item, iv)
