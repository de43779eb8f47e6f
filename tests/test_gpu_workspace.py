"""Workspace sizes are exact for every path of the fast engine: a call given exactly the bytes the size function
advertises runs and returns what the exact engine returns, bit for bit; one byte less returns NABO_EWORKSPACE.  The
sizes come from running each pass's workspace carve, so this checks the carves and the plan they share.  The 256-key
tensor-core plan has the same check in tests/test_gpu_tc_large_k.py."""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu

EWORKSPACE = -2

# (name, metric, g, n_query, n_ref, k, dist_factor, kernel launches per drop_first (one-shot, prepared)).  The launch
# counts tell the paths apart: the tensor-core pass counts its preparation (6, or 3 with a prepared reference), the
# emit kernel and the threshold reduction of a split call; the sliced pass reports 10 and the exact engine 1.  A call
# that runs the exact engine for every drop_first needs no workspace, so its prepared size is 0.
CASES = [
    ("tc_fused", "euclidean", 50, 3001, 6000, 30, 0.25, {0: (10, 7), 1: (10, 7)}),
    ("tc_emit", "cosine", 50, 3001, 20011, 60, 0.25, {0: (11, 8), 1: (11, 8)}),
    ("tc_split", "euclidean", 50, 300, 100000, 30, 0.25, {0: (12, 9), 1: (12, 9)}),
    ("sliced", "mod_canberra", 50, 3001, 6000, 30, 0.25, {0: (10, 10), 1: (10, 10)}),
    ("sliced_split", "mod_canberra", 50, 300, 100000, 30, 0.25, {0: (10, 10), 1: (10, 10)}),
    # dist_factor < 1e-6 runs the exact engine; the one-shot size (which has no dist_factor) is still the sliced carve
    ("vanishing_f", "mod_canberra", 50, 3001, 20011, 30, 1e-7, {0: (1, 1), 1: (1, 1)}),
    # k + drop_first = 57 is past the sliced pass: drop_first runs the exact engine on a workspace sized for the
    # sliced pass that the same k takes without it
    ("exact", "mod_canberra", 50, 2001, 20011, 56, 0.25, {0: (10, 10), 1: (1, 1)}),
]


@pytest.fixture(scope="module")
def core():
    from nabo_b200 import build, core as c
    build.build()
    return c


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_workspace_is_exact_on_every_path(core, case):
    from nabo_b200 import _lib, synth
    _, metric, g, n, m, k, f, launches = case
    L = _lib.lib()
    mi = _lib.METRICS[metric]
    r = torch.from_numpy(synth.pc_mixture(m, g, seed=5)).cuda()
    q = torch.from_numpy(synth.pc_mixture(n, g, seed=6)).cuda()
    pr = core.prepare_reference(r, metric)
    idx = torch.empty((n, k), dtype=torch.int32, device="cuda")
    dst = torch.empty((n, k), dtype=torch.float64, device="cuda")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    full = int(L.nabo_knn_workspace_bytes(n, m, g, k, mi, 1))
    prep = int(L.nabo_knn_prepared_workspace_bytes(n, C.byref(pr.desc), k, f, 1))
    if case[0] == "vanishing_f":
        assert prep == 0 and full > 0
    else:
        assert 0 < prep <= full
    if case[0] not in ("vanishing_f", "exact"):
        assert prep < full                              # the prepared operands replace the reference's share
    ws = torch.empty(full, dtype=torch.uint8, device="cuda")
    stats = (C.c_int64 * 8)()

    def one_shot(nbytes, drop_first):
        return L.nabo_knn(C.c_void_p(q.data_ptr()), g, C.c_void_p(r.data_ptr()), g, n, m, g, k, mi, f, None,
                          drop_first, 0, 1, C.c_void_p(idx.data_ptr()), C.c_void_p(dst.data_ptr()),
                          C.c_void_p(ws.data_ptr()), nbytes, stats, st)

    def prepared(nbytes, drop_first):
        return L.nabo_knn_prepared(C.c_void_p(q.data_ptr()), g, n, C.byref(pr.desc), k, f, drop_first, 0, 1,
                                   C.c_void_p(idx.data_ptr()), C.c_void_p(dst.data_ptr()), C.c_void_p(ws.data_ptr()),
                                   nbytes, stats, st)

    for drop_first in (0, 1):
        ei, ed = core.knn(q, r, k, metric, dist_factor=f, drop_first=bool(drop_first), mode="exact")
        for call, nbytes, nl in ((one_shot, full, launches[drop_first][0]), (prepared, prep, launches[drop_first][1])):
            idx.fill_(-7)
            dst.fill_(-7.0)
            assert call(nbytes, drop_first) == 0, (call.__name__, drop_first)
            torch.cuda.synchronize()
            assert stats[3] == nl, (call.__name__, drop_first, list(stats))
            assert torch.equal(idx, ei) and torch.equal(dst.view(torch.int64), ed.view(torch.int64)), \
                (call.__name__, drop_first)
            if nbytes > 0:
                assert call(nbytes - 1, drop_first) == EWORKSPACE, (call.__name__, drop_first)
