"""Correlation distance on the B200: full tiles, both kNN engines, prepared references, routed rows, workspace sizes
and the Mapping facade.  Every comparison is bit for bit, in indices and FP64 distances (NaN equals NaN)."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import nabo_oracle as O
from correlation_oracle import centre_rows, correlation_dist
import correlation_oracle as CO

pytestmark = pytest.mark.gpu

EWORKSPACE = -2


@pytest.fixture(scope="module")
def core():
    from nabo_b200 import build, core as c
    build.build()
    return c


def same_bits(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return a.shape == b.shape and bool(((a == b) | (np.isnan(a) & np.isnan(b))).all())


def _data(n, m, g, seed, nan=True, const=True, dup=True):
    rng = np.random.default_rng(seed)
    centers = rng.normal(size=(6, g)) * 3
    scale = 10.0 ** rng.uniform(-1, 1, size=g)
    r = (centers[rng.integers(0, 6, m)] + rng.normal(size=(m, g))) * scale
    q = (centers[rng.integers(0, 6, n)] + rng.normal(size=(n, g))) * scale
    if dup:
        r[rng.integers(0, m, m // 20)] = r[rng.integers(0, m)]
        q[rng.integers(0, n, max(1, n // 20))] = r[rng.integers(0, m)]
    if nan:
        r[rng.integers(0, m, 3), rng.integers(0, g, 3)] = np.nan
        q[rng.integers(0, n), rng.integers(0, g)] = np.nan
    if const:
        r[rng.integers(0, m, 2)] = 2.5                 # exact sum: centres to zero
        r[rng.integers(0, m)] = 0.1                    # inexact sum: a tiny constant residual
        q[rng.integers(0, n)] = -4.0
    return q, r


# ------------------------------------------------------------------ 1. full tiles
@pytest.mark.parametrize("g", [1, 2, 3, 50, 128])
def test_full_tiles_equal_oracle(core, g):
    q, r = _data(67, 131, g, seed=g)
    d = core.correlation_dist(q, r)
    assert same_bits(d, correlation_dist(q, r))
    out = np.empty((len(q), len(r)))                    # the caller's buffer, filled in place
    assert core.correlation_dist(q, r, out) is out and same_bits(out, d)


def test_centring_order_is_pinned(core):
    x = np.array([[1e16, 1.0, -1e16, 1.0], [1.0, 2.0, 3.0, 5.0], [0.0, 1.0, 0.0, 0.0]])
    assert same_bits(core.correlation_dist(x, x), correlation_dist(x, x))
    i, d = core.knn(x, x, 2, "correlation", mode="exact")
    oi, od = CO.knn(x, x, 2)
    assert np.array_equal(i, oi) and same_bits(d, od)


# ------------------------------------------------------------------ 2. both engines against the oracle
GRID = [(g, k, df) for g in (1, 3, 25, 50, 52, 53, 100, 128) for (k, df) in
        ((1, False), (10, False), (30, False), (60, False), (88, False), (89, False), (127, True))]


@pytest.mark.parametrize("g,k,drop_first", GRID, ids=["g%d-k%d-d%d" % c for c in GRID])
def test_knn_grid_equals_oracle(core, g, k, drop_first):
    q, r = _data(400, 3000, g, seed=1000 + 7 * g + k)
    rng = np.random.default_rng(k)
    mask = rng.random(len(r)) < 0.1 if k % 2 == 0 else None
    off = 1000 if k % 3 == 0 else 0
    if drop_first:
        q = r[:400]
    oi, od = CO.knn(q, r, k, mask=mask, drop_first=drop_first)
    oi = np.where(oi >= 0, oi + off, oi)
    for mode in ("exact", "fast"):
        i, d = core.knn(q, r, k, "correlation", ref_mask=mask, drop_first=drop_first, idx_offset=off, mode=mode)
        assert np.array_equal(i, oi) and same_bits(d, od), mode


def test_knn_k_beyond_unmasked_cells(core):
    q, r = _data(300, 2000, 50, seed=3)
    mask = np.ones(len(r), bool)
    mask[::100] = False                                   # 20 unmasked cells, k = 30
    oi, od = CO.knn(q, r, 30, mask=mask)
    for mode in ("exact", "fast"):
        i, d = core.knn(q, r, 30, "correlation", ref_mask=mask, mode=mode)
        assert np.array_equal(i, oi) and same_bits(d, od), mode
        assert np.isnan(d[:, 20:]).all()


def _case(seed):
    rng = np.random.default_rng(seed)
    g = int(rng.choice([1, 2, 3, 7, 16, 17, 25, 33, 50, 57, 64, 100, 128]))
    m = int(rng.choice([40, 129, 300, 1000, 2049, 5000]))
    n = int(rng.choice([1, 31, 33, 100, 385, 700]))
    k = int(min(rng.choice([1, 5, 15, 30, 33, 60, 90, 120]), m - 2))
    q, r = _data(n, m, g, seed, nan=rng.random() < 0.3, const=rng.random() < 0.3, dup=rng.random() < 0.5)
    if rng.random() < 0.3:                                # rows of one constant offset from a reference row
        q[rng.integers(0, n)] = r[rng.integers(0, m)] + 3.0
    mask = (rng.random(m) < rng.choice([0.05, 0.5])) if rng.random() < 0.4 else None
    if mask is not None and (~mask).sum() < k + 2:
        mask = None
    return q, r, k, mask, int(rng.choice([0, 0, 1000]))


@pytest.mark.parametrize("seed", range(60))
def test_random_fast_equals_exact_equals_oracle(core, seed):
    q, r, k, mask, off = _case(seed)
    fi, fd = core.knn(q, r, k, "correlation", ref_mask=mask, idx_offset=off, mode="fast")
    ei, ed = core.knn(q, r, k, "correlation", ref_mask=mask, idx_offset=off, mode="exact")
    assert np.array_equal(fi, ei) and same_bits(fd, ed), "fast != exact"
    oi, od = CO.knn(q, r, k, mask=mask)
    assert np.array_equal(ei, np.where(oi >= 0, oi + off, oi)) and same_bits(ed, od), "exact != oracle"


# ------------------------------------------------------------------ 3. the fast path is taken
def test_fast_path_taken(core):
    from nabo_b200 import synth
    n = 20000
    r = torch.from_numpy(synth.pc_mixture(n, 50, seed=11)).cuda()
    q = torch.from_numpy(synth.pc_mixture(n, 50, seed=12)).cuda()
    _, _, sc = core.knn(q, r, 30, "cosine", mode="fast", return_stats=True)
    i, d, st = core.knn(q, r, 30, "correlation", mode="fast", return_stats=True)
    print("\ncorrelation 20k x 20k g=50 k=30: rows to the exact fallback %d (cosine %d), centring %.3f ms"
          % (st["rows_exact_fallback"], sc["rows_exact_fallback"], st["prep_ms"]))
    assert st["rows_reranked"] == n and st["candidates_per_row"] == sc["candidates_per_row"]
    assert st["kernel_launches"] == sc["kernel_launches"] + 2
    ci, cd = core.knn(torch.from_numpy(centre_rows(q.cpu().numpy())).cuda(),
                      torch.from_numpy(centre_rows(r.cpu().numpy())).cuda(), 30, "cosine", mode="fast")
    assert torch.equal(i, ci) and torch.equal(d.view(torch.int64), cd.view(torch.int64))


# ------------------------------------------------------------------ 4. workspace sizes are exact
WS_CASES = [(50, 3001, 6000, 30), (50, 3001, 20011, 100), (53, 300, 100000, 30)]


@pytest.mark.parametrize("case", WS_CASES, ids=[str(c) for c in WS_CASES])
def test_workspace_is_exact(core, case):
    from nabo_b200 import _lib, synth
    g, n, m, k = case
    L = _lib.lib()
    mi = _lib.CORRELATION
    r = torch.from_numpy(synth.pc_mixture(m, g, seed=5)).cuda()
    q = torch.from_numpy(synth.pc_mixture(n, g, seed=6)).cuda()
    pr = core.prepare_reference(r, "correlation")
    idx = torch.empty((n, k), dtype=torch.int32, device="cuda")
    dst = torch.empty((n, k), dtype=torch.float64, device="cuda")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    stats = (C.c_int64 * 8)()
    big = int(L.nabo_knn_workspace_bytes(n, m, g, k, mi, 1))
    ws = torch.empty(big, dtype=torch.uint8, device="cuda")

    def one_shot(nbytes, drop_first, mode):
        return L.nabo_knn(C.c_void_p(q.data_ptr()), g, C.c_void_p(r.data_ptr()), g, n, m, g, k, mi, 0.25, None,
                          drop_first, 0, mode, C.c_void_p(idx.data_ptr()), C.c_void_p(dst.data_ptr()),
                          C.c_void_p(ws.data_ptr()), nbytes, stats, st)

    def prepared(nbytes, drop_first, mode):
        return L.nabo_knn_prepared(C.c_void_p(q.data_ptr()), g, n, C.byref(pr.desc), k, 0.25, drop_first, 0, mode,
                                   C.c_void_p(idx.data_ptr()), C.c_void_p(dst.data_ptr()), C.c_void_p(ws.data_ptr()),
                                   nbytes, stats, st)

    for drop_first in (0, 1):
        ei, ed = core.knn(q, r, k, "correlation", drop_first=bool(drop_first), mode="exact")
        _, _, cs = core.knn(q, r, k, "cosine", drop_first=bool(drop_first), mode="fast", return_stats=True)
        for mode in (1, 0):
            for call in (one_shot, prepared):
                nbytes = int(L.nabo_knn_workspace_bytes(n, m, g, k, mi, mode)) if call is one_shot else \
                    int(L.nabo_knn_prepared_workspace_bytes(n, C.byref(pr.desc), k, 0.25, mode))
                assert 0 < nbytes <= big
                idx.fill_(-7)
                dst.fill_(-7.0)
                assert call(nbytes, drop_first, mode) == 0, (call.__name__, drop_first, mode)
                torch.cuda.synchronize()
                assert torch.equal(idx, ei) and torch.equal(dst.view(torch.int64), ed.view(torch.int64)), \
                    (call.__name__, drop_first, mode)
                centring = 2 if call is one_shot else 1
                if mode == 0:
                    assert stats[3] == 1 + centring and stats[1] == n
                elif call is one_shot:
                    assert stats[3] == cs["kernel_launches"] + centring, list(stats)
                assert stats[7] > 0
                assert call(nbytes - 1, drop_first, mode) == EWORKSPACE, (call.__name__, drop_first, mode)


# ------------------------------------------------------------------ 5. prepared reference
def test_prepared_batches_equal_one_shot(core):
    from nabo_b200 import _lib, synth
    g, m = 50, 60000
    r = torch.from_numpy(synth.pc_mixture(m, g, seed=21)).cuda()
    r[5] = 1.5                                           # a constant reference row
    keep = r.clone()
    mask = torch.from_numpy(np.random.default_rng(2).random(m) < 0.05).cuda()
    pr = core.prepare_reference(r, "correlation")
    prm = core.prepare_reference(r, "correlation", ref_mask=mask)
    assert pr.nbytes == int(_lib.lib().nabo_ref_prepared_bytes(m, g, _lib.CORRELATION))
    assert pr.desc.r == pr.buffer.data_ptr() and pr.desc.ldr == g
    for b, (n, k, extra) in enumerate([(1, 88, {}), (500, 100, dict(drop_first=True)),
                                       (3001, 30, dict(mode="exact")), (20000, 88, dict(idx_offset=1000)),
                                       (3001, 100, dict(masked=True)), (500, 127, dict(drop_first=True, mode="exact"))]):
        q = torch.from_numpy(synth.pc_mixture(n, g, seed=300 + b)).cuda()
        if extra.get("drop_first"):
            q = r[:n].clone()
        kw = {x: v for x, v in extra.items() if x != "masked"}
        p = prm if extra.get("masked") else pr
        mk = mask if extra.get("masked") else None
        pi, pd = core.knn(q, p, k, **kw)
        oi, od = core.knn(q, r, k, "correlation", ref_mask=mk, **kw)
        assert torch.equal(pi, oi) and torch.equal(pd.view(torch.int64), od.view(torch.int64)), (n, k, extra)
    assert torch.equal(r.view(torch.int64), keep.view(torch.int64))            # the caller's rows are unchanged
    L = _lib.lib()
    buf = torch.empty(1 << 20, dtype=torch.uint8, device="cuda")
    d = _lib.PreparedDesc()
    w = torch.zeros((1000, 129), dtype=torch.float64, device="cuda")
    assert L.nabo_ref_prepare(C.c_void_p(w.data_ptr()), 129, 1000, 129, _lib.CORRELATION, None,
                              C.c_void_p(buf.data_ptr()), buf.numel(), C.byref(d), None) == -3


# ------------------------------------------------------------------ 6. routed rows
def test_routed_equals_unrouted(core):
    from nabo_b200 import synth
    g, k, n = 50, 30, 5000
    r = torch.from_numpy(synth.pc_mixture(20000, g, seed=31)).cuda()
    q = torch.from_numpy(synth.pc_mixture(n, g, seed=32)).cuda()
    pr = core.prepare_reference(r, "correlation")
    bounds = [0, 1234, 1234, 5000]
    for ref, mode in ((r, "fast"), (r, "exact"), (pr, "fast")):
        ib = [torch.full((bounds[p + 1] - bounds[p], k), -7, dtype=torch.int32, device="cuda") for p in range(3)]
        db = [torch.zeros((bounds[p + 1] - bounds[p], k), dtype=torch.float64, device="cuda") for p in range(3)]
        core.knn(q, ref, k, "correlation", idx_offset=77, mode=mode,
                 out_parts=(bounds, [b.data_ptr() if b.numel() else 0 for b in ib],
                            [b.data_ptr() if b.numel() else 0 for b in db]))
        ui, ud = core.knn(q, r, k, "correlation", idx_offset=77, mode=mode)
        assert torch.equal(torch.cat(ib), ui) and torch.equal(torch.cat(db).view(torch.int64), ud.view(torch.int64))


# ------------------------------------------------------------------ 7. full size
def test_full_size(core):
    from nabo_b200 import synth
    n, g, k = 100000, 50, 30
    r = torch.from_numpy(synth.pc_mixture(n, g, seed=41)).cuda()
    q = torch.from_numpy(synth.pc_mixture(n, g, seed=42)).cuda()
    fi, fd, st = core.knn(q, r, k, "correlation", mode="fast", return_stats=True)
    print("\ncorrelation 100k x 100k g=50 k=30: rows to the exact fallback %d" % st["rows_exact_fallback"])
    rows = torch.from_numpy(np.random.default_rng(0).choice(n, 768, replace=False)).cuda()
    ei, ed = core.knn(q[rows], r, k, "correlation", mode="exact")
    assert torch.equal(fi[rows], ei) and torch.equal(fd[rows].view(torch.int64), ed.view(torch.int64))
    sub = rows[:32].cpu().numpy()
    oi, od = CO.knn(q.cpu().numpy()[sub], r.cpu().numpy(), k)
    assert np.array_equal(fi[rows[:32]].cpu().numpy(), oi) and same_bits(fd[rows[:32]].cpu().numpy(), od)


# ------------------------------------------------------------------ 8. the Mapping facade
def test_mapping_facade(core, tmp_path):
    import random
    from nabo_b200 import Graph, Mapping, store, synth
    g, k = 20, 11
    ref = synth.pc_mixture(1500, g, seed=1)
    tgt = synth.pc_mixture(700, g, seed=101)
    rn, tn = synth.cell_names(len(ref), "R"), synth.cell_names(len(tgt), "T")
    ref_fn, tgt_fn, map_fn = (str(tmp_path / x) for x in ("ref.h5", "tgt.h5", "map.h5"))
    for fn, names, mat in ((ref_fn, rn, ref), (tgt_fn, tn, tgt)):
        h = store.File(fn, "w")
        h.create_row_group("data", names, mat)
        h.close()
    random.seed(5)
    m = Mapping(map_fn, "REF", ref_fn, "data", overwrite=True)
    m.set_parameters(g, k, 0.25, 64)
    m.make_ref_graph(metric="correlation")
    m.map_target("TGT", tgt_fn, "data", metric="correlation")
    h5 = store.File(map_fn, "r")
    ruid = h5["name_stash/ref_name"][1].decode()
    tuid = [i[1].decode() for i in h5["name_stash/target_names"] if i[0] == b"TGT"][0]
    rk = np.array([h5[ruid + "_sortedDist"][c][:k] for c in rn])
    rd = np.array([h5[ruid + "_dist"][c][:k] for c in rn])
    tk = np.array([h5[tuid + "_sortedDist"][c][:k] for c in tn])
    td = np.array([h5[tuid + "_dist"][c][:k] for c in tn])
    h5.close()
    ori, ord_ = CO.knn(ref, ref, k, drop_first=True)
    oti, otd = CO.knn(tgt, ref, k)
    assert np.array_equal(rk, ori) and same_bits(rd, ord_)
    assert np.array_equal(tk, oti) and same_bits(td, otd)
    cnt, w = O.snn_weights(oti, ori, k)
    gph = Graph()
    gph.load_from_h5(map_fn, "REF", "reference")
    gph.load_from_h5(map_fn, "TGT", "target")
    got = {(a, b) if a.endswith("_TGT") else (b, a): d["weight"] for a, b, d in gph.edges(data=True)
           if a.endswith("_TGT") or b.endswith("_TGT")}
    exp = {(tn[t] + "_TGT", rn[int(oti[t, j])] + "_REF"): float(w[t, j])
           for t in range(len(tn)) for j in range(k) if cnt[t, j] > 0}
    assert got == exp
    sc = gph.get_mapping_score("TGT")
    arr = np.array([sc[c + "_REF"] for c in rn])
    np.testing.assert_allclose(arr, O.mapping_scores(oti, w, len(rn), counts=cnt), rtol=1e-12, atol=0)
    res = core.map_cells(tgt, ref, ori.astype(np.int32), k, metric="correlation")
    assert np.array_equal(res["idx"], oti) and same_bits(res["dist"], otd)
    assert np.array_equal(res["counts"], cnt) and same_bits(res["weights"], w)
    np.testing.assert_allclose(res["scores"], O.mapping_scores(oti, w, len(rn), counts=cnt), rtol=1e-12, atol=0)


def test_cosine_certificate_covers_rounded_down_distances(core):
    """Parallel rows: the FP64 cosine distance rounds to a few ulps below zero, differently per row, while the
    candidate scores tie.  Every centred row at g = 2 is such a row; the certificate must send these rows to the exact
    fallback rather than pass a candidate list that misses a rounded-down neighbour."""
    rng = np.random.default_rng(1)
    a = rng.normal(size=2049)
    for x in (np.stack([a, -a], 1), _case(14)[1]):
        for metric in ("cosine", "correlation"):
            fi, fd = core.knn(x[:100], x, 15, metric, mode="fast")
            ei, ed = core.knn(x[:100], x, 15, metric, mode="exact")
            assert np.array_equal(fi, ei) and same_bits(fd, ed), metric
