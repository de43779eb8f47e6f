"""256-key plan of the tensor-core candidate pass (k + drop_first from 89 to 128, K' = 111 .. 160): the fast engine must
return exactly what the exact engine (and the oracle) returns - indices and FP64 distances, bit for bit - through every
entry point, while the certificate clears nearly every row.  k + drop_first <= 88 keeps the 128-key plan."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import nabo_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def core():
    from nabo_b200 import build, core as c
    build.build()
    return c


def same_bits(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return a.shape == b.shape and bool(((a == b) | (np.isnan(a) & np.isnan(b))).all())


def kprime(ksel):
    return ksel + max(ksel // 4, 8)


def fast_vs_exact(core, q, r, k, metric, **kw):
    fi, fd, st = core.knn(q, r, k, metric, mode="fast", return_stats=True, **kw)
    ei, ed = core.knn(q, r, k, metric, mode="exact", **kw)
    assert same_bits(fd, ed) and np.array_equal(fi, ei), (metric, k, kw.keys())
    return fi, fd, st


def check_fast_plan(st, n, ksel):
    assert st["rows_reranked"] == n, st                               # the tensor-core pass ran
    assert st["candidates_per_row"] == kprime(ksel), st
    assert st["rows_exact_fallback"] <= max(2, n // 50), st


@pytest.mark.parametrize("metric", ["euclidean", "cosine"])
@pytest.mark.parametrize("g", [25, 50, 64, 100, 128])
def test_large_k_fast_equals_exact(core, metric, g):
    from nabo_b200 import synth
    for i, k in enumerate([89, 100, 128]):
        n, m = 1500 + 7 * g + 101 * i, 9001 + 14 * g + 517 * i
        assert n % 128 and m % 128
        q = synth.pc_mixture(n, g, seed=101 + i)
        r = synth.pc_mixture(m, g, seed=1 + i)
        q[5] = np.nan
        q[9, g // 2] = np.nan
        r[17, 0] = np.nan
        mask = np.random.default_rng(g + i).random(m) < 0.1
        for kw in (dict(), dict(ref_mask=mask, idx_offset=4321)):
            _, _, st = fast_vs_exact(core, q, r, k, metric, **kw)
            check_fast_plan(st, n, k)


@pytest.mark.parametrize("metric", ["euclidean", "cosine"])
def test_plan_boundary(core, metric):
    """ksel = 88 keeps the 128-key plan (K' = 96); ksel = 89 and 128 (k = 88 / 127 with drop_first) take the 256-key
    plan.  The self-kNN rows also match the C oracle."""
    from nabo_b200 import synth
    g = 50
    r = synth.pc_mixture(6000, g, seed=1)
    r[7] = r[8]
    q = synth.pc_mixture(2000, g, seed=2)
    _, _, st = fast_vs_exact(core, q, r, 88, metric)
    assert st["rows_reranked"] == len(q) and st["candidates_per_row"] == 96, st
    for k in (88, 127):
        fi, fd, st = fast_vs_exact(core, r, r, k, metric, drop_first=True)
        check_fast_plan(st, len(r), k + 1)
        rows = np.random.default_rng(k).choice(len(r), 200, replace=False)
        oi, od = O.knn(r[rows], r, k, metric, drop_first=True)
        assert same_bits(fd[rows], od) and np.array_equal(fi[rows], oi)


@pytest.mark.parametrize("metric", ["euclidean", "cosine"])
def test_tie_class_larger_than_kprime(core, metric):
    """200 identical references nearest to a block of queries: more ties than the K' = 125 candidates (k = 100), so these rows
    fail the certificate and the exact fallback answers them, in index order inside the tie class."""
    from nabo_b200 import synth
    g = 100
    r = synth.pc_mixture(9000, g, seed=11)
    q = synth.pc_mixture(700, g, seed=12)
    r[2000:2200] = r[2000]
    q[50:90] = r[2000]
    assert O.dist_matrix(q[50:51], r[2000:2001], metric)[0, 0] == 0.0
    fi, fd, st = fast_vs_exact(core, q, r, 100, metric)
    assert (fi[50:90] == np.arange(2000, 2100)[None, :]).all()
    assert 40 <= st["rows_exact_fallback"] < 100, st


@pytest.mark.parametrize("metric", ["euclidean", "cosine"])
def test_schedules(core, metric):
    """g = 50 (384 queries per item, 148 SMs): grid + 1 and 2 grid - 1 items against a reference that fits in half of
    L2 (items cut at CTA boundaries, tails resume the heads' 256-key buffers); grid + 1 items against 260 k references
    (no cuts); 1 and 500 queries against 300 k references (one partial wave)."""
    from nabo_b200 import synth
    g, k = 50, 100
    r = synth.pc_mixture(30011, g, seed=3)
    for n in (148 * 384 + 100, 294 * 384 + 50):
        q = synth.pc_mixture(n, g, seed=n)
        _, _, st = fast_vs_exact(core, q, r, k, metric)
        check_fast_plan(st, n, k)
    big = synth.pc_mixture(300000, g, seed=4)
    q = synth.pc_mixture(148 * 384 + 100, g, seed=5)
    _, _, st = fast_vs_exact(core, q, big[:260000], k, metric)
    check_fast_plan(st, len(q), k)
    for n in (1, 500):
        q = synth.pc_mixture(n, g, seed=6 + n)
        _, _, st = fast_vs_exact(core, q, big, k, metric, drop_first=True)
        check_fast_plan(st, n, k + 1)


def test_routed_output(core):
    from nabo_b200 import synth
    g, k = 100, 110
    q = torch.from_numpy(synth.pc_mixture(5000, g, seed=101)).cuda()
    r = torch.from_numpy(synth.pc_mixture(20000, g, seed=1)).cuda()
    pi, pd = core.knn(q, r, k, "cosine", idx_offset=7)
    bounds = [0, 2345, 2345, 5000]
    bi = [torch.full((bounds[p + 1] - bounds[p], k), -9, dtype=torch.int32, device="cuda") for p in range(3)]
    bd = [torch.full((bounds[p + 1] - bounds[p], k), -9.0, dtype=torch.float64, device="cuda") for p in range(3)]
    _, _, st = core.knn(q, r, k, "cosine", idx_offset=7, return_stats=True,
                        out_parts=(bounds, [b.data_ptr() for b in bi], [b.data_ptr() for b in bd]))
    check_fast_plan(st, 5000, k)
    assert torch.equal(torch.cat(bi), pi) and torch.equal(torch.cat(bd).view(torch.int64), pd.view(torch.int64))
    ei, ed = core.knn(q, r, k, "cosine", idx_offset=7, mode="exact")
    assert torch.equal(pi, ei) and torch.equal(pd.view(torch.int64), ed.view(torch.int64))


@pytest.mark.parametrize("metric", ["euclidean", "cosine"])
def test_prepared_reference(core, metric):
    from nabo_b200 import synth
    g, k = 64, 100
    r = synth.pc_mixture(12007, g, seed=2)
    mask = np.random.default_rng(1).random(len(r)) < 0.1
    pr = core.prepare_reference(r, metric, mask)
    for n, drop_first in ((3001, False), (700, True)):
        q = r[:n] if drop_first else synth.pc_mixture(n, g, seed=n)
        pi, pd, st = core.knn(q, pr, k, drop_first=drop_first, idx_offset=3, return_stats=True)
        check_fast_plan(st, n, k + drop_first)
        oi, od = core.knn(q, r, k, metric, ref_mask=mask, drop_first=drop_first, idx_offset=3)
        ei, ed = core.knn(q, r, k, metric, ref_mask=mask, drop_first=drop_first, idx_offset=3, mode="exact")
        assert np.array_equal(pi, oi) and same_bits(pd, od)
        assert np.array_equal(pi, ei) and same_bits(pd, ed)


def test_workspace_sizes_are_exact(core):
    """At k = 100 a call given exactly the advertised workspace runs; one byte less returns NABO_EWORKSPACE - for the
    one-shot call (with and without drop_first) and for a prepared reference."""
    from nabo_b200 import _lib, synth
    L = _lib.lib()
    g, m, n, k = 50, 20011, 3001, 100
    r = torch.from_numpy(synth.pc_mixture(m, g, seed=5)).cuda()
    q = torch.from_numpy(synth.pc_mixture(n, g, seed=6)).cuda()
    pr = core.prepare_reference(r, "euclidean")
    idx = torch.empty((n, k), dtype=torch.int32, device="cuda")
    dst = torch.empty((n, k), dtype=torch.float64, device="cuda")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    full = int(L.nabo_knn_workspace_bytes(n, m, g, k, 0, 1))
    prep = int(L.nabo_knn_prepared_workspace_bytes(n, C.byref(pr.desc), k, 0.25, 1))
    assert 0 < prep < full
    ws = torch.empty(full, dtype=torch.uint8, device="cuda")
    stats = (C.c_int64 * 8)()

    def one_shot(nbytes, drop_first):
        return L.nabo_knn(C.c_void_p(q.data_ptr()), g, C.c_void_p(r.data_ptr()), g, n, m, g, k, 0, 0.25, None,
                          drop_first, 0, 1, C.c_void_p(idx.data_ptr()), C.c_void_p(dst.data_ptr()),
                          C.c_void_p(ws.data_ptr()), nbytes, stats, st)

    def prepared(nbytes):
        return L.nabo_knn_prepared(C.c_void_p(q.data_ptr()), g, n, C.byref(pr.desc), k, 0.25, 0, 0, 1,
                                   C.c_void_p(idx.data_ptr()), C.c_void_p(dst.data_ptr()), C.c_void_p(ws.data_ptr()),
                                   nbytes, stats, st)

    for drop_first in (0, 1):
        assert one_shot(full, drop_first) == 0 and stats[2] == kprime(k + drop_first)
        assert one_shot(full - 1, drop_first) == -2
    assert prepared(prep) == 0 and stats[2] == kprime(k)
    assert prepared(prep - 1) == -2
    torch.cuda.synchronize()
    ei, ed = core.knn(q, r, k, "euclidean", mode="exact")
    assert torch.equal(idx, ei) and torch.equal(dst.view(torch.int64), ed.view(torch.int64))


def test_mapping_drop_in(core, tmp_path, monkeypatch):
    """Mapping with k = 100: the reference graph (Euclidean self-kNN, ksel = 101) and a cosine target mapping store
    the same neighbour tables and edges whether the fast or the exact engine computed them, and the fast Mapping's own
    kNN calls ran the 256-key tensor-core plan (their stats are recorded through a wrapper of core.knn)."""
    from nabo_b200 import Mapping, Graph, store, synth
    knn, seen = core.knn, []

    def recording_knn(q, r, k, *a, **kw):
        idx, dst, st = knn(q, r, k, *a, return_stats=True, **kw)
        seen.append((k, kw.get("drop_first", False), kw.get("mode", "fast"), len(q), st))
        return idx, dst

    monkeypatch.setattr(core, "knn", recording_knn)
    g, k = 50, 100
    ref, tgt = synth.pc_mixture(3000, g, seed=1), synth.pc_mixture(2000, g, seed=2)
    rn, tn = synth.cell_names(len(ref), "R"), synth.cell_names(len(tgt), "T")
    ref_fn, tgt_fn = str(tmp_path / "ref.h5"), str(tmp_path / "tgt.h5")
    for fn, names, mat in ((ref_fn, rn, ref), (tgt_fn, tn, tgt)):
        h = store.File(fn, "w")
        h.create_row_group("data", names, mat)
        h.close()
    found = {}
    for mode in ("fast", "exact"):
        map_fn = str(tmp_path / ("map_%s.h5" % mode))
        m = Mapping(map_fn, "REF", ref_fn, "data", overwrite=True)
        m.set_parameters(g, k, 0.25, 64)
        m.make_ref_graph(mode=mode)
        m.map_target("TGT", tgt_fn, "data", metric="cosine", mode=mode)
        h5 = store.File(map_fn, "r")
        ruid = h5["name_stash/ref_name"][1].decode()
        tuid = [i[1].decode() for i in h5["name_stash/target_names"] if i[0] == b"TGT"][0]
        tables = [np.array([h5[uid + grp][c][:k] for c in names])
                  for uid, names in ((ruid, rn), (tuid, tn)) for grp in ("_sortedDist", "_dist")]
        h5.close()
        gph = Graph()
        gph.load_from_h5(map_fn, "REF", "reference")
        gph.load_from_h5(map_fn, "TGT", "target")
        edges = sorted((a, b, d["weight"]) if a < b else (b, a, d["weight"]) for a, b, d in gph.edges(data=True))
        found[mode] = (tables, edges)
    (tf, ef), (te, ee) = found["fast"], found["exact"]
    assert all(same_bits(a, b) for a, b in zip(tf, te))
    assert len(ef) > 0 and ef == ee
    fast = [(kk, drop, n, st) for kk, drop, mode, n, st in seen if mode == "fast" and kk == k]
    assert sorted((kk, drop) for kk, drop, _, _ in fast) == [(k, False), (k, True)], seen
    for kk, drop, n, st in fast:
        check_fast_plan(st, n, kk + drop)


def test_downstream_consumers_at_k128(core):
    """Neighbour tables from the 256-key plan at k = 128 feed the SNN weights, mapping scores, classification and the
    16-part merge of the reference-sharded mode unchanged: each matches the oracle / the unsharded result."""
    from nabo_b200 import synth
    g, k = 50, 128
    ref = torch.from_numpy(synth.pc_mixture(9000, g, seed=1)).cuda()
    tgt = torch.from_numpy(synth.pc_mixture(1200, g, seed=2)).cuda()
    ri, _, st = core.knn(ref, ref, k, "euclidean", return_stats=True)
    check_fast_plan(st, len(ref), k)
    ti, td, st = core.knn(tgt, ref, k, "euclidean", return_stats=True)
    check_fast_plan(st, len(tgt), k)
    ref_knn, tgt_knn = ri.cpu().numpy(), ti.cpu().numpy()
    cnt, w = core.snn_weights(tgt_knn, ref_knn, k)
    oc, ow = O.snn_weights(tgt_knn, ref_knn, k)
    assert np.array_equal(cnt, oc) and np.array_equal(w, ow)
    np.testing.assert_allclose(core.mapping_scores(tgt_knn, cnt, len(ref), k),
                               O.mapping_scores(tgt_knn, ow, len(ref), counts=oc), rtol=1e-13, atol=0)
    labels = np.random.default_rng(3).integers(-1, 7, size=len(ref)).astype(np.int32)
    got = core.classify_targets(tgt_knn, cnt, labels, 7, k)
    assert np.array_equal(got, O.classify_targets(tgt_knn, w, labels, 7, min_weight=0.1, counts=oc))
    bounds = [len(ref) * p // 16 for p in range(17)]
    parts = [core.knn(tgt, ref[a:b], k, "euclidean", idx_offset=a) for a, b in zip(bounds, bounds[1:])]
    mi, md = core.merge_topk_parts([p[0].data_ptr() for p in parts], [p[1].data_ptr() for p in parts], len(tgt), k,
                                   tgt.device)
    assert torch.equal(mi, ti) and torch.equal(md.view(torch.int64), td.view(torch.int64))
