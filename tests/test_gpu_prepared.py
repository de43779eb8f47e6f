"""Prepared references (core.prepare_reference / nabo_ref_prepare + nabo_knn_prepared): one reference packed once
serves many query batches, and every result is bit-identical to core.knn with the raw rows and to the exact engine -
indices, FP64 distances, tie and NaN order - across both tensor-core tile plans, the sliced Canberra pass, the
exact-engine branches (k beyond the fast plans, a vanishing dist_factor), every batch schedule (reference split, one
wave, balanced cuts, several waves), masks, drop_first, idx_offset, routed output, and queries far outside the
reference's scale."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def core():
    from nabo_b200 import build, core as c
    build.build()
    return c


@pytest.fixture(scope="module")
def synth():
    from nabo_b200 import synth as s
    return s


def same_bits(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return a.shape == b.shape and bool(((a == b) | (np.isnan(a) & np.isnan(b))).all())


def check_batch(core, q, r, pr, k, metric, f=0.25, mask=None, drop_first=False, idx_offset=0):
    """prepared == one-shot fast == exact, bit for bit; returns the prepared call's stats."""
    pi, pd, ps = core.knn(q, pr, k, dist_factor=f, drop_first=drop_first, idx_offset=idx_offset, return_stats=True)
    oi, od = core.knn(q, r, k, metric, f, ref_mask=mask, drop_first=drop_first, idx_offset=idx_offset)
    ei, ed = core.knn(q, r, k, metric, f, ref_mask=mask, drop_first=drop_first, idx_offset=idx_offset, mode="exact")
    assert np.array_equal(pi, oi) and same_bits(pd, od), (metric, k, len(q))
    assert np.array_equal(pi, ei) and same_bits(pd, ed), (metric, k, len(q))
    return ps


def queries(synth, n, g, seed, nan_rows=True):
    q = synth.pc_mixture(n, g, seed=seed)
    if nan_rows and n > 10:
        q[3] = np.nan
        q[7, g // 2] = np.nan
    return q


@pytest.mark.parametrize("metric", ["euclidean", "cosine"])
@pytest.mark.parametrize("g", [25, 50, 64, 100, 128])
def test_tc_prepared_serves_several_batches(core, synth, metric, g):
    m = 9001 + 3 * g
    r = synth.pc_mixture(m, g, seed=1)
    mask = np.random.default_rng(g).random(m) < 0.1
    for msk in (None, mask):
        pr = core.prepare_reference(r, metric, msk)
        for i, (n, k) in enumerate([(1, 30), (500, 1), (3001, 30), (20000, 88), (500, 30)]):
            q = queries(synth, n, g, 100 + i)
            st = check_batch(core, q, r, pr, k, metric, mask=msk)
            if k <= 30:
                assert st["rows_reranked"] == n, st                  # the prepared operands were used
        # reference <-> reference rows, global indices
        check_batch(core, r[:700], r, pr, 30, metric, mask=msk, drop_first=True, idx_offset=12345)


@pytest.mark.parametrize("g", [24, 50, 77, 100, 128])
def test_canberra_prepared_serves_several_batches(core, synth, g):
    m = 8001 + 5 * g
    r = synth.pc_mixture(m, g, seed=2)
    mask = np.random.default_rng(g).random(m) < 0.1
    for msk in (None, mask):
        pr = core.prepare_reference(r, "mod_canberra", msk)
        for f in (0.25, 1e-7):                                       # sliced pass / exact engine
            for i, (n, k) in enumerate([(1, 30), (500, 1), (2500, 30), (1200, 88)]):
                q = queries(synth, n, g, 200 + i)
                st = check_batch(core, q, r, pr, k, "mod_canberra", f=f, mask=msk)
                if k == 88 or f < 1e-6:
                    assert st["rows_exact_fallback"] == n, st         # past the fast plan or its f: the exact engine
            check_batch(core, r[:300], r, pr, 30, "mod_canberra", f=f, mask=msk, drop_first=True, idx_offset=7)


@pytest.mark.parametrize("metric,m", [("euclidean", 30011), ("cosine", 30011), ("mod_canberra", 12007)])
def test_prepared_batch_schedules(core, synth, metric, m):
    """1 query (reference split), 500 (one partial wave), 20 000 (split items), 57 000 (one wave + balanced cuts),
    120 000 (several waves) against one prepared reference."""
    g = 50
    r = synth.pc_mixture(m, g, seed=3)
    pr = core.prepare_reference(r, metric)
    for i, n in enumerate([1, 500, 20000, 57000, 120000]):
        q = queries(synth, n, g, 300 + i)
        st = check_batch(core, q, r, pr, 30, metric)
        assert st["rows_reranked"] == n and st["rows_exact_fallback"] <= max(4, n // 200), st


def test_prepared_outlier_queries(core, synth):
    """The prepared scale comes from the reference alone.  Queries at 400x the largest reference norm still fit FP16
    (scaled norm < 25 600); queries at 5 000x with the norm on one axis overflow it (scaled coordinate >= 160 000):
    they must go to the exact fallback, be counted there, and come out bit-identical."""
    rng = np.random.default_rng(9)
    g = 50
    r = synth.pc_mixture(6000, g, seed=1) * 0.02
    q = synth.pc_mixture(900, g, seed=101) * 0.02
    rmax = np.linalg.norm(r, axis=1).max()
    for t in range(1, 60):                                           # near ties around the k-th rank
        v = rng.normal(size=g)
        v /= np.linalg.norm(v)
        r[100 + 2 * t] = q[t] + 0.05 * v
        r[101 + 2 * t] = q[t] - 0.05 * (1 + 3e-8) * v
    for i in range(60, 70):
        v = rng.normal(size=g)
        q[i] = v / np.linalg.norm(v) * 400.0 * rmax
    big = list(range(70, 75))
    for j, i in enumerate(big):
        q[i] = 1e-3 * rng.normal(size=g) * rmax
        q[i, j] = 5000.0 * rmax * (1 if j % 2 else -1)
    pr = core.prepare_reference(r, "euclidean")
    for k in (1, 12, 30):
        st = check_batch(core, q, r, pr, k, "euclidean")
        assert st["rows_exact_fallback"] >= len(big), st
        _, _, only = core.knn(q[big], pr, k, return_stats=True)
        assert only["rows_exact_fallback"] == len(big), only


@pytest.mark.parametrize("metric", ["euclidean", "mod_canberra"])
@pytest.mark.parametrize("n_parts", [2, 3])
def test_prepared_routed_equals_knn_routed(core, synth, metric, n_parts):
    g, m, n, k = 50, 20011, 7001, 31
    r = synth.pc_mixture(m, g, seed=4)
    q = torch.from_numpy(queries(synth, n, g, 400)).cuda()
    pr = core.prepare_reference(r, metric)
    bounds = [n * p // n_parts for p in range(n_parts + 1)]

    def routed(ref, **kw):
        ib = [torch.full((bounds[p + 1] - bounds[p], k), -7, dtype=torch.int32, device="cuda") for p in range(n_parts)]
        db = [torch.zeros((bounds[p + 1] - bounds[p], k), dtype=torch.float64, device="cuda") for p in range(n_parts)]
        core.knn(q, ref, k, dist_factor=0.25, idx_offset=1000,
                 out_parts=(bounds, [b.data_ptr() for b in ib], [b.data_ptr() for b in db]), **kw)
        return torch.cat(ib).cpu().numpy(), torch.cat(db).cpu().numpy()

    pi, pd = routed(pr)
    oi, od = routed(r, metric=metric)
    assert np.array_equal(pi, oi) and same_bits(pd, od)
    ei, ed = core.knn(q, r, k, metric, 0.25, idx_offset=1000, mode="exact")       # host r: NumPy results
    assert np.array_equal(pi, ei) and same_bits(pd, ed)


def test_prepared_descriptor_status(core, synth):
    from nabo_b200 import _lib
    L = _lib.lib()
    g, m, n, k = 50, 3000, 64, 10
    r = torch.from_numpy(synth.pc_mixture(m, g, seed=5)).cuda()
    q = torch.from_numpy(synth.pc_mixture(n, g, seed=6)).cuda()
    pr = core.prepare_reference(r, "euclidean")
    idx = torch.empty((n, k), dtype=torch.int32, device="cuda")
    dst = torch.empty((n, k), dtype=torch.float64, device="cuda")
    ws = torch.empty(int(L.nabo_knn_prepared_workspace_bytes(n, C.byref(pr.desc), k, 0.25, 1)), dtype=torch.uint8,
                     device="cuda")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(d, kk=k, ldq=g):
        return L.nabo_knn_prepared(C.c_void_p(q.data_ptr()), ldq, n, C.byref(d), kk, 0.25, 0, 0, 1,
                                   C.c_void_p(idx.data_ptr()), C.c_void_p(dst.data_ptr()), C.c_void_p(ws.data_ptr()),
                                   ws.numel(), None, st)

    def edited(**fields):
        d = _lib.PreparedDesc()
        C.pointer(d)[0] = pr.desc
        for f_, v in fields.items():
            setattr(d, f_, v)
        return d

    assert call(pr.desc) == 0
    assert call(edited(magic=0)) == -1
    assert call(edited(abi_version=2)) == -3
    assert call(edited(metric=1)) == -1                       # a Canberra metric on tensor-core operands
    assert call(edited(metric=7)) == -3
    assert call(edited(g=129)) == -3
    assert call(edited(buffer_bytes=100)) == -1
    assert call(edited(ldr=g - 1)) == -1
    assert call(edited(ops=(C.c_void_p * 3)(16, 32, 0))) == -1
    assert call(pr.desc, kk=129) == -3                          # k + drop_first > 128
    assert call(pr.desc, ldq=g - 1) == -1
    assert L.nabo_knn_prepared_workspace_bytes(n, C.byref(edited(magic=0)), k, 0.25, 1) == 0
    # the query-side workspace is smaller than the one-shot workspace by the reference's share
    full = L.nabo_knn_workspace_bytes(n, m, g, k, 0, 1)
    assert ws.numel() < full and full - ws.numel() >= L.nabo_ref_prepared_bytes(m, g, 0) - 4096
    assert L.nabo_ref_prepared_bytes(m, 129, 0) == 0 and L.nabo_ref_prepared_bytes(m, g, 5) == 0
    d = _lib.PreparedDesc()
    buf = torch.empty(1 << 20, dtype=torch.uint8, device="cuda")
    assert L.nabo_ref_prepare(C.c_void_p(r.data_ptr()), g, m, 129, 0, None, C.c_void_p(buf.data_ptr()), buf.numel(),
                              C.byref(d), st) == -3
    assert L.nabo_ref_prepare(C.c_void_p(r.data_ptr()), g, m, g, 0, None, C.c_void_p(buf.data_ptr()), 1000,
                              C.byref(d), st) == -1
    # Python: conflicting arguments and a source modified in place
    with pytest.raises(ValueError, match="conflicts"):
        core.knn(q, pr, k, "cosine")
    with pytest.raises(ValueError, match="columns"):
        core.knn(q[:, :10].contiguous(), pr, k)
    r[0, 0] += 1.0
    with pytest.raises(ValueError, match="modified in place"):
        core.knn(q, pr, k)


def test_map_cells_with_prepared_reference(core, synth):
    from nabo_b200 import parallel
    g, m, n, k = 50, 15013, 9000, 11
    r = synth.pc_mixture(m, g, seed=7)
    t = synth.pc_mixture(n, g, seed=8)
    mask = np.random.default_rng(1).random(m) < 0.05
    ref_knn, _ = core.knn(r, r, k, "euclidean", drop_first=True)
    pr = core.prepare_reference(r, "mod_canberra", mask)
    for tgt in (t, t[:777]):
        a = core.map_cells(tgt, pr, ref_knn, k)
        b = core.map_cells(tgt, r, ref_knn, k, ref_mask=mask)
        assert set(a) == set(b)
        for key in ("idx", "counts"):
            assert np.array_equal(a[key], b[key]), key
        for key in ("dist", "weights", "scores"):
            assert same_bits(a[key], b[key]), key
    # the pipelined host form and the sharded mappers (one rank) take the prepared reference too
    th = torch.from_numpy(t).pin_memory()
    ha = {x: v.clone() for x, v in core.map_cells_host(th, pr, ref_knn, k).items()}
    hb = core.map_cells_host(th, r, ref_knn, k, ref_mask=mask)
    for key in ha:
        assert same_bits(ha[key].numpy(), hb[key].numpy()), key
    td, rd = torch.from_numpy(t).cuda(), torch.from_numpy(r).cuda()
    rk = torch.from_numpy(ref_knn).cuda()
    sa = parallel.map_targets_sharded(td, pr, rk, k, n)
    sb = parallel.map_targets_sharded(td, rd, rk, k, n, ref_mask=mask)
    ra = parallel.map_reference_sharded(td, pr, 0, m, rk, k)
    rb = parallel.map_reference_sharded(td, rd, 0, m, rk, k, ref_mask_shard=mask)
    for x, y in ((sa, sb), (ra, rb)):
        for key in ("idx", "dist", "counts", "weights", "scores"):
            assert same_bits(x[key].double().cpu().numpy(), y[key].double().cpu().numpy()), key


def test_mapping_keeps_the_prepared_reference(tmp_path, core, synth, monkeypatch):
    """Two targets mapped in a row onto one Mapping: the second map_target neither packs nor uploads the reference
    again, and both give what the host-matrix path gives."""
    from nabo_b200 import Mapping, store
    g, m, k = 20, 3000, 11
    ref = synth.pc_mixture(m, g, seed=11)
    tgts = [synth.pc_mixture(900, g, seed=12), synth.pc_mixture(1100, g, seed=13)]
    rn = synth.cell_names(m, "R")
    fns = {x: str(tmp_path / (x + ".h5")) for x in ("ref", "t0", "t1", "map")}
    for name, mat in (("ref", ref), ("t0", tgts[0]), ("t1", tgts[1])):
        h = store.File(fns[name], "w")
        h.create_row_group("data", rn if name == "ref" else synth.cell_names(len(mat), name.upper()), mat)
        h.close()
    calls = {"prepare": 0, "ref_uploads": 0}
    real_prepare, real_dev = core.prepare_reference, core._dev

    def counting_prepare(*a, **kw):
        calls["prepare"] += 1
        return real_prepare(*a, **kw)

    mp = Mapping(fns["map"], "REF", fns["ref"], "data", overwrite=True)

    def counting_dev(x, *a, **kw):
        if x is not None and x is mp._refMatCache:
            calls["ref_uploads"] += 1
        return real_dev(x, *a, **kw)

    monkeypatch.setattr(core, "prepare_reference", counting_prepare)
    monkeypatch.setattr(core, "_dev", counting_dev)
    mp.set_parameters(g, k, 0.25, 64)
    mp.make_ref_graph()
    mp.map_target("T0", fns["t0"], "data")
    after_first = dict(calls)
    assert after_first["prepare"] == 2                          # Euclidean for the graph, Canberra for the targets
    mp.map_target("T1", fns["t1"], "data")
    assert calls == after_first, calls                          # no repack, no upload of the reference
    h5 = store.File(fns["map"], "r")
    for i, name in enumerate(("T0", "T1")):
        uid = [x[1].decode() for x in h5["name_stash/target_names"] if x[0] == name.encode()][0]
        tn = synth.cell_names(len(tgts[i]), "T%d" % i)
        got_i = np.array([h5[uid + "_sortedDist"][c][:k] for c in tn])
        got_d = np.array([h5[uid + "_dist"][c][:k] for c in tn])
        want_i, want_d = core.knn(tgts[i], ref, k, "mod_canberra", 0.25)
        assert np.array_equal(got_i, want_i) and same_bits(got_d, want_d)
    h5.close()
    mp.set_parameters(g, k, 0.25, 64)
    assert mp._refPrepCache is None                            # new parameters drop the packed reference
