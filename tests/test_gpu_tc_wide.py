"""Wide tile plan of the tensor-core candidate pass (53 <= g <= 128: two query tiles per work item, reference tiles
streamed in K-slabs): the fast engine must return exactly what the exact engine (and the oracle) returns, through
every entry point, and the certificate constant must still hold at K = 3g + 3 up to 387."""
import numpy as np
import pytest

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


def fast_vs_exact(core, q, r, k, metric, **kw):
    fi, fd, st = core.knn(q, r, k, metric, mode="fast", return_stats=True, **kw)
    ei, ed = core.knn(q, r, k, metric, mode="exact", **kw)
    assert same_bits(fd, ed) and np.array_equal(fi, ei)
    return fi, fd, st


@pytest.mark.parametrize("metric", ["euclidean", "cosine"])
@pytest.mark.parametrize("g", [53, 57, 64, 65, 80, 100, 101, 127, 128])
def test_wide_fast_equals_exact(core, metric, g):
    from nabo_b200 import synth
    for i, k in enumerate([1, 10, 30, 60]):
        n, m = 1500 + 7 * g + 101 * i, 9001 + 14 * g + 517 * i
        assert n % 256 and m % 128
        q = synth.pc_mixture(n, g, seed=101 + i)
        r = synth.pc_mixture(m, g, seed=1 + i)
        _, _, st = fast_vs_exact(core, q, r, k, metric)
        assert st["rows_reranked"] == n, st                          # the tensor-core pass ran
        assert st["rows_exact_fallback"] <= max(2, n // 50), st


@pytest.mark.parametrize("metric", ["euclidean", "cosine"])
def test_wide_mask_nan_offset(core, metric):
    from nabo_b200 import synth
    g = 100
    q = synth.pc_mixture(1700, g, seed=101)
    r = synth.pc_mixture(7000, g, seed=1)
    q[5, 3] = np.nan
    r[17, 0] = np.nan
    mask = np.zeros(len(r), bool)
    mask[::3] = True
    for kw in (dict(ref_mask=mask), dict(idx_offset=12345), dict(ref_mask=mask, idx_offset=7)):
        fi, fd, st = fast_vs_exact(core, q, r, 20, metric, **kw)
        assert st["rows_reranked"] == len(q)
        oi, od = O.knn(q[:200], r, 20, metric, mask=kw.get("ref_mask"))
        assert same_bits(fd[:200], od) and np.array_equal(fi[:200] - kw.get("idx_offset", 0), oi)


@pytest.mark.parametrize("metric", ["euclidean", "cosine"])
def test_wide_tie_class_larger_than_kprime(core, metric):
    """100 identical references nearest to a block of queries: more ties than K' candidates, so these rows fail the
    certificate and the exact fallback answers them, in index order inside the tie class."""
    from nabo_b200 import synth
    g = 100
    r = synth.pc_mixture(9000, g, seed=11)
    q = synth.pc_mixture(700, g, seed=12)
    r[2000:2100] = r[2000]
    q[50:90] = r[2000]
    # exact distance 0: a tie whose reference-arithmetic distance rounds below 0 (cosine of a rescaled copy can) passes
    # the certificate's clamped lower bound and needs no fallback
    assert O.dist_matrix(q[50:51], r[2000:2001], metric)[0, 0] == 0.0
    fi, fd, st = fast_vs_exact(core, q, r, 30, metric)
    assert (fi[50:90] == np.arange(2000, 2030)[None, :]).all()
    assert 40 <= st["rows_exact_fallback"] < 100


@pytest.mark.parametrize("g", [64, 128])
def test_wide_self_knn_with_duplicates(core, g):
    from nabo_b200 import synth
    r = synth.pc_mixture(6000, g, seed=1)
    r[100:140] = r[100]                   # 40 identical cells: more ties than candidates for k = 15
    r[7] = r[8]
    fi, fd, st = fast_vs_exact(core, r, r, 15, "euclidean", drop_first=True)
    assert st["rows_reranked"] == len(r)
    oi, od = O.knn(r[:300], r, 15, "euclidean", drop_first=True)
    assert same_bits(fd[:300], od) and np.array_equal(fi[:300], oi)


def _split16(x):
    hi = x.astype(np.float16).astype(np.float64)
    lo = (x - hi).astype(np.float16).astype(np.float64)
    return hi, lo


def test_wide_score_error_bound(core):
    """The certificate assumes |score_tc - score_fp64| <= 2^-16 (4|q||r| + |r|^2 + |q|^2); the wide plan sums up to
    K = 387 products per score.  Measure it on the threshold candidates of many queries and require a >= 4x margin."""
    from nabo_b200 import synth
    worst = {}
    for seed, (n, m, g, k) in enumerate([(6000, 30000, 64, 30), (4000, 20000, 100, 10), (3000, 12000, 128, 60)]):
        q = synth.pc_mixture(n, g, seed=200 + seed)
        r = synth.pc_mixture(m, g, seed=300 + seed)
        c = core.knn_candidates(q, r, k, "euclidean")
        sc = c["scal"][0]
        kp = c["cand"].shape[1]
        fin = np.isfinite(c["tau"]) & (c["cand"][:, kp - 1] >= 0)
        assert fin.mean() > 0.99
        qi = np.nonzero(fin)[0]
        rj = c["cand"][qi, kp - 1]
        qh, ql = _split16(q[qi] * sc)
        rh, rl = _split16(r[rj] * sc)
        rt, qt = rh + rl, qh + ql
        nn = (rt * rt).sum(1)
        n1 = nn.astype(np.float16).astype(np.float64)
        n2 = (nn - n1).astype(np.float16).astype(np.float64)
        n3 = (nn - n1 - n2).astype(np.float16).astype(np.float64)
        s64 = (n1 + n2 + n3) - 2.0 * ((qh * rh).sum(1) + (qh * rl).sum(1) + (ql * rh).sum(1))
        qn, rn = np.sqrt((qt * qt).sum(1)), np.sqrt(nn)
        np.testing.assert_allclose(c["qn2"][qi], (qt * qt).sum(1), rtol=1e-12)
        rel = np.abs(c["tau"][qi].astype(np.float64) - s64) / (4 * qn * rn + rn * rn + qn * qn)
        worst[g] = float(rel.max())
    print("max tensor-core score error / bound term by g: %s (certificate constant 2^-16 = %.3e)"
          % (", ".join("%d: %.3e" % kv for kv in worst.items()), 2.0 ** -16))
    assert max(worst.values()) < 2.0 ** -18


@pytest.mark.parametrize("stats", [False, True])
def test_wide_partial_last_wave(core, stats):
    """235 work items of 256 queries on 148 SMs: the re-rank of the full wave runs as a dependent launch under the
    partly filled second wave (without stats), or after the candidate kernel (with stats)."""
    from nabo_b200 import synth
    g = 100
    q = synth.pc_mixture(60000, g, seed=101)
    r = synth.pc_mixture(12500, g, seed=1)
    out = core.knn(q, r, 30, "euclidean", mode="fast", return_stats=stats)
    ei, ed = core.knn(q, r, 30, "euclidean", mode="exact")
    assert same_bits(out[1], ed) and np.array_equal(out[0], ei)
    if stats:
        assert out[2]["rows_reranked"] == len(q)


@pytest.mark.parametrize("metric", ["euclidean", "cosine"])
def test_wide_few_queries_reference_split(core, metric):
    """12 work items: every item's reference range is cut into pieces (the SPLIT instances of the kernel)."""
    from nabo_b200 import synth
    g = 100
    q = synth.pc_mixture(3000, g, seed=101)
    r = synth.pc_mixture(40000, g, seed=1)
    _, _, st = fast_vs_exact(core, q, r, 30, metric)
    assert st["rows_reranked"] == len(q)


def test_wide_routed_output(core):
    import torch
    from nabo_b200 import synth
    g, k = 100, 30
    q = torch.from_numpy(synth.pc_mixture(5000, g, seed=101)).cuda()
    r = torch.from_numpy(synth.pc_mixture(20000, g, seed=1)).cuda()
    pi, pd = core.knn(q, r, k, "euclidean", idx_offset=7)
    bounds = [0, 2345, 5000]
    bi = [torch.full((bounds[p + 1] - bounds[p], k), -9, dtype=torch.int32, device="cuda") for p in range(2)]
    bd = [torch.full((bounds[p + 1] - bounds[p], k), -9.0, dtype=torch.float64, device="cuda") for p in range(2)]
    core.knn(q, r, k, "euclidean", idx_offset=7,
             out_parts=(bounds, [b.data_ptr() for b in bi], [b.data_ptr() for b in bd]))
    assert torch.equal(torch.cat(bi), pi) and torch.equal(torch.cat(bd).view(torch.int64), pd.view(torch.int64))


def test_wide_mapping_drop_in(core, tmp_path):
    """Mapping with use_comps = 100: the reference graph (Euclidean) and a cosine target mapping store the same
    neighbour tables and edges whether the fast or the exact engine computed them."""
    from nabo_b200 import Mapping, Graph, store, synth
    g, k = 100, 15
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
        m.set_parameters(100, k, 0.25, 64)
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
