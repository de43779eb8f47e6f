"""Tensor-core candidate pass (tcgen05) + certificate: the fast engine must return exactly
what the exact engine (and the oracle) returns, and the certificate constant must hold."""
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


@pytest.mark.parametrize("metric", ["euclidean", "cosine"])
@pytest.mark.parametrize("n,m,g,k", [(3000, 20000, 50, 30), (500, 1300, 25, 10), (1000, 5000, 15, 64), (129, 385, 52, 5)])
def test_fast_equals_exact(core, metric, n, m, g, k):
    from nabo_b200 import synth
    q = synth.pc_mixture(n, g, seed=101)
    r = synth.pc_mixture(m, g, seed=1)
    fi, fd, st = core.knn(q, r, k, metric, mode="fast", return_stats=True)
    ei, ed = core.knn(q, r, k, metric, mode="exact")
    assert same_bits(fd, ed) and np.array_equal(fi, ei)
    assert st["rows_reranked"] == n
    assert st["rows_exact_fallback"] <= max(2, n // 50), st     # the certificate clears almost every row


def test_fast_self_knn_with_duplicates(core):
    from nabo_b200 import synth
    r = synth.pc_mixture(6000, 50, seed=1)
    r[100:140] = r[100]                   # 40 identical cells: more ties than candidates for k=15
    r[7] = r[8]
    fi, fd, st = core.knn(r, r, 15, "euclidean", drop_first=True, mode="fast", return_stats=True)
    ei, ed = core.knn(r, r, 15, "euclidean", drop_first=True, mode="exact")
    assert same_bits(fd, ed) and np.array_equal(fi, ei)
    oi, od = O.knn(r[:300], r, 15, "euclidean", drop_first=True)
    assert same_bits(fd[:300], od) and np.array_equal(fi[:300], oi)


@pytest.mark.parametrize("metric", ["euclidean", "cosine"])
def test_fast_tie_class_larger_than_the_rerank_width(core, metric):
    """100 identical reference cells that are the nearest neighbours of a block of queries: the final histogram cut
    of the fused re-rank keeps more than its 64 slots, the sort path takes over, the certificate fails on the tie
    and the exact engine answers - index order inside the tie class."""
    from nabo_b200 import synth
    r = synth.pc_mixture(9000, 50, seed=11)
    q = synth.pc_mixture(700, 50, seed=12)
    r[2000:2100] = r[2000]
    q[50:90] = r[2000] * (1.0 + 1e-9)
    fi, fd, st = core.knn(q, r, 30, metric, mode="fast", return_stats=True)
    ei, ed = core.knn(q, r, 30, metric, mode="exact")
    assert same_bits(fd, ed) and np.array_equal(fi, ei)
    assert (fi[50:90] == np.arange(2000, 2030)[None, :]).all()
    assert 40 <= st["rows_exact_fallback"] < 100


def test_fast_mask_nan_offset(core):
    from nabo_b200 import synth
    q = synth.pc_mixture(700, 30, seed=101)
    r = synth.pc_mixture(3000, 30, seed=1)
    q[5, 3] = np.nan
    r[17, 0] = np.nan
    mask = np.zeros(3000, bool)
    mask[::3] = True
    for kw in (dict(ref_mask=mask), dict(idx_offset=12345), dict(ref_mask=mask, idx_offset=7)):
        fi, fd = core.knn(q, r, 20, "euclidean", mode="fast", **kw)
        ei, ed = core.knn(q, r, 20, "euclidean", mode="exact", **kw)
        assert same_bits(fd, ed) and np.array_equal(fi, ei)
    off = mask.copy()
    off[:] = True
    off[:10] = False                       # only 10 usable references, k = 20 -> masked tail
    fi, fd = core.knn(q, r, 20, "euclidean", ref_mask=off, mode="fast")
    ei, ed = core.knn(q, r, 20, "euclidean", ref_mask=off, mode="exact")
    assert same_bits(fd, ed) and np.array_equal(fi, ei)


def test_fast_badly_scaled_inputs(core):
    """Power-of-two rescaling keeps huge / tiny coordinates inside FP16 range."""
    from nabo_b200 import synth
    for scale in (1e-6, 1.0, 3e5):
        q = synth.pc_mixture(400, 20, seed=101) * scale
        r = synth.pc_mixture(2500, 20, seed=1) * scale
        fi, fd, st = core.knn(q, r, 12, "euclidean", mode="fast", return_stats=True)
        ei, ed = core.knn(q, r, 12, "euclidean", mode="exact")
        assert same_bits(fd, ed) and np.array_equal(fi, ei)
        assert st["rows_exact_fallback"] <= 8, (scale, st)


def test_fast_outlier_query_shrinks_the_scale(core):
    """One query ~400x larger than every reference norm fixes the power-of-two scale, so all other vectors land
    below 0.25 in scaled units, where the FP16 low halves are subnormal and the split error is absolute, not
    relative; the certificate carries an absolute slack term for that (fast.cu, cert.abs_slack).  Near-tie rows
    must still come out exactly as the exact engine gives them."""
    from nabo_b200 import synth
    rng = np.random.default_rng(9)
    r = synth.pc_mixture(6000, 50, seed=1) * 0.02
    q = synth.pc_mixture(900, 50, seed=101) * 0.02
    q[0] *= 400.0
    # near ties around the k-th rank: pairs of references at almost the same distance from a query
    for t in range(1, 60):
        v = rng.normal(size=50)
        v /= np.linalg.norm(v)
        r[100 + 2 * t] = q[t] + 0.05 * v
        r[101 + 2 * t] = q[t] - 0.05 * (1 + 3e-8) * v
    for k in (1, 2, 12):
        fi, fd, st = core.knn(q, r, k, "euclidean", mode="fast", return_stats=True)
        ei, ed = core.knn(q, r, k, "euclidean", mode="exact")
        assert same_bits(fd, ed) and np.array_equal(fi, ei), k


def _split16(x):
    hi = x.astype(np.float16).astype(np.float64)
    lo = (x - hi).astype(np.float16).astype(np.float64)
    return hi, lo


def test_tc_score_error_bound(core):
    """The certificate assumes |score_tc - score_fp64| <= 2^-16 (4|q||r| + |r|^2 + |q|^2).
    Measure it on the threshold candidates of many queries and require a >= 4x margin."""
    from nabo_b200 import synth
    worst = 0.0
    for seed, (n, m, g, k) in enumerate([(6000, 30000, 50, 30), (4000, 9000, 25, 10), (3000, 4000, 52, 60)]):
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
        worst = max(worst, float(rel.max()))
    print("max tensor-core score error / bound term = %.3e (certificate constant 2^-16 = %.3e)" % (worst, 2.0 ** -16))
    assert worst < 2.0 ** -18


@pytest.mark.parametrize("n_bad", [5, 700, 3000])
def test_fallback_paths(core, n_bad):
    """Uncertified rows: few -> reference-split exact pass + merge; many (> 2048) -> row-parallel exact pass."""
    from nabo_b200 import synth
    q = synth.pc_mixture(4000, 25, seed=101)
    r = synth.pc_mixture(9000, 25, seed=1)
    r[100:160] = r[100]                                   # 60 identical references
    bad = np.random.default_rng(1).choice(4000, n_bad, replace=False)
    q[bad] = r[100]                                       # ... that are the nearest cells of these queries: ties > K'
    q[bad[: n_bad // 2], 3] = np.nan                      # and NaN rows
    for kw in (dict(), dict(drop_first=True), dict(idx_offset=77)):
        fi, fd, st = core.knn(q, r, 20, "euclidean", mode="fast", return_stats=True, **kw)
        ei, ed = core.knn(q, r, 20, "euclidean", mode="exact", **kw)
        assert st["rows_exact_fallback"] >= n_bad
        assert same_bits(fd, ed) and np.array_equal(fi, ei)
    fi, fd, st = core.knn(q, r, 20, "mod_canberra", 0.25, mode="fast", return_stats=True)
    ei, ed = core.knn(q, r, 20, "mod_canberra", 0.25, mode="exact")
    assert same_bits(fd, ed) and np.array_equal(fi, ei)


@pytest.mark.parametrize("f", [0.05, 0.25, 1.5])
def test_canberra_threshold_adversarial(core, f):
    """Modified Canberra fast path: the sliced pass over-counts unsaturated dimensions over widened bin intervals
    and scores the survivors in FP32; both must stay LOWER bounds.  References are built so that, for their query, most
    dimensions sit within 1e-3 .. 1e-7 (relative) of the saturation boundary |x-y| = f|x|, with column
    magnitudes from 1e-6 to 1e5 and a few zeros / tiny values; a violated bound would drop a true neighbour."""
    rng = np.random.default_rng(int(f * 100))
    nq, per, g, k = 300, 12, 24, 10
    mag = 10.0 ** rng.uniform(-6, 5, size=g)
    q = rng.normal(size=(nq, g)) * mag
    q[:, 3] *= 1e-3
    q[rng.random((nq, g)) < 0.02] = 0.0
    refs = []
    for rep in range(per):
        delta = rng.choice([1e-3, -1e-3, 1e-4, -1e-4, 1e-5, -1e-5, 1e-7, -1e-7, 0.0], size=(nq, g))
        sign = rng.choice([-1.0, 1.0], size=(nq, g))
        y = q * (1.0 + sign * f * (1.0 - delta))
        far = rng.random((nq, g)) < 0.25 + 0.05 * rep           # some dimensions clearly saturated
        y[far] = (q * 3.0 + mag[None, :])[far]
        refs.append(y)
    r = np.concatenate(refs + [rng.normal(size=(2000, g)) * mag])
    r = r[rng.permutation(len(r))]
    fi, fd, st = core.knn(q, r, k, "mod_canberra", f, mode="fast", return_stats=True)
    ei, ed = core.knn(q, r, k, "mod_canberra", f, mode="exact")
    assert same_bits(fd, ed) and np.array_equal(fi, ei)
    oi, od = O.knn(q[:64], r, k, "mod_canberra", f)
    assert same_bits(fd[:64], od) and np.array_equal(fi[:64], oi)


@pytest.mark.parametrize("n,m,g,k,f", [
    (1, 200, 50, 30, 0.25),            # one query, one warp, two reference tiles
    (33, 129, 5, 3, 0.25),             # ragged everywhere: 2 query groups, 1 reference beyond a tile, g < 8
    (1000, 4097, 13, 15, 0.1),         # g = 8 + 5
    (5000, 30000, 25, 10, 0.25),       # config-1 width
    (4800, 20000, 50, 30, 0.5),        # 150 query groups: every SM gets one or two
    (700, 9000, 56, 20, 0.25),         # widest g of the sliced pass
    (700, 9000, 64, 20, 0.25),         # past it: the wide plan
    (300, 3000, 80, 8, 2.0),           # wide plan; f > 1 (intervals straddle zero)
    (300, 3000, 40, 8, 2.0),
    (300, 3000, 20, 8, 1e-9),          # vanishing dist_factor: exact engine (margin of the sliced pass too thin)
    (300, 3000, 20, 8, 1e-4),
])
def test_canberra_sliced_shapes(core, n, m, g, k, f):
    """Bit-sliced Canberra pass (bin planes + carry-save count + FP32 evaluation): same result as the exact
    engine over ragged shapes, and the certificate must actually clear the rows (a silently wrong bound
    would show up as mass fallback, not as a wrong answer)."""
    from nabo_b200 import synth
    q = synth.pc_mixture(n, g, seed=7)
    r = synth.pc_mixture(m, g, seed=8)
    fi, fd, st = core.knn(q, r, k, "mod_canberra", f, mode="fast", return_stats=True)
    ei, ed = core.knn(q, r, k, "mod_canberra", f, mode="exact")
    assert same_bits(fd, ed) and np.array_equal(fi, ei)
    if g <= 64 and f >= 0.05:            # wider inputs run on the exact engine; with a vanishing f every pair ties at d = g
        assert st["rows_exact_fallback"] <= max(2, n // 50)


def test_canberra_sliced_degenerate_values(core):
    """Bin edges and interval ends on awkward data: integer-valued columns (every value sits on a bin edge),
    constant and all-zero columns (all edges equal, empty intervals), huge / tiny magnitudes, NaN and inf
    entries, masked references and self-mapping with the first neighbour dropped."""
    rng = np.random.default_rng(5)
    n, m, g, k = 900, 6000, 20, 12
    r = rng.normal(size=(m, g))
    r[:, 0] = rng.integers(-3, 4, size=m)                 # few distinct values, many exact ties with the edges
    r[:, 1] = 2.5                                         # constant
    r[:, 2] = 0.0                                         # zero: |x - y| < f|x| is never true
    r[:, 3] *= 1e30
    r[:, 4] *= 1e-30
    r[:, 5] = np.round(r[:, 5], 1)
    q = r[rng.choice(m, n, replace=False)] * (1.0 + 0.05 * rng.normal(size=(n, g)))
    q[:, 0] = rng.integers(-3, 4, size=n)
    q[5, 7] = np.nan
    q[6, 8] = np.inf
    r[17, 9] = np.nan
    r[18, 9] = -np.inf
    mask = rng.random(m) < 0.3
    for kw in (dict(), dict(ref_mask=mask), dict(idx_offset=11)):
        fi, fd, st = core.knn(q, r, k, "mod_canberra", 0.25, mode="fast", return_stats=True, **kw)
        ei, ed = core.knn(q, r, k, "mod_canberra", 0.25, mode="exact", **kw)
        assert same_bits(fd, ed) and np.array_equal(fi, ei)
    oi, od = O.knn(q[:40], r, k, "mod_canberra", 0.25, mask=mask)
    fi, fd = core.knn(q[:40], r, k, "mod_canberra", 0.25, ref_mask=mask, mode="fast")
    assert same_bits(fd, od) and np.array_equal(fi, oi)
    si, sd = core.knn(r[:2000], r[:2000], k, "mod_canberra", 0.25, drop_first=True, mode="fast")
    ei, ed = core.knn(r[:2000], r[:2000], k, "mod_canberra", 0.25, drop_first=True, mode="exact")
    assert same_bits(sd, ed) and np.array_equal(si, ei)


@pytest.mark.parametrize("metric", ["euclidean", "cosine", "mod_canberra"])
@pytest.mark.parametrize("n,m", [(700, 20000), (3000, 40000), (9000, 30000)])
def test_reference_split_for_small_query_sets(core, metric, n, m):
    """Few queries: the candidate kernels cut the reference range into pieces swept by different CTAs and the
    re-rank takes the union of the pieces' K' lists with the smallest threshold.  Same result as the exact engine,
    with masks, duplicates, drop_first and an index offset, and the rows must still certify."""
    from nabo_b200 import synth
    rng = np.random.default_rng(n + m)
    r = synth.pc_mixture(m, 50, seed=1)
    q = synth.pc_mixture(n, 50, seed=2)
    r[rng.integers(0, m, 50)] = r[7]                       # ties that straddle the pieces
    q[:20] = r[rng.integers(0, m, 20)]
    mask = rng.random(m) < 0.1
    for kw in (dict(), dict(ref_mask=mask, idx_offset=5)):
        fi, fd, st = core.knn(q, r, 30, metric, 0.25, mode="fast", return_stats=True, **kw)
        ei, ed = core.knn(q, r, 30, metric, 0.25, mode="exact", **kw)
        assert same_bits(fd, ed) and np.array_equal(fi, ei)
        assert st["rows_exact_fallback"] <= max(60, n // 20)
    si, sd = core.knn(r[:n], r, 15, metric, 0.25, drop_first=True, mode="fast")
    ei, ed = core.knn(r[:n], r, 15, metric, 0.25, drop_first=True, mode="exact")
    assert same_bits(sd, ed) and np.array_equal(si, ei)


@pytest.mark.parametrize("metric", ["euclidean", "cosine"])
@pytest.mark.parametrize("n,m", [(65000, 13000), (100000, 12500), (75000, 20011)])
def test_partial_last_wave_equals_exact(core, metric, n, m):
    """More query items than SMs with a partly filled last wave: the re-rank of the queries of the full waves is a
    dependent launch that runs under the candidate kernel's last wave.  The per-stage timing pass (return_stats) runs
    the same call without that overlap.  Both must return exactly what the exact engine returns."""
    import torch
    from nabo_b200 import synth
    g, k = 50, 30
    q = torch.from_numpy(synth.pc_mixture(n, g, seed=101)).cuda()
    r = torch.from_numpy(synth.pc_mixture(m, g, seed=1)).cuda()
    r[17] = r[m - 5]                                    # a tie between the first and the last reference tile
    q[3] = r[17]
    mask = torch.zeros(m, dtype=torch.bool, device="cuda")
    mask[::7] = True
    for kw in (dict(), dict(ref_mask=mask, idx_offset=11)):
        oi, od = core.knn(q, r, k, metric, mode="fast", **kw)
        fi, fd, st = core.knn(q, r, k, metric, mode="fast", return_stats=True, **kw)
        ei, ed = core.knn(q, r, k, metric, mode="exact", **kw)
        assert torch.equal(oi, ei) and torch.equal(od.view(torch.int64), ed.view(torch.int64))
        assert torch.equal(fi, ei) and torch.equal(fd.view(torch.int64), ed.view(torch.int64))
        assert st["candidates_per_row"] == 38 and st["rows_exact_fallback"] < n // 100


def test_few_uncertified_rows_against_a_large_reference(core):
    """A handful of rows the certificate cannot clear (NaN coordinate, more exact ties than candidates) against
    >= 262 144 references take the few-rows split of the exact fallback (two reference pieces per SM, block-wide
    merge); more rows take the 48-piece split.  Both must return what the exact engine returns."""
    import torch
    from nabo_b200 import synth
    m, g, k = 300_000, 20, 10
    r = synth.pc_mixture(m, g, seed=1)
    r[1000:1060] = r[1000]                          # 60 identical cells: a tie class larger than K'
    for n_bad in (3, 200):
        q = synth.pc_mixture(3000, g, seed=101)
        q[9] = r[1000]
        q[11] = r[1000] + 1e-9
        bad = np.arange(20, 20 + n_bad)
        q[bad, 3] = np.nan
        qd, rd = torch.from_numpy(q).cuda(), torch.from_numpy(r).cuda()
        for kw in (dict(), dict(drop_first=True, idx_offset=5)):
            fi, fd, st = core.knn(qd, rd, k, "euclidean", mode="fast", return_stats=True, **kw)
            ei, ed = core.knn(qd, rd, k, "euclidean", mode="exact", **kw)
            assert st["rows_exact_fallback"] >= n_bad + 1
            assert torch.equal(fi, ei)
            assert same_bits(fd.cpu().numpy(), ed.cpu().numpy())
