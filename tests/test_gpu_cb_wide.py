"""Wide plan of the bit-sliced modified-Canberra candidate pass (57 <= g <= 128: 8 warps per CTA, 8-bit sliced
counters, 64- or 32-reference tiles over the pass's own [tile32][k][32] FP32 reference copy): the fast engine must
return exactly what the exact engine (and the oracle) returns, through every entry point, and the FP32 evaluation
must stay a lower bound within nabo_cb_eps(g) at these widths."""
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


def fast_vs_exact(core, q, r, k, f, **kw):
    fi, fd, st = core.knn(q, r, k, "mod_canberra", f, mode="fast", return_stats=True, **kw)
    ei, ed = core.knn(q, r, k, "mod_canberra", f, mode="exact", **kw)
    assert same_bits(fd, ed) and np.array_equal(fi, ei)
    return fi, fd, st


@pytest.mark.parametrize("f", [0.1, 0.25, 2.0])
@pytest.mark.parametrize("g", [57, 63, 64, 65, 72, 77, 78, 100, 101, 120, 127, 128])
def test_cb_wide_fast_equals_exact(core, g, f):
    from nabo_b200 import synth
    for i, k in enumerate([1, 10, 30, 55]):
        n, m = 1500 + 7 * g + 101 * i, 9001 + 14 * g + 517 * i
        n, m = n + (n % 32 == 0), m + (m % 32 == 0)                  # ragged: no whole last group or tile
        q = synth.pc_mixture(n, g, seed=101 + i)
        r = synth.pc_mixture(m, g, seed=1 + i)
        _, _, st = fast_vs_exact(core, q, r, k, f)
        assert st["rows_reranked"] == n, st                          # the candidate pass ran
        assert st["rows_exact_fallback"] <= max(2, n // 50), st


@pytest.mark.parametrize("f", [0.05, 0.25, 1.5])
@pytest.mark.parametrize("g", [100, 128])
def test_cb_wide_threshold_adversarial(core, g, f):
    """Most dimensions of the planted references sit within 1e-3 .. 1e-7 (relative) of the saturation boundary
    |x - y| = f|x| of their query, with column magnitudes from 1e-6 to 1e5 and a few zeros: a violated lower bound
    (count over-estimate or FP32 score within nabo_cb_eps) would drop a true neighbour."""
    rng = np.random.default_rng(g + int(f * 100))
    nq, per, k = 300, 12, 10
    mag = 10.0 ** rng.uniform(-6, 5, size=g)
    q = rng.normal(size=(nq, g)) * mag
    q[:, 3] *= 1e-3
    q[rng.random((nq, g)) < 0.02] = 0.0
    refs = []
    for rep in range(per):
        delta = rng.choice([1e-3, -1e-3, 1e-4, -1e-4, 1e-5, -1e-5, 1e-7, -1e-7, 0.0], size=(nq, g))
        sign = rng.choice([-1.0, 1.0], size=(nq, g))
        y = q * (1.0 + sign * f * (1.0 - delta))
        far = rng.random((nq, g)) < 0.25 + 0.05 * rep
        y[far] = (q * 3.0 + mag[None, :])[far]
        refs.append(y)
    r = np.concatenate(refs + [rng.normal(size=(2000, g)) * mag])
    r = r[rng.permutation(len(r))]
    fi, fd, st = fast_vs_exact(core, q, r, k, f)
    assert st["rows_reranked"] == nq
    oi, od = O.knn(q[:64], r, k, "mod_canberra", f)
    assert same_bits(fd[:64], od) and np.array_equal(fi[:64], oi)


def test_cb_wide_degenerate_values(core):
    """Integer, constant and zero columns, huge / tiny magnitudes, NaN and inf, with masks, an index offset and a
    self-kNN that drops the first neighbour."""
    rng = np.random.default_rng(5)
    n, m, g, k = 900, 6000, 100, 12
    r = rng.normal(size=(m, g))
    r[:, 0] = rng.integers(-3, 4, size=m)
    r[:, 1] = 2.5
    r[:, 2] = 0.0
    r[:, 3] *= 1e30
    r[:, 4] *= 1e-30
    r[:, 5] = np.round(r[:, 5], 1)
    r[:, 60] = rng.integers(-2, 3, size=m)
    r[:, 99] = 0.0
    q = r[rng.choice(m, n, replace=False)] * (1.0 + 0.05 * rng.normal(size=(n, g)))
    q[:, 0] = rng.integers(-3, 4, size=n)
    q[5, 7] = np.nan
    q[6, 8] = np.inf
    q[7, 90] = -np.inf
    r[17, 9] = np.nan
    r[18, 9] = -np.inf
    r[19, 97] = np.inf
    mask = rng.random(m) < 0.3
    for kw in (dict(), dict(ref_mask=mask), dict(idx_offset=11), dict(ref_mask=mask, idx_offset=3)):
        fast_vs_exact(core, q, r, k, 0.25, **kw)
    oi, od = O.knn(q[:40], r, k, "mod_canberra", 0.25, mask=mask)
    fi, fd = core.knn(q[:40], r, k, "mod_canberra", 0.25, ref_mask=mask, mode="fast")
    assert same_bits(fd, od) and np.array_equal(fi, oi)
    fast_vs_exact(core, r[:2000], r[:2000], k, 0.25, drop_first=True)


def test_cb_wide_counter_top_bits(core):
    """g = 128: references that equal their query (all 128 dimensions unsaturated: count 128, the counter's top
    bit), or differ from it in 64 or in 1 saturated dimension (counts 64 and 127), and a class of 100 identical
    references nearest to a block of queries - more ties than K', answered by the fallback in index order."""
    from nabo_b200 import synth
    rng = np.random.default_rng(3)
    g, k = 128, 30
    r = synth.pc_mixture(9000, g, seed=11)
    q = synth.pc_mixture(700, g, seed=12)
    assert (q != 0).all() and (r != 0).all()
    r[2000:2100] = r[2000]                                  # tie class of 100 > K'
    q[50:90] = r[2000]
    for i in range(100, 300):                               # planted partners with 128, 127 or 64 unsaturated dims
        j = 3000 + 3 * i
        r[j] = q[i]
        r[j + 1] = q[i] * (1.0 + 0.01 * rng.normal(size=g))
        d = rng.integers(g)
        r[j + 1, d] = q[i, d] * 3.0 + np.sign(q[i, d])
        r[j + 2] = q[i] * (1.0 + 0.01 * rng.normal(size=g))
        sat = rng.choice(g, 64, replace=False)
        r[j + 2, sat] = q[i, sat] * 3.0 + np.sign(q[i, sat])
    fi, fd, st = fast_vs_exact(core, q, r, k, 0.25)
    assert (fi[50:90] == np.arange(2000, 2000 + k)[None, :]).all()
    assert 40 <= st["rows_exact_fallback"] < 100
    assert (fi[100:300, 0] == 3000 + 3 * np.arange(100, 300)).all() and (fd[100:300, 0] == 0.0).all()
    oi, od = O.knn(q[90:154], r, k, "mod_canberra", 0.25)
    assert same_bits(fd[90:154], od) and np.array_equal(fi[90:154], oi)


@pytest.mark.parametrize("n,m", [(700, 20000), (3000, 40000), (60000, 12000)])
def test_cb_wide_reference_split_and_rounds(core, n, m):
    """Few queries: the reference range is cut into pieces (the SPLIT instances).  60 000 queries on 148 CTAs of
    8 warps: every CTA sweeps the reference more than once."""
    from nabo_b200 import synth
    rng = np.random.default_rng(n + m)
    g = 100
    r = synth.pc_mixture(m, g, seed=1)
    q = synth.pc_mixture(n, g, seed=2)
    r[rng.integers(0, m, 50)] = r[7]
    q[:20] = r[rng.integers(0, m, 20)]
    mask = rng.random(m) < 0.1
    for kw in (dict(), dict(ref_mask=mask, idx_offset=5)):
        _, _, st = fast_vs_exact(core, q, r, 30, 0.25, **kw)
        assert st["rows_reranked"] == n
        assert st["rows_exact_fallback"] <= max(60, n // 20)
    fast_vs_exact(core, r[:min(n, m)], r, 15, 0.25, drop_first=True)


def test_cb_wide_routed_output(core):
    import torch
    from nabo_b200 import synth
    g, k = 100, 30
    q = torch.from_numpy(synth.pc_mixture(5000, g, seed=101)).cuda()
    r = torch.from_numpy(synth.pc_mixture(20000, g, seed=1)).cuda()
    pi, pd = core.knn(q, r, k, "mod_canberra", 0.25, idx_offset=7)
    bounds = [0, 2345, 5000]
    bi = [torch.full((bounds[p + 1] - bounds[p], k), -9, dtype=torch.int32, device="cuda") for p in range(2)]
    bd = [torch.full((bounds[p + 1] - bounds[p], k), -9.0, dtype=torch.float64, device="cuda") for p in range(2)]
    core.knn(q, r, k, "mod_canberra", 0.25, idx_offset=7,
             out_parts=(bounds, [b.data_ptr() for b in bi], [b.data_ptr() for b in bd]))
    assert torch.equal(torch.cat(bi), pi) and torch.equal(torch.cat(bd).view(torch.int64), pd.view(torch.int64))


def test_cb_wide_mapping_drop_in(core, tmp_path):
    """Mapping with use_comps = 100 and map_target's default metric (modified Canberra): the stored neighbour tables
    and graph edges are the same whether the fast or the exact engine computed them."""
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
        m.map_target("TGT", tgt_fn, "data", mode=mode)
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


def test_cb_wide_vanishing_dist_factor(core):
    """f = 1e-9 is below the sliced pass's interval margin: the call runs on the exact engine at every width."""
    from nabo_b200 import synth
    for g in (20, 50, 100):
        q = synth.pc_mixture(300, g, seed=7)
        r = synth.pc_mixture(3000, g, seed=8)
        _, _, st = fast_vs_exact(core, q, r, 8, 1e-9)
        assert st["rows_exact_fallback"] == len(q) and st["kernel_launches"] == 1, (g, st)
