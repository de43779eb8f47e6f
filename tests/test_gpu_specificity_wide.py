"""Mapping specificity for targets with 65 to 128 mapped reference cells: the 128-source (two-word) instance of the
bit-parallel multi-source search must give the oracle's means bit for bit, flag unconnected pairs, agree with the
64-source instance wherever both apply, and run end to end through Mapping and Graph at k = 100."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp
from scipy.sparse.csgraph import shortest_path

from oracle import nabo_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def core():
    from nabo_b200 import build, core as c
    build.build()
    return c


def csr(a, b, m):
    keep = a != b
    adj = sp.coo_matrix((np.ones(2 * keep.sum(), np.int8), (np.r_[a[keep], b[keep]], np.r_[b[keep], a[keep]])),
                        shape=(m, m)).tocsr()
    adj.sum_duplicates()
    return adj


def hop_means(adj, knn, cnt):
    """Exact per-target means from one scipy BFS per mapped cell, for graphs where the Python oracle would be slow on
    every row (it is then run on a subset).  NaN below two mapped cells, None without a path."""
    mapped = [[int(r) for r, c in zip(knn[t], cnt[t]) if c > 0 and r >= 0] for t in range(len(knn))]
    cells = sorted({r for row in mapped for r in row})
    pos = {r: i for i, r in enumerate(cells)}
    d = shortest_path(adj, unweighted=True, indices=cells) if cells else None
    out = []
    for row in mapped:
        if len(row) < 2:
            out.append(np.nan)
            continue
        s = [d[pos[row[i]], row[j]] for i in range(len(row)) for j in range(i + 1, len(row))]
        out.append(None if np.isinf(s).any() else float(sum(int(x) for x in s)) / len(s))
    return out


def raw_call(knn, cnt, adj, nbytes=None):
    """nabo_mapping_specificity itself: (status, out_sum, out_pairs, out_nmapped)."""
    import torch
    from nabo_b200 import _lib
    L = _lib.lib()
    n, k = knn.shape
    ip = torch.from_numpy(adj.indptr.astype(np.int64)).cuda()
    ix = torch.from_numpy(adj.indices.astype(np.int32)).cuda()
    td = torch.from_numpy(np.ascontiguousarray(knn, np.int32)).cuda()
    cd = torch.from_numpy(np.ascontiguousarray(cnt, np.uint8)).cuda()
    osum = torch.full((n,), -7, dtype=torch.int64, device="cuda")
    opairs = torch.full((n,), -7, dtype=torch.int32, device="cuda")
    onm = torch.full((n,), -7, dtype=torch.int32, device="cuda")
    if nbytes is None:
        nbytes = L.nabo_specificity_workspace_bytes_k(adj.shape[0], n, k)
    ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device="cuda")
    p = lambda x: C.c_void_p(x.data_ptr())
    rc = L.nabo_mapping_specificity(p(ip), p(ix), adj.shape[0], p(td), p(cd), n, k, p(osum), p(opairs), p(onm), p(ws),
                                    nbytes, C.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return rc, osum.cpu().numpy(), opairs.cpu().numpy(), onm.cpu().numpy()


def random_graph(m, deg, comps, rng):
    comp = rng.integers(0, comps, size=m)
    a, b = [], []
    for c in range(comps):
        nodes = np.nonzero(comp == c)[0]
        a += list(nodes); b += list(np.roll(nodes, 1))                # connected inside a component
        for _ in range(deg - 1):
            a += list(nodes); b += list(rng.permutation(nodes))
    return np.array(a), np.array(b), comp


@pytest.mark.parametrize("m,n,k,deg,comps", [(700, 150, 65, 3, 1), (1500, 150, 100, 2, 1), (1200, 150, 128, 2, 3),
                                             (400, 150, 128, 4, 1), (3000, 100, 100, 2, 2)])
def test_random_graphs_match_oracle(core, m, n, k, deg, comps):
    """Long paths, several components, targets with 0 / 1 / all k mapped cells and -1 padding."""
    rng = np.random.default_rng(m + k)
    a, b, comp = random_graph(m, deg, comps, rng)
    adj = csr(a, b, m)
    knn = np.stack([rng.choice(m, k, replace=False) for _ in range(n)]).astype(np.int32)
    cnt = (rng.random((n, k)) < 0.6).astype(np.uint8)
    cnt[0] = 0                                                      # nothing mapped
    cnt[1] = 0; cnt[1, k - 1] = 1                                   # one cell mapped, in the second word
    knn[2, ::2] = -1                                                # padding entries are not edges
    knn[3, 5:70] = -1
    cnt[4] = 1                                                      # every cell mapped
    cnt[5] = 0; cnt[5, 0] = cnt[5, k - 1] = 1                       # one cell in each word
    if comps > 1:                                                   # targets inside one component (row 6: all mapped)
        for t in range(6, 30):
            knn[t] = rng.choice(np.nonzero(comp == comp[t])[0], k, replace=False)
        cnt[6] = 1
    same = np.array([len({comp[r] for r, c in zip(knn[t], cnt[t]) if c and r >= 0}) <= 1 for t in range(n)])
    assert (~same).any() == (comps > 1)
    mean, connected = core.mapping_specificity(adj.indptr.astype(np.int64), adj.indices.astype(np.int32), knn, cnt)
    assert np.array_equal(connected, same)
    sel = np.nonzero(same)[0]
    assert np.array_equal(mean[sel], O.mapping_specificity(a, b, m, knn[sel], cnt[sel]), equal_nan=True)
    assert np.isnan(mean[0]) and np.isnan(mean[1]) and np.isfinite(mean[5]) and np.isfinite(mean[6])
    rc, osum, opairs, onm = raw_call(knn, cnt, adj)
    assert rc == 0
    nm = ((cnt > 0) & (knn >= 0)).sum(1)
    assert np.array_equal(onm, nm) and onm[4] == k
    assert np.array_equal(opairs[same], (nm * (nm - 1))[same])      # ordered pairs
    assert (opairs[~same] < (nm * (nm - 1))[~same]).all()


def structured(shape):
    if shape == "path":
        m = 300; a = np.arange(m - 1); b = a + 1
    elif shape == "cycle":
        m = 257; a = np.arange(m); b = (a + 1) % m
    elif shape == "star":
        m = 400; a = np.zeros(m - 1, dtype=int); b = np.arange(1, m)
    elif shape == "tree":
        m = 511; b = np.arange(1, m); a = (b - 1) // 2
    elif shape == "grid":
        side = 21; m = side * side
        idx = np.arange(m).reshape(side, side)
        a = np.r_[idx[:, :-1].ravel(), idx[:-1, :].ravel()]; b = np.r_[idx[:, 1:].ravel(), idx[1:, :].ravel()]
    else:
        m = 140; a, b = np.triu_indices(m, 1)
    return m, a, b


@pytest.mark.parametrize("shape", ["path", "cycle", "star", "tree", "grid", "clique"])
def test_structured_graphs_k128(core, shape):
    """Odd and even distances, long paths and hubs with 128 sources.  In the star every leaf source reaches the hub in
    the same level from both words: the hub must enter the next frontier exactly once."""
    m, a, b = structured(shape)
    adj = csr(a, b, m)
    rng = np.random.default_rng(len(shape))
    n, k = 12, 128
    knn = np.stack([rng.choice(m, k, replace=False) for _ in range(n)]).astype(np.int32)
    ext = np.r_[np.arange(32), m - 1 - np.arange(32), m // 2 + np.arange(32), m // 3 + np.arange(32)]
    knn[0] = ext if len(set(ext)) == k else rng.choice(m, k, replace=False)   # the extremes together
    if shape == "star":
        knn[1] = np.arange(1, k + 1)                                # leaves only: all meet at the hub in level 1
        knn[2] = np.arange(k)                                       # the hub and 127 leaves
    cnt = (rng.random((n, k)) < 0.8).astype(np.uint8)
    cnt[:3] = 1
    mean, connected = core.mapping_specificity(adj.indptr.astype(np.int64), adj.indices.astype(np.int32), knn, cnt)
    assert connected.all()
    exp = O.mapping_specificity(a, b, m, knn, cnt)
    assert np.array_equal(mean, exp, equal_nan=True)
    if shape == "star":
        assert mean[1] == 2.0 and mean[2] == (127 * 1 + 127 * 126 // 2 * 2) / (128 * 127 // 2)


def test_both_instances_agree(core):
    """A 40-wide table (64-source instance) and the same table spread over 100 columns with -1 padding (128-source
    instance): the same sums, pair counts and mapped-cell counts."""
    rng = np.random.default_rng(40)
    m, n, k = 2500, 400, 40
    a, b, _ = random_graph(m, 2, 2, rng)
    adj = csr(a, b, m)
    knn = np.stack([rng.choice(m, k, replace=False) for _ in range(n)]).astype(np.int32)
    cnt = (rng.random((n, k)) < 0.7).astype(np.uint8)
    cnt[0] = 0
    wide = np.full((n, 100), -1, dtype=np.int32)
    wcnt = rng.integers(0, 3, size=(n, 100)).astype(np.uint8)      # padding is skipped whatever its count
    cols = np.sort(rng.choice(100, k, replace=False))
    wide[:, cols], wcnt[:, cols] = knn, cnt
    narrow_out, wide_out = raw_call(knn, cnt, adj), raw_call(wide, wcnt, adj)
    assert narrow_out[0] == 0 and wide_out[0] == 0
    for x, y in zip(narrow_out[1:], wide_out[1:]):
        assert np.array_equal(x, y)
    nm = narrow_out[3].astype(np.int64)
    assert (narrow_out[2] < nm * (nm - 1)).any() and (narrow_out[2] == nm * (nm - 1)).any()


def _write(fn, names, mat):
    from nabo_b200 import store
    h = store.File(fn, "w")
    h.create_row_group("data", names, mat)
    h.close()


def _target_tables(gph, ref_names, tgt_names):
    """The graph's own edges as (target x mapped reference cell) tables padded with -1, and the reference edges."""
    pos = {c + "_REF": i for i, c in enumerate(ref_names)}
    rows = [[pos[x] for x in gph.neighbors(t + "_TGT") if x in pos] for t in tgt_names]
    w = max(len(r) for r in rows)
    knn = np.full((len(rows), w), -1, dtype=np.int32)
    for i, r in enumerate(rows):
        knn[i, :len(r)] = r
    ea = np.array([pos[x] for x, y in gph.refG.edges()])
    eb = np.array([pos[y] for x, y in gph.refG.edges()])
    return knn, ea, eb


@pytest.mark.parametrize("layout", ["columnar", "reference"])
def test_mapping_k100_end_to_end(core, tmp_path, layout):
    """Mapping at k = 100 (make_ref_graph, map_target) -> Graph.load_from_h5 -> get_mapping_specificity: the oracle's
    values on the stored edges, with and without fill_na, and get_ref_specificity on top."""
    from nabo_b200 import Graph, Mapping, synth
    g, k = 20, 100
    ref, tgt = synth.pc_mixture(1200, g, seed=1), synth.pc_mixture(300, g, seed=2)
    rn, tn = synth.cell_names(len(ref), "R"), synth.cell_names(len(tgt), "T")
    ref_fn, tgt_fn, map_fn = (str(tmp_path / x) for x in ("ref.h5", "tgt.h5", "map.h5"))
    _write(ref_fn, rn, ref)
    _write(tgt_fn, tn, tgt)
    m = Mapping(map_fn, "REF", ref_fn, "data", overwrite=True)
    m.graph_layout = layout
    m.set_parameters(g, k, 0.25, 64)
    m.make_ref_graph()
    m.map_target("TGT", tgt_fn, "data")
    gph = Graph()
    gph.load_from_h5(map_fn, "REF", "reference")
    gph.load_from_h5(map_fn, "TGT", "target")
    assert gph._samples["TGT"].knn.shape[1] > 64                    # the 128-source instance ran
    knn, ea, eb = _target_tables(gph, rn, tn)
    assert ((knn >= 0).sum(1) > 64).any()
    sp_raw = gph.get_mapping_specificity("TGT", fill_na=False)
    got = np.array([sp_raw[c + "_TGT"] for c in tn])
    adj = csr(ea, eb, len(rn))
    assert np.array_equal(got, np.array(hop_means(adj, knn, knn >= 0), dtype=np.float64), equal_nan=True)
    rows = np.r_[np.argsort(-(knn >= 0).sum(1))[:3], np.arange(0, len(tn), 60)]
    assert np.array_equal(got[rows], O.mapping_specificity(ea, eb, len(rn), knn[rows], knn[rows] >= 0), equal_nan=True)
    sp_fill = gph.get_mapping_specificity("TGT")
    top = max(sp_raw.values())                                      # upstream: builtin max, then fillna
    assert sp_fill == {c: (top if np.isnan(v) else v) for c, v in sp_raw.items()}
    rs = gph.get_ref_specificity("TGT", sp_fill)
    assert len(rs) > 0 and all(np.isfinite(v) for v in rs.values())


def test_disconnected_reference_raises_no_path(core, tmp_path):
    """Two far-apart mirror-image clusters with the reference-graph repair switched off: targets at the centre map
    into both components at k = 100, and get_mapping_specificity raises NetworkXNoPath as the reference does."""
    import networkx as nx
    from nabo_b200 import Graph, Mapping, synth
    g, k = 10, 100
    half = synth.pc_mixture(300, g, seed=3) * 0.1
    off = np.zeros(g); off[0] = 1000.0
    ref = np.r_[half, off - half]
    tgt = np.r_[np.tile(off / 2, (5, 1)), half[:20] + 0.01]        # the centre is as near one cluster as the other
    rn, tn = synth.cell_names(len(ref), "R"), synth.cell_names(len(tgt), "T")
    ref_fn, tgt_fn, map_fn = (str(tmp_path / x) for x in ("ref.h5", "tgt.h5", "map.h5"))
    _write(ref_fn, rn, ref)
    _write(tgt_fn, tn, tgt)
    m = Mapping(map_fn, "REF", ref_fn, "data", overwrite=True)
    m.set_parameters(g, k, 0.25, 64)
    m.make_ref_graph()
    m.calc_snn(m._refSortedDistGrp, "REF", m._refGraphGrpName, fix_graph_attempts=0)
    m.map_target("TGT", tgt_fn, "data", metric="euclidean")
    gph = Graph()
    gph.load_from_h5(map_fn, "REF", "reference")
    gph.load_from_h5(map_fn, "TGT", "target")
    assert nx.number_connected_components(gph.refG) == 2
    knn, _, _ = _target_tables(gph, rn, tn)
    both = [(r[r >= 0] < 300).any() and (r[r >= 0] >= 300).any() for r in knn]
    assert any(both) and knn.shape[1] > 64
    with pytest.raises(nx.NetworkXNoPath):
        gph.get_mapping_specificity("TGT")


def test_limits_and_exact_workspace(core):
    """A 129-wide table is refused with a message that names 128; a one-target k = 128 call runs with exactly the
    advertised workspace, and not with one byte less or with the 64-source size."""
    from nabo_b200 import _lib
    L = _lib.lib()
    rng = np.random.default_rng(129)
    m = 2000
    a, b, _ = random_graph(m, 3, 1, rng)
    adj = csr(a, b, m)
    wide = rng.choice(m, (3, 129)).astype(np.int32)
    with pytest.raises(RuntimeError, match="128"):
        core.mapping_specificity(adj.indptr.astype(np.int64), adj.indices.astype(np.int32), wide, np.ones_like(wide))
    knn = rng.choice(m, 128, replace=False).astype(np.int32)[None, :]
    cnt = np.ones_like(knn, dtype=np.uint8)
    need = L.nabo_specificity_workspace_bytes_k(m, 1, 128)
    assert need > L.nabo_specificity_workspace_bytes(m, 1)
    rc, osum, opairs, onm = raw_call(knn, cnt, adj, need)
    assert rc == 0 and onm[0] == 128 and opairs[0] == 128 * 127
    exp = O.mapping_specificity(a, b, m, knn, cnt)[0]
    assert (osum[0] // 2) / (128 * 127 // 2) == exp
    assert raw_call(knn, cnt, adj, need - 1)[0] == -2
    assert raw_call(knn, cnt, adj, L.nabo_specificity_workspace_bytes(m, 1))[0] == -2
