"""``Mapping``: the reference's mapping call surface on top of the CUDA path.

Drop-in for ``nabo.Mapping`` (nabo/_mapping.py:280-621): same constructor and methods,
same exceptions, same mapping-file group names (``name_stash``, ``ref_cells``,
``<uid>_dist``, ``<uid>_sortedDist``, ``<uid>_graph``).  What changes:

* distances + sorting are one fused CUDA call (``core.knn``); the N x M matrix and the
  N x M argsort are never materialised, so ``<uid>_dist`` / ``<uid>_sortedDist`` hold the
  k(+1) best entries of each row (everything ``_calc_snn`` ever reads, :190/:193) as
  columnar ``RowGroup``s; ``<uid>_dist/<cell>[j]`` is the distance to
  ``<uid>_sortedDist/<cell>[j]``;
* ``<uid>_graph`` is columnar (``nodes``, ``knn``, ``snn``, ``k``, optional repair edges)
  instead of one string-encoded dataset per node (:252-273); ``Graph.load_from_h5``
  reads both layouts, and ``Mapping.graph_layout = 'reference'`` (or ``calc_snn(...,
  graph_layout='reference')``) writes the reference's own per-node layout, which the unmodified
  ``nabo.Graph`` reads (tests/golden/verify_reference_reader.py);
* ``chunk_size`` is accepted and validated but has no effect (results never depended on
  it, :106-128);
* new keyword-only extensions with reference-preserving defaults: ``metric`` (None ->
  Euclidean for the reference graph, modified Canberra for targets, :433-440; or any of
  'euclidean', 'mod_canberra', 'cosine', 'correlation' - Pearson correlation distance, scanpy's
  and scipy's ``correlation``) and ``mode`` ('fast' | 'exact').
"""
from __future__ import annotations

import os
import random
import string
from typing import Dict, List, Optional, Tuple

import numpy as np

from . import core
from .store import batched_writes, RowGroup, open_file

__all__ = ["Mapping", "read_matrix"]


def random_string(n: int = 30) -> str:
    # nabo/_mapping.py:276-277 (global `random`, so random.seed() controls it as upstream)
    return "".join(random.choice(string.ascii_lowercase) for _ in range(n))


def read_matrix(grp, use_comps: Optional[int] = None) -> Tuple[List[str], np.ndarray]:
    """(cell names in HDF5 iteration order = bytewise sorted, matrix of their vectors).

    Accepts the reference layout (one dataset per cell, nabo/_dataset.py:1028) and the
    columnar ``RowGroup``.  Neighbour indices everywhere are positions in this order
    (nabo/_mapping.py:79, 403-405)."""
    if isinstance(grp, RowGroup):
        names = list(grp)                                   # sorted
        pos = grp._idx()
        rows = np.fromiter((pos[n] for n in names), dtype=np.int64, count=len(names))
        mat = np.asarray(grp.data)[rows]
    else:
        names = [x for x in grp]
        mat = np.array([np.asarray(grp[n][:]) for n in names], dtype=np.float64) if names else np.zeros((0, 0))
    mat = np.ascontiguousarray(mat, dtype=np.float64)
    if use_comps is not None:
        mat = np.ascontiguousarray(mat[:, :use_comps])
    return names, mat


class Mapping:
    """See nabo.Mapping.  :param mapping_h5_fn: output file; :param ref_name: label of the
    reference sample; :param ref_pca_fn / ref_pca_grp_name: PCA file + group of the reference;
    :param overwrite: wipe the mapping file first."""

    def __init__(self, mapping_h5_fn: str, ref_name: str, ref_pca_fn: str, ref_pca_grp_name: str,
                 overwrite: bool = False):
        self._h5Fn: str = mapping_h5_fn
        if ref_name.find("__") != -1:
            raise ValueError("ERROR: Underscores are not allowed in the value for `ref_name` parameter")
        self.refName: str = ref_name
        self._refPcaFn: str = ref_pca_fn
        self._refPcaGrp: str = ref_pca_grp_name
        if self._h5Fn == self._refPcaFn:
            raise ValueError("ERROR: Input HDF5 and output HDF5 file cannot be same")
        self._check_h5(self._refPcaFn, self._refPcaGrp)
        self.refCells: List[str] = []
        self._nameStash: Dict[str, str] = {}
        self._check_preload(overwrite)
        uid = self._nameStash[self.refName]
        self._refDistGrp = uid + "_dist"
        self._refSortedDistGrp = uid + "_sortedDist"
        self._refGraphGrpName = uid + "_graph"
        self._useComps = None
        self._k = None
        self.graph_layout = "columnar"      # 'reference' = per-node datasets as nabo's _dump_graph writes them
        self._distFactor = None
        self._chunkSize = None
        self._refMatCache = None
        self._refPrepCache = None       # (key, core.PreparedReference) of the last calc_dist, see _prepared_ref

    # ------------------------------------------------------------------ files
    @staticmethod
    def _check_h5(fn: str, group: str) -> bool:
        if os.path.exists(fn) is False:
            raise ValueError("File %s doesn't exist" % fn)
        h5 = open_file(fn, mode="r")
        ok = group in h5
        h5.close()
        if not ok:
            raise ValueError("Group %s does not exist in file %s" % (group, fn))
        return True

    def _load_ref_cells(self) -> List[str]:
        h5 = open_file(self._refPcaFn, mode="r")
        cells = [x for x in h5[self._refPcaGrp]]
        h5.close()
        return cells

    def _create_metadata(self, h5) -> bool:
        for i in list(h5.keys()):
            del h5[i]
        grp = h5.create_group("name_stash")
        rs = random_string(30)
        self._nameStash[self.refName] = rs
        grp.create_dataset("ref_name", data=[self.refName.encode("ascii"), rs.encode("ascii")])
        self.refCells = self._load_ref_cells()
        grp = h5.create_group("ref_cells")
        grp.create_dataset("ref_cells", data=[x.encode("ascii") for x in self.refCells])
        return True

    def _check_preload(self, overwrite: bool):
        h5 = open_file(self._h5Fn, mode="a")
        if overwrite is True:
            self._create_metadata(h5)
        else:
            if "ref_cells" in h5 and "ref_cells" in h5["ref_cells"] and "name_stash" in h5 and \
                    "ref_name" in h5["name_stash"]:
                ref_name = h5["name_stash/ref_name"][0].decode("UTF-8")
                if ref_name != self.refName:
                    h5.close()
                    raise ValueError("ERROR: A different ref_name was used before for this mapping file. "
                                     "Please set overwrite=True if you want to overwrite all the saved data.")
                if "target_names" in h5["name_stash"]:
                    for i in h5["name_stash/target_names"]:
                        self._nameStash[i[0].decode("UTF-8")] = i[1].decode("UTF-8")
                self._nameStash[self.refName] = h5["name_stash/ref_name"][1].decode("UTF-8")
                saved_cells = [x.decode("UTF-8") for x in h5["ref_cells/ref_cells"][:]]
                pca_cells = self._load_ref_cells()
                intersect = set(saved_cells).intersection(pca_cells)
                if len(saved_cells) == len(pca_cells) == len(intersect):
                    self.refCells = saved_cells
                else:
                    h5.close()
                    raise ValueError("ERROR: Cell names in PCA file does not match those used before in this "
                                     "mapping file. Please set overwrite=True if you want to overwrite all the "
                                     "saved data.")
            else:
                self._create_metadata(h5)
        h5.close()

    def _stash_target_name(self, target: str):
        h5 = open_file(self._h5Fn, mode="a")
        if "target_names" in h5["name_stash"]:
            del h5["name_stash/target_names"]
        self._nameStash[target] = random_string(30)
        stash = [[i.encode("ascii"), self._nameStash[i].encode("ascii")] for i in self._nameStash
                 if i != self.refName]
        h5["name_stash"].create_dataset("target_names", data=stash)
        h5.close()

    # ------------------------------------------------------------------ parameters
    def set_parameters(self, use_comps: int, k: int, dist_factor: float, chunk_size: int) -> None:
        """nabo/_mapping.py:495-524."""
        self._useComps = use_comps
        self._k = k
        try:
            float(dist_factor)
            assert (dist_factor > 0)
        except (ValueError, AssertionError, TypeError):
            raise ValueError('ERROR: "dist_factor" must be a non-zero float value')
        self._distFactor = dist_factor
        self._chunkSize = chunk_size
        self._refMatCache = None
        self._refPrepCache = None
        return None

    def _ref_matrix(self) -> np.ndarray:
        """Reference PCA rows in self.refCells order, first use_comps columns."""
        if self._refMatCache is None:
            h5 = open_file(self._refPcaFn, mode="r")
            names, mat = read_matrix(h5[self._refPcaGrp], self._useComps)
            h5.close()
            if names != self.refCells:                     # saved order wins (_mapping.py:383)
                pos = {n: i for i, n in enumerate(names)}
                mat = np.ascontiguousarray(mat[[pos[c] for c in self.refCells]])
            self._refMatCache = mat
        return self._refMatCache

    def _prepared_ref(self, metric: str, ignore_ref_cells: List[str], mask) -> Optional["core.PreparedReference"]:
        """The reference packed for (use_comps, metric, ignore_ref_cells), kept between calc_dist calls so that
        mapping several targets uploads and packs the reference once.  One is kept at a time (its device memory:
        the FP64 rows plus about 31 MB per 100 k references at use_comps = 50, and for correlation the centred
        copy of the rows, 40 MB per 100 k references at use_comps = 50).  None where no prepared form
        exists (use_comps > core.PREPARED_MAX_G): the call then takes the host matrix."""
        key = (self._useComps, metric, frozenset(ignore_ref_cells))
        if self._refPrepCache is not None and self._refPrepCache[0] == key:
            return self._refPrepCache[1]
        ref = self._ref_matrix()
        if ref.shape[1] > core.PREPARED_MAX_G:
            return None
        self._refPrepCache = None                           # release the previous one before packing
        pr = core.prepare_reference(ref, metric, mask)
        self._refPrepCache = (key, pr)
        return pr

    # ------------------------------------------------------------------ distances + top-k
    def calc_dist(self, target_fn: str, target_grp: str, dist_grp: str, sorted_dist_grp: str,
                  ignore_ref_cells: List[str], *, metric: Optional[str] = None, mode: str = "fast") -> None:
        """nabo/_mapping.py:408-444 + _calc_dist :48-148, fused on the GPU.  Writes the k (+1 for
        the reference) best (distance, index) pairs of every row."""
        if self._useComps is None or self._chunkSize is None or self._distFactor is None:
            raise ValueError('ERROR: Please set the parameters first using "set_parameters" method')
        if self._k is None:
            raise ValueError("ERROR: Set parameters first")
        if ignore_ref_cells is None:
            ignore_ref_cells = []
        intra_ref = target_fn == self._refPcaFn and target_grp == self._refPcaGrp
        metric = core.resolve_metric(metric, intra_ref)
        ref = self._ref_matrix()
        if intra_ref:
            tnames, tmat = self.refCells, ref
        else:
            h5 = open_file(target_fn, mode="r")
            tnames, tmat = read_matrix(h5[target_grp], self._useComps)
            h5.close()
        mask = None
        if len(ignore_ref_cells) > 0:
            ign = set(ignore_ref_cells)
            mask = np.fromiter((c in ign for c in self.refCells), dtype=bool, count=len(self.refCells))
        m = len(self.refCells)
        drop = bool(intra_ref)                              # np.argsort(a)[1:], :141-142
        keep = min(self._k, m - (1 if drop else 0))
        if keep < 1:
            raise ValueError("ERROR: k=%s needs at least %d reference cells" % (self._k, 2 if drop else 1))
        pr = self._prepared_ref(metric, ignore_ref_cells, mask)
        if pr is not None:
            idx, dst = core.knn(tmat, pr, keep, metric, float(self._distFactor), drop_first=drop, mode=mode)
        else:
            idx, dst = core.knn(tmat, ref, keep, metric, float(self._distFactor), ref_mask=mask, drop_first=drop,
                                mode=mode)
        out = open_file(self._h5Fn, mode="a")
        for g in (dist_grp, sorted_dist_grp):
            if g in out:
                del out[g]
        out.create_row_group(dist_grp, tnames, np.asarray(dst, dtype=np.float64))
        out.create_row_group(sorted_dist_grp, tnames, np.asarray(idx, dtype=np.int64))
        out.flush()
        out.close()
        return None

    # ------------------------------------------------------------------ SNN graph
    def calc_snn(self, target_sorted_dist_grp: str, target_name: str, graph_grp: str,
                 fix_graph_attempts: int = 5, fix_weight: float = None, *, graph_layout: Optional[str] = None) -> None:
        """nabo/_mapping.py:446-493 + _calc_snn :151-200 (+ _fix_disconnected_graph :203-249 for the
        reference graph, re-expressed as masked nearest-neighbour queries).  ``graph_layout='reference'``
        writes the group the way ``_dump_graph`` does (:252-273: one dataset per node, rows of
        [neighbour name, str(weight)]) so that the reference's own ``Graph.load_from_h5`` can read it."""
        layout = graph_layout or self.graph_layout
        if layout not in ("columnar", "reference"):
            raise ValueError("ERROR: graph_layout must be 'columnar' or 'reference'")
        if self._k is None:
            raise ValueError("ERROR: Set parameters first")
        k = self._k
        h5 = open_file(self._h5Fn, mode="r")
        if self._refSortedDistGrp not in h5:
            h5.close()
            raise KeyError("ERROR: Please make sure that the distances between reference cells has already "
                           "been calculated")
        if target_sorted_dist_grp not in h5:
            h5.close()
            raise KeyError("ERROR: Please make sure that the distances between reference and target cells has "
                           "already been calculated")
        rnames, rknn = _rows_in_order(h5[self._refSortedDistGrp], self.refCells)
        tnames, tknn = _rows_in_order(h5[target_sorted_dist_grp], None)
        h5.close()
        # calc_dist stores the k (+1) best entries of a row, not upstream's full argsort: a k raised after the
        # distances were stored cannot be served from them (a narrower table is only legitimate when the
        # reference itself has fewer cells than k)
        m = len(self.refCells)
        if tknn.shape[1] < k and tknn.shape[1] != m - (1 if target_name == self.refName else 0):
            raise ValueError("ERROR: the stored distances of %r hold the %d nearest reference cells of each cell but "
                             "k is now %d. Recompute them (use_stored_distances=False) with the current parameters."
                             % (target_name, tknn.shape[1], k))
        if rknn.shape[1] < k and rknn.shape[1] != m - 1:
            raise ValueError("ERROR: the stored reference distances hold the %d nearest cells of each reference cell "
                             "but k is now %d. Run make_ref_graph(use_stored_distances=False) with the current "
                             "parameters first." % (rknn.shape[1], k))
        kk = min(k, tknn.shape[1])
        tk = np.ascontiguousarray(tknn[:, :kk], dtype=np.int32)
        rk = np.ascontiguousarray(rknn[:, :min(k, rknn.shape[1])], dtype=np.int32)
        cnt, _ = core.snn_weights(tk, rk, kk) if kk == k else _snn_with_k(tk, rk, k)
        if 2 * (k - 1) <= k and int(np.asarray(cnt).max(initial=0)) == 2 * (k - 1):
            raise ZeroDivisionError("division by zero")     # snn == 2 (k - 1): upstream's weight divides by zero (:194)
        fix_edges = np.zeros((0, 2), dtype=np.int64)
        fw = None
        if target_name == self.refName:
            fix_edges, fw = self._repair_reference_graph(tk, cnt, fix_graph_attempts, fix_weight)
        out = open_file(self._h5Fn, mode="a")
        if graph_grp in out:
            del out[graph_grp]
        g = out.create_group(graph_grp)
        if layout == "reference":
            _write_reference_layout(g, tnames, target_name, rnames, self.refName, tk, np.asarray(cnt), k,
                                    fix_edges, fw, undirected=target_name == self.refName)
            out.flush()
            out.close()
            return None
        g.create_dataset("nodes", data=np.array([(n + "_" + target_name).encode("ascii") for n in tnames]))
        g.create_dataset("knn", data=tk)
        g.create_dataset("snn", data=np.asarray(cnt, dtype=np.uint8))
        g.create_dataset("k", data=np.array([k], dtype=np.int64))
        g.create_dataset("ref_suffix", data=np.array([self.refName.encode("ascii")]))
        if len(fix_edges):
            g.create_dataset("fix_edges", data=fix_edges)
            g.create_dataset("fix_weight", data=np.array([fw], dtype=np.float64))
        out.flush()
        out.close()

    def _repair_reference_graph(self, knn: np.ndarray, cnt: np.ndarray, attempts: int, fix_weight):
        """Connect components the way _fix_disconnected_graph does (nabo/_mapping.py:203-249): every
        component gets one edge of weight `fix_weight` from the member whose nearest cell inside any
        strictly larger component is closest.  The "walk the full sorted row to the first candidate"
        of the reference is a k=1 query with every non-candidate masked."""
        m = knn.shape[0]
        rows = np.repeat(np.arange(m), knn.shape[1])
        sel = (cnt.ravel() > 0) & (knn.ravel() >= 0)
        a, b = rows[sel], knn.ravel()[sel].astype(np.int64)
        fixes: List[Tuple[int, int]] = []
        fw = fix_weight

        def components(ea, eb):
            # union-find on the GPU (nabo_connected_components); labels renumbered 0..ncomp-1
            lab_min = core.connected_components(ea.astype(np.int32), eb.astype(np.int32), m)
            uniq, lab = np.unique(lab_min, return_inverse=True)
            return len(uniq), lab

        ncomp, lab = components(a, b)
        if ncomp > 1:
            if fw is None:
                fw = core.fix_weight(self._k)
            print("INFO: Reference graph is disconnected. Trying to fix..")
        ref = None
        for _ in range(attempts):
            if ncomp <= 1:
                if fixes:
                    print("INFO: Reference graph is no longer disconnected.")
                break
            sizes = np.bincount(lab, minlength=ncomp)
            new = []
            for s in np.unique(sizes):
                cand = sizes[lab] > s                       # cells of strictly larger components
                if not cand.any():
                    continue
                members = np.nonzero(sizes[lab] == s)[0]
                if ref is None:                             # the reference goes to the device once, not per size class
                    import torch
                    ref = torch.from_numpy(np.ascontiguousarray(self._ref_matrix())).cuda()
                idx, dst = core.knn(ref[torch.from_numpy(members).cuda()], ref, 1, "euclidean",
                                    ref_mask=torch.from_numpy(~cand).cuda(), mode="fast")
                idx, dst = idx.cpu().numpy(), dst.cpu().numpy()
                for comp in np.unique(lab[members]):
                    loc = np.nonzero(lab[members] == comp)[0]
                    best = loc[np.argsort(dst[loc, 0], kind="stable")[0]]
                    new.append((int(members[best]), int(idx[best, 0])))
            fixes.extend(new)
            ea = np.concatenate([a, np.array([f[0] for f in fixes], dtype=np.int64)])
            eb = np.concatenate([b, np.array([f[1] for f in fixes], dtype=np.int64)])
            ncomp, lab = components(ea, eb)
        if ncomp > 1:
            print("WARNING: Output graph is disconnected.")
        return np.array(fixes, dtype=np.int64).reshape(-1, 2), fw

    # ------------------------------------------------------------------ wrappers
    def make_ref_graph(self, use_stored_distances: bool = False, *, metric: Optional[str] = None,
                       mode: str = "fast"):
        """nabo/_mapping.py:526-541."""
        with batched_writes(self._h5Fn):                   # distances + graph: one rewrite of the mapping file
            if use_stored_distances is False:
                self.calc_dist(self._refPcaFn, self._refPcaGrp, self._refDistGrp, self._refSortedDistGrp, [],
                               metric=metric, mode=mode)
            self.calc_snn(self._refSortedDistGrp, self.refName, self._refGraphGrpName)

    def map_target(self, target_name: str, target_pca_fn: str, target_pca_grp_name: str,
                   ignore_ref_cells: List[str] = None, use_stored_distances: bool = False,
                   overwrite: bool = False, *, metric: Optional[str] = None, mode: str = "fast") -> None:
        """nabo/_mapping.py:557-621."""
        if target_pca_fn == self._refPcaFn:
            if target_pca_grp_name == self._refPcaGrp:
                raise ValueError("ERROR: Target PCA file name and group name can not be same as that of reference")
        if target_pca_fn == self._h5Fn:
            raise ValueError("ERROR: Input HDF5 and output HDF5 file cannot be same")
        if target_name == self.refName:
            raise ValueError("ERROR: Target name cannot be same as reference name. Please provide a different name.")
        if target_name.find("__") != -1:
            raise ValueError("ERROR: Underscores are not allowed in the value for `target_name` parameter")
        if ignore_ref_cells is None:
            ignore_ref_cells = []
        if use_stored_distances is True:
            if target_name not in self._nameStash:
                print("WARNING: Target data not saved. use_stored_distances will have no effect")
            else:
                if overwrite is True:
                    print("WARNING: overwrite has no effect as use_stored_distances is set to True")
                self.calc_snn(self._nameStash[target_name] + "_sortedDist", target_name,
                              self._nameStash[target_name] + "_graph")
                return None
        else:
            if overwrite is False and target_name in self._nameStash:
                raise ValueError("ERROR: Data with this target name exists. Please set overwrite=True if you "
                                 "want to map this target again.")
        with batched_writes(self._h5Fn):                   # name stash + distances + graph: one rewrite
            self._stash_target_name(target_name)
            self._check_h5(target_pca_fn, target_pca_grp_name)
            uid = self._nameStash[target_name]
            self.calc_dist(target_pca_fn, target_pca_grp_name, uid + "_dist", uid + "_sortedDist", ignore_ref_cells,
                           metric=metric, mode=mode)
            self.calc_snn(uid + "_sortedDist", target_name, uid + "_graph")
            return None


def _write_reference_layout(g, tnames, target_name, rnames, ref_name, knn, cnt, k, fix_edges, fix_w, undirected):
    """The reference's ``_dump_graph`` layout (nabo/_mapping.py:252-273): one dataset per node holding its
    incident edges as rows [neighbour node name, weight]; NumPy coerces a (bytes, float) row to byte strings, so
    the weight is stored as its decimal string, exactly like upstream.  For the reference graph (undirected,
    targets = reference cells) a node lists every incident edge, with the weight of the LAST add_edge for that
    pair (:196-198) and the repair edges."""
    lut = core.snn_weight_lut(k, strict=False)
    rows, cols = np.nonzero(cnt > 0)
    nb = knn[rows, cols].astype(np.int64)
    w = lut[cnt[rows, cols]]
    ref_nodes = [c + "_" + ref_name for c in rnames]
    own_nodes = [c + "_" + target_name for c in tnames]
    if undirected:
        hi, lo = np.maximum(rows, nb), np.minimum(rows, nb)
        order = np.lexsort((rows >= nb, lo, hi))            # per pair: the edge seen from max(a, b) is added last
        hi, lo, w = hi[order], lo[order], w[order]
        last = np.ones(len(hi), dtype=bool)
        last[:-1] = (hi[:-1] != hi[1:]) | (lo[:-1] != lo[1:])
        hi, lo, w = hi[last], lo[last], w[last]
        if len(fix_edges):
            lo = np.concatenate([lo, fix_edges[:, 0]])
            hi = np.concatenate([hi, fix_edges[:, 1]])
            w = np.concatenate([w, np.full(len(fix_edges), fix_w)])
        src = np.concatenate([lo, hi])
        dst = np.concatenate([hi, lo])
        w = np.concatenate([w, w])
        names_dst = own_nodes
    else:
        src, dst, names_dst = rows, nb, ref_nodes
    order = np.argsort(src, kind="stable")
    src, dst, w = src[order], dst[order], w[order]
    bounds = np.searchsorted(src, np.arange(len(own_nodes) + 1))
    for i, node in enumerate(own_nodes):
        lo_, hi_ = bounds[i], bounds[i + 1]
        temp = [(names_dst[int(j)].encode("ascii"), float(x)) for j, x in zip(dst[lo_:hi_], w[lo_:hi_])]
        g.create_dataset(node, data=np.array(temp) if temp else np.zeros((0, 2), dtype="S32"))


def _rows_in_order(grp, order: Optional[List[str]]):
    """(names, 2-D int array) of a sorted-distance group, rows in `order` (default: sorted names)."""
    if isinstance(grp, RowGroup):
        names = list(grp) if order is None else list(order)
        pos = grp._idx()
        rows = np.fromiter((pos[n] for n in names), dtype=np.int64, count=len(names))
        return names, np.asarray(grp.data)[rows]
    names = [x for x in grp] if order is None else list(order)
    width = min(len(grp[n]) for n in names) if names else 0
    return names, np.array([np.asarray(grp[n][:width]) for n in names], dtype=np.int64)


def _snn_with_k(tk: np.ndarray, rk: np.ndarray, k: int):
    """Stored rows shorter than k (fewer reference cells than k): counts with the weight table of k."""
    cnt, _ = core.snn_weights(tk, rk, tk.shape[1])
    return cnt, core.snn_weight_lut(k, strict=False)[cnt]
