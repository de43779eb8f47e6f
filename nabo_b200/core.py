"""Array-level public API of the hot path (host side of the C ABI).

Each function mirrors one reference operator (file:line in the docstrings) and
accepts either NumPy arrays (host buffers: copied to the device through pinned
memory, results copied back) or ``torch`` CUDA tensors (used in place, results
stay on the device).  PyTorch is used only for device memory and streams; every
computation is a call into ``libnabo_b200.so``.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional

import numpy as np
import torch

from ._lib import METRICS, MODE_EXACT, MODE_FAST, PreparedDesc, check, lib, require_device

__all__ = ["euclidean_dist", "mod_canberra_dist", "cosine_dist", "correlation_dist", "knn", "prepare_reference", "PreparedReference", "knn_candidates", "rerank_exact", "merge_topk",
           "merge_topk_parts", "snn_int_weights", "score_accumulate", "scores_finalize", "snn_weight_lut", "fix_weight", "snn_weights", "mapping_scores", "classify_targets", "mapping_specificity", "sparse_row_stats", "connected_components",
           "project", "project_csr", "scale_counts", "map_cells", "map_cells_host", "resolve_metric"]


# ----------------------------------------------------------------------------- helpers
def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _is_host(*xs) -> bool:
    return any(isinstance(x, np.ndarray) or (x is not None and not isinstance(x, torch.Tensor)) for x in xs
               if x is not None)


def _dev(x, dtype: torch.dtype, name: str = "array") -> Optional[torch.Tensor]:
    """Device tensor of `dtype`, row-major contiguous.  Host arrays are copied from pageable memory: pinning a
    buffer for a single use costs more than it saves (map_cells_host is the pre-pinned, pipelined path)."""
    if x is None:
        return None
    if isinstance(x, torch.Tensor):
        if not x.is_cuda:
            x = x.cuda()
        if x.dtype != dtype:
            x = x.to(dtype)
        return x.contiguous()
    a = np.ascontiguousarray(x)
    t = torch.from_numpy(a)
    if t.dtype != dtype:
        t = t.to(dtype)
    return t.cuda()


def _mask_dev(mask) -> Optional[torch.Tensor]:
    if mask is None:
        return None
    if isinstance(mask, torch.Tensor):
        return _dev(mask.to(torch.uint8), torch.uint8)
    return _dev(np.asarray(mask).astype(np.uint8), torch.uint8)


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _out(t: torch.Tensor, host: bool):
    return t.cpu().numpy() if host else t


def resolve_metric(metric: Optional[str], intra_ref: bool) -> str:
    """Reference dispatch (nabo/_mapping.py:119-124, 433-440): Euclidean when the query
    set is the reference itself, modified Canberra otherwise; an explicit name overrides."""
    if metric is None:
        return "euclidean" if intra_ref else "mod_canberra"
    if metric not in METRICS:
        raise ValueError("ERROR: unknown metric %r (choose from %s)" % (metric, sorted(METRICS)))
    return metric


# ----------------------------------------------------------------------------- (1) distance tiles
def _dist(fn_name: str, x, y, d, f: Optional[float]):
    require_device()
    host = _is_host(x, y, d)
    xd, yd = _dev(x, torch.float64), _dev(y, torch.float64)
    if xd.dim() != 2 or yd.dim() != 2 or xd.shape[1] != yd.shape[1]:
        raise ValueError("ERROR: x and y must be 2-D with the same number of columns")
    m, g = xd.shape
    n = yd.shape[0]
    if d is None:
        dd = torch.empty((m, n), dtype=torch.float64, device=xd.device)
    elif isinstance(d, torch.Tensor):
        if tuple(d.shape) != (m, n) or d.dtype != torch.float64 or not d.is_contiguous() or not d.is_cuda:
            raise ValueError("ERROR: d must be a contiguous float64 CUDA tensor of shape (%d, %d)" % (m, n))
        dd = d
    else:
        if d.shape != (m, n) or d.dtype != np.float64:
            raise ValueError("ERROR: d must be a float64 array of shape (%d, %d)" % (m, n))
        dd = torch.empty((m, n), dtype=torch.float64, device=xd.device)
    fn = getattr(lib(), fn_name)
    args = [_ptr(xd), g, _ptr(yd), g, _ptr(dd), n, m, n, g]
    if f is not None:
        args.append(float(f))
    args.append(C.c_void_p(_stream()))
    check(fn(*args), fn_name)
    if isinstance(d, np.ndarray):
        d[...] = dd.cpu().numpy()      # the reference kernels fill the caller's buffer in place
        return d
    return _out(dd, host) if d is None else dd


def euclidean_dist(x, y, d=None):
    """``_euclidean_dist(x, y, d)`` (nabo/_mapping.py:16-26): fills ``d`` (m x n float64) in
    place, bit-identical to the numba kernel.  ``d=None`` allocates and returns it."""
    return _dist("nabo_euclidean_dist", x, y, d, None)


def mod_canberra_dist(x, y, d=None, f: float = 0.25):
    """``_mod_canberra_dist(x, y, d, f)`` (nabo/_mapping.py:29-45); x = target, y = reference."""
    if not (float(f) > 0):
        raise ValueError('ERROR: "dist_factor" must be a non-zero float value')
    return _dist("nabo_mod_canberra_dist", x, y, d, f)


def cosine_dist(x, y, d=None):
    """Extension metric: 1 - x.y/(|x||y|), sequential FP64 (no reference counterpart)."""
    return _dist("nabo_cosine_dist", x, y, d, None)


def correlation_dist(x, y, d=None):
    """Extension metric: Pearson correlation distance, the cosine distance of the row-centred vectors (each row
    minus its mean, summed sequentially in FP64; see NABO_CORRELATION in include/nabo_b200.h).  Constant rows give
    NaN, like zero rows under cosine."""
    return _dist("nabo_correlation_dist", x, y, d, None)


# ----------------------------------------------------------------------------- (2) kNN
PREPARED_MAX_G = 128      # widest PCA space with a prepared form (the fast plans' limit, nabo_ref_prepared_bytes)


class PreparedReference:
    """A reference packed once for any number of ``knn`` calls (``nabo_ref_prepare``): the reference-side operands
    of the fast engine for one (rows, g, metric, mask) in a device buffer this object owns, plus the FP64 rows and
    the mask it keeps on the device (the exact re-rank and fallback read them).  Results are bit-identical to
    ``knn`` with the raw rows.  Device memory: the packed tensor-core tiles take 2 * ceil16(3g + 3) bytes per
    reference (about 31 MB per 100 k references at g = 50); correlation adds the centred FP64 copy of the rows
    (8g bytes per reference), which the calls read instead of ``r``; see ``nbytes``.

    The rows must not change while the object is in use: a CUDA tensor passed in (or the float64 copy made of
    it) that is modified in place afterwards makes every later call raise ``ValueError``.  NumPy input is copied
    at preparation, so later changes to the array are not seen at all."""

    def __init__(self, r, metric: str, ref_mask=None):
        require_device()
        if metric not in METRICS:
            raise ValueError("ERROR: unknown metric %r" % (metric,))
        rd = _dev(r, torch.float64)
        if rd.dim() != 2 or rd.shape[0] < 1:
            raise ValueError("ERROR: the reference must be a non-empty 2-D array")
        md = _mask_dev(ref_mask)
        if md is not None and md.numel() != rd.shape[0]:
            raise ValueError("ERROR: ref_mask must have one entry per reference cell")
        self.metric = metric
        self.n_ref, self.g = int(rd.shape[0]), int(rd.shape[1])
        self.r, self.mask, self._mask_src = rd, md, ref_mask
        self._sources = [(t, t._version) for t in {id(x): x for x in (r, rd, ref_mask, md)
                                                   if isinstance(x, torch.Tensor)}.values()]
        L = lib()
        nbytes = int(L.nabo_ref_prepared_bytes(self.n_ref, self.g, METRICS[metric]))
        if nbytes == 0:
            raise ValueError("ERROR: metric %r with g=%d has no prepared form (1 <= g <= 128)" % (metric, self.g))
        self.buffer = torch.empty(nbytes, dtype=torch.uint8, device=rd.device)
        self.desc = PreparedDesc()
        check(L.nabo_ref_prepare(_ptr(rd), self.g, self.n_ref, self.g, METRICS[metric], _ptr(md), _ptr(self.buffer),
                                 nbytes, C.byref(self.desc), C.c_void_p(_stream())), "ref_prepare")

    @property
    def shape(self):
        return (self.n_ref, self.g)

    @property
    def device(self):
        return self.r.device

    @property
    def nbytes(self) -> int:
        """Device bytes of the packed operands (the FP64 rows and the mask not included)."""
        return self.buffer.numel()

    def check_unchanged(self) -> None:
        for t, v in self._sources:
            if t._version != v:
                raise ValueError("ERROR: the reference rows or mask were modified in place after prepare_reference; "
                                 "prepare the reference again")


def prepare_reference(r, metric: str, ref_mask=None) -> PreparedReference:
    """Pack the reference ``r`` (M,g) once for ``metric`` (and ``ref_mask``); pass the result to ``knn`` /
    ``map_cells`` / the sharded mappers in place of ``r``."""
    return PreparedReference(r, metric, ref_mask)


def _check_prepared_args(pr: PreparedReference, metric, ref_mask, g: int) -> str:
    """Metric, mask and g of a call on a prepared reference come from the object; conflicting arguments raise."""
    if metric is not None and metric != pr.metric:
        raise ValueError("ERROR: metric %r conflicts with the prepared reference's %r" % (metric, pr.metric))
    if ref_mask is not None and ref_mask is not pr._mask_src and ref_mask is not pr.mask:
        raise ValueError("ERROR: ref_mask comes from the prepared reference; do not pass another one")
    if g != pr.g:
        raise ValueError("ERROR: queries have %d columns, the prepared reference %d" % (g, pr.g))
    pr.check_unchanged()
    return pr.metric


def knn(q, r, k: int, metric: Optional[str] = None, dist_factor: float = 0.25, ref_mask=None,
        drop_first: bool = False, idx_offset: int = 0, mode: str = "fast", return_stats: bool = False, out=None,
        out_parts=None):
    """Fused distance + per-query top-k: what ``_calc_dist`` (nabo/_mapping.py:48-148) leaves
    for ``_calc_snn`` to read (``[:k]`` of each sorted row), without the N x M matrix.

    q (N,g), r (M,g) float64.  ``ref_mask`` (M,) bool marks ``ignore_ref_cells`` (sorted last,
    :135-140); ``drop_first`` is the reference<->reference ``[1:]`` (:141-142).  ``metric`` defaults to
    Euclidean.  ``r`` may be a ``PreparedReference``: metric, mask and g then come from it (a conflicting
    ``metric`` / ``ref_mask`` / query width raises ``ValueError``) and the reference is not packed again.
    Returns (idx int32 (N,k), dist float64 (N,k)) [+ stats dict].

    ``out_parts=(bounds, idx_ptrs, dist_ptrs)`` routes the result rows instead (``nabo_knn_routed``): row t
    with bounds[p] <= t < bounds[p+1] is written to row t - bounds[p] of the (rows_p, k) int32 / float64
    blocks at the device ADDRESSES idx_ptrs[p] / dist_ptrs[p] (local buffers or NVLink-mapped peer memory);
    the call then returns (None, None)."""
    pr = r if isinstance(r, PreparedReference) else None
    if pr is not None:
        metric = _check_prepared_args(pr, metric, ref_mask, _ncols(q))
    elif metric is None:
        metric = "euclidean"
    require_device()
    if metric not in METRICS:
        raise ValueError("ERROR: unknown metric %r" % (metric,))
    if mode not in ("fast", "exact"):
        raise ValueError("ERROR: mode must be 'fast' or 'exact'")
    host = _is_host(q) if pr is not None else _is_host(q, r)
    qd = _dev(q, torch.float64)
    rd = pr.r if pr is not None else _dev(r, torch.float64)
    if qd.dim() != 2 or rd.dim() != 2 or qd.shape[1] != rd.shape[1]:
        raise ValueError("ERROR: q and r must be 2-D with the same number of columns")
    n, g = qd.shape
    m = rd.shape[0]
    k = int(k)
    if k < 1 or k + (1 if drop_first else 0) > m:
        raise ValueError("ERROR: k=%d is not in 1..%d" % (k, m - (1 if drop_first else 0)))
    md = pr.mask if pr is not None else _mask_dev(ref_mask)
    if md is not None and md.numel() != m:
        raise ValueError("ERROR: ref_mask must have one entry per reference cell")
    if out_parts is not None:
        return _knn_routed(qd, rd, n, m, g, k, metric, dist_factor, md, drop_first, idx_offset, mode, out_parts,
                           return_stats, pr)
    if out is not None:                                    # caller-owned (n, k) int32 / float64 device buffers
        idx, dst = out
        if tuple(idx.shape) != (n, k) or tuple(dst.shape) != (n, k) or idx.dtype != torch.int32 or \
                dst.dtype != torch.float64 or not (idx.is_contiguous() and dst.is_contiguous() and idx.is_cuda):
            raise ValueError("ERROR: out must be contiguous CUDA (n, k) int32 and float64 tensors")
    else:
        idx = torch.empty((n, k), dtype=torch.int32, device=qd.device)
        dst = torch.empty((n, k), dtype=torch.float64, device=qd.device)
    mode_i = MODE_FAST if mode == "fast" else MODE_EXACT
    L = lib()
    stats = (C.c_int64 * 8)() if return_stats else None
    if pr is not None:
        ws_bytes = int(L.nabo_knn_prepared_workspace_bytes(n, C.byref(pr.desc), k, float(dist_factor), mode_i))
        ws = torch.empty(max(ws_bytes, 256), dtype=torch.uint8, device=qd.device)
        check(L.nabo_knn_prepared(_ptr(qd), g, n, C.byref(pr.desc), k, float(dist_factor), 1 if drop_first else 0,
                                  int(idx_offset), mode_i, _ptr(idx), _ptr(dst), _ptr(ws), ws.numel(), stats,
                                  C.c_void_p(_stream())), "knn_prepared")
    else:
        ws_bytes = int(L.nabo_knn_workspace_bytes(n, m, g, k, METRICS[metric], mode_i))
        ws = torch.empty(max(ws_bytes, 256), dtype=torch.uint8, device=qd.device)
        check(L.nabo_knn(_ptr(qd), g, _ptr(rd), g, n, m, g, k, METRICS[metric], float(dist_factor), _ptr(md),
                         1 if drop_first else 0, int(idx_offset), mode_i, _ptr(idx), _ptr(dst), _ptr(ws),
                         ws.numel(), stats, C.c_void_p(_stream())), "knn")
    res = (_out(idx, host), _out(dst, host))
    if return_stats:
        res = res + (_stats_dict(stats),)
    return res


def _stats_dict(stats):
    return {"rows_reranked": int(stats[0]), "rows_exact_fallback": int(stats[1]),
            "candidates_per_row": int(stats[2]), "kernel_launches": int(stats[3]),
            "main_kernel_ms": stats[4] / 1e6, "rerank_ms": stats[5] / 1e6,
            "fallback_ms": stats[6] / 1e6, "prep_ms": stats[7] / 1e6}


def _ncols(x) -> int:
    return int(x.shape[1]) if getattr(x, "ndim", 0) == 2 else -1


def _knn_routed(qd, rd, n, m, g, k, metric, dist_factor, md, drop_first, idx_offset, mode, out_parts, return_stats,
                pr=None):
    bounds, idx_ptrs, dist_ptrs = out_parts
    n_parts = len(idx_ptrs)
    if len(bounds) != n_parts + 1 or len(dist_ptrs) != n_parts:
        raise ValueError("ERROR: out_parts needs n_parts + 1 bounds and n_parts idx / dist addresses")
    mode_i = MODE_FAST if mode == "fast" else MODE_EXACT
    L = lib()
    stats = (C.c_int64 * 8)() if return_stats else None
    b = (C.c_int * (n_parts + 1))(*[int(x) for x in bounds])
    pi = (C.c_void_p * n_parts)(*[int(x) if x else None for x in idx_ptrs])
    pd = (C.c_void_p * n_parts)(*[int(x) if x else None for x in dist_ptrs])
    if pr is not None:
        ws_bytes = int(L.nabo_knn_prepared_workspace_bytes(n, C.byref(pr.desc), k, float(dist_factor), mode_i))
        ws = torch.empty(max(ws_bytes, 256), dtype=torch.uint8, device=qd.device)
        check(L.nabo_knn_prepared_routed(_ptr(qd), g, n, C.byref(pr.desc), k, float(dist_factor), 1 if drop_first else 0,
                                         int(idx_offset), mode_i, n_parts, b, pi, pd, _ptr(ws), ws.numel(), stats,
                                         C.c_void_p(_stream())), "knn_prepared_routed")
    else:
        ws_bytes = int(L.nabo_knn_workspace_bytes(n, m, g, k, METRICS[metric], mode_i))
        ws = torch.empty(max(ws_bytes, 256), dtype=torch.uint8, device=qd.device)
        check(L.nabo_knn_routed(_ptr(qd), g, _ptr(rd), g, n, m, g, k, METRICS[metric], float(dist_factor), _ptr(md),
                                1 if drop_first else 0, int(idx_offset), mode_i, n_parts, b, pi, pd, _ptr(ws),
                                ws.numel(), stats, C.c_void_p(_stream())), "knn_routed")
    return (None, None, _stats_dict(stats)) if return_stats else (None, None)


def _rows_as_given(metric: str, what: str) -> None:
    if metric == "correlation":
        raise ValueError("ERROR: %s takes rows as given and has no correlation form; centre the rows and pass "
                         "metric='cosine'" % what)


def knn_candidates(q, r, k: int, metric: str = "euclidean", ref_mask=None, drop_first: bool = False):
    """Tensor-core candidate pass alone (Euclidean / cosine).  Returns dict(cand int32 (N,K'),
    tau float32 (N,), qn2 float64 (N,), scal float64 (4,)); see include/nabo_b200.h.  Rows are taken as
    given: for correlation, pass row-centred rows with ``metric="cosine"``."""
    _rows_as_given(metric, "knn_candidates")
    require_device()
    host = _is_host(q, r)
    qd, rd = _dev(q, torch.float64), _dev(r, torch.float64)
    n, g = qd.shape
    m = rd.shape[0]
    md = _mask_dev(ref_mask)
    L = lib()
    kp = int(L.nabo_knn_candidates_width(int(k), 1 if drop_first else 0))
    cand = torch.empty((n, kp), dtype=torch.int32, device=qd.device)
    tau = torch.empty(n, dtype=torch.float32, device=qd.device)
    qn2 = torch.empty(n, dtype=torch.float64, device=qd.device)
    scal = torch.empty(4, dtype=torch.float64, device=qd.device)
    ws = torch.empty(int(L.nabo_knn_candidates_workspace_bytes(n, m, g, int(k), 1 if drop_first else 0)),
                     dtype=torch.uint8, device=qd.device)
    check(L.nabo_knn_candidates(_ptr(qd), g, _ptr(rd), g, n, m, g, int(k), METRICS[metric], _ptr(md),
                                1 if drop_first else 0, _ptr(cand), _ptr(tau), _ptr(qn2), _ptr(scal), _ptr(ws),
                                ws.numel(), C.c_void_p(_stream())), "knn_candidates")
    return {"cand": _out(cand, host), "tau": _out(tau, host), "qn2": _out(qn2, host), "scal": _out(scal, host)}


def rerank_exact(q, r, cand, k: int, metric: str = "euclidean", dist_factor: float = 0.25, ref_mask=None,
                 drop_first: bool = False, idx_offset: int = 0):
    """Exact FP64 re-rank (reference arithmetic order) of caller-supplied candidates.  Rows are taken as given:
    for correlation, pass row-centred rows with ``metric="cosine"``."""
    _rows_as_given(metric, "rerank_exact")
    require_device()
    host = _is_host(q, r, cand)
    qd, rd = _dev(q, torch.float64), _dev(r, torch.float64)
    cd = _dev(cand, torch.int32)
    n, g = qd.shape
    m = rd.shape[0]
    md = _mask_dev(ref_mask)
    idx = torch.empty((n, k), dtype=torch.int32, device=qd.device)
    dst = torch.empty((n, k), dtype=torch.float64, device=qd.device)
    check(lib().nabo_rerank_exact(_ptr(qd), g, _ptr(rd), g, n, m, g, int(k), METRICS[metric], float(dist_factor),
                                  _ptr(md), 1 if drop_first else 0, int(idx_offset), _ptr(cd), cd.shape[1],
                                  _ptr(idx), _ptr(dst), C.c_void_p(_stream())), "rerank_exact")
    return _out(idx, host), _out(dst, host)


def merge_topk(idx, dist, k: Optional[int] = None):
    """Merge shard-major candidates (S,N,k) by (dist, idx): the reference-sharded result."""
    require_device()
    host = _is_host(idx, dist)
    i_d, d_d = _dev(idx, torch.int32), _dev(dist, torch.float64)
    if i_d.dim() != 3 or i_d.shape != d_d.shape:
        raise ValueError("ERROR: idx and dist must both be (n_shards, n_query, k)")
    s, n, kk = i_d.shape
    if k is not None and k != kk:
        raise ValueError("ERROR: k must equal the per-shard k")
    oi = torch.empty((n, kk), dtype=torch.int32, device=i_d.device)
    od = torch.empty((n, kk), dtype=torch.float64, device=i_d.device)
    check(lib().nabo_merge_topk(_ptr(i_d), _ptr(d_d), s, n, kk, _ptr(oi), _ptr(od), C.c_void_p(_stream())),
          "merge_topk")
    return _out(oi, host), _out(od, host)


def merge_topk_parts(idx_ptrs, dist_ptrs, n_query: int, k: int, device, drop_first: bool = False, out=None):
    """``nabo_merge_topk_parts``: merge one (n_query, k) idx / dist block per shard, given by device ADDRESS
    (the per-source blocks of an all-to-all / peer-written receive buffer, consumed in place).
    Returns (idx int32, dist float64) of shape (n_query, k - drop_first) on ``device``."""
    require_device()
    s = len(idx_ptrs)
    ko = int(k) - (1 if drop_first else 0)
    if out is not None:
        oi, od = out
    else:
        oi = torch.empty((n_query, ko), dtype=torch.int32, device=device)
        od = torch.empty((n_query, ko), dtype=torch.float64, device=device)
    pi = (C.c_void_p * s)(*[int(x) for x in idx_ptrs])
    pd = (C.c_void_p * s)(*[int(x) for x in dist_ptrs])
    check(lib().nabo_merge_topk_parts(s, pi, pd, int(n_query), int(k), 1 if drop_first else 0, _ptr(oi), _ptr(od),
                                      C.c_void_p(_stream())), "merge_topk_parts")
    return oi, od


# ----------------------------------------------------------------------------- (4) SNN weights
def snn_weight_lut(k: int, strict: bool = True) -> np.ndarray:
    """weight(snn) = round(snn / (2*(k-1) - snn), 2) with Python's round() on a double
    (nabo/_mapping.py:185, 194).  Entry 0 = 0.0 (no edge, :195).

    k = 2 has no weight for snn = 2 (division by zero).  Upstream raises ZeroDivisionError only when some
    pair really shares both neighbours; ``strict=False`` fills that entry with NaN so that callers can raise
    on an actual count of 2 (``Mapping.calc_snn`` does), ``strict=True`` raises as soon as the table is built."""
    factor = 2 * (k - 1)
    lut = np.zeros(k + 1, dtype=np.float64)
    for snn in range(1, k + 1):
        if factor == snn:
            if strict:
                raise ZeroDivisionError("division by zero")
            lut[snn] = np.nan
        else:
            lut[snn] = round(snn / (factor - snn), 2)
    return lut


_LUT_DEV: Dict[tuple, "torch.Tensor"] = {}


def _lut_dev(k: int, device) -> "torch.Tensor":
    """Device copy of the weight table, cached: a fresh pageable host->device copy per call would block the
    host until the stream's earlier kernels have finished and expose every later launch latency."""
    key = (int(k), str(device))
    t = _LUT_DEV.get(key)
    if t is None:
        t = _LUT_DEV[key] = torch.from_numpy(snn_weight_lut(k, strict=False)).to(device)
    return t


def fix_weight(k: int) -> float:
    """Default weight of repair edges (nabo/_mapping.py:478-479)."""
    return 0.5 / ((2 * (k - 1)) - 0.5)


def snn_weights(tgt_knn, ref_knn, k: Optional[int] = None, out=None):
    """``_calc_snn`` (nabo/_mapping.py:151-200) in array form.
    Returns (counts uint8 (N,k), weights float64 (N,k)); an edge exists where counts > 0."""
    require_device()
    host = _is_host(tgt_knn, ref_knn)
    td, rd = _dev(tgt_knn, torch.int32), _dev(ref_knn, torch.int32)
    n, kk = td.shape
    if k is None:
        k = kk
    if k != kk:
        td = td[:, :k].contiguous()
    lut = _lut_dev(k, td.device)
    if out is not None:
        cnt, w = out
    else:
        cnt = torch.empty((n, k), dtype=torch.uint8, device=td.device)
        w = torch.empty((n, k), dtype=torch.float64, device=td.device)
    check(lib().nabo_snn_weights(_ptr(td), n, k, _ptr(rd), rd.shape[0], rd.shape[1], _ptr(lut), _ptr(cnt),
                                 _ptr(w), C.c_void_p(_stream())), "snn_weights")
    return _out(cnt, host), _out(w, host)


# ----------------------------------------------------------------------------- (5) scores
def mapping_scores(tgt_knn, counts, n_ref: int, k: Optional[int] = None, include=None, min_weight: float = 0.0,
                   min_score: float = 0.0, weighted: bool = True, score_multiplier: float = 1000.0,
                   n_targets_total: Optional[int] = None):
    """Core of ``Graph.get_mapping_score`` (nabo/_graph.py:643-653, 690-693) in array form.
    ``n_targets_total`` overrides the divisor (a rank's partial score in the sharded modes)."""
    require_device()
    host = _is_host(tgt_knn, counts)
    td, cd = _dev(tgt_knn, torch.int32), _dev(counts, torch.uint8)
    n, kk = td.shape
    k = kk if k is None else k
    lut = _lut_dev(k, td.device)
    inc = None
    n_inc = n if n_targets_total is None else int(n_targets_total)
    if include is not None:
        inc_h = np.asarray(include.cpu() if isinstance(include, torch.Tensor) else include)
        if inc_h.dtype != np.bool_ and inc_h.dtype != np.uint8:
            b = np.zeros(n, dtype=np.uint8)
            b[inc_h] = 1
            inc_h = b
        inc_h = inc_h.astype(np.uint8)
        n_inc = int(inc_h.sum())
        inc = _dev(inc_h, torch.uint8)
    out = torch.empty(n_ref, dtype=torch.float64, device=td.device)
    L = lib()
    ws_bytes = int(L.nabo_scores_workspace_bytes(n, kk, n_ref))
    ws = torch.empty(max(ws_bytes, 256), dtype=torch.uint8, device=td.device)
    check(L.nabo_mapping_scores(_ptr(td), _ptr(cd), _ptr(lut), n, kk, int(n_ref), _ptr(inc), n_inc,
                                float(min_weight), 1 if weighted else 0, float(score_multiplier),
                                float(min_score), _ptr(out), _ptr(ws), ws.numel(), C.c_void_p(_stream())),
          "mapping_scores")
    return _out(out, host)


SCORE_UNITS = 100        # the reference's weights are round(w, 2): integers in hundredths


def snn_int_weights(k: int, min_weight: float = 0.0, weighted: bool = True) -> np.ndarray:
    """The SNN weight table in integer units for ``score_accumulate``: entry c = round(lut[c] * 100) (exact,
    every weight is ``round(x, 2)``, nabo/_mapping.py:185, 194), 0 where the edge does not count
    (c = 0, or weight <= min_weight, nabo/_graph.py:647-648); unweighted: 1 per counted edge (:649-650)."""
    lut = snn_weight_lut(k, strict=False)     # NaN (k = 2, snn = 2) never occurs in a stored graph
    iw = np.zeros(k + 1, dtype=np.int64)
    for c in range(1, k + 1):
        if weighted:
            if lut[c] > min_weight:                     # False for NaN
                iw[c] = int(round(lut[c] * SCORE_UNITS))
                if abs(iw[c] / SCORE_UNITS - lut[c]) > 1e-12:
                    raise ValueError("ERROR: weight table entry %r is not a multiple of 1/%d" % (lut[c], SCORE_UNITS))
        else:
            iw[c] = 1
    return iw


_IW_DEV: Dict[tuple, "torch.Tensor"] = {}


def score_accumulate(tgt_knn, counts, n_ref: int, k: Optional[int] = None, acc=None, include=None,
                     min_weight: float = 0.0, weighted: bool = True):
    """Integer accumulation of the edge weights per reference cell (``nabo_score_accumulate``): adds this
    batch of targets to ``acc`` (int64 (n_ref,), created zeroed when None) and returns it.  ``acc`` can be
    summed over target batches and all-reduced over GPUs as integers: the resulting scores have the same bits
    for any number of GPUs."""
    require_device()
    td, cd = _dev(tgt_knn, torch.int32), _dev(counts, torch.uint8)
    n, kk = td.shape
    k = kk if k is None else int(k)
    key = (k, float(min_weight), bool(weighted), str(td.device))
    iw = _IW_DEV.get(key)
    if iw is None:
        iw = _IW_DEV[key] = torch.from_numpy(snn_int_weights(k, min_weight, weighted)).to(td.device)
    if acc is None:
        acc = torch.zeros(int(n_ref), dtype=torch.int64, device=td.device)
    inc = None if include is None else _mask_dev(include)
    check(lib().nabo_score_accumulate(_ptr(td), _ptr(cd), _ptr(iw), n, kk, int(n_ref), _ptr(inc), _ptr(acc),
                                      C.c_void_p(_stream())), "score_accumulate")
    return acc


def scores_finalize(acc, n_include: int, score_multiplier: float = 1000.0, min_score: float = 0.0,
                    weighted: bool = True):
    """score = score_multiplier * (acc / units) / n_include, zero below min_score (nabo/_graph.py:651-653, 690-693)."""
    require_device()
    host = _is_host(acc)
    ad = _dev(acc, torch.int64)
    out = torch.empty(ad.numel(), dtype=torch.float64, device=ad.device)
    check(lib().nabo_scores_finalize(_ptr(ad), ad.numel(), float(SCORE_UNITS if weighted else 1),
                                     float(score_multiplier), int(n_include), float(min_score), _ptr(out),
                                     C.c_void_p(_stream())), "scores_finalize")
    return _out(out, host)


def classify_targets(tgt_knn, counts, ref_labels, n_labels: int, k: Optional[int] = None,
                     weight_frac: float = 0.5, min_degree: int = 2, min_weight: float = 0.1):
    """Array form of ``Graph.classify_target`` (nabo/_graph.py:722-792); -1 = na_label."""
    require_device()
    host = _is_host(tgt_knn, counts, ref_labels)
    td, cd, ld = _dev(tgt_knn, torch.int32), _dev(counts, torch.uint8), _dev(ref_labels, torch.int32)
    n, kk = td.shape
    lut = _lut_dev(kk if k is None else k, td.device)
    out = torch.empty(n, dtype=torch.int32, device=td.device)
    check(lib().nabo_classify_targets(_ptr(td), _ptr(cd), _ptr(lut), n, kk, _ptr(ld), int(n_labels),
                                      float(weight_frac), int(min_degree), float(min_weight), _ptr(out),
                                      C.c_void_p(_stream())), "classify_targets")
    return _out(out, host)


def mapping_specificity(indptr, indices, tgt_knn, counts):
    """Array form of ``Graph.get_mapping_specificity`` (nabo/_graph.py:794-824): per target, the mean
    unweighted shortest-path length in the reference graph (symmetric CSR ``indptr`` int64, ``indices``
    int32) between all pairs of reference cells the target has an edge to (``counts > 0``).
    ``tgt_knn`` / ``counts`` are (N, k) with k <= 128 (every k the kNN engines take); wider tables raise.
    Returns (mean float64 (N,) with NaN where fewer than two cells are mapped, connected bool (N,) -
    False where some pair has no path, which is where the reference raises NetworkXNoPath)."""
    require_device()
    host = _is_host(indptr, indices, tgt_knn, counts)
    ip, ix = _dev(indptr, torch.int64), _dev(indices, torch.int32)
    td, cd = _dev(tgt_knn, torch.int32), _dev(counts, torch.uint8)
    n, kk = td.shape
    m = ip.numel() - 1
    if cd.shape != td.shape:
        raise ValueError("ERROR: tgt_knn and counts must have the same shape")
    osum = torch.empty(n, dtype=torch.int64, device=td.device)
    opairs = torch.empty(n, dtype=torch.int32, device=td.device)
    onm = torch.empty(n, dtype=torch.int32, device=td.device)
    wb = lib().nabo_specificity_workspace_bytes_k(m, n, kk)
    ws = torch.empty(max(wb, 1), dtype=torch.uint8, device=td.device)
    check(lib().nabo_mapping_specificity(_ptr(ip), _ptr(ix), m, _ptr(td), _ptr(cd), n, kk, _ptr(osum), _ptr(opairs),
                                         _ptr(onm), _ptr(ws), ws.numel(), C.c_void_p(_stream())), "mapping_specificity")
    nm = onm.to(torch.int64)
    want = nm * (nm - 1)
    mean = torch.where(nm >= 2, (osum // 2).to(torch.float64) / (want // 2).clamp(min=1).to(torch.float64),
                       torch.full((n,), float("nan"), dtype=torch.float64, device=td.device))
    connected = opairs.to(torch.int64) >= want
    return _out(mean, host), _out(connected, host)


def connected_components(edge_a, edge_b, n_nodes: int):
    """Component label (= smallest node id of the component) of every node of the undirected graph given by
    the edge list; the ``nx.connected_components`` of the reference-graph repair (nabo/_mapping.py:203-249)."""
    require_device()
    host = _is_host(edge_a, edge_b)
    ea, eb = _dev(edge_a, torch.int32), _dev(edge_b, torch.int32)
    if ea.numel() != eb.numel():
        raise ValueError("ERROR: edge_a and edge_b must have the same length")
    dev = ea.device
    lab = torch.empty(int(n_nodes), dtype=torch.int32, device=dev)
    ws = torch.empty(int(n_nodes) * 4 + 1024, dtype=torch.uint8, device=dev)
    check(lib().nabo_connected_components(_ptr(ea), _ptr(eb), ea.numel(), int(n_nodes), _ptr(lab), _ptr(ws), ws.numel(),
                                          C.c_void_p(_stream())), "connected_components")
    return _out(lab, host)


def sparse_row_stats(indptr, idx, val, pos_of_col, n_dense: int, scale=None, moments: bool = True):
    """Float32 row statistics of a CSR count matrix in NumPy's pairwise order (``Dataset.set_sf`` /
    ``set_gene_stats``, nabo/_dataset.py:573-583, 609-622): for every row, the dense vector of length
    ``n_dense`` (column c sits at ``pos_of_col[c]``, -1 = dropped; values times ``scale``) is reduced exactly
    like ``temp.sum()``, ``temp.mean()``, ``temp[temp > 0].mean()``, ``temp.var()``, ``(temp > 0).sum()``.
    Returns dict(sum[, mean, nzmean, var, npos]) - NumPy if the inputs were."""
    require_device()
    host = _is_host(indptr, idx, val)
    ip, ix, vl = _dev(indptr, torch.int64), _dev(idx, torch.int32), _dev(val, torch.float32)
    pc = _dev(pos_of_col, torch.int32)
    sc = _dev(scale, torch.float32) if scale is not None else None
    n_rows = ip.numel() - 1
    if sc is not None and sc.numel() != n_dense:
        raise ValueError("ERROR: scale must have one entry per dense position")
    dev = ip.device
    out = {"sum": torch.empty(n_rows, dtype=torch.float32, device=dev)}
    if moments:
        out.update(mean=torch.empty(n_rows, dtype=torch.float32, device=dev),
                   nzmean=torch.empty(n_rows, dtype=torch.float32, device=dev),
                   var=torch.empty(n_rows, dtype=torch.float32, device=dev),
                   npos=torch.empty(n_rows, dtype=torch.int32, device=dev))
    check(lib().nabo_sparse_row_stats(_ptr(ip), _ptr(ix), _ptr(vl), n_rows, pc.numel(), _ptr(pc), _ptr(sc), int(n_dense),
                                      1 if moments else 0, _ptr(out["sum"]), _ptr(out.get("mean")), _ptr(out.get("nzmean")),
                                      _ptr(out.get("var")), _ptr(out.get("npos")), C.c_void_p(_stream())), "sparse_row_stats")
    return {k_: _out(v, host) for k_, v in out.items()}


# ----------------------------------------------------------------------------- (6) projection
def project(counts, gene_idx, sf, mu, sigma, components, mean, engine: str = "mma", out=None):
    """``get_scaled_values`` + ``transform_pca`` (nabo/_dataset.py:905-913, 1028) on a dense
    (cells x genes) count block.  ``gene_idx`` = column of each model gene (-1 = missing).
    ``engine='mma'``: one FP64 tensor-core GEMM with the per-gene constants folded into the component matrix
    (``nabo_project_dense_mma``); ``'simple'``: the straightforward FP64 CUDA-core kernel (``nabo_project_dense``)."""
    require_device()
    host = _is_host(counts)
    cd = _dev(counts, torch.float32)
    gi = _dev(gene_idx, torch.int32)
    sfd = _dev(sf, torch.float32)
    mud, sgd = _dev(mu, torch.float64), _dev(sigma, torch.float64)
    cm, mn = _dev(components, torch.float64), _dev(mean, torch.float64)
    n, ld = cd.shape
    nc, G = cm.shape
    if not (gi.numel() == G == mud.numel() == sgd.numel() == mn.numel()):
        raise ValueError("ERROR: gene_idx, mu, sigma, mean and components disagree on the number of genes")
    if sfd.numel() != n:
        raise ValueError("ERROR: one size factor per cell is required")
    if out is None:
        out = torch.empty((n, nc), dtype=torch.float64, device=cd.device)
    if engine == "simple":
        check(lib().nabo_project_dense(_ptr(cd), ld, n, _ptr(gi), G, _ptr(sfd), _ptr(mud), _ptr(sgd), _ptr(cm),
                                       _ptr(mn), nc, _ptr(out), nc, C.c_void_p(_stream())), "project_dense")
    else:
        L = lib()
        ws = torch.empty(int(L.nabo_project_dense_workspace_bytes(G, nc)), dtype=torch.uint8, device=cd.device)
        check(L.nabo_project_dense_mma(_ptr(cd), ld, n, _ptr(gi), G, _ptr(sfd), _ptr(mud), _ptr(sgd), _ptr(cm),
                                       _ptr(mn), nc, _ptr(out), nc, _ptr(ws), ws.numel(), C.c_void_p(_stream())),
              "project_dense_mma")
    return _out(out, host)


def scale_counts(counts, gene_idx, sf, mu, sigma):
    """``get_scaled_values`` core (nabo/_dataset.py:905-913) on a dense count block -> z (cells x G) float64."""
    require_device()
    host = _is_host(counts)
    cd = _dev(counts, torch.float32)
    gi = _dev(gene_idx, torch.int32)
    sfd = _dev(sf, torch.float32)
    mud, sgd = _dev(mu, torch.float64), _dev(sigma, torch.float64)
    n, ld = cd.shape
    G = gi.numel()
    out = torch.empty((n, G), dtype=torch.float64, device=cd.device)
    check(lib().nabo_scale_dense(_ptr(cd), ld, n, _ptr(gi), G, _ptr(sfd), _ptr(mud), _ptr(sgd), _ptr(out), G,
                                 C.c_void_p(_stream())), "scale_dense")
    return _out(out, host)


def project_csr(indptr, col, val, gene_pos, sf, mu, sigma, components, mean):
    """Same projection from CSR counts over all genes of the dataset (the layout of the
    reference's ``cell_data`` group, nabo/_io.py:103).  ``gene_pos[j]`` = position of dataset
    gene j in the model's gene order, or -1."""
    require_device()
    host = _is_host(indptr, col, val)
    ip, cl, vl = _dev(indptr, torch.int64), _dev(col, torch.int32), _dev(val, torch.float32)
    gp = _dev(gene_pos, torch.int32)
    sfd = _dev(sf, torch.float32)
    mud, sgd = _dev(mu, torch.float64), _dev(sigma, torch.float64)
    cm, mn = _dev(components, torch.float64), _dev(mean, torch.float64)
    n = ip.numel() - 1
    nc, G = cm.shape
    out = torch.empty((n, nc), dtype=torch.float64, device=ip.device)
    L = lib()
    ws = torch.empty(int(L.nabo_project_csr_workspace_bytes(G, nc)), dtype=torch.uint8, device=ip.device)
    check(L.nabo_project_csr(_ptr(ip), _ptr(cl), _ptr(vl), n, _ptr(gp), gp.numel(), G, _ptr(sfd), _ptr(mud),
                             _ptr(sgd), _ptr(cm), _ptr(mn), nc, _ptr(out), nc, _ptr(ws), ws.numel(),
                             C.c_void_p(_stream())), "project_csr")
    return _out(out, host)


# ----------------------------------------------------------------------------- whole path
def _call_metric(pr: Optional[PreparedReference], metric: Optional[str]) -> str:
    """The mapping metric of a call: the prepared reference's when one is given (``knn`` rejects a conflicting
    ``metric``), else the reference's dispatch (modified Canberra for targets)."""
    if pr is not None:
        if metric is not None and metric != pr.metric:
            raise ValueError("ERROR: metric %r conflicts with the prepared reference's %r" % (metric, pr.metric))
        return pr.metric
    return resolve_metric(metric, False)


def map_cells(target, ref, ref_knn, k: int, metric: Optional[str] = None, dist_factor: float = 0.25,
              ref_mask=None, mode: str = "fast", pca_model: Optional[Dict] = None,
              scores: bool = True) -> Dict[str, object]:
    """The hot path end to end for one target sample (what ``Dataset.transform_pca`` ->
    ``Mapping.map_target`` -> ``Graph.get_mapping_score`` compute, minus the files):

      target   (N,g) float64 PCA coordinates, or raw counts (N,genes) when ``pca_model`` is
               given as dict(gene_idx, sf, mu, sigma, components, mean)
      ref      (M,g) float64 reference PCA coordinates
      ref_knn  (M,k) int32 reference self-kNN (``make_ref_graph``'s sorted rows)

    ``ref`` may be a ``PreparedReference`` (``prepare_reference``): the metric and mask then come from it.
    Returns dict(idx, dist, counts, weights, scores[, pca]) - NumPy if the inputs were."""
    pr = ref if isinstance(ref, PreparedReference) else None
    m = _call_metric(pr, metric)
    host = _is_host(target, ref_knn) if pr is not None else _is_host(target, ref, ref_knn)
    res: Dict[str, object] = {}
    rd = pr.r if pr is not None else _dev(ref, torch.float64)
    if pca_model is not None:
        tq = project(_dev(target, torch.float32), pca_model["gene_idx"], pca_model["sf"], pca_model["mu"],
                     pca_model["sigma"], pca_model["components"], pca_model["mean"])
        g = rd.shape[1]
        res["pca"] = tq
        tq = tq[:, :g].contiguous()
    else:
        tq = _dev(target, torch.float64)
    rk = _dev(ref_knn, torch.int32)
    idx, dst = knn(tq, pr if pr is not None else rd, k, m, dist_factor, ref_mask, False, 0, mode)
    cnt, w = snn_weights(idx, rk, k)
    res.update(idx=idx, dist=dst, counts=cnt, weights=w)
    if scores:
        res["scores"] = mapping_scores(idx, cnt, rd.shape[0], k)
    if host:
        res = {k_: (v.cpu().numpy() if isinstance(v, torch.Tensor) else v) for k_, v in res.items()}
    return res


class _HostPipeline:
    """Reusable device / pinned-host buffers and streams of ``map_cells_host`` for one shape."""

    def __init__(self, n, g, k, m, device):
        self.key = (n, g, k, m, str(device))
        self.dev_in = torch.empty((n, g), dtype=torch.float64, device=device)
        self.idx = torch.empty((n, k), dtype=torch.int32, device=device)
        self.dist = torch.empty((n, k), dtype=torch.float64, device=device)
        self.cnt = torch.empty((n, k), dtype=torch.uint8, device=device)
        self.w = torch.empty((n, k), dtype=torch.float64, device=device)
        self.acc = torch.zeros(m, dtype=torch.int64, device=device)
        self.host = {"idx": torch.empty((n, k), dtype=torch.int32, pin_memory=True),
                     "dist": torch.empty((n, k), dtype=torch.float64, pin_memory=True),
                     "weights": torch.empty((n, k), dtype=torch.float64, pin_memory=True),
                     "scores": torch.empty(m, dtype=torch.float64, pin_memory=True)}
        self.s_in, self.s_out = torch.cuda.Stream(device), torch.cuda.Stream(device)


_PIPE: Dict[tuple, _HostPipeline] = {}
_WAVE = 148 * 384         # queries one wave of the persistent candidate kernel maps (one 384-query work item per SM)


def map_cells_host(target_host: torch.Tensor, ref, ref_knn, k: int, metric: Optional[str] = None,
                   dist_factor: float = 0.25, ref_mask=None, mode: str = "fast", chunks: int = 2,
                   min_piece: int = 32768) -> Dict[str, torch.Tensor]:
    """Host-buffer form of ``map_cells``: ``target_host`` is a pinned CPU float64 (N, g) tensor; the results
    land in pinned host tensors (idx, dist, weights, scores).  The targets are processed in ``chunks``
    pieces so that the host->device copy of piece i+1 and the device->host copy of piece i-1 overlap the
    kernels of piece i (three CUDA streams); the per-reference scores are integer weight sums accumulated piece by
    piece (``score_accumulate``), finalised once.  ``ref`` may be a ``PreparedReference``."""
    require_device()
    pr = ref if isinstance(ref, PreparedReference) else None
    rd = pr.r if pr is not None else _dev(ref, torch.float64)
    rk = _dev(ref_knn, torch.int32)
    n, g = target_host.shape
    m = rd.shape[0]
    key = (n, g, int(k), m, str(rd.device))
    pipe = _PIPE.get(key)
    if pipe is None:
        _PIPE.clear()
        pipe = _PIPE[key] = _HostPipeline(n, g, int(k), m, rd.device)
    met = _call_metric(pr, metric)
    comp = torch.cuda.current_stream()
    chunks = max(1, min(int(chunks), n // int(min_piece) if n >= 2 * int(min_piece) else 1))
    bounds = [n * i // chunks for i in range(chunks + 1)]
    if chunks == 2 and n > _WAVE:
        # the first piece's upload and the last piece's download are the exposed copies: make the first piece the
        # smaller one, and the last one whole waves of the persistent candidate kernel (148 SMs x 384 queries)
        last = (n // 2 + _WAVE - 1) // _WAVE * _WAVE
        if 0 < n - last < n:
            bounds = [0, n - last, n]
    pipe.s_in.wait_stream(comp)
    pipe.s_out.wait_stream(comp)
    pipe.acc.zero_()
    ready = []
    for lo, hi in zip(bounds, bounds[1:]):
        with torch.cuda.stream(pipe.s_in):
            pipe.dev_in[lo:hi].copy_(target_host[lo:hi], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(pipe.s_in)
        ready.append(ev)
    for (lo, hi), ev in zip(zip(bounds, bounds[1:]), ready):
        comp.wait_event(ev)
        knn(pipe.dev_in[lo:hi], pr if pr is not None else rd, k, met, dist_factor, ref_mask, False, 0, mode, out=(pipe.idx[lo:hi], pipe.dist[lo:hi]))
        found = torch.cuda.Event()
        found.record(comp)
        with torch.cuda.stream(pipe.s_out):                 # neighbours go home while the weights are still being made
            pipe.s_out.wait_event(found)
            pipe.host["idx"][lo:hi].copy_(pipe.idx[lo:hi], non_blocking=True)
            pipe.host["dist"][lo:hi].copy_(pipe.dist[lo:hi], non_blocking=True)
        snn_weights(pipe.idx[lo:hi], rk, k, out=(pipe.cnt[lo:hi], pipe.w[lo:hi]))
        done = torch.cuda.Event()
        done.record(comp)
        with torch.cuda.stream(pipe.s_out):
            pipe.s_out.wait_event(done)
            pipe.host["weights"][lo:hi].copy_(pipe.w[lo:hi], non_blocking=True)
        score_accumulate(pipe.idx[lo:hi], pipe.cnt[lo:hi], m, k, acc=pipe.acc)     # integer sums: piece order is immaterial
    sc = scores_finalize(pipe.acc, n)
    pipe.host["scores"].copy_(sc, non_blocking=True)
    comp.synchronize()
    pipe.s_out.synchronize()
    return pipe.host
