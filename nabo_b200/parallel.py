"""Multi-GPU execution of the hot path: one process per GPU, ``torch.distributed`` (NCCL over
NVLink/NVSwitch) for the plumbing.  The reference has no parallelism at all (SURVEY.md section 2);
the path shards because every target cell is an independent query (nabo/_mapping.py:98-130,
186-198).  Two layouts (SURVEY.md 8e):

* **target-sharded** - reference, its self-kNN table and the PCA model are replicated, each rank
  maps a contiguous block of targets.  No data-path collective: neighbour lists and weights stay
  on the rank that made them; only the per-reference scores (a sum over targets) need one
  all-reduce - of INTEGER weight sums (``core.score_accumulate``), so the scores have the same bits
  for any number of GPUs.
* **reference-sharded** - the reference rows are split, every rank sees all targets and produces a
  local top-k with GLOBAL indices (``idx_offset``); rank d merges the block of targets
  ``shard_bounds(N, world, d)``.  The exchange is an all-to-all in which each rank receives only
  its own block (world x fewer bytes than an all-gather), and it is fused into the producer: the
  re-rank kernel writes every result row straight to its destination (``nabo_knn_routed``) -
  either into the receive buffer of the owning GPU, mapped over NVLink through
  ``torch.distributed._symmetric_memory`` (transport ``"p2p"``: no copy kernel, no NCCL call, one
  device-side barrier), or into a per-destination send buffer moved by ONE ``all_to_all_single``
  (transport ``"a2a"``; also what the CPU/gloo tests run).  ``nabo_merge_topk_parts`` then merges
  the per-source blocks in place by (distance, index) - bit-identical to the unsharded result.

Wherever a function takes ``ref`` / ``ref_shard`` it also takes a ``core.PreparedReference`` of it: a rank that
maps many target batches against the same reference (or shard) prepares it once, and every step reuses the packed
operands.  The metric and mask then come from the prepared object (pass ``ref_mask`` / ``ref_mask_shard`` = None).

The compute engine is a parameter so that the host-side logic (bounds, offsets, block layout,
merge slices) is testable on CPU with ``gloo``; the default engine is the CUDA library and
raises without a GPU.
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional, Tuple

import torch
import torch.distributed as dist

__all__ = ["shard_bounds", "CudaEngine", "CandidateExchange", "map_targets_sharded", "knn_reference_sharded",
           "map_reference_sharded"]


def shard_bounds(n: int, world: int, rank: int) -> Tuple[int, int]:
    """Contiguous, balanced block [lo, hi) of `n` rows for `rank` (name-sorted order is preserved)."""
    base, rem = divmod(n, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def _world() -> Tuple[int, int]:
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def _metric_for(ref, metric: Optional[str]) -> str:
    """The call's metric: an explicit one, else the prepared reference's, else modified Canberra (targets)."""
    if metric:
        return metric
    from .core import PreparedReference
    return ref.metric if isinstance(ref, PreparedReference) else "mod_canberra"


# ----------------------------------------------------------------------------- engines
class CudaEngine:
    """Default engine: thin pass-through to nabo_b200.core on the current CUDA device."""

    routed = True          # knn() can deliver rows straight to device addresses (nabo_knn_routed)

    def knn(self, q, r, k, metric, dist_factor, ref_mask, drop_first, idx_offset, mode, out_parts=None):
        from . import core
        return core.knn(q, r, k, metric, dist_factor, ref_mask=ref_mask, drop_first=drop_first,
                        idx_offset=idx_offset, mode=mode, out_parts=out_parts)[:2]

    def merge_parts(self, idx_blocks, dist_blocks, n_rows, k, drop_first):
        from . import core
        return core.merge_topk_parts([b.data_ptr() for b in idx_blocks], [b.data_ptr() for b in dist_blocks],
                                     n_rows, k, idx_blocks[0].device, drop_first)

    def merge_topk(self, idx, dst):
        from . import core
        return core.merge_topk(idx, dst)

    def snn_weights(self, tgt_knn, ref_knn, k):
        from . import core
        return core.snn_weights(tgt_knn, ref_knn, k)

    def score_accumulate(self, tgt_knn, counts, n_ref, k):
        from . import core
        return core.score_accumulate(tgt_knn, counts, n_ref, k)

    def scores_finalize(self, acc, n_total):
        from . import core
        return core.scores_finalize(acc, n_total)


# ----------------------------------------------------------------------------- candidate exchange
def _align(x: int, a: int = 16) -> int:
    return (x + a - 1) // a * a


class CandidateExchange:
    """Buffers and transport of the reference-sharded candidate exchange for one (n_query, k) shape.

    Block layout (bytes), the same in a send buffer and in a receive buffer: the candidates one rank s
    holds for the target block of rank d are ``rows_d x k`` float64 distances followed by ``rows_d x k``
    int32 global indices (``blk_d`` bytes, 16-byte aligned).
      receive buffer of rank d : world blocks of blk_d bytes, block s = what rank s found
      send buffer of rank s    : blocks for d = 0 .. world-1 back to back (a2a transport only)
    """

    def __init__(self, n_query: int, k: int, device, transport: str = "auto"):
        self.rank, self.world = _world()
        self.n, self.k, self.device = int(n_query), int(k), torch.device(device)
        self.bounds = [shard_bounds(self.n, self.world, d)[0] for d in range(self.world)] + [self.n]
        self.rows = [self.bounds[d + 1] - self.bounds[d] for d in range(self.world)]
        self.blk = [_align(r * self.k * 12) for r in self.rows]
        self.max_blk = max(self.blk)
        if transport == "auto":
            transport = os.environ.get("NABO_EXCHANGE", "p2p" if (self.device.type == "cuda" and self.world > 1) else "a2a")
        self.step = 0
        self.hdl = None
        self.p2p_error = None
        if transport == "p2p" and self.world > 1:
            ok = 1
            try:
                import torch.distributed._symmetric_memory as symm
                # two receive buffers used alternately: a rank may run one step ahead of the slowest rank's merge
                self.recv = symm.empty(2 * self.world * self.max_blk, dtype=torch.uint8, device=self.device)
                self.hdl = symm.rendezvous(self.recv, dist.group.WORLD)
                self.peer_base = [int(p) for p in self.hdl.buffer_ptrs]
                self.send = None
            except Exception as e:                                  # no peer mapping on this box: NCCL all-to-all
                ok = 0
                self.p2p_error = repr(e)
            flag = torch.tensor([ok], dtype=torch.int32, device=self.device)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)             # all ranks take the same transport
            if int(flag.item()) == 0:
                transport = "a2a"
                self.hdl = None
        self.transport = transport
        if self.transport != "p2p" or self.world == 1:
            self.transport = "a2a"
            self.recv = torch.empty(max(16, self.world * self.blk[self.rank]), dtype=torch.uint8, device=self.device)
            self.send = torch.empty(max(16, sum(self.blk)), dtype=torch.uint8, device=self.device)
            self.send_off = [sum(self.blk[:d]) for d in range(self.world)]

    # -- where this rank's rows for destination d go
    def _half(self) -> int:
        return (self.step & 1) * self.world * self.max_blk

    def route(self) -> Tuple[List[int], List[int], List[int]]:
        """(bounds, idx addresses, dist addresses) for ``core.knn(out_parts=...)``."""
        ip, dp = [], []
        for d in range(self.world):
            if self.transport == "p2p":
                base = self.peer_base[d] + self._half() + self.rank * self.max_blk
            else:
                base = self.send.data_ptr() + self.send_off[d]
            dp.append(base)
            ip.append(base + self.rows[d] * self.k * 8)
        return self.bounds, ip, dp

    def send_views(self, d: int) -> Tuple[torch.Tensor, torch.Tensor]:
        """(idx, dist) views of the a2a send block for destination d (engines without routed output)."""
        o, r, k = self.send_off[d], self.rows[d], self.k
        dv = self.send[o:o + r * k * 8].view(torch.float64).view(r, k)
        iv = self.send[o + r * k * 8:o + r * k * 12].view(torch.int32).view(r, k)
        return iv, dv

    def exchange(self) -> None:
        """Make every rank's rows for my block visible in my receive buffer (stream-ordered)."""
        if self.world == 1:
            self.recv, self.send = self.send, self.recv            # my only block is the one I wrote
            return
        if self.transport == "p2p":
            self.hdl.barrier(channel=self.step & 1)                # all peers' kernels that write to me are done
        else:
            b = self.blk[self.rank]
            dist.all_to_all_single(self.recv[:self.world * b], self.send[:sum(self.blk)],
                                   output_split_sizes=[b] * self.world, input_split_sizes=self.blk)

    def recv_blocks(self) -> Tuple[List[torch.Tensor], List[torch.Tensor]]:
        """Per-source (idx, dist) views of my receive buffer, in rank (= global index) order."""
        r, k = self.rows[self.rank], self.k
        stride = self.max_blk if self.transport == "p2p" else self.blk[self.rank]
        base = self._half() if self.transport == "p2p" else 0
        buf = self.recv
        ib, db = [], []
        for s in range(self.world):
            o = base + s * stride
            db.append(buf[o:o + r * k * 8].view(torch.float64).view(r, k))
            ib.append(buf[o + r * k * 8:o + r * k * 12].view(torch.int32).view(r, k))
        return ib, db

    def bytes_sent(self) -> int:
        """Bytes this rank ships to OTHER ranks per step."""
        return sum(self.rows[d] * self.k * 12 for d in range(self.world) if d != self.rank)

    def advance(self) -> None:
        self.step += 1


_EXCHANGES: Dict[tuple, CandidateExchange] = {}


def _exchange_for(n: int, k: int, device, transport: str) -> CandidateExchange:
    key = (n, k, str(device), transport, _world())
    ex = _EXCHANGES.get(key)
    if ex is None:
        if len(_EXCHANGES) > 4:
            _EXCHANGES.clear()
        ex = _EXCHANGES[key] = CandidateExchange(n, k, device, transport)
    return ex


# ----------------------------------------------------------------------------- target-sharded
def map_targets_sharded(target_shard, ref, ref_knn, k: int, n_targets_total: int, metric: Optional[str] = None,
                        dist_factor: float = 0.25, ref_mask=None, mode: str = "fast", engine=None,
                        scores: bool = True) -> Dict[str, torch.Tensor]:
    """Target-sharded mapping of this rank's block of target cells.

    Returns this rank's idx / dist / counts / weights and (if ``scores``) the GLOBAL per-reference
    mapping scores (identical on every rank, and for every world size, after the integer all-reduce)."""
    engine = engine or CudaEngine()
    rank, world = _world()
    metric = _metric_for(ref, metric)
    idx, dst = engine.knn(target_shard, ref, k, metric, dist_factor, ref_mask, False, 0, mode)
    cnt, w = engine.snn_weights(idx, ref_knn, k)
    out = {"idx": idx, "dist": dst, "counts": cnt, "weights": w}
    if scores:
        acc = engine.score_accumulate(idx, cnt, ref.shape[0], k)
        if world > 1:
            dist.all_reduce(acc, op=dist.ReduceOp.SUM)
        out["score_acc"] = acc
        out["scores"] = engine.scores_finalize(acc, n_targets_total)
    return out


# ----------------------------------------------------------------------------- reference-sharded
def knn_reference_sharded(q, ref_shard, ref_offset: int, k: int, metric: str, dist_factor: float = 0.25,
                          ref_mask_shard=None, drop_first: bool = False, mode: str = "fast", engine=None,
                          merge_slice: bool = True, transport: str = "auto", timings: Optional[dict] = None):
    """kNN of ALL queries against a row-sharded reference.

    Each rank computes a local top-(k [+1]) with global indices whose rows are delivered to the rank that
    owns the query block (see the module docstring); every rank merges its own block and returns
    (lo, hi, idx, dist) for it.  ``merge_slice=False`` additionally all-gathers the merged blocks so that
    every rank returns all queries (lo, hi = 0, N).  ``timings`` (dict of lists of (start, end) CUDA event
    pairs keyed by stage) is filled when given."""
    engine = engine or CudaEngine()
    rank, world = _world()
    kk = k + (1 if drop_first else 0)                  # the dropped "first" element is global, decide after merge
    n = q.shape[0]
    ex = _exchange_for(n, kk, q.device, transport)
    kk_local = min(kk, ref_shard.shape[0])

    def stage(name):
        if timings is None:
            return None
        ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        timings.setdefault(name, []).append(ev)
        ev[0].record()
        return ev

    def done(ev):
        if ev is not None:
            ev[1].record()

    ev = stage("knn")
    if getattr(engine, "routed", False) and kk_local == kk:
        engine.knn(q, ref_shard, kk, metric, dist_factor, ref_mask_shard, False, ref_offset, mode,
                   out_parts=ex.route())
    else:
        idx, dst = engine.knn(q, ref_shard, kk_local, metric, dist_factor, ref_mask_shard, False, ref_offset, mode)
        if kk_local < kk:                              # tiny shard: pad with "missing"
            pad_i = torch.full((n, kk - kk_local), -1, dtype=idx.dtype, device=idx.device)
            pad_d = torch.full((n, kk - kk_local), float("nan"), dtype=dst.dtype, device=dst.device)
            idx, dst = torch.cat([idx, pad_i], 1), torch.cat([dst, pad_d], 1)
        if ex.transport == "p2p":
            raise RuntimeError("nabo_b200.parallel: the p2p transport needs an engine with routed output")
        for d in range(world):
            iv, dv = ex.send_views(d)
            iv.copy_(idx[ex.bounds[d]:ex.bounds[d + 1]])
            dv.copy_(dst[ex.bounds[d]:ex.bounds[d + 1]])
    done(ev)
    ev = stage("exchange")
    ex.exchange()
    done(ev)
    ev = stage("merge")
    ib, db = ex.recv_blocks()
    lo, hi = ex.bounds[rank], ex.bounds[rank + 1]
    mi, md = engine.merge_parts(ib, db, hi - lo, kk, drop_first)
    done(ev)
    ex.advance()
    if not merge_slice and world > 1:
        # equal-sized padded blocks: all_gather_into_tensor wants one shape everywhere
        rows = max(ex.rows)
        pi = torch.full((rows, k), -1, dtype=mi.dtype, device=mi.device)
        pd = torch.full((rows, k), float("nan"), dtype=md.dtype, device=md.device)
        pi[:hi - lo], pd[:hi - lo] = mi, md
        gi = torch.empty((world * rows, k), dtype=mi.dtype, device=mi.device)
        gd = torch.empty((world * rows, k), dtype=md.dtype, device=md.device)
        dist.all_gather_into_tensor(gi, pi)
        dist.all_gather_into_tensor(gd, pd)
        keep = torch.cat([torch.arange(ex.rows[d], device=mi.device) + d * rows for d in range(world)])
        return 0, n, gi[keep].contiguous(), gd[keep].contiguous()
    return lo, hi, mi, md


def map_reference_sharded(targets, ref_shard, ref_offset: int, n_ref_total: int, ref_knn, k: int,
                          metric: Optional[str] = None, dist_factor: float = 0.25, ref_mask_shard=None,
                          mode: str = "fast", engine=None, scores: bool = True, transport: str = "auto",
                          timings: Optional[dict] = None) -> Dict[str, object]:
    """Reference-sharded mapping (BASELINE config 4): all targets against this rank's reference rows,
    fused candidate exchange + merge, then SNN weights with the replicated reference kNN table (global
    indices) and an all-reduce of the integer per-reference weight sums.  Returns results for this rank's
    target block [lo, hi)."""
    engine = engine or CudaEngine()
    rank, world = _world()
    metric = _metric_for(ref_shard, metric)
    lo, hi, idx, dst = knn_reference_sharded(targets, ref_shard, ref_offset, k, metric, dist_factor, ref_mask_shard,
                                             False, mode, engine, merge_slice=True, transport=transport,
                                             timings=timings)

    def stage(name):
        if timings is None:
            return None
        ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        timings.setdefault(name, []).append(ev)
        ev[0].record()
        return ev

    ev = stage("snn")
    cnt, w = engine.snn_weights(idx, ref_knn, k)
    if ev:
        ev[1].record()
    out = {"lo": lo, "hi": hi, "idx": idx, "dist": dst, "counts": cnt, "weights": w}
    if scores:
        ev = stage("scores")
        acc = engine.score_accumulate(idx, cnt, n_ref_total, k)
        if world > 1:
            dist.all_reduce(acc, op=dist.ReduceOp.SUM)
        out["score_acc"] = acc
        out["scores"] = engine.scores_finalize(acc, targets.shape[0])
        if ev:
            ev[1].record()
    return out
