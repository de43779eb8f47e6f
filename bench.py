#!/usr/bin/env python
"""Benchmark of the nabo cell-projection hot path on B200 (contract: see task statement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--metric ...] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): 100 000 target cells mapped onto a 100 000-cell
reference, 50 PCs, k = 30.  One *step* = one pass of the hot path over one batch of target
cells: fused distance + per-query top-k (`Mapping.map_target`'s `_calc_dist`), SNN neighbour
weights (`_calc_snn`) and per-reference mapping scores (`Graph.get_mapping_score`).  The
reference self-kNN table those weights need (`make_ref_graph`) is built once in setup.
Headline metric = target cells mapped per second; the Euclidean metric is the headline
(north_star quotes its targets on it), modified Canberra - the reference's own target->ref
metric - is measured in the same run and reported under "mod_canberra".

N > 1 (torchrun, one rank per GPU): targets are sharded, the reference is replicated, no
data-path collective -> weak scaling; value = all ranks' cells / max-over-ranks time.

`--impl reference`: the reference's CPU algorithm (oracle/nabo_oracle.c, a loop-for-loop
port pinned against the unmodified reference; nabo itself is Python + numba and
/root/reference does not exist on the GPU box) on all host threads, on a bounded sample of
the same workload per step.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--metric", default="euclidean", choices=["euclidean", "mod_canberra", "cosine"])
    ap.add_argument("--n-ref", type=int, default=100_000)
    ap.add_argument("--n-query", type=int, default=100_000, help="target cells per GPU per step")
    ap.add_argument("--comps", type=int, default=50)
    ap.add_argument("--k", type=int, default=30)
    ap.add_argument("--engine", default="fast", choices=["fast", "exact"])
    ap.add_argument("--shard", default="targets", choices=["targets", "reference"],
                    help="targets: every GPU maps its own --n-query targets against the same --n-ref reference "
                         "(no collective); reference: every GPU holds --n-ref reference rows of a --gpus x larger "
                         "reference, all GPUs map the same --n-query targets, candidates are all-gathered and merged "
                         "(BASELINE config 4)")
    ap.add_argument("--workload", default="config2", choices=["config2", "config5"],
                    help="config2 (default): the headline line; config5: counts -> projection -> cosine kNN -> scores per sample")
    ap.add_argument("--c5-cells", type=int, default=500_000)
    ap.add_argument("--c5-ref", type=int, default=2_000_000)
    ap.add_argument("--c5-genes", type=int, default=2000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-config5", action="store_true", help="skip the config-5 block (one sample per GPU)")
    ap.add_argument("--no-projection", action="store_true", help="skip the projection (A1/A2) measurement")
    ap.add_argument("--no-ref-sharded", action="store_true", help="skip the reference-sharded (config 4) block")
    ap.add_argument("--ref-rows-per-gpu", type=int, default=1_250_000)
    ap.add_argument("--ref-batch", type=int, default=227_328,
                    help="targets per step of the reference-sharded block (default 4 x 148 SMs x 384 queries per work item: "
                         "whole waves of the persistent candidate kernel; 5 batches = 1.14 M targets)")
    ap.add_argument("--no-secondary", action="store_true", help="skip the modified-Canberra measurement")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU work per cpu_baseline sample")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (neighbour indices and "
                         "distances, SNN counts and weights, per-reference scores) as DIR/<name>.npy in float32 / "
                         "float64, at most 64 MB in all: a fixed, seeded sample of target rows when the whole output "
                         "is larger (DIR/rows.npy lists them).  Default workload only")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "b200" or a.workload != "config2" or a.shard != "targets"):
        ap.error("--dump-outputs covers the default workload (--impl b200 --workload config2 --shard targets)")
    return a


WORKLOAD = "config2: {nq} target x {nr} reference cells, {g} PCs, k={k}, {metric}"


def canberra_roofline(g, n, m, kernel_ms):
    """Roofline of the bit-sliced modified-Canberra candidate pass (canberra_sliced.cu).  The pipe that bounds it is
    the integer ALU (148 SM x 64 lanes per clock at the max SM clock - nominal, MEASURED_PEAKS.json has no integer
    figure): a pair is rejected by the count bound for 3.25 / 32 LOP3 per dimension (1 interval test + 2.25
    carry-save adder ops per 32 references), and `frac` is that EXECUTED work against that pipe.  SURVEY 8(d)'s
    algorithmic figure (5 FP ops per (pair, dimension) on the FP32 pipe) is kept as a side key: ~98 % of it is
    never executed, so its ratio to the FP32 peak is not a roofline fraction."""
    t = kernel_ms * 1e-3
    lop = 3.25 / 32.0 * g * n * m / t / 1e12
    lop_peak = 148 * 64 * 1.965e9 / 1e12
    alg = 5.0 * g * n * m / t / 1e12
    fp32_peak = 148 * 128 * 2 * 1.965e9 / 1e12
    return {"bound": "alu", "kernel": "cbs::sliced_kernel", "achieved": lop, "unit": "TLOP3/s", "peak": lop_peak,
            "frac": lop / lop_peak, "peak_source": "nominal B200 integer-ALU issue rate at max SM clock",
            "pairs_per_s": n * m / t,
            "algorithmic_fp32": {"achieved": alg, "unit": "TFLOP/s", "nominal_fp32_peak": fp32_peak,
                                 "note": "5 FP ops per (pair, dimension) of the full metric; the count bound prunes "
                                         "~98 % of it before the FP32 pipe, so achieved / peak is not a fraction of a roof"},
            "traffic": None}


DUMP_BYTES = 64_000_000


def dump_outputs(path, out, budget=DUMP_BYTES, suffix=""):
    """Write the arrays of one mapping step (`out`: name -> host array; "scores" per reference cell, the others per
    target row) as path/<name><suffix>.npy.  Integers are stored exactly as float64 (indices) or float32 (counts).
    When the per-target arrays do not fit in `budget` bytes, only a sample of target rows drawn with a fixed seed is
    written; rows.npy holds the row numbers, so that two runs with the same arguments give the same files."""
    exact = {np.dtype(np.int32): np.float64, np.dtype(np.int64): np.float64, np.dtype(np.uint8): np.float32}
    out = {name: np.ascontiguousarray(v, dtype=exact.get(v.dtype, v.dtype)) for name, v in out.items()}
    per_row = [name for name in out if name != "scores"]
    n = out[per_row[0]].shape[0]
    row_bytes = 8 + sum(out[name][:1].nbytes for name in per_row)           # + the row number itself
    keep = min(n, max(0, budget - out["scores"].nbytes - 4096) // row_bytes)   # 4 KB for the .npy headers
    rows = np.arange(n) if keep == n else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    out.update({name: out[name][rows] for name in per_row}, rows=rows.astype(np.float64))
    os.makedirs(path, exist_ok=True)
    for name, v in out.items():
        np.save(os.path.join(path, name + suffix + ".npy"), v, allow_pickle=False)
    return keep, n


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


# ----------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index: int, period: float = 0.02):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._halt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {}
        for n in dir(nv):
            if n.startswith("nvmlClocksEventReason") or n.startswith("nvmlClocksThrottleReason"):
                v = getattr(nv, n)
                if isinstance(v, int) and v:
                    names.setdefault(v, n.replace("nvmlClocksEventReason", "").replace("nvmlClocksThrottleReason", ""))
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if r & bit and nm not in ("GpuIdle", "None", "All"):
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        snake = {"SwPowerCap": "sw_power_cap", "HwSlowdown": "hw_slowdown", "HwThermalSlowdown": "hw_thermal_slowdown",
                 "SwThermalSlowdown": "sw_thermal_slowdown", "HwPowerBrakeSlowdown": "hw_power_brake_slowdown",
                 "SyncBoost": "sync_boost", "ApplicationsClocksSetting": "applications_clocks_setting",
                 "DisplayClockSetting": "display_clock_setting"}
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "samples": len(self.samples),
                "reasons": sorted(snake.get(r, r) for r in self.reasons)}


# ----------------------------------------------------------------------------- CPU baseline / reference arm
def cpu_reference_rate(ref, tgt, ref_knn, k, metric, seconds, threads):
    """Targets/s of the reference algorithm (C port) on `threads` host threads, on a bounded
    sample of the workload: distances to every reference cell, full-row sort, SNN counts, scores."""
    from oracle import c_port, nabo_oracle as O
    c_port.build()
    m = "euclidean" if metric == "euclidean" else "mod_canberra"
    if metric == "cosine":
        raise SystemExit("the reference has no cosine metric; no CPU baseline for it")
    t0 = time.perf_counter()
    c_port.knn(tgt[:4], ref, k, m, 0.25, nthreads=1)
    per = (time.perf_counter() - t0) / 4
    n = int(max(threads * 2, min(len(tgt), seconds * threads / max(per, 1e-6))))
    n = max(threads, n // threads * threads)
    sample = tgt[:n]
    lut = O.snn_weight_lut(k)
    t0 = time.perf_counter()
    idx, _ = c_port.knn(sample, ref, k, m, 0.25, nthreads=threads)
    cnt = c_port.snn_counts(idx, ref_knn, nthreads=threads)
    c_port.scores(idx, cnt, lut, ref.shape[0])
    dt = time.perf_counter() - t0
    return n / dt, n, dt


def run_reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from nabo_b200 import synth
    from oracle import c_port
    threads = os.cpu_count() or 1
    ref = synth.pc_mixture(a.n_ref, a.comps, seed=1)
    tgt = synth.pc_mixture(min(a.n_query, 4096 * 4), a.comps, seed=101)
    # the reference table the SNN step needs: built with the same CPU port on a subset is too slow
    # at 100k x 100k (hours), so the bounded sample uses random neighbour lists of the right shape;
    # the SNN/score cost does not depend on their values.
    rng = np.random.default_rng(0)
    ref_knn = rng.integers(0, a.n_ref, size=(a.n_ref, a.k), dtype=np.int32)
    # size each step to ~3 s of wall time
    rate0, n0, _ = cpu_reference_rate(ref, tgt, ref_knn, a.k, a.metric, 1.0, threads)
    per_step = int(max(threads, min(len(tgt), rate0 * 3.0)) // threads * threads)
    times = []
    for s in range(a.warmup + a.steps):
        t0 = time.perf_counter()
        idx, _ = c_port.knn(tgt[:per_step], ref, a.k, "euclidean" if a.metric == "euclidean" else "mod_canberra",
                            0.25, nthreads=threads)
        cnt = c_port.snn_counts(idx, ref_knn, nthreads=threads)
        c_port.scores(idx, cnt, np.zeros(a.k + 1), a.n_ref)
        dt = time.perf_counter() - t0
        if s >= a.warmup:
            times.append(dt)
    ms = 1e3 * sum(times) / len(times)
    value = per_step / (ms / 1e3)
    line = {
        "impl": "reference", "metric": "target_cells_mapped_per_s", "value": value, "unit": "cells/s",
        "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD.format(nq=a.n_query, nr=a.n_ref, g=a.comps, k=a.k, metric=a.metric),
                   "sample": "%d target cells per step against all %d reference cells" % (per_step, a.n_ref),
                   "substitutions": "the reference kNN table the SNN step reads is a random table of the right shape and the "
                                    "weight table is zero (building the true table with the CPU port would take hours at "
                                    "this size); the cost of the SNN / score loops does not depend on the values"},
        "cpu_baseline": {"value": value, "unit": "cells/s", "cores": threads, "kind": "port",
                         "sample": "%d targets x %d references per step, %d host threads; C port of "
                                   "nabo/_mapping.py:16-45,135-146,186-198 + _graph.py:643-653" % (per_step, a.n_ref, threads)},
        "e2e": {"value": value, "unit": "cells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- B200 arm, reference-sharded
def _ev_ms(pairs):
    return [s.elapsed_time(e) for s, e in pairs]


def ref_sharded_block(a, dev, rank, world, rows_per_gpu, n_batch, n_batches, steps, warmup, metric="euclidean",
                      check_rows=1024):
    """BASELINE config 4 (the north-star shape at 8 GPUs): a reference of world x rows_per_gpu cells split by rows,
    every rank maps the same batches of targets against its rows; the re-rank kernel delivers each result row to
    the rank that owns the target (peer memory over NVLink, or one all_to_all_single), which merges the per-source
    lists in place, computes the SNN weights against the replicated TRUE reference kNN table and adds its integer
    weight sums to the all-reduced per-reference score accumulator.  One step = one batch of n_batch targets.
    Untimed, in the same run: the merged (idx, dist) of check_rows sampled targets is compared bit for bit with
    the unsharded exact engine over the whole reference on rank 0."""
    import torch
    import torch.distributed as dist
    from nabo_b200 import core, parallel, synth

    g, k = a.comps, a.k
    M = rows_per_gpu
    m_total = M * world
    t_setup = time.perf_counter()
    ref = synth.pc_mixture_device(M, g, seed=1 + 1000 * rank, device=dev)            # this rank's rows
    if world > 1:
        full = torch.empty((m_total, g), dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(full, ref)
    else:
        full = ref
    # the replicated reference kNN table (make_ref_graph's sorted rows), built by the same sharded path:
    # every rank queries all cells against its rows, self dropped after the global merge
    ref_knn = torch.empty((m_total, k), dtype=torch.int32, device=dev)
    chunk = n_batch
    for lo in range(0, m_total, chunk):
        hi = min(m_total, lo + chunk)
        _, _, ri, _ = parallel.knn_reference_sharded(full[lo:hi], ref, rank * M, k, "euclidean", drop_first=True,
                                                     mode=a.engine, merge_slice=False)
        ref_knn[lo:hi] = ri
    batches = [synth.pc_mixture_device(n_batch, g, seed=101 + b, device=dev) for b in range(n_batches)]
    torch.cuda.synchronize()
    setup_s = time.perf_counter() - t_setup
    flush = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def step(q, timings=None):
        return parallel.map_reference_sharded(q, ref, rank * M, m_total, ref_knn, k, metric=metric, dist_factor=0.25,
                                              mode=a.engine, timings=timings)

    for i in range(warmup):
        step(batches[i % n_batches])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    sampler = ClockSampler(dev.index)
    sampler.start()
    for i in range(steps):
        flush.zero_()
        ev[i][0].record()
        step(batches[i % n_batches])
        ev[i][1].record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clocks = sampler.stop()
    t = torch.tensor([sum(_ev_ms(ev))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / steps

    # per-stage pass (untimed): CUDA events around the stages + the library's own events inside the kNN call
    stages = {}
    kstats = []
    for i in range(min(steps, n_batches)):
        flush.zero_()
        step(batches[i], timings=stages)
        r = core.knn(batches[i], ref, k, metric, 0.25, idx_offset=rank * M, mode=a.engine, return_stats=True)
        kstats.append(r[2])
    torch.cuda.synchronize()
    stage_ms = {name: sum(_ev_ms(p)) / len(p) for name, p in stages.items()}
    if kstats:
        stage_ms["knn_candidates"] = sum(x["main_kernel_ms"] for x in kstats) / len(kstats)
        stage_ms["knn_rerank"] = sum(x["rerank_ms"] for x in kstats) / len(kstats)
        stage_ms["knn_prepare"] = sum(x["prep_ms"] for x in kstats) / len(kstats)
        stage_ms["knn_exact_fallback"] = sum(x["fallback_ms"] for x in kstats) / len(kstats)
        stage_ms["knn_rows_to_exact_fallback"] = sum(x["rows_exact_fallback"] for x in kstats) / len(kstats)
    st = torch.tensor([stage_ms.get(n_, 0.0) for n_ in sorted(stage_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(st, op=dist.ReduceOp.MAX)
    stage_ms = {n_: float(v) for n_, v in zip(sorted(stage_ms), st.tolist())}

    # in-run parity (untimed): sampled targets of batch 0, sharded result vs the unsharded exact engine
    out = step(batches[0])
    sel = torch.linspace(0, n_batch - 1, check_rows, device=dev).long().unique()
    mine = sel[(sel >= out["lo"]) & (sel < out["hi"])]
    rows_i = out["idx"][mine - out["lo"]]
    rows_d = out["dist"][mine - out["lo"]]
    rows_w = out["weights"][mine - out["lo"]]
    if world > 1:
        sizes = [None] * world
        dist.all_gather_object(sizes, int(mine.numel()))
        pad = max(sizes)
        def padded(x):
            p = torch.zeros((pad,) + tuple(x.shape[1:]), dtype=x.dtype, device=dev)
            p[:x.shape[0]] = x
            return p
        gi = [torch.empty((pad, k), dtype=torch.int32, device=dev) for _ in range(world)]
        gd = [torch.empty((pad, k), dtype=torch.float64, device=dev) for _ in range(world)]
        gw = [torch.empty((pad, k), dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(gi, padded(rows_i))
        dist.all_gather(gd, padded(rows_d))
        dist.all_gather(gw, padded(rows_w))
        rows_i = torch.cat([x[:n_] for x, n_ in zip(gi, sizes)])
        rows_d = torch.cat([x[:n_] for x, n_ in zip(gd, sizes)])
        rows_w = torch.cat([x[:n_] for x, n_ in zip(gw, sizes)])
    parity = None
    if rank == 0:
        xi, xd = core.knn(batches[0][sel], full, k, metric, 0.25, mode="exact")
        _, xw = core.snn_weights(xi, ref_knn, k)
        parity = {"rows": int(sel.numel()), "against": "unsharded exact engine (FP64 brute force) over all %d reference "
                                                        "cells + SNN weights on the true reference kNN table" % m_total,
                  "idx_equal": bool(torch.equal(rows_i, xi)),
                  "dist_bit_equal": bool(torch.equal(rows_d.view(torch.int64), xd.view(torch.int64))),
                  "weights_bit_equal": bool(torch.equal(rows_w.view(torch.int64), xw.view(torch.int64)))}
        if not (parity["idx_equal"] and parity["dist_bit_equal"] and parity["weights_bit_equal"]):
            raise SystemExit("ref_sharded parity check FAILED: %r" % (parity,))
    ex = parallel._exchange_for(n_batch, k, dev, "auto")
    peaks = load_peaks()
    kern = stage_ms.get("knn_candidates", 0.0)
    flops = 2.0 * g * n_batch * M
    block = {
        "workload": "config4: %d targets per step (%d batches = %d targets) x %d reference cells row-sharded over %d GPU(s) "
                    "(%d rows each), %d PCs, k=%d, %s" % (n_batch, n_batches, n_batch * n_batches, m_total, world, M, g, k, metric),
        "value": n_batch / (ms_step / 1e3), "unit": "cells/s", "ms_per_step": ms_step, "steps": steps, "warmup": warmup,
        "targets_per_step": n_batch, "n_ref_total": m_total, "rows_per_gpu": M,
        "pairs_per_s": float(n_batch) * m_total / (ms_step / 1e3),
        "stage_ms": stage_ms,
        "exchange": {"transport": ex.transport, "bytes_sent_per_rank_per_step": ex.bytes_sent(),
                     "all_gather_equivalent_bytes_received": (world - 1) * n_batch * k * 12,
                     "what": "(float64 distance, int32 global index) x k per target, written by rerank_kernel "
                             "straight into the owner's receive block; merged in place by merge_kernel"},
        "score_reduce": {"all_reduce_bytes": m_total * 8, "dtype": "int64 weight sums (hundredths)"},
        "ref_knn": "true table: %d-cell self-kNN (k=%d) built in setup by the same sharded path" % (m_total, k),
        "parity": parity, "setup_s": setup_s, "clocks": clocks,
        "roofline": {"bound": "tensor", "kernel": "tc::candidates_kernel", "achieved": flops / (kern * 1e-3) / 1e12 if kern else None,
                     "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                     "frac": (flops / (kern * 1e-3) / 1e12 / peaks["bf16_tflops_sustained"]) if kern else None,
                     "peak_source": "%s bf16 sustained (kernel timed inside a long step)" % peaks["source"],
                     "executed_tflops": (flops * (((3 * g + 3 + 15) // 16 * 16) / g) / (kern * 1e-3) / 1e12) if kern else None,
                     "traffic": None},
    }
    del full, ref_knn, batches, flush
    torch.cuda.empty_cache()
    return block


def projection_block(dev, steps=5, warmup=2, shapes=None):
    """A1/A2 of the path (get_scaled_values + transform_pca, nabo/_dataset.py:905-913, 1028) on dense count blocks
    of the BASELINE shapes: config 1 (5 000 cells, 2 000 HVGs -> 25 PCs) and a config-5 sample slice (262 144 of
    the 500 000 cells, 2 000 HVGs -> 50 PCs; the kernel is linear in cells).  Algorithmic work (SURVEY 8d):
    2*G*C flop per cell, 4*G bytes of counts per cell in, 8*C out.  Both engines are timed: the FP64 tensor-core
    GEMM (nabo_project_dense_mma, the product path) and the simple FP64 CUDA-core kernel it replaced."""
    import torch
    from nabo_b200 import core, synth
    out = {}
    fp64_peak = 40.0        # TFLOP/s, NVIDIA's B200 FP64 figure (no measured FP64 peak in MEASURED_PEAKS.json)
    peaks = load_peaks()
    for name, n, G, nc in (shapes or (("config1", 5000, 2000, 25), ("config5_slice", 262144, 2000, 50))):
        counts = synth.nb_counts_device(n, G, seed=11, device=dev)
        tot = counts.sum(1)
        sf = (1000.0 / torch.where(tot > 0, tot, torch.ones_like(tot))).to(torch.float32)
        x = counts[:4096] * sf[:4096, None]
        mu = x.mean(0).to(torch.float64)
        sigma = x.std(0).to(torch.float64) + 1e-3
        gen = torch.Generator(device=dev)
        gen.manual_seed(5)
        comps = torch.linalg.qr(torch.randn((G, nc), generator=gen, device=dev, dtype=torch.float64))[0].T.contiguous()
        mean = 0.1 * torch.randn(G, generator=gen, device=dev, dtype=torch.float64)
        gi = torch.arange(G, dtype=torch.int32, device=dev)
        res = torch.empty((n, nc), dtype=torch.float64, device=dev)
        entry = {"cells": n, "genes": G, "comps": nc, "nonzero_fraction": float((counts > 0).float().mean())}
        for engine in ("mma", "simple"):
            for _ in range(warmup):
                core.project(counts, gi, sf, mu, sigma, comps, mean, engine=engine, out=res)
            torch.cuda.synchronize()
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
            for s_, e_ in ev:
                s_.record()
                core.project(counts, gi, sf, mu, sigma, comps, mean, engine=engine, out=res)
                e_.record()
            torch.cuda.synchronize()
            ms = sum(_ev_ms(ev)) / steps
            flops, nbytes = 2.0 * G * nc * n, 4.0 * n * G + 8.0 * n * nc
            entry[engine] = {"ms": ms, "cells_per_s": n / (ms / 1e3), "fp64_tflops": flops / (ms * 1e-3) / 1e12,
                             "frac_fp64_peak": flops / (ms * 1e-3) / 1e12 / fp64_peak, "gb_per_s": nbytes / (ms * 1e-3) / 1e9,
                             "frac_hbm_peak": nbytes / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"]}
        entry["bound"] = "fp64 pipe (nominal %.0f TFLOP/s); the counts (4*G B per cell) stream once from HBM" % fp64_peak
        out[name] = entry
        del counts, res
    torch.cuda.empty_cache()
    return out


def score_determinism_check(dev, rank, world, ref, ref_knn, k, n_targets=65_536):
    """The same fixed problem (n_targets targets, the config-2 reference) mapped three ways - unsharded on one
    GPU, target-sharded and reference-sharded over all ranks - must give the SAME per-reference score bits: the
    score reduction is an integer sum (core.score_accumulate), so it does not depend on the GPU count.  The
    SHA-256 of the score vector is reported; it is the same string at --gpus 1, 2, 4 and 8."""
    import hashlib
    import torch
    from nabo_b200 import core, parallel, synth
    M = ref.shape[0]
    tgt = synth.pc_mixture_device(n_targets, ref.shape[1], seed=4242, device=dev)
    ref_knn = ref_knn.contiguous()
    i0, _ = core.knn(tgt, ref, k, "euclidean", mode="fast")
    c0, _ = core.snn_weights(i0, ref_knn, k)
    single = core.scores_finalize(core.score_accumulate(i0, c0, M, k), n_targets)
    lo, hi = parallel.shard_bounds(n_targets, world, rank)
    a_ = parallel.map_targets_sharded(tgt[lo:hi].contiguous(), ref, ref_knn, k, n_targets, metric="euclidean")
    rlo, rhi = parallel.shard_bounds(M, world, rank)
    b_ = parallel.map_reference_sharded(tgt, ref[rlo:rhi].contiguous(), rlo, M, ref_knn, k, metric="euclidean")
    same = bool(torch.equal(single.view(torch.int64), a_["scores"].view(torch.int64)) and
                torch.equal(single.view(torch.int64), b_["scores"].view(torch.int64)))
    if not same:
        raise SystemExit("score determinism check FAILED on rank %d" % rank)
    return {"targets": n_targets, "n_ref": M, "bit_identical_single_vs_target_sharded_vs_reference_sharded": same,
            "scores_sha256": hashlib.sha256(single.cpu().numpy().tobytes()).hexdigest()}


def config5_block(a, dev, rank, world, steps, warmup, samples_per_gpu=None):
    """BASELINE config 5: 8 target samples x --c5-cells cells of raw counts (--c5-genes HVG columns) against a
    --c5-ref-cell reference in 50-PC space, cosine, k = 30, target-sharded: rank r maps samples r, r + world, ...
    (samples_per_gpu = 1 inside the default line: ONE sample per GPU, so the block takes seconds at any GPU count).
    One step = one sample through the whole path: counts -> scaling + projection (FP64 tensor-core GEMM) -> cosine
    kNN (tcgen05 candidates + FP64 re-rank) -> SNN weights -> integer score accumulation.  The per-reference scores
    of all samples are all-reduced once at the end (integers: same bits for any GPU count)."""
    import torch
    import torch.distributed as dist
    from nabo_b200 import core, synth

    local = dev.index
    M, N, G, nc, k, n_samples = a.c5_ref, a.c5_cells, a.c5_genes, a.comps, a.k, 8
    t0 = time.perf_counter()
    ref = synth.pc_mixture_device(M, nc, seed=1, device=dev)
    ref_knn = torch.empty((M, k), dtype=torch.int32, device=dev)
    for lo in range(0, M, 500_000):                                  # make_ref_graph's table, cosine
        hi = min(M, lo + 500_000)
        ref_knn[lo:hi] = core.knn(ref[lo:hi], ref, k + 1, "cosine", mode=a.engine)[0][:, 1:]
    gen = torch.Generator(device=dev)
    gen.manual_seed(5)
    comps = torch.linalg.qr(torch.randn((G, nc), generator=gen, device=dev, dtype=torch.float64))[0].T.contiguous()
    mean = 0.1 * torch.randn(G, generator=gen, device=dev, dtype=torch.float64)
    probe = synth.nb_counts_device(4096, G, seed=99, device=dev)
    ptot = probe.sum(1)
    x = probe * (1000.0 / torch.where(ptot > 0, ptot, torch.ones_like(ptot)))[:, None]
    mu, sigma = x.mean(0).to(torch.float64), x.std(0).to(torch.float64) + 1e-3
    gi = torch.arange(G, dtype=torch.int32, device=dev)
    mine = list(range(rank, n_samples, world)) if samples_per_gpu is None else [rank % n_samples][:samples_per_gpu]
    samples = []
    for s_ in mine:
        c = synth.nb_counts_device(N, G, seed=100 + s_, device=dev)
        tot = c.sum(1)
        samples.append((c, (1000.0 / torch.where(tot > 0, tot, torch.ones_like(tot))).to(torch.float32)))
    torch.cuda.synchronize()
    setup_s = time.perf_counter() - t0
    acc = torch.zeros(M, dtype=torch.int64, device=dev)
    pca = torch.empty((N, nc), dtype=torch.float64, device=dev)
    stage = {n_: [] for n_ in ("projection", "knn", "snn", "scores")}

    def step(i, timed_stages=False):
        counts, sf = samples[i % len(samples)]
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(5)] if timed_stages else None
        if marks: marks[0].record()
        core.project(counts, gi, sf, mu, sigma, comps, mean, engine="mma", out=pca)
        if marks: marks[1].record()
        idx, dst = core.knn(pca, ref, k, "cosine", mode=a.engine)
        if marks: marks[2].record()
        cnt, w = core.snn_weights(idx, ref_knn, k)
        if marks: marks[3].record()
        core.score_accumulate(idx, cnt, M, k, acc=acc)
        if marks:
            marks[4].record()
            for j_, n_ in enumerate(("projection", "knn", "snn", "scores")):
                stage[n_].append((marks[j_], marks[j_ + 1]))
        return idx, dst, w

    for i in range(warmup):
        step(i)
    acc.zero_()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    sampler = ClockSampler(local)
    sampler.start()
    for i in range(steps):
        ev[i][0].record()
        step(i)
        ev[i][1].record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clocks = sampler.stop()
    t = torch.tensor([sum(_ev_ms(ev))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(acc, op=dist.ReduceOp.SUM)
    scores = core.scores_finalize(acc, world * steps * N)
    for i in range(min(2, steps)):
        step(i, timed_stages=True)
    torch.cuda.synchronize()
    ms_step = float(t.item()) / steps
    mean_ms = {n_: sum(_ev_ms(p_)) / max(1, len(p_)) for n_, p_ in stage.items()}
    block = {
        "workload": "config5: %d cells x %d HVG counts per sample -> %d PCs -> cosine kNN (k=%d) against %d reference cells -> "
                    "SNN weights -> mapping scores; target-sharded, %d sample(s) per GPU" % (N, G, nc, k, M, len(mine)),
        "value": world * N / (ms_step / 1e3), "unit": "cells/s", "ms_per_step": ms_step, "steps": steps, "warmup": warmup,
        "stage_ms": mean_ms,
        "projection_tflops_fp64": 2.0 * G * nc * N / (max(1e-9, mean_ms["projection"]) * 1e-3) / 1e12,
        "knn_pairs_per_s": float(N) * M / (max(1e-9, mean_ms["knn"]) * 1e-3),
        "reference_cells_with_a_score": int((scores > 0).sum()), "setup_s": setup_s, "clocks": clocks,
    }
    del samples, ref, ref_knn, acc, pca
    torch.cuda.empty_cache()
    return block


def run_b200_config5(a):
    """`--workload config5`: the config-5 block with all 8 samples dealt over the GPUs, as the whole line."""
    import torch
    import torch.distributed as dist
    from nabo_b200 import build

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if a.gpus > 1 and world != a.gpus:
        raise SystemExit("--gpus %d needs torchrun --nproc-per-node %d (WORLD_SIZE=%d)" % (a.gpus, a.gpus, world))
    build.build()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    b = config5_block(a, dev, rank, world, a.steps, a.warmup)
    peaks = load_peaks()
    ach = 2.0 * a.comps * b["knn_pairs_per_s"] / 1e12
    line = {
        "metric": "target_cells_mapped_per_s", "value": b["value"], "unit": "cells/s", "n_gpus": world,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": b["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64 (projection: f64 DMMA; candidates: f16x2-split tcgen05, f32 accumulate)",
        "data": "synthetic",
        "config": {"workload": b["workload"], "engine": a.engine, "l2": "inputs (4 GB of counts per sample) exceed L2",
                   "inputs_resident": True},
        "clocks": b["clocks"], "stage_ms": b["stage_ms"], "projection_tflops_fp64": b["projection_tflops_fp64"],
        "knn_pairs_per_s": b["knn_pairs_per_s"], "e2e": None, "gpu_launches": None, "cpu_baseline": None,
        "setup_s": b["setup_s"],
        "roofline": {"bound": "tmem-read / tensor", "kernel": "tc::candidates_kernel", "unit": "TFLOP/s", "achieved": ach,
                     "peak": peaks["bf16_tflops_sustained"], "frac": ach / peaks["bf16_tflops_sustained"], "traffic": None,
                     "note": "whole kNN call (candidates + re-rank), 2*g flop per pair"},
    }
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_b200_refshard(a):
    """`--shard reference`: only the reference-sharded block, as the whole line."""
    import torch
    import torch.distributed as dist
    from nabo_b200 import build

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if a.gpus > 1 and world != a.gpus:
        raise SystemExit("--gpus %d needs torchrun --nproc-per-node %d (WORLD_SIZE=%d)" % (a.gpus, a.gpus, world))
    build.build()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    b = ref_sharded_block(a, dev, rank, world, a.n_ref, a.n_query, 5, a.steps, a.warmup, metric=a.metric)
    line = {"metric": "target_cells_mapped_per_s", "value": b["value"], "unit": "cells/s", "n_gpus": world,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": b["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64 (candidates: f16x2-split tcgen05, f32 accumulate)",
            "data": "synthetic", "config": {"workload": b["workload"], "engine": a.engine,
                                            "l2": "512 MB buffer rewritten between timed iterations"},
            "clocks": b["clocks"], "ref_sharded": b, "roofline": b["roofline"], "cpu_baseline": None,
            "gpu_launches": None}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ----------------------------------------------------------------------------- B200 arm
def run_b200(a):
    import torch
    import torch.distributed as dist
    from nabo_b200 import build, core, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if a.gpus > 1 and world != a.gpus:
        raise SystemExit("--gpus %d needs torchrun --nproc-per-node %d (WORLD_SIZE=%d)" % (a.gpus, a.gpus, world))
    build.build()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    peaks = load_peaks()

    g, k, M, N = a.comps, a.k, a.n_ref, a.n_query
    ref_h = synth.pc_mixture(M, g, seed=1)
    tgt_h = synth.pc_mixture(N, g, seed=101 + rank)             # this rank's target shard
    ref = torch.from_numpy(ref_h).to(dev)
    tgt = torch.from_numpy(tgt_h).to(dev)
    tgt_pin = torch.from_numpy(tgt_h).pin_memory()
    # setup (untimed): reference self-kNN = make_ref_graph's sorted rows
    ref_knn, _ = core.knn(ref, ref, k, "euclidean", drop_first=True, mode=a.engine)
    flush = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2

    score_acc = torch.zeros(M, dtype=torch.int64, device=dev)

    def step(metric, q, stats=False):
        r = core.knn(q, ref, k, metric, 0.25, mode=a.engine, return_stats=stats)
        idx, dst = r[0], r[1]
        cnt, w = core.snn_weights(idx, ref_knn, k)
        score_acc.zero_()
        core.score_accumulate(idx, cnt, M, k, acc=score_acc)        # integer weight sums: same bits on any GPU count
        sc = core.scores_finalize(score_acc, N)
        return idx, dst, cnt, w, sc, (r[2] if stats else None)

    def timed(metric, steps, warmup, e2e=False, keep_last=False):
        for _ in range(warmup):
            if e2e:
                host_step(metric)
            else:
                step(metric, tgt)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        kern_ms, launches, fallback, last = [], 0, 0, None
        sampler = ClockSampler(local)
        sampler.start()
        t0 = time.perf_counter()
        for i in range(steps):
            flush.zero_()                                   # evict L2 between timed iterations (untimed)
            ev[i][0].record()
            if e2e:
                host_step(metric)
            elif keep_last and i == steps - 1:
                last = step(metric, tgt)
            else:
                step(metric, tgt)
            ev[i][1].record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        if world > 1:
            dist.barrier()
        clocks = sampler.stop()
        if last is not None:
            last = {name: x.cpu().numpy() for name, x in zip(("idx", "dist", "counts", "weights", "scores"), last)}
        if not e2e:
            # kernel timing pass: the same steps again with the library's per-stage CUDA events (recorded on the
            # launch stream around the candidate kernel).  Kept out of the timed region because reading the
            # events needs a host synchronisation inside every call, which the product path does not have.
            for i in range(steps):
                flush.zero_()
                st = step(metric, tgt, stats=True)[5]
                kern_ms.append(st["main_kernel_ms"])
                launches += st["kernel_launches"] + 1 + SCORE_LAUNCHES
                fallback += st["rows_exact_fallback"]
            torch.cuda.synchronize()
        total_ms = sum(s.elapsed_time(e) for s, e in ev)
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return {"ms_total": float(t.item()), "kern_ms": kern_ms, "launches": launches, "fallback": fallback,
                "clocks": clocks, "wall_s": wall, "last": last}

    SCORE_LAUNCHES = 3          # memset of the accumulator, score_accumulate_kernel, score_finalize_kernel

    def host_step(metric):
        """Public host-buffer API: pinned host targets in, pinned host results out (copies pipelined)."""
        core.map_cells_host(tgt_pin, ref, ref_knn, k, metric=metric, dist_factor=0.25, mode=a.engine)

    main = timed(a.metric, a.steps, a.warmup, keep_last=bool(a.dump_outputs))
    e2e = timed(a.metric, max(3, a.steps // 2), 2, e2e=True)
    ms_step = main["ms_total"] / a.steps
    value = world * N / (ms_step / 1e3)
    e2e_steps = max(3, a.steps // 2)
    e2e_value = world * N / (e2e["ms_total"] / e2e_steps / 1e3)
    h2d = N * g * 8
    d2h = N * k * (4 + 8 + 8) + M * 8

    kern = sum(main["kern_ms"]) / max(1, len(main["kern_ms"]))
    if a.metric in ("euclidean", "cosine") and a.engine == "fast":
        flops = 2.0 * g * N * M                                   # SURVEY 8(d): 2*g flop per pair, true g
        roof = {"bound": "tensor", "achieved": flops / (kern * 1e-3) / 1e12, "peak": peaks["bf16_tflops"],
                "unit": "TFLOP/s", "kernel": "tc::candidates_kernel",
                "peak_source": "%s bf16 burst (kernel timed per launch)" % peaks["source"],
                "executed_tflops": flops * (((3 * g + 3 + 15) // 16 * 16) / g) / (kern * 1e-3) / 1e12,
                # the resource that really binds this kernel: every 128 x 128 FP32 accumulator tile has to leave TMEM
                # through tcgen05.ld at 64 B per clock per SM = 16 pairs per clock per SM (DESIGN.md 4.1), whatever K is
                "tmem_readout": {"achieved_pairs_per_s": float(N) * M / (kern * 1e-3),
                                 "peak_pairs_per_s": 148 * 16 * 1.965e9,
                                 "frac": float(N) * M / (kern * 1e-3) / (148 * 16 * 1.965e9),
                                 "peak_source": "64 B/clk/SM TMEM read port (B300_MICROARCH.md; reproduced here: the kernel "
                                                "with selection compiled out runs at 1 049 clk per tile), 148 SMs, max SM clock"},
                "traffic": None}
    elif a.metric == "mod_canberra" and a.engine == "fast":
        roof = canberra_roofline(g, N, M, kern)
    else:
        ops = 5.0 * g * N * M if a.metric == "mod_canberra" else 3.0 * g * N * M
        roof = {"bound": "fp64", "achieved": ops / (kern * 1e-3) / 1e12, "peak": 37.0,
                "unit": "TFLOP/s", "kernel": "knn_exact_kernel",
                "peak_source": "nominal B200 FP64 (no measured FP64 peak in MEASURED_PEAKS.json)", "traffic": None}
    roof["frac"] = roof["achieved"] / roof["peak"]
    tr = os.path.join(ROOT, "profiles", "bench_traffic.json")
    if os.path.exists(tr):
        trj = json.load(open(tr))
        roof["traffic"] = trj.get(roof["kernel"])
        roof["traffic_source"] = "static, not measured in this run: " + trj.get("source", "profiles/bench_traffic.json")

    line = {
        "metric": "target_cells_mapped_per_s", "value": value, "unit": "cells/s", "n_gpus": world,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None,
        "dtype": ("f64 (candidates: f16x2-split tcgen05, f32 accumulate)" if a.metric != "mod_canberra" else
                  "f64 (candidates: bit-sliced u32 count bound, f32 evaluation)"),
        "data": "synthetic",
        "config": {"workload": WORKLOAD.format(nq=N, nr=M, g=g, k=k, metric=a.metric), "engine": a.engine,
                   "per_gpu_targets": N, "sharding": "targets (reference replicated, no collective)",
                   "l2": "512 MB buffer rewritten between timed iterations", "inputs_resident": True},
        "clocks": {"sm_mhz": main["clocks"]["sm_mhz"], "sm_max_mhz": main["clocks"]["sm_max_mhz"],
                   "reasons": main["clocks"]["reasons"], "samples": main["clocks"]["samples"]},
        "e2e": {"value": e2e_value, "unit": "cells/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e["ms_total"] / e2e_steps, "api": "nabo_b200.core.map_cells_host (pinned host in/out, 2-piece copy/compute pipeline)"},
        "gpu_launches": main["launches"],
        "roofline": roof,
        "kernel_ms_per_step": kern,
        "rows_exact_fallback_per_step": main["fallback"] / a.steps,
    }

    if rank == 0 and world == 1 and not a.no_secondary and a.metric == "euclidean":
        sec_steps = max(2, a.steps // 5)
        sec = timed("mod_canberra", sec_steps, 1)
        sk = sum(sec["kern_ms"]) / len(sec["kern_ms"])
        line["mod_canberra"] = {"value": N / (sec["ms_total"] / sec_steps / 1e3), "unit": "cells/s",
                                "ms_per_step": sec["ms_total"] / sec_steps, "kernel_ms_per_step": sk,
                                "rows_exact_fallback_per_step": sec["fallback"] / sec_steps,
                                "roofline": canberra_roofline(g, N, M, sk)}
        if os.path.exists(tr):
            line["mod_canberra"]["roofline"]["traffic"] = trj.get("cbs::sliced_kernel")
            line["mod_canberra"]["roofline"]["traffic_source"] = roof.get("traffic_source")

    if not a.no_ref_sharded and a.metric == "euclidean" and a.engine == "fast":
        # BASELINE config 4 under the same clock: world x 1.25 M reference rows, 5 batches of --ref-batch targets
        line["ref_sharded"] = ref_sharded_block(a, dev, rank, world, a.ref_rows_per_gpu, a.ref_batch, 5,
                                                max(5, a.steps // 2), 2)
        line["score_determinism"] = score_determinism_check(dev, rank, world, ref, ref_knn, k)
        if not a.no_config5:
            # BASELINE config 5 under the same clock: one sample (500 k cells of counts) per GPU against a 2 M reference
            line["config5"] = config5_block(a, dev, rank, world, 2, 1, samples_per_gpu=1)
    if rank == 0 and not a.no_projection:
        line["projection"] = projection_block(dev)
    if world > 1:
        dist.barrier()

    if rank == 0 and world == 1 and not a.no_cpu_baseline and a.metric != "cosine":
        threads = os.cpu_count() or 1
        rate, n, dt = cpu_reference_rate(ref_h, tgt_h, ref_knn.cpu().numpy(), k, a.metric, a.cpu_seconds, threads)
        line["cpu_baseline"] = {"value": rate, "unit": "cells/s", "cores": threads, "kind": "port",
                                "sample": "%d of the %d target cells against all %d reference cells in %.1f s "
                                          "(C port of the reference loops, %d host threads)" % (n, N, M, dt, threads)}
    elif rank == 0:
        line["cpu_baseline"] = None
    if a.dump_outputs:
        # every rank maps its own targets: one file set per rank when there are several, sharing the size budget
        dump_outputs(a.dump_outputs, main["last"], DUMP_BYTES // world, "" if world == 1 else "_rank%d" % rank)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference_arm(args)
    elif args.workload == "config5":
        run_b200_config5(args)
    elif args.shard == "reference":
        run_b200_refshard(args)
    else:
        run_b200(args)
