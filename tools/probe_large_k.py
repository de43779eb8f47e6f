"""Fast kNN engine at large k: the 256-key plan of the tensor-core candidate pass (k + drop_first from 89 to 128) and
the 128-key plan next to it (k = 60, 88).  Development probe.

Cases (Euclidean and cosine unless noted): 100 000 x 100 000 at g = 50 for k = 60, 88, 89, 100, 128; g = 100, k = 100;
a 1 000 000-cell self-kNN at k = 100 (g = 50, Euclidean; the exact engine on a 20 000-row subsample); the 56 832 x
1 250 000 shard shape at k = 100 (Euclidean).  Per case: fast ms per call (CUDA events, warmed up, mean of REPS calls),
the return_stats stage split, K', fallback rows, the exact engine's ms on the same call and bit parity.

  python tools/probe_large_k.py [quick]      quick: the 100 k x 100 k g = 50 cases and 100 k x 190 k at k = 100 (the
                                             largest reference whose packed tiles, 61 MB, still get cut items) only,
                                             for an A/B of library builds selected with NABO_B200_LIB
  python tools/probe_large_k.py stats        needs the -DNABO_TC_STATS build: compactions per query and the epilogue
                                             cycle split of the candidate kernel at 100 k x 100 k, g = 50, k = 30 .. 128
"""
import ctypes as C
import subprocess
import sys

import torch

sys.path.insert(0, ".")
from nabo_b200 import _lib, core, synth  # noqa: E402

REPS = 5


def timed(fn, reps=REPS, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def same(a, b):
    return torch.equal(a[0], b[0]) and torch.equal(a[1].view(torch.int64), b[1].view(torch.int64))


def case(name, q, r, k, metric, drop=False, exact_rows=None, reps=REPS):
    run = lambda: core.knn(q, r, k, metric, drop_first=drop)  # noqa: E731
    ms = timed(run, reps=reps)
    fi, fd, st = core.knn(q, r, k, metric, drop_first=drop, return_stats=True)
    fast = run()
    if exact_rows is None:
        ms_exact = timed(lambda: core.knn(q, r, k, metric, drop_first=drop, mode="exact"), reps=1, warm=1)
        ok = same(fast, core.knn(q, r, k, metric, drop_first=drop, mode="exact"))
        ex = "exact %9.2f ms (%.0fx)" % (ms_exact, ms_exact / ms)
    else:
        ex_i, ex_d = core.knn(q[exact_rows], r, k, metric, drop_first=drop, mode="exact")
        ok = same((fast[0][exact_rows], fast[1][exact_rows]), (ex_i, ex_d))
        ex = "exact on %d rows" % len(exact_rows)
    pairs = q.shape[0] * r.shape[0]
    print("%-34s k=%3d: fast %9.3f ms %.3e pairs/s | %s | bit-identical %s" % (name, k, ms, pairs / ms * 1e3, ex, ok))
    print("      stages: prep %.3f, candidates %.3f, re-rank %.3f, fallback %.3f ms | K' %d | fallback rows %d of %d"
          % (st["prep_ms"], st["main_kernel_ms"], st["rerank_ms"], st["fallback_ms"], st["candidates_per_row"],
             st["rows_exact_fallback"], st["rows_reranked"]), flush=True)


def tc_stats():
    TC_NST = 12 + 64 + 2048
    L = _lib.lib()
    out = (C.c_ulonglong * TC_NST)()
    g, n = 50, 100000
    q = torch.from_numpy(synth.pc_mixture(n, g, seed=101)).cuda()
    r = torch.from_numpy(synth.pc_mixture(n, g, seed=1)).cuda()
    for k in (30, 60, 88, 89, 100, 128):
        core.knn(q, r, k, "euclidean")
        L.nabo_dbg_tc_stats(out, 1)
        _, _, st = core.knn(q, r, k, "euclidean", return_stats=True)
        L.nabo_dbg_tc_stats(out, 1)
        ch, hit, lanes, app, comp = out[0], out[1], out[2], out[3], out[4]
        tot = max(out[10], 1)
        print("k=%3d K'=%3d: appends per query %.1f, running compactions per query %.2f (%.1f appends each); epilogue "
              "cycles: compaction %.1f %%, filter %.1f %%, accumulator wait %.1f %%, tcgen05.ld %.1f %%; %.0f cycles per "
              "compaction" % (k, st["candidates_per_row"], app / n, comp / n, app / max(comp, 1), 100.0 * out[5] / tot,
                              100.0 * out[6] / tot, 100.0 * out[7] / tot, 100.0 * out[8] / tot, out[5] / max(comp, 1)),
              flush=True)


def main():
    props = torch.cuda.get_device_properties(0)
    smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                          "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    print("GPU: %s | %d SMs | nvidia-smi: %s | library %s" % (props.name, props.multi_processor_count, smi,
                                                               _lib.LIB_PATH))
    if sys.argv[1:] == ["stats"]:
        tc_stats()
        return
    quick = sys.argv[1:] == ["quick"]
    n = m = 100000
    g = 50
    q = torch.from_numpy(synth.pc_mixture(n, g, seed=101)).cuda()
    r = torch.from_numpy(synth.pc_mixture(m, g, seed=1)).cuda()
    for metric in ("euclidean", "cosine"):
        for k in (60, 88, 89, 100, 128):
            case("100k x 100k g=50 %s" % metric, q, r, k, metric)
    if quick:
        r = torch.from_numpy(synth.pc_mixture(190000, g, seed=1)).cuda()
        for metric in ("euclidean", "cosine"):
            case("100k x 190k g=50 %s" % metric, q, r, 100, metric)
        return
    g = 100
    q = torch.from_numpy(synth.pc_mixture(n, g, seed=101)).cuda()
    r = torch.from_numpy(synth.pc_mixture(m, g, seed=1)).cuda()
    for metric in ("euclidean", "cosine"):
        case("100k x 100k g=100 %s" % metric, q, r, 100, metric)
    del q, r
    g = 50
    big = torch.from_numpy(synth.pc_mixture(1250000, g, seed=2)).cuda()
    rows = torch.from_numpy(torch.randperm(1000000, generator=torch.Generator().manual_seed(0))[:20000].numpy()).cuda()
    case("1M self-kNN g=50 euclidean", big[:1000000], big[:1000000], 100, "euclidean", drop=True, exact_rows=rows,
         reps=2)
    q = torch.from_numpy(synth.pc_mixture(56832, g, seed=3)).cuda()
    case("56832 x 1.25M g=50 euclidean", q, big, 100, "euclidean", reps=3)


if __name__ == "__main__":
    main()
