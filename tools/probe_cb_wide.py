"""Fast modified-Canberra kNN across PCA widths, on both sides of the wide plan of the bit-sliced candidate pass
(g <= 56: 12 warps, 128-reference tiles; 57 <= g <= 128: 8 warps, 64- or 32-reference tiles, 8-bit counters).

For g in {50, 64, 77, 100, 128}: 100 000 x 100 000, k = 30, f = 0.25; then a map_target-shaped call at g = 100
(core.map_cells: 100 000 targets against a 100 000-cell reference, k = 30, default metric, SNN weights and scores).
Per case: fast ms per call (CUDA events, warmed up, mean of REPS calls), the return_stats stage split, the exact
engine's ms on the same call (one timed repetition), whether fast and exact are bit-identical, and the fallback rows.
Select another build of the library with NABO_B200_LIB=<path> (tools/build_variant.py)."""
import os
import subprocess
import sys

import torch

sys.path.insert(0, ".")
from nabo_b200 import core, synth  # noqa: E402

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


def main():
    gs = [int(x) for x in sys.argv[1].split(",")] if len(sys.argv) > 1 else [50, 64, 77, 100, 128]
    props = torch.cuda.get_device_properties(0)
    smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                          "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    print("GPU: %s | %d SMs | nvidia-smi: %s | library: %s"
          % (props.name, props.multi_processor_count, smi, os.environ.get("NABO_B200_LIB", "in-tree")))
    n = m = 100000
    k, f = 30, 0.25
    for g in gs:
        r = torch.from_numpy(synth.pc_mixture(m, g, seed=1)).cuda()
        q = torch.from_numpy(synth.pc_mixture(n, g, seed=101)).cuda()
        ms = timed(lambda: core.knn(q, r, k, "mod_canberra", f, mode="fast"))
        _, _, st = core.knn(q, r, k, "mod_canberra", f, mode="fast", return_stats=True)
        ms_exact = timed(lambda: core.knn(q, r, k, "mod_canberra", f, mode="exact"), reps=1, warm=1)
        ei, ed = core.knn(q, r, k, "mod_canberra", f, mode="exact")
        fi, fd = core.knn(q, r, k, "mod_canberra", f, mode="fast")
        same = torch.equal(fi, ei) and torch.equal(fd.view(torch.int64), ed.view(torch.int64))
        print("g=%3d mod_canberra k=%d f=%.2f: fast %8.3f ms  %.3e pairs/s | exact %9.2f ms (%.1fx) | bit-identical %s"
              % (g, k, f, ms, n * m / ms * 1e3, ms_exact, ms_exact / ms, same))
        print("      stages: candidates %.3f, re-rank %.3f, fallback %.3f ms | fallback rows %d of %d (%.3f %%)"
              " | K' %d | launches %d"
              % (st["main_kernel_ms"], st["rerank_ms"], st["fallback_ms"], st["rows_exact_fallback"],
                 st["rows_reranked"], 100.0 * st["rows_exact_fallback"] / max(1, st["rows_reranked"]),
                 st["candidates_per_row"], st["kernel_launches"]))
        if g == 100:
            ridx, _ = core.knn(r, r, k, "euclidean", drop_first=True, mode="fast")
            call = {mode: (lambda mode=mode: core.map_cells(q, r, ridx, k, dist_factor=f, mode=mode))
                    for mode in ("fast", "exact")}
            ms = timed(call["fast"])
            ms_exact = timed(call["exact"], reps=1, warm=1)
            a, b = call["fast"](), call["exact"]()
            same = all(torch.equal(a[key].view(torch.int64) if a[key].dtype == torch.float64 else a[key],
                                   b[key].view(torch.int64) if b[key].dtype == torch.float64 else b[key])
                       for key in ("idx", "dist", "counts", "weights", "scores"))
            print("g=100 map_cells (map_target shape, default metric) k=%d: fast %8.3f ms | exact %9.2f ms (%.1fx)"
                  " | bit-identical %s" % (k, ms, ms_exact, ms_exact / ms, same))
        del q, r
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
