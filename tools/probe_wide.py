"""Fast kNN engine across PCA widths, on both sides of the wide tile plan of the tensor-core candidate pass (g <= 52:
three query tiles per work item; 53 <= g <= 128: two, reference tiles streamed in K-slabs).

For g in {50, 64, 100, 128}: 100 000 x 100 000, k = 30, Euclidean and cosine, and a 100 000-cell Euclidean self-kNN
(k = 15, drop_first).  Per case: fast ms per call (CUDA events, warmed up, mean of REPS calls), the return_stats stage
split, pairs/s of the call and of the candidate kernel, the kernel against the per-tile bound (the larger of the MMA
time, 64 clocks per K step of a 128 x 128 tile, and the 1 024-clock TMEM read-out of the tile, at the card's maximum
SM clock on all SMs), the exact engine's ms on the same call, and whether fast and exact are bit-identical."""
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
    props = torch.cuda.get_device_properties(0)
    smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                          "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    print("GPU: %s | %d SMs | nvidia-smi: %s" % (props.name, props.multi_processor_count, smi))
    try:
        clk_hz = float(smi.split(",")[-1].split()[0]) * 1e6
    except (ValueError, IndexError):
        clk_hz = float("nan")
    n = m = 100000
    for g in (50, 64, 100, 128):
        kp = (3 * g + 3 + 15) // 16 * 16
        ksteps = kp // 16
        mma_clk, ldtm_clk = 64 * ksteps, 1024
        bound = {"MMA": 128 * 128 / mma_clk * clk_hz * props.multi_processor_count,
                 "TMEM read-out": 128 * 128 / ldtm_clk * clk_hz * props.multi_processor_count}
        r = torch.from_numpy(synth.pc_mixture(m, g, seed=1)).cuda()
        q = torch.from_numpy(synth.pc_mixture(n, g, seed=101)).cuda()
        cases = [("euclidean", q, r, 30, False), ("cosine", q, r, 30, False), ("euclidean self", r, r, 15, True)]
        for name, qq, rr, k, drop in cases:
            metric = name.split()[0]
            fast = lambda: core.knn(qq, rr, k, metric, drop_first=drop, mode="fast")  # noqa: E731
            ms = timed(fast)
            fi, fd, st = core.knn(qq, rr, k, metric, drop_first=drop, mode="fast", return_stats=True)
            ms_exact = timed(lambda: core.knn(qq, rr, k, metric, drop_first=drop, mode="exact"), reps=1, warm=1)
            ei, ed = core.knn(qq, rr, k, metric, drop_first=drop, mode="exact")
            fi, fd = core.knn(qq, rr, k, metric, drop_first=drop, mode="fast")
            same = torch.equal(fi, ei) and torch.equal(fd.view(torch.int64), ed.view(torch.int64))
            pairs = qq.shape[0] * rr.shape[0]
            kern = pairs / (st["main_kernel_ms"] * 1e-3) if st["main_kernel_ms"] > 0 else float("nan")
            which = min(bound, key=bound.get)          # the smaller rate is the bound
            print("g=%3d kp=%3d %-15s k=%2d: fast %8.3f ms  %.3e pairs/s | exact %9.2f ms (%.1fx) | bit-identical %s"
                  % (g, kp, name, k, ms, pairs / ms * 1e3, ms_exact, ms_exact / ms, same))
            print("      stages: prep %.3f, candidates %.3f, re-rank %.3f, fallback %.3f ms | fallback rows %d of %d (%.3f %%)"
                  " | K' %d | launches %d"
                  % (st["prep_ms"], st["main_kernel_ms"], st["rerank_ms"], st["fallback_ms"], st["rows_exact_fallback"],
                     st["rows_reranked"], 100.0 * st["rows_exact_fallback"] / max(1, st["rows_reranked"]),
                     st["candidates_per_row"], st["kernel_launches"]))
            print("      candidate kernel %.3e pairs/s = %.1f %% of the %s bound %.3e (MMA %d clk vs read-out %d clk per tile)"
                  % (kern, 100.0 * kern / bound[which], which, bound[which], mma_clk, ldtm_clk))
        del q, r
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
