"""Fast kNN with the correlation metric against cosine, on one GPU.

Correlation runs the cosine engines on row-centred copies (include/nabo_b200.h), so the difference between the two
is the centring launches and whatever the centred data changes in the candidate pass (certificate failures -> exact
fallback).  Shapes (g = 50, synth.pc_mixture): config 2 (100 000 x 100 000, k = 30), the same at k = 100 (the
256-key plan), and 4 096 queries x 2 000 000 references through a prepared reference (k = 30).  Per shape: ms per
call of core.knn from CUDA events over REPS calls after warm-up, the two metrics in alternating blocks of BLOCK calls
so that clock drift hits both alike; the rows each sends to the exact fallback; the centring time on its own, from a
separate call with stats: stats_host[7] (operand preparation) of correlation minus that of cosine.  Prints the card
name, power limit and max SM clock.
Usage: python tools/probe_correlation.py [reps-scale]  (1.0 = 200 calls per metric and shape)."""
import subprocess
import sys

import torch

sys.path.insert(0, ".")
from nabo_b200 import core, synth  # noqa: E402

BLOCK = 20


def timed_block(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def compare(fns, reps):
    for _ in range(3):
        for fn in fns.values():
            fn()
    torch.cuda.synchronize()
    t = {k: [] for k in fns}
    blocks = max(2, reps // BLOCK)
    names = list(fns)
    for i in range(blocks):
        for name in (names if i % 2 == 0 else names[::-1]):
            t[name].append(timed_block(fns[name], BLOCK) / BLOCK)
    return {k: (sum(v) / len(v), max(v) - min(v)) for k, v in t.items()}, blocks * BLOCK


def main():
    scale = float(sys.argv[1]) if len(sys.argv) > 1 else 1.0
    reps = max(2 * BLOCK, int(200 * scale))
    props = torch.cuda.get_device_properties(0)
    smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                          "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    print("GPU: %s | %d SMs | nvidia-smi (name, power limit, max SM clock): %s"
          % (props.name, props.multi_processor_count, smi))
    g = 50
    dev = torch.device("cuda")
    shapes = [("config 2, k=30", 100000, 100000, 30, False),
              ("config 2, k=100", 100000, 100000, 100, False),
              ("4096 x 2M prepared, k=30", 4096, 2000000, 30, True)]
    for label, n, m, k, prep in shapes:
        r = synth.pc_mixture_device(m, g, seed=1, device=dev)
        q = synth.pc_mixture_device(n, g, seed=101, device=dev)
        refs = {mt: (core.prepare_reference(r, mt) if prep else r) for mt in ("cosine", "correlation")}
        out = {mt: (torch.empty((n, k), dtype=torch.int32, device=dev),
                    torch.empty((n, k), dtype=torch.float64, device=dev)) for mt in refs}
        fns = {mt: (lambda mt=mt: core.knn(q, refs[mt], k, None if prep else mt, out=out[mt])) for mt in refs}
        res, calls = compare(fns, reps)
        stats = {mt: core.knn(q, refs[mt], k, None if prep else mt, return_stats=True)[2] for mt in refs}
        print("%-26s n=%d m=%d g=%d k=%d  (%d calls per metric)" % (label, n, m, g, k, calls))
        for mt in refs:
            st = stats[mt]
            print("  %-12s %8.3f ms/call (block spread %.3f)  fallback rows %6d  operand preparation %.3f ms  launches %d"
                  % (mt, res[mt][0], res[mt][1], st["rows_exact_fallback"], st["prep_ms"], st["kernel_launches"]))
        centring = stats["correlation"]["prep_ms"] - stats["cosine"]["prep_ms"]
        print("  correlation / cosine = %.4f; centring %.3f ms = %.1f %% of the correlation call"
              % (res["correlation"][0] / res["cosine"][0], centring, 100.0 * centring / res["correlation"][0]))
        del refs, out, fns, r, q
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
