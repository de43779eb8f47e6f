"""Per-call kNN time with and without a prepared reference (core.prepare_reference), on one GPU.

Shapes (g = 50, k = 30): config 2 (100 000 x 100 000, Euclidean and modified Canberra f = 0.25), 4 096 queries x
2 000 000 references (cosine), and the config-4 shard shape (227 328 targets x 1 250 000 references, Euclidean and
modified Canberra).  Per shape: ms per call of core.knn(q, r) and of core.knn(q, prepared) from CUDA events over
REPS calls after warm-up, taken in alternating blocks of BLOCK calls so that clock drift hits both alike; the
one-off nabo_ref_prepare time; and whether both give the same bits.  Prints the card name and power limit.
Usage: python tools/probe_prepared.py [reps-scale]  (1.0 = 400 calls per side on the small shapes, 100 on the shard)."""
import subprocess
import sys

import torch

sys.path.insert(0, ".")
from nabo_b200 import core, synth  # noqa: E402

BLOCK = 25


def timed_block(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def compare(one_shot, prepared, reps):
    for _ in range(3):
        one_shot()
        prepared()
    torch.cuda.synchronize()
    t = {"one-shot": [], "prepared": []}
    blocks = max(1, reps // BLOCK)
    for i in range(blocks):
        order = (("one-shot", one_shot), ("prepared", prepared)) if i % 2 == 0 else \
                (("prepared", prepared), ("one-shot", one_shot))
        for name, fn in order:
            t[name].append(timed_block(fn, BLOCK) / BLOCK)
    mean = {k: sum(v) / len(v) for k, v in t.items()}
    spread = {k: (max(v) - min(v)) for k, v in t.items()}
    return mean, spread, blocks * BLOCK


def main():
    scale = float(sys.argv[1]) if len(sys.argv) > 1 else 1.0
    props = torch.cuda.get_device_properties(0)
    smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                          "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    print("GPU: %s | %d SMs | nvidia-smi: %s" % (props.name, props.multi_processor_count, smi))
    g, k = 50, 30
    dev = torch.device("cuda")
    shapes = [("config 2", 100000, 100000, ["euclidean", "mod_canberra"], 400),
              ("4096 x 2M", 4096, 2000000, ["cosine"], 400),
              ("config-4 shard", 227328, 1250000, ["euclidean", "mod_canberra"], 100)]
    for label, n, m, metrics, reps in shapes:
        r = synth.pc_mixture_device(m, g, seed=1, device=dev)
        q = synth.pc_mixture_device(n, g, seed=101, device=dev)
        for metric in metrics:
            pr = core.prepare_reference(r, metric)
            prep_ms = timed_block(lambda: core.prepare_reference(r, metric), 10) / 10
            one = lambda: core.knn(q, r, k, metric)                 # noqa: E731
            pre = lambda: core.knn(q, pr, k)                        # noqa: E731
            oi, od = one()
            pi, pd = pre()
            same = torch.equal(oi, pi) and torch.equal(od.view(torch.int64), pd.view(torch.int64))
            mean, spread, calls = compare(one, pre, max(BLOCK, int(reps * scale)))
            _, _, st = core.knn(q, pr, k, return_stats=True)
            print("%-15s %-12s %7d x %8d: one-shot %8.3f ms (block spread %.3f) | prepared %8.3f ms (%.3f) | "
                  "saved %7.3f ms = %5.1f %% | %d calls each | nabo_ref_prepare %.3f ms, %.1f MB | prep stage %.3f ms "
                  "| same bits %s" % (label, metric, n, m, mean["one-shot"], spread["one-shot"], mean["prepared"],
                                      spread["prepared"], mean["one-shot"] - mean["prepared"],
                                      100 * (mean["one-shot"] - mean["prepared"]) / mean["one-shot"], calls, prep_ms,
                                      pr.nbytes / 1e6, st["prep_ms"], same), flush=True)
            del pr
        del r, q
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
