"""Candidate pass alone (knn_candidates, packing included) over a few shapes; run with NABO_B200_LIB pointing at an
A/B variant (tools/build_variant.py) to separate MMA / accumulator read-out / selection cost.  Development probe."""
import os, sys
import torch
sys.path.insert(0, ".")
from nabo_b200 import core, synth

g, k = 50, int(os.environ.get("PROBE_K", "30"))
shapes = [(100000, 100000), (56832, 100000), (100000, 200000), (100000, 400000), (56832, 1250000)]
if len(sys.argv) > 1:
    shapes = [tuple(int(x) for x in a.split("x")) for a in sys.argv[1:]]
for n, m in shapes:
    q = torch.from_numpy(synth.pc_mixture(n, g, 101)).cuda()
    r = torch.from_numpy(synth.pc_mixture(m, g, 1)).cuda()
    for _ in range(2):
        core.knn_candidates(q, r, k, "euclidean")
    torch.cuda.synchronize()
    a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(3):
        core.knn_candidates(q, r, k, "euclidean")
    b.record(); torch.cuda.synchronize()
    ms = a.elapsed_time(b) / 3
    waves = -(-(-(-n // 384)) // 148)
    jobs = waves * 3 * -(-m // 128)
    print("k=%d %s  %7d x %7d: %.3f ms  %.3e pairs/s  %.3f us per (128x128) job on the critical SM" % (
        k, os.path.basename(os.environ.get("NABO_B200_LIB", "product")), n, m, ms, n * m / ms * 1e3, ms * 1e3 / jobs))
