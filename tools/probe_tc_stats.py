"""Selection statistics of the candidate kernel (needs the NABO_TC_STATS variant: tools/build_variant.py stats
-DNABO_TC_STATS, then NABO_B200_LIB=tools/_variants/lib_stats.so).  Development probe."""
import ctypes as C, sys
import torch
sys.path.insert(0, ".")
from nabo_b200 import core, synth, _lib
g, k = 50, 30
L = _lib.lib()
for n, m in ((100000, 100000), (56832, 1250000)):
    q = torch.from_numpy(synth.pc_mixture(n, g, 101)).cuda()
    r = torch.from_numpy(synth.pc_mixture(m, g, 1)).cuda()
    out = (C.c_ulonglong * 12)()
    L.nabo_dbg_tc_stats(out, 1)
    core.knn_candidates(q, r, k, "euclidean")
    L.nabo_dbg_tc_stats(out, 1)
    ch, hit, lanes, app, comp = out[0], out[1], out[2], out[3], out[4]
    print("%d x %d: warp chunks %d, with a hit %.1f %%, hit lanes per hit chunk %.2f, appends per query %.1f, "
          "appends per hit lane %.2f, running compactions per query %.2f" % (
              n, m, ch, 100.0 * hit / ch, lanes / max(hit, 1), app / n, app / max(lanes, 1), comp / n))
    tot = max(out[10], 1)
    print("   epilogue warp cycles: item loop 100 %% = %.3e; wait for accumulator %.1f %%, tcgen05.ld+wait %.1f %%, filter_chunk %.1f %%, "
          "running compaction %.1f %%, final emit %.1f %%; per compaction %.0f cycles, per final emit (32 queries) %.0f cycles" % (
              tot, 100.0 * out[7] / tot, 100.0 * out[8] / tot, 100.0 * out[6] / tot, 100.0 * out[5] / tot, 100.0 * out[9] / tot,
              out[5] / max(comp, 1), out[9] / max(n / 32, 1)))
