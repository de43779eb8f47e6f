"""Selection statistics of the candidate kernel (needs the NABO_TC_STATS variant: tools/build_variant.py stats
-DNABO_TC_STATS, then NABO_B200_LIB=tools/_variants/lib_stats.so).  Development probe.  Besides the counters it prints the
epilogue cycles per warp-tile by sweep position (log2 buckets), the fit of the schedule's cost model
F(x) = x + beta j0 ln(1 + x / j0) (tc::sweep_cost: beta = 16.2, j0 = K' / 20) to them (j0 free, and j0 = K' / 128), and the spread of the CTAs' finish times."""
import ctypes as C, sys
import numpy as np
import torch
sys.path.insert(0, ".")
from nabo_b200 import core, synth, _lib
g, k = 50, 30
KP = 39                       # K' of k = 30
TC_HIST, TC_TIME, NST = 12, 12 + 64, 12 + 64 + 2048
L = _lib.lib()
print(torch.cuda.get_device_name(0))
for n, m in ((100000, 100000), (56832, 1250000)):
    q = torch.from_numpy(synth.pc_mixture(n, g, 101)).cuda()
    r = torch.from_numpy(synth.pc_mixture(m, g, 1)).cuda()
    out = (C.c_ulonglong * NST)()
    core.knn_candidates(q, r, k, "euclidean")
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
    n_rt = (m + 127) // 128
    cyc = np.array([out[TC_HIST + b] for b in range(32)], float)
    cnt = np.array([out[TC_HIST + 32 + b] for b in range(32)], float)
    nb = int(np.nonzero(cnt)[0].max()) + 1
    lo = np.array([2 ** b - 1 for b in range(nb)], float)
    hi = np.minimum(np.array([2 ** (b + 1) - 1 for b in range(nb)], float), n_rt)
    mean = cyc[:nb] / np.maximum(cnt[:nb], 1)
    print("   cycles per warp-tile by sweep position: " + ", ".join(
        "[%d,%d) %.0f" % (lo[b], hi[b], mean[b]) for b in range(nb)))
    # the schedule uses only the SHAPE of the cumulative cost, F(x) / F(n): fit it (minimax over the bucket edges)
    x = np.concatenate([[0.0], hi])
    cum = np.concatenate([[0.0], np.cumsum(mean * (hi - lo))])
    shape = cum / cum[-1]
    def err(beta, j0):
        f = x + beta * j0 * np.log1p(x / j0)
        return np.max(np.abs(f / f[-1] - shape))
    fits = [min((err(b, j), b, j) for j in np.geomspace(0.05, 20, 300) for b in np.geomspace(1, 500, 400)),
            min((err(b, KP / 128.0), b, KP / 128.0) for b in np.geomspace(1, 500, 2000))]
    for e, b, j in fits:
        print("   fit of F(x) = x + beta j0 ln(1 + x / j0): j0 = %.3f tiles (= K' / %.1f), beta = %.1f; largest error of "
              "F(x) / F(n) %.2f %% of an item" % (j, KP / j, b, 100 * e))
    for b, j in ((16.2, KP / 20.0),):
        print("   tc::sweep_cost (beta %.1f, j0 = K' / 20): largest error %.2f %% of an item" % (b, 100 * err(b, j)))
    t = np.array([out[TC_TIME + i] for i in range(2048)], float).reshape(1024, 2)
    t = t[t[:, 1] > 0]
    if len(t):
        span = t[:, 1].max() - t[:, 0].min()
        print("   %d CTAs: kernel %.3f ms (globaltimer), finish times spread %.3f ms (%.1f %%), first finish at %.1f %%" % (
            len(t), span / 1e6, (t[:, 1].max() - t[:, 1].min()) / 1e6, 100 * (t[:, 1].max() - t[:, 1].min()) / span,
            100 * (t[:, 1].min() - t[:, 0].min()) / span))
