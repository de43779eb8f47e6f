"""mapping_specificity at config-2 scale: 100 k targets x 100 k references, g = 50, the target mapping at k (default 30;
k > 64 runs the 128-source search) and the reference graph at min(k, 127), the widest self-kNN with drop_first.
Usage: python tools/probe_specificity.py [k ...]"""
import sys, time, torch, numpy as np
sys.path.insert(0, ".")
from nabo_b200 import core, synth
import scipy.sparse as sp
n, g = 100000, 50
ref = torch.from_numpy(synth.pc_mixture(n, g, 1)).cuda()
tgt = torch.from_numpy(synth.pc_mixture(n, g, 101)).cuda()
for k in [int(a) for a in sys.argv[1:]] or [30]:
    kr = min(k, 127)
    rk, _ = core.knn(ref, ref, kr, "euclidean", drop_first=True)
    tk, _ = core.knn(tgt, ref, k, "mod_canberra", 0.25)
    rc, _ = core.snn_weights(rk, rk, kr)
    tc, _ = core.snn_weights(tk, rk, k)
    rows, cols = np.nonzero(rc.cpu().numpy() > 0)
    a = rows; b = rk.cpu().numpy()[rows, cols]
    adj = sp.coo_matrix((np.ones(2 * len(a), np.int8), (np.r_[a, b], np.r_[b, a])), shape=(n, n)).tocsr(); adj.sum_duplicates()
    ip = torch.from_numpy(adj.indptr.astype(np.int64)).cuda(); ix = torch.from_numpy(adj.indices.astype(np.int32)).cuda()
    cnt = (tc > 0).to(torch.uint8)
    for _ in range(3):
        torch.cuda.synchronize(); t = time.perf_counter()
        mean, conn = core.mapping_specificity(ip, ix, tk, cnt)
        torch.cuda.synchronize()
        print("k %d: specificity kernel path: %.3f s; mean of means %.6f; mapped/target %.1f (max %d); edges %d"
              % (k, time.perf_counter() - t, float(torch.nanmean(mean)), float(cnt.sum()) / n,
                 int(cnt.sum(1).max()), adj.nnz), flush=True)
