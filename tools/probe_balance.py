"""Config-2 kNN (100 k x 100 k, g = 50, k = 30, Euclidean) with the reference in random row order and sorted by mixture
cluster (cold starts of the running selection then differ between reference ranges): ms per call and stage times.
Run once per library (NABO_B200_LIB=...) for an A/B.  Development probe."""
import sys
import numpy as np
import torch
sys.path.insert(0, ".")
from nabo_b200 import core, synth
n = m = 100000
g, k = 50, 30
print(torch.cuda.get_device_name(0))
q = torch.from_numpy(synth.pc_mixture(n, g, 101)).cuda()
r_np = synth.pc_mixture(m, g, 1)
lab = np.random.default_rng(1).integers(0, 32, size=m)          # the labels pc_mixture drew (same generator)
for name, r_host in (("random order", r_np), ("sorted by cluster", r_np[np.argsort(lab, kind="stable")])):
    r = torch.from_numpy(np.ascontiguousarray(r_host)).cuda()
    for _ in range(3):
        core.knn(q, r, k, "euclidean")
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(20):
        idx, dist = core.knn(q, r, k, "euclidean")
    b.record()
    torch.cuda.synchronize()
    st = core.knn(q, r, k, "euclidean", return_stats=True)[2]
    print("%s: knn %.3f ms per call; stages %s; idx checksum %d" % (
        name, a.elapsed_time(b) / 20, {kk: (round(v, 3) if isinstance(v, float) else v) for kk, v in st.items()},
        int(idx.to(torch.int64).sum())))
