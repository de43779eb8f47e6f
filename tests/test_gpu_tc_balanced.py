"""Balanced schedule of the unsplit tensor-core candidate pass: with more work items than SMs the items are dealt out
on a line of modelled cost, and an item cut at a CTA boundary is swept as a head on one CTA and a tail that resumes the
head's selection state on another.  The buffers it leaves must be exactly those of an unsplit sweep, so the candidates
must be bit-identical to the same queries run in slices of at most one wave (one whole item per CTA), and the fast
engine must return what the exact engine returns."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def core():
    from nabo_b200 import build, core as c
    build.build()
    return c


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def item_rows(g):
    return 384 if g <= 52 else 256            # query rows per work item: three or two 128-row tiles (plan_smem)


def data(n, m, g, seed=0):
    from nabo_b200 import synth
    q = torch.from_numpy(synth.pc_mixture(n, g, seed=101 + seed)).cuda()
    r = torch.from_numpy(synth.pc_mixture(m, g, seed=1 + seed)).cuda()
    return q, r


@pytest.mark.parametrize("metric,g,k,masked", [("euclidean", 50, 30, False), ("cosine", 50, 60, True),
                                               ("euclidean", 100, 1, False), ("cosine", 25, 30, True),
                                               ("euclidean", 64, 30, True)])
def test_candidates_equal_one_wave_slices(core, metric, g, k, masked):
    n, m = 100_000, 30_011
    q, r = data(n, m, g)
    kw = {}
    if masked:
        mask = torch.zeros(m, dtype=torch.bool, device="cuda")
        mask[::5] = True
        kw = dict(ref_mask=mask, drop_first=True)
    whole = core.knn_candidates(q, r, k, metric, **kw)
    step = sms() * item_rows(g)                      # one wave: every CTA sweeps one whole item, nothing is cut
    assert n > step and n % step
    for a in range(0, n, step):
        part = core.knn_candidates(q[a:a + step], r, k, metric, **kw)
        assert torch.equal(part["cand"], whole["cand"][a:a + step]), a
        assert torch.equal(part["tau"].view(torch.int32), whole["tau"][a:a + step].view(torch.int32)), a


def knn_equal(core, q, r, k, metric, **kw):
    fi, fd = core.knn(q, r, k, metric, mode="fast", **kw)
    ei, ed = core.knn(q, r, k, metric, mode="exact", **kw)
    assert torch.equal(fi, ei)
    assert torch.equal(fd.view(torch.int64), ed.view(torch.int64))


@pytest.mark.parametrize("items", ["grid+1", "1.5grid", "2grid-1", "2grid+1"])
@pytest.mark.parametrize("metric,g,k", [("euclidean", 50, 30), ("cosine", 50, 1), ("euclidean", 25, 60),
                                        ("cosine", 100, 30)])
def test_knn_equals_exact_at_partial_waves(core, items, metric, g, k):
    grid = sms()
    n_items = {"grid+1": grid + 1, "1.5grid": (3 * grid) // 2, "2grid-1": 2 * grid - 1, "2grid+1": 2 * grid + 1}[items]
    n = n_items * item_rows(g) - 77                  # a ragged last item
    m = 12_007
    q, r = data(n, m, g, seed=3)
    r[17] = r[m - 5]                                 # a tie between the first and the last reference tile
    q[3] = r[17]
    mask = torch.zeros(m, dtype=torch.bool, device="cuda")
    mask[::7] = True
    knn_equal(core, q, r, k, metric)
    knn_equal(core, q, r, k, metric, ref_mask=mask, idx_offset=11)
    s, _ = data(n, 1, g, seed=4)                     # self-kNN with drop_first over the same number of items
    knn_equal(core, s, s, k, metric, drop_first=True)


@pytest.mark.parametrize("metric,g,k", [("euclidean", 50, 30), ("cosine", 50, 60), ("euclidean", 100, 30)])
def test_knn_equals_exact_at_100k(core, metric, g, k):
    q, r = data(100_000, 50_000, g, seed=5)
    knn_equal(core, q, r, k, metric)
    mask = torch.zeros(50_000, dtype=torch.bool, device="cuda")
    mask[3::11] = True
    knn_equal(core, q, r, k, metric, ref_mask=mask, drop_first=True, idx_offset=4)


def test_knn_equals_exact_without_cuts(core):
    """A packed reference larger than half of L2 (250 k x g = 50: 78 MB) is not cut: every CTA sweeps the items c,
    c + grid, ... and the re-rank of the full waves runs as a dependent launch under the partly filled last wave (no
    stage timing, which would turn that overlap off)."""
    grid = sms()
    n = (grid + 9) * item_rows(50) - 5
    q, r = data(n, 250_000, 50, seed=7)
    knn_equal(core, q, r, 30, "euclidean")
    mask = torch.zeros(250_000, dtype=torch.bool, device="cuda")
    mask[::13] = True
    knn_equal(core, q, r, 30, "cosine", ref_mask=mask, idx_offset=3)
