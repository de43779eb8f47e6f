"""CPU checks of the correlation metric: the test oracle against scipy, the pinned centring order, NaN rows, the
header / binding constants, the workspace and prepared-buffer sizes, and the Python refusals."""
import ctypes as C
import math
import re

import numpy as np
import pytest
from scipy.spatial.distance import cdist

from nabo_b200 import _lib, build, core
from correlation_oracle import centre_rows, correlation_dist


def _al(b):
    return (b + 255) // 256 * 256


def test_oracle_matches_scipy():
    rng = np.random.default_rng(3)
    for g in (2, 3, 17, 50, 128):
        x = rng.normal(size=(40, g)) * rng.uniform(0.1, 10.0, size=g)
        y = rng.normal(size=(70, g)) + 0.5
        np.testing.assert_allclose(correlation_dist(x, y), cdist(x, y, "correlation"), rtol=0, atol=1e-12)


def test_centring_order_is_sequential():
    # ((1e16 + 1) - 1e16) + 1 = 1 in sequential FP64 (the first 1 is lost), while the exact and the pairwise sums are 2
    row = np.array([[1e16, 1.0, -1e16, 1.0]])
    assert math.fsum(row[0]) == 2.0 and (row[0, 0] + row[0, 2]) + (row[0, 1] + row[0, 3]) == 2.0
    c = centre_rows(row)
    assert c.tolist() == [[1e16, 0.75, -1e16, 0.75]]           # mu = 1 / 4
    y = np.array([[1.0, 2.0, 3.0, 5.0]])
    cy = centre_rows(y)
    assert cy.tolist() == [[-1.75, -0.75, 0.25, 2.25]]
    dot = 1e16 * -1.75 + 0.75 * -0.75 + -1e16 * 0.25 + 0.75 * 2.25
    nx = math.sqrt(1e16 * 1e16 + 0.75 * 0.75 + 1e16 * 1e16 + 0.75 * 0.75)
    ny = math.sqrt(1.75 * 1.75 + 0.75 * 0.75 + 0.25 * 0.25 + 2.25 * 2.25)
    assert correlation_dist(row, y)[0, 0] == 1.0 - dot / (nx * ny)


def test_constant_and_nonfinite_rows_give_nan():
    y = np.random.default_rng(0).normal(size=(5, 6))
    x = np.vstack([np.full(6, 2.5), np.full(6, -3.0), y[0], y[1], y[2]])
    x[3, 2] = np.nan
    x[4, 5] = np.inf
    d = correlation_dist(x, y)
    assert np.isnan(d).all(axis=1).tolist() == [True, True, False, True, True]
    assert np.isnan(correlation_dist(y, x)[:, [0, 1, 3, 4]]).all()
    assert np.isnan(correlation_dist(y[:, :1], y[:, :1])).all()          # g = 1: every row is constant


def test_header_constant_and_binding():
    txt = open(_lib.HEADER).read()
    assert int(re.search(r"#define NABO_CORRELATION (\d+)", txt).group(1)) == _lib.CORRELATION == 3
    assert _lib.METRICS["correlation"] == _lib.CORRELATION
    assert "nabo_correlation_dist" in _lib.declared_symbols() and "nabo_correlation_dist" in _lib.SIGNATURES
    build.build()
    assert hasattr(_lib.lib(), "nabo_correlation_dist")
    assert core.resolve_metric("correlation", False) == "correlation"


SHAPES = [(1, 200, 1, 1), (3001, 6000, 50, 30), (300, 100000, 50, 30), (3001, 20011, 50, 60), (2000, 20011, 53, 100),
          (4096, 2000000, 50, 30), (100, 5000, 128, 127), (10, 1000, 129, 10), (1000, 50, 25, 88)]


@pytest.mark.parametrize("shape", SHAPES, ids=[str(s) for s in SHAPES])
def test_workspace_sizes(shape):
    build.build()
    L = _lib.lib()
    n, m, g, k = shape
    copies = _al(8 * n * g) + _al(8 * m * g)
    for mode in (0, 1):
        cos = L.nabo_knn_workspace_bytes(n, m, g, k, _lib.COSINE, mode)
        assert L.nabo_knn_workspace_bytes(n, m, g, k, _lib.CORRELATION, mode) == copies + cos
    assert L.nabo_knn_workspace_bytes(n, m, g, k, _lib.CORRELATION, 0) == copies + 256
    for metric in (_lib.EUCLIDEAN, _lib.MOD_CANBERRA, _lib.COSINE):
        assert L.nabo_knn_workspace_bytes(n, m, g, k, metric, 0) == 256


def _desc(n_ref, g, metric, L):
    """A descriptor as nabo_ref_prepare fills it, at made-up device addresses: the size functions only compare
    addresses, they read no memory."""
    d = _lib.PreparedDesc()
    base = 1 << 40
    d.magic, d.abi_version, d.n_ref, d.g, d.metric, d.plan = 0x5250424e, 1, n_ref, g, metric, 1
    d.buffer = base
    d.buffer_bytes = L.nabo_ref_prepared_bytes(n_ref, g, metric)
    head = _al(8 * n_ref * g) if metric == _lib.CORRELATION else 0
    d.r, d.ldr = (base if metric == _lib.CORRELATION else 1 << 41), g
    d.ops[0], d.ops[1] = base + head, base + head + 256
    return d


@pytest.mark.parametrize("shape", SHAPES, ids=[str(s) for s in SHAPES])
def test_prepared_sizes(shape):
    build.build()
    L = _lib.lib()
    n, m, g, k = shape
    pc = L.nabo_ref_prepared_bytes(m, g, _lib.CORRELATION)
    if g > 128:
        assert pc == 0 and L.nabo_ref_prepared_bytes(m, g, _lib.COSINE) == 0
        return
    assert pc == _al(8 * m * g) + L.nabo_ref_prepared_bytes(m, g, _lib.COSINE)
    dc, dk = _desc(m, g, _lib.CORRELATION, L), _desc(m, g, _lib.COSINE, L)
    for mode in (0, 1):
        cos = L.nabo_knn_prepared_workspace_bytes(n, C.byref(dk), k, 0.25, mode)
        cor = L.nabo_knn_prepared_workspace_bytes(n, C.byref(dc), k, 0.25, mode)
        assert cos == 256 or mode == 1
        assert cor == _al(8 * n * g) + cos, (mode, cor, cos)
    # a correlation descriptor whose rows are not the copy in its buffer is not one nabo_ref_prepare made
    dc.r = 1 << 41
    assert L.nabo_knn_prepared_workspace_bytes(n, C.byref(dc), k, 0.25, 1) == 0


def test_prepare_refuses_wide_correlation():
    build.build()
    L = _lib.lib()
    d = _lib.PreparedDesc()
    assert L.nabo_ref_prepared_bytes(1000, 129, _lib.CORRELATION) == 0
    assert L.nabo_ref_prepare(None, 129, 1000, 129, _lib.CORRELATION, None, None, 0, d, None) == -3
    assert L.nabo_ref_prepared_bytes(1000, 50, 5) == 0


def test_rows_as_given_entry_points_refuse_correlation(monkeypatch):
    def refuse(*a, **kw):
        raise AssertionError("the library was called")
    monkeypatch.setattr(core, "lib", refuse)
    monkeypatch.setattr(core, "require_device", refuse)
    q = np.zeros((3, 4))
    with pytest.raises(ValueError, match="centre the rows"):
        core.knn_candidates(q, q, 2, "correlation")
    with pytest.raises(ValueError, match="centre the rows"):
        core.rerank_exact(q, q, np.zeros((3, 2), np.int32), 2, "correlation")
