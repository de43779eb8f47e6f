"""CPU checks of the prepared-reference surface: every new header symbol is exported and typed, and the Python
argument validation of a call on a prepared reference (metric / mask / g conflicts, a source modified in place)
raises before the library is called."""
import numpy as np
import pytest
import torch

from nabo_b200 import _lib, build, core

NEW_SYMBOLS = ["nabo_ref_prepared_bytes", "nabo_ref_prepare", "nabo_knn_prepared_workspace_bytes",
               "nabo_knn_prepared", "nabo_knn_prepared_routed"]


def test_prepared_symbols_exported_and_typed():
    build.build()
    L = _lib.lib()
    declared = _lib.declared_symbols()
    for name in NEW_SYMBOLS:
        assert name in declared and name in _lib.SIGNATURES, name
        assert hasattr(L, name), name
    # shape queries need no device
    assert L.nabo_ref_prepared_bytes(100000, 50, _lib.EUCLIDEAN) > 100000 * 320
    assert L.nabo_ref_prepared_bytes(100000, 129, _lib.EUCLIDEAN) == 0
    assert L.nabo_ref_prepared_bytes(0, 50, _lib.MOD_CANBERRA) == 0
    assert L.nabo_knn_prepared_workspace_bytes(10, None, 5, 0.25, 1) == 0
    assert L.nabo_knn_prepared(None, 50, 10, None, 5, 0.25, 0, 0, 1, None, None, None, 0, None, None) == -1
    d = _lib.PreparedDesc()
    assert L.nabo_knn_prepared(None, 50, 10, d, 5, 0.25, 0, 0, 1, None, None, None, 0, None, None) == -1
    assert b"magic" in L.nabo_last_error()
    assert L.nabo_ref_prepare(None, 50, 1000, 200, 0, None, None, 0, d, None) == -3


class _Stub(core.PreparedReference):
    """A prepared reference without a device: what the validation sees, nothing the library could use."""

    def __init__(self, metric="euclidean", g=4, mask=None):
        self.metric, self.n_ref, self.g = metric, 10, g
        self.r = torch.zeros((10, g), dtype=torch.float64)
        self.mask, self._mask_src = None, mask
        self._sources = [(self.r, self.r._version)]


@pytest.fixture
def no_library(monkeypatch):
    def refuse(*a, **kw):
        raise AssertionError("the library was called")
    monkeypatch.setattr(core, "lib", refuse)
    monkeypatch.setattr(core, "require_device", refuse)


def test_prepared_argument_conflicts_raise_first(no_library):
    q = np.zeros((3, 4))
    with pytest.raises(ValueError, match="conflicts"):
        core.knn(q, _Stub("euclidean"), 2, "mod_canberra")
    with pytest.raises(ValueError, match="ref_mask"):
        core.knn(q, _Stub(), 2, ref_mask=np.zeros(10, bool))
    own = np.zeros(10, bool)
    with pytest.raises(AssertionError, match="library was called"):     # its own mask is no conflict
        core.knn(q, _Stub(mask=own), 2, ref_mask=own)
    with pytest.raises(ValueError, match="columns"):
        core.knn(np.zeros((3, 5)), _Stub(g=4), 2)
    with pytest.raises(ValueError, match="conflicts"):
        core.map_cells(q, _Stub("cosine"), np.zeros((10, 2), np.int32), 2, metric="euclidean")


def test_prepared_modified_source_raises_first(no_library):
    st = _Stub()
    st.r[0, 0] = 1.0                                   # in place: bumps the tensor's version counter
    with pytest.raises(ValueError, match="modified in place"):
        core.knn(np.zeros((3, 4)), st, 2)
