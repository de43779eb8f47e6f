"""Workspace sizes of the mapping-specificity search without a GPU (the SM count then falls back to 148): tables up
to 64 wide keep the size nabo_specificity_workspace_bytes always returned; 65 to 128 wide need the larger per-node
scratch of the 128-source search; wider tables are refused (0)."""
import pytest

from nabo_b200 import _lib, build


@pytest.fixture(scope="module")
def L():
    build.build()
    return _lib.lib()


@pytest.mark.parametrize("n_ref,n_query", [(1, 1), (1000, 3), (100000, 100000), (3_000_000, 2)])
def test_workspace_size_by_width(L, n_ref, n_query):
    old = L.nabo_specificity_workspace_bytes(n_ref, n_query)
    assert old > 0
    for k in range(1, 65):
        assert L.nabo_specificity_workspace_bytes_k(n_ref, n_query, k) == old
    wide = L.nabo_specificity_workspace_bytes_k(n_ref, n_query, 65)
    assert wide > old
    for k in range(65, 129):
        assert L.nabo_specificity_workspace_bytes_k(n_ref, n_query, k) == wide
    assert L.nabo_specificity_workspace_bytes_k(n_ref, n_query, 129) == 0


def test_workspace_per_node_bytes(L):
    # one CTA (one target): 45 bytes per reference cell (rounded up to 64 cells) below 65 mapped cells, 81 above
    assert L.nabo_specificity_workspace_bytes_k(6400, 1, 64) == 6400 * 45 + 1024
    assert L.nabo_specificity_workspace_bytes_k(6400, 1, 128) == 6400 * 81 + 1024
    assert L.nabo_specificity_workspace_bytes_k(6401, 1, 100) == 6464 * 81 + 1024
