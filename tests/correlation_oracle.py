"""CPU restatement of the correlation metric for the tests (NABO_CORRELATION in include/nabo_b200.h): each row minus
its mean, the sum sequential in ascending k, then the oracle's cosine distance on the centred rows.  NumPy's
elementwise add, divide and subtract are the IEEE operations the kernels use, so results are bit-identical."""
import numpy as np

from oracle import nabo_oracle as O


def centre_rows(x) -> np.ndarray:
    x = np.ascontiguousarray(x, dtype=np.float64)
    s = np.zeros(x.shape[0], dtype=np.float64)
    for k in range(x.shape[1]):
        s = s + x[:, k]
    with np.errstate(invalid="ignore"):
        return x - (s / x.shape[1])[:, None]


def correlation_dist(x, y) -> np.ndarray:
    return O.cosine_dist(centre_rows(x), centre_rows(y))


def knn(x, y, k: int, mask=None, drop_first: bool = False):
    """``oracle.knn`` for the correlation metric: (idx int64 (N,k), dist float64 (N,k))."""
    return O.knn(centre_rows(x), centre_rows(y), k, "cosine", mask=mask, drop_first=drop_first)
