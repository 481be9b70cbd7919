"""Restatement of the speckle filter (cv::filterSpeckles, stereo_ctx_set_speckle_filter) for the tests: numpy and scipy on
the host, never part of the product."""
import numpy as np
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components


def filter_speckles(d, new_val, max_size, max_diff):
    """The map after the filter, in its own dtype (any integer dtype).  Two 4-neighbours are connected when neither equals
    new_val and |a - b| <= max_diff (computed in 64 bits); every pixel of a connected component of at most max_size pixels
    becomes new_val, every other pixel keeps its value."""
    d = np.asarray(d)
    if d.ndim != 2 or not np.issubdtype(d.dtype, np.integer):
        raise ValueError("the map must be a 2-D integer array")
    if max_size < 0 or max_diff < 0:
        raise ValueError("max_size and max_diff must be >= 0")
    rows, cols = d.shape
    v = d.astype(np.int64)
    ok = v != new_val
    idx = np.arange(rows * cols).reshape(rows, cols)
    a, b = [], []
    for s0, s1 in (((slice(None), slice(None, -1)), (slice(None), slice(1, None))),      # left-right neighbours
                   ((slice(None, -1), slice(None)), (slice(1, None), slice(None)))):     # up-down neighbours
        e = ok[s0] & ok[s1] & (np.abs(v[s0] - v[s1]) <= max_diff)
        a.append(idx[s0][e])
        b.append(idx[s1][e])
    a, b = np.concatenate(a), np.concatenate(b)
    n = rows * cols
    g = coo_matrix((np.ones(a.size, np.int8), (a, b)), shape=(n, n))
    _, lab = connected_components(g, directed=False)
    size = np.bincount(lab)[lab].reshape(rows, cols)
    out = d.copy()
    out[ok & (size <= max_size)] = new_val
    return out
