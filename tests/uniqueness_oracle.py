"""Restatement of the uniqueness ratio (stereo_ctx_set_uniqueness, StereoSGBM's uniquenessRatio) for the tests: numpy on
the host, never part of the product.  V is the value a map minimises over its candidates - S from sgm_oracle.aggregate
(SSD or sgm_ncc_oracle's NCC cost), or the block matcher's window sums C from sgm_oracle.cost_volume."""
import numpy as np

BM_NO_WINNER = 99999999      # the block matcher's initial best cost: a pixel whose every cost reaches it keeps the default 0


def unique(V, present, u, block_matcher=False):
    """(rows, cols) mask of the pixels the ratio keeps.  j* is the first minimum of V over the present candidates and V* its
    value; a pixel is rejected when some present candidate d with |d - j*| > 1 has V(d) (100 - u) < V* 100 (int64), and,
    for block-matcher maps, when every present V is >= 99999999."""
    V = np.asarray(V, np.int64)
    present = np.asarray(present, bool)
    if not 0 <= u <= 99:
        raise ValueError("u must be in [0, 99]")
    Vm = np.where(present, V, np.iinfo(np.int64).max)
    j = Vm.argmin(axis=-1)
    vstar = np.take_along_axis(Vm, j[..., None], axis=-1)
    far = np.abs(np.arange(V.shape[-1]) - j[..., None]) > 1
    keep = ~(present & far & (V * (100 - u) < vstar * 100)).any(axis=-1)
    if block_matcher:
        keep &= vstar[..., 0] < BM_NO_WINNER
    return keep


def apply(d, keep, disparity_range):
    """The map d with every pixel the mask rejects set to the sentinel -(disparity_range + 1), in d's dtype."""
    d = np.asarray(d)
    return np.where(keep, d, -(disparity_range + 1)).astype(d.dtype)
