"""Restatement of the left-right consistency check (stereo_ctx_set_lr_check) for the tests: numpy on the host, never part
of the product."""
import numpy as np


def lr_check(dl, dr, disparity_range, max_diff):
    """Both maps of a pair after the check.  The left pixel x with value dL is kept when x + dL lies in [0, cols) and
    |dL + dR(x + dL)| <= max_diff, the right pixel likewise with the maps swapped, both against the unchecked maps; every
    other pixel becomes -(disparity_range + 1).  Returns the two checked maps in the input maps' dtype."""
    dl, dr = np.asarray(dl), np.asarray(dr)
    if dl.ndim != 2 or dl.shape != dr.shape:
        raise ValueError("maps must be 2-D arrays of equal shape")
    if disparity_range < 0 or max_diff < 0:
        raise ValueError("disparity_range and max_diff must be >= 0")
    cols = dl.shape[1]

    def one(own, partner):
        d, q = own.astype(np.int64), partner.astype(np.int64)
        p = np.arange(cols)[None, :] + d
        inside = (p >= 0) & (p < cols)
        s = d + np.take_along_axis(q, np.clip(p, 0, cols - 1), axis=1)
        return np.where(inside & (np.abs(s) <= max_diff), d, -(disparity_range + 1)).astype(own.dtype)

    return one(dl, dr), one(dr, dl)
