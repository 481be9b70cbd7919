"""Semi-global matching of one NCC direction restated in numpy (stereo_ctx_set_sgm_ncc_scale, include/stereo_b200.h).

scores restates the float32 TM_CCORR_NORMED score of every candidate of every pixel in the literal oracle's arithmetic, as
ncc_check.score_at does one named candidate at a time: products in double summed per cell in (wy, k) order and rounded to
float32, double window energies in the same order, the 10·FLT_EPSILON zero-energy rule and the 1.125·t rule.  The loop runs
over the window offsets and is vectorised over pixels and candidates, so every cell still sums in (wy, k) order.
cost_volume turns the scores into C = q - floor(fl32(q·s)) and the present mask 0 <= x + d <= cols - 1; the aggregation
and the winner are sgm_oracle's, unchanged.
"""
import numpy as np

from sgm_oracle import aggregate, winner

FLT_EPSILON = float(np.finfo(np.float32).eps)


def present_mask(rows, cols, dmin, dmax):
    """(rows, cols, D) mask of the candidates d in [dmin, dmax] present at (y, x): 0 <= x + d <= cols - 1."""
    s = np.arange(cols)[:, None] + np.arange(dmin, dmax + 1)[None, :]
    return np.broadcast_to(((s >= 0) & (s <= cols - 1))[None], (rows, cols, dmax - dmin + 1))


def scores(ref, tgt, R, dmin, dmax):
    """(s, present): float32 scores (rows, cols, dmax - dmin + 1), 0 at absent candidates, and the present mask."""
    ref = np.asarray(ref, np.float32)
    tgt = np.asarray(tgt, np.float32)
    rows, cols = ref.shape
    w = 2 * R + 1
    Lp = np.pad(ref, R, mode="edge").astype(np.float64)
    Rp = np.pad(tgt, R, mode="edge").astype(np.float64)
    present = present_mask(rows, cols, dmin, dmax)
    tcol = np.clip(np.arange(cols)[:, None] + np.arange(dmin, dmax + 1)[None, :], 0, cols - 1)      # (cols, D), x + d
    acc = np.zeros(present.shape)
    el = np.zeros((rows, cols))
    er = np.zeros((rows, cols))                  # window energy of the target at every unpadded column
    for wy in range(w):
        for k in range(w):
            a = Lp[wy:wy + rows, k:k + cols]
            b = Rp[wy:wy + rows, k:k + cols]
            acc += a[:, :, None] * b[:, tcol]
            el += a * a
            er += b * b
    num = acc.astype(np.float32).astype(np.float64)
    ert = er[:, tcol]
    diff2 = np.where(ert > 0, ert, 0.0)
    lim = np.minimum(0.5, 10 * FLT_EPSILON * ert)
    t = np.where(diff2 <= lim, 0.0, np.sqrt(diff2)) * np.sqrt(el)[:, :, None]
    with np.errstate(divide="ignore", invalid="ignore"):
        sc = np.where(np.abs(num) < t, num / t, np.where(np.abs(num) < t * 1.125, np.sign(num), 0.0))
    return np.where(present, sc, 0.0).astype(np.float32), present


def quantise(s, q):
    """floor(fl32(q·s)) as int64: the float32 product rounded once, as the kernels compute it."""
    return np.floor(np.float32(q) * np.asarray(s, np.float32)).astype(np.int64)


def cost_volume(ref, tgt, R, dmin, dmax, q):
    """(C, present): C = q - floor(fl32(q·s)) in [0, 2q] (int64) and the present-candidate mask."""
    s, present = scores(ref, tgt, R, dmin, dmax)
    return q - quantise(s, q), present


def sgm(ref, tgt, R, dmin, dmax, q, paths, P1, P2):
    C, present = cost_volume(ref, tgt, R, dmin, dmax, q)
    return winner(aggregate(C, present, paths, P1, P2), present, dmin)


def clip_range(cols, rng):
    """A pair range clipped to the candidates some pixel has present: |d| <= cols - 1."""
    return min(rng, cols - 1)


def sgm_pair(left, right, R, rng, q, paths, P1, P2):
    """Both maps of an NCC pair call: L->R over [-rng, 0] on the left image, R->L over [0, rng] with the images swapped."""
    cols = np.asarray(left).shape[1]
    r = clip_range(cols, rng)
    return sgm(left, right, R, -r, 0, q, paths, P1, P2), sgm(right, left, R, 0, r, q, paths, P1, P2)
