"""Semi-global matching of one SSD direction restated in numpy (stereo_ctx_set_sgm, include/stereo_b200.h).

cost_volume restates the single-direction SSD call's window sums for every candidate: replicate padding, the flat-index
reads of the target that wrap into the neighbouring padded row or the zero guard, and per element round(f32(f32(l - r)^2))
rounded half away from zero, accumulated as an integer.  aggregate restates the path recurrence as row-by-row and
column-by-column sweeps; aggregate_literal is the same definition as a plain per-pixel loop, for tiny images.
"""
import numpy as np

PATHS8 = [(0, 1), (0, -1), (1, 0), (-1, 0), (1, 1), (1, -1), (-1, 1), (-1, -1)]
_BIG = np.int64(1) << 40       # stands for an absent candidate: above every present L_r + P2


def _elem(a, b):
    d = np.float32(a) - np.float32(b)
    q = (d * d).astype(np.float32)
    return np.floor(q.astype(np.float64) + 0.5).astype(np.int64)


def cost_volume(ref, tgt, R, dmin, dmax):
    """(C, present): int64 window sums (rows, cols, dmax - dmin + 1) and the present-candidate mask."""
    ref = np.asarray(ref, np.float32)
    tgt = np.asarray(tgt, np.float32)
    rows, cols = ref.shape
    Hp, Wp, w = rows + 2 * R, cols + 2 * R, 2 * R + 1
    Lp = np.pad(ref, R, mode="edge")
    flat = np.pad(tgt, R, mode="edge").reshape(-1)
    r, c = np.mgrid[:Hp, :Wp]
    D = dmax - dmin + 1
    C = np.empty((rows, cols, D), np.int64)
    for j in range(D):
        f = r * Wp + c + (dmin + j)
        ok = (f >= 0) & (f < Hp * Wp)
        T = np.where(ok, flat[np.clip(f, 0, Hp * Wp - 1)], np.float32(0))     # the zero guard outside the buffer
        E = _elem(Lp, T)
        I = np.zeros((Hp + 1, Wp + 1), np.int64)
        I[1:, 1:] = E.cumsum(0).cumsum(1)
        C[:, :, j] = I[w:, w:] - I[:-w, w:] - I[w:, :-w] + I[:-w, :-w]
    xp = np.arange(cols) + R
    s = xp[:, None] + np.arange(dmin, dmax + 1)[None, :]
    present = np.broadcast_to(((s >= 0) & (s <= Wp - 1))[None], C.shape)
    return C, present


def _step(Lq, Cp, pres_p, P1, P2):
    """L_r at a set of pixels p from L_r at their predecessors q (absent candidates of q hold _BIG)."""
    m = Lq.min(axis=-1, keepdims=True)
    big = np.full(Lq.shape[:-1] + (1,), _BIG)
    nb = np.minimum(np.concatenate([big, Lq[..., :-1]], -1), np.concatenate([Lq[..., 1:], big], -1))
    L = Cp + np.minimum(np.minimum(Lq, nb + P1), m + P2) - m
    return np.where(pres_p, L, _BIG)


def path_cost(C, present, dy, dx, P1, P2):
    """L_r for r = (dy, dx) over the whole image, by sweeps along the rows (dy != 0) or the columns (dy == 0)."""
    rows, cols, _ = C.shape
    Cb = np.where(present, C, _BIG)
    L = np.empty_like(Cb)
    if dy != 0:
        ys = range(rows) if dy > 0 else range(rows - 1, -1, -1)
        prev = None
        for y in ys:
            if prev is None:
                L[y] = Cb[y]
            else:
                L[y] = Cb[y]
                x0, x1 = max(0, dx), min(cols, cols + dx)        # columns whose predecessor (y - dy, x - dx) exists
                L[y, x0:x1] = _step(prev[x0 - dx:x1 - dx], C[y, x0:x1], present[y, x0:x1], P1, P2)
            prev = L[y]
    else:
        xs = range(cols) if dx > 0 else range(cols - 1, -1, -1)
        prev = None
        for x in xs:
            L[:, x] = Cb[:, x] if prev is None else _step(prev, C[:, x], present[:, x], P1, P2)
            prev = L[:, x]
    return L


def aggregate(C, present, paths, P1, P2):
    S = np.zeros(C.shape, np.int64)
    for dy, dx in PATHS8[:paths]:
        S += path_cost(C, present, dy, dx, P1, P2)
    return S


def winner(S, present, dmin):
    """The first minimum of S over the present candidates, as a disparity."""
    return np.where(present, S, np.iinfo(np.int64).max).argmin(axis=-1) + dmin


def sgm(ref, tgt, R, dmin, dmax, paths, P1, P2):
    C, present = cost_volume(ref, tgt, R, dmin, dmax)
    return winner(aggregate(C, present, paths, P1, P2), present, dmin)


def sgm_pair(left, right, R, rng, paths, P1, P2):
    """Both maps of a pair call: L->R over [-rng, 0] on the left image, R->L over [0, rng] with the images swapped."""
    return sgm(left, right, R, -rng, 0, paths, P1, P2), sgm(right, left, R, 0, rng, paths, P1, P2)


def aggregate_literal(C, present, paths, P1, P2):
    """The definition, pixel by pixel and candidate by candidate (tiny images only)."""
    rows, cols, D = C.shape
    S = np.zeros(C.shape, np.int64)
    for dy, dx in PATHS8[:paths]:
        L = {}
        ys = range(rows) if dy >= 0 else range(rows - 1, -1, -1)
        xs = list(range(cols) if dx >= 0 else range(cols - 1, -1, -1))
        for y in ys:
            for x in xs:
                qy, qx = y - dy, x - dx
                inside = 0 <= qy < rows and 0 <= qx < cols
                if inside:
                    m = min(L[qy, qx, e] for e in range(D) if present[qy, qx, e])
                for d in range(D):
                    if not present[y, x, d]:
                        continue
                    if not inside:
                        v = int(C[y, x, d])
                    else:
                        terms = [m + P2]
                        for e, pen in ((d, 0), (d - 1, P1), (d + 1, P1)):
                            if 0 <= e < D and present[qy, qx, e]:
                                terms.append(L[qy, qx, e] + pen)
                        v = int(C[y, x, d]) + min(terms) - m
                    L[y, x, d] = v
                    S[y, x, d] += v
    return S
