"""Restatement of the sub-pixel disparity (stereo_ctx_set_subpixel, StereoSGBM's 1/16-pixel fixed point) for the tests:
numpy on the host, never part of the product.  V is the value a map minimises over its candidates - S from
sgm_oracle.aggregate (SSD or sgm_ncc_oracle's NCC cost), or the block matcher's window sums C from sgm_oracle.cost_volume.
bm_window_sums3 evaluates the block matcher's V only at d - 1, d and d + 1 of each pixel, for full-size maps whose whole
cost volume would not fit in memory."""
import numpy as np


def offset(vm, v0, vp):
    """((V(d-1) - V(d+1)) 16 + den) / (2 den), den = max(V(d-1) + V(d+1) - 2 V(d), 1), in int64 with C division (toward
    zero; numpy's // floors)."""
    vm, v0, vp = (np.asarray(a, np.int64) for a in (vm, v0, vp))
    den = np.maximum(vm + vp - 2 * v0, 1)
    num = (vm - vp) * 16 + den
    return np.sign(num) * (np.abs(num) // (2 * den))


def refine3(d, vm, v0, vp, ok, sentinel):
    """16 d + offset where ok (d - 1 and d + 1 present, d not the sentinel), 16 d elsewhere (int64)."""
    d = np.asarray(d, np.int64)
    ok = np.asarray(ok, bool) & (d != sentinel)
    return np.where(ok, 16 * d + offset(np.where(ok, vm, 0), np.where(ok, v0, 0), np.where(ok, vp, 0)), 16 * d)


def refine(V, present, d, dmin, sentinel):
    """The refined map (int64) of the integer map d from the full volume V (rows, cols, D) of candidates dmin .. dmin + D - 1
    and its present mask."""
    V = np.asarray(V, np.int64)
    present = np.asarray(present, bool)
    d = np.asarray(d, np.int64)
    D = V.shape[-1]
    j = d - dmin
    inside = (j - 1 >= 0) & (j + 1 <= D - 1)
    jc = np.clip(j, 1, max(D - 2, 1))

    def at(a, jj):
        return np.take_along_axis(a, np.clip(jj, 0, D - 1)[..., None], -1)[..., 0]

    ok = inside & at(present, jc - 1) & at(present, jc + 1)
    return refine3(d, at(V, jc - 1), at(V, jc), at(V, jc + 1), ok, sentinel)


def refine_literal(V, present, d, dmin, sentinel):
    """The rule pixel by pixel in Python integers (tiny maps only)."""
    rows, cols, D = np.shape(V)
    out = np.empty((rows, cols), np.int64)
    for y in range(rows):
        for x in range(cols):
            dv = int(d[y, x])
            j = dv - dmin
            if dv != sentinel and 1 <= j <= D - 2 and present[y, x, j - 1] and present[y, x, j + 1]:
                vm, v0, vp = int(V[y, x, j - 1]), int(V[y, x, j]), int(V[y, x, j + 1])
                den = max(vm + vp - 2 * v0, 1)
                num = (vm - vp) * 16 + den
                q = abs(num) // (2 * den)
                out[y, x] = 16 * dv + (q if num >= 0 else -q)
            else:
                out[y, x] = 16 * dv
    return out


def bm_window_sums3(ref, tgt, R, d, ys, chunk=16):
    """V(d - 1), V(d), V(d + 1) (int64, (len(ys), cols) each) of the single-direction SSD call at the output rows ys, d the
    map's rows ys: replicate padding, flat-index target reads that wrap into the neighbouring padded row or the zero guard,
    per element round(f32(f32(l - r)^2)) half away from zero.  Evaluated chunk rows at a time."""
    ref = np.asarray(ref, np.float32)
    tgt = np.asarray(tgt, np.float32)
    rows, cols = ref.shape
    Hp, Wp, w = rows + 2 * R, cols + 2 * R, 2 * R + 1
    Lp = np.pad(ref, R, mode="edge")
    flat = np.pad(tgt, R, mode="edge").reshape(-1)
    d = np.asarray(d, np.int64)
    ys = np.asarray(ys)
    out = np.zeros((3, len(ys), cols), np.int64)
    x = np.arange(cols)
    for c0 in range(0, len(ys), chunk):
        yy = ys[c0:c0 + chunk]
        dd = d[c0:c0 + chunk]
        for wy in range(w):
            r = (yy + wy)[:, None]
            for k in range(w):
                lv = Lp[r, x[None, :] + k]
                for i, delta in enumerate((-1, 0, 1)):
                    f = r * Wp + x[None, :] + k + dd + delta
                    ok = (f >= 0) & (f < Hp * Wp)
                    tv = np.where(ok, flat[np.clip(f, 0, Hp * Wp - 1)], np.float32(0))
                    e = (lv - tv).astype(np.float32)
                    q = (e * e).astype(np.float32)
                    out[i, c0:c0 + chunk] += np.floor(q.astype(np.float64) + 0.5).astype(np.int64)
    return out[0], out[1], out[2]


def bm_refine_rows(ref, tgt, R, d, ys, dmin, dmax, sentinel):
    """The refined rows ys of a block-matcher SSD map d (the rows ys of the integer map) of candidates [dmin, dmax]."""
    d = np.asarray(d, np.int64)
    cols = d.shape[1]
    Wp = cols + 2 * R
    s = np.arange(cols)[None, :] + R + d
    ok = (d - 1 >= dmin) & (d + 1 <= dmax) & (s - 1 >= 0) & (s + 1 <= Wp - 1)
    return refine3(d, *bm_window_sums3(ref, tgt, R, np.where(ok, d, 0), ys), ok, sentinel)
