"""The prefilter / texture-threshold restatement (prefilter_oracle) against executed OpenCV: interior pixels against
cv2.Sobel, the texture rule and the prefilter's border-column and odd-last-row rules against cv2.StereoBM matching an image
with itself; then planted cases of the float extension and of tiny shapes.  CPU only."""
import numpy as np
import pytest

from prefilter_oracle import pf, texture_keep, texture_sum


def _image(rng, rows, cols, kind):
    if kind == "noise":
        return rng.integers(0, 256, (rows, cols)).astype(np.uint8)
    # smooth texture with flat patches, so that window sums spread across the threshold
    base = rng.integers(0, 256, (rows // 4 + 2, cols // 4 + 2)).astype(np.float64)
    up = np.kron(base, np.ones((4, 4)))[:rows, :cols]
    up[rows // 3: rows // 2, :] = 128
    return np.clip(up + rng.normal(0, 3, (rows, cols)), 0, 255).astype(np.uint8)


# ---- 1. interior pixels against cv2.Sobel ------------------------------------------------------------------------------

@pytest.mark.parametrize("rows,cols", [(31, 47), (32, 48), (2, 9), (3, 5), (64, 3)])
@pytest.mark.parametrize("cap", [1, 7, 31, 63])
def test_interior_equals_cv2_sobel(rows, cols, cap):
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(rows * 1000 + cols + cap)
    for kind in ("noise", "smooth"):
        img = _image(rng, rows, cols, kind)
        s = cv2.Sobel(img, cv2.CV_16S, 1, 0, ksize=3, borderType=cv2.BORDER_REFLECT_101).astype(np.int64)
        want = (np.clip(s, -cap, cap) + cap).astype(np.uint8)
        n = rows - (rows & 1)
        got = pf(img, cap)
        assert np.array_equal(got[:n, 1:cols - 1], want[:n, 1:cols - 1]), (rows, cols, cap, kind)
        assert (got[:, [0, cols - 1]] == cap).all()
        if rows & 1:
            assert (got[-1] == cap).all()


# ---- 2. texture rule and prefilter quirks against cv2.StereoBM(left == right) ------------------------------------------

@pytest.mark.parametrize("rows", [60, 61])
@pytest.mark.parametrize("block", [5, 9, 15])
@pytest.mark.parametrize("cap", [1, 13, 31, 63])
def test_texture_rule_equals_cv2_stereobm(rows, block, cap):
    cv2 = pytest.importorskip("cv2")
    R, cols = block // 2, 96
    rng = np.random.default_rng(rows * 100 + block * 7 + cap)
    compared = 0
    for kind in ("smooth", "noise"):
        img = _image(rng, rows, cols, kind)
        P = pf(img, cap)
        tsum = texture_sum(P, cap, R)
        ys, xs = slice(R, rows - R), slice(15 + R, cols - R)
        # thresholds across this image's distribution of window sums (and 0, which never fires)
        for T in [0, *np.unique(np.quantile(tsum[ys, xs], [0.05, 0.3, 0.6, 0.95]).round().astype(int) + 1)]:
            bm = cv2.StereoBM_create(16, block)
            bm.setPreFilterType(cv2.STEREO_BM_PREFILTER_XSOBEL)
            bm.setPreFilterCap(cap)
            bm.setTextureThreshold(int(T))
            bm.setUniquenessRatio(0)
            bm.setSpeckleWindowSize(0)
            bm.setDisp12MaxDiff(-1)
            d = bm.compute(img, img)
            rejected = d[ys, xs] == -16
            want = ~texture_keep(P, cap, R, int(T))[ys, xs]
            assert np.array_equal(rejected, want), (rows, block, cap, kind, int(T), int((rejected != want).sum()))
            compared += rejected.size
    assert compared > 0


# ---- 3. planted cases -------------------------------------------------------------------------------------------------

def test_f32_rounds_half_to_even():
    cap = 20
    img = np.zeros((2, 3), np.float32)
    # rows 0 and 1 reflect onto each other: with t at (0, 2) and zeros elsewhere, v = 2 t at (0, 1) (centre row) and
    # t + t at (1, 1) (both neighbour rows), exactly
    for v, want in ((0.5, 0), (1.5, 2), (2.5, 2), (3.5, 4), (-0.5, 0), (-1.5, -2), (-2.5, -2), (-3.5, -4), (7.5, 8)):
        img[0, 2] = np.float32(v / 2)
        P = pf(img, cap)
        assert P[0, 1] == cap + want and P[1, 1] == cap + want, (v, P[:, 1])


def test_f32_non_finite_neighbourhoods():
    cap = 31
    img = np.full((6, 7), 100, np.float32)
    img[2, 3] = np.nan
    img[4, 5] = np.inf
    P = pf(img, cap)
    # NaN at (2, 3): every output whose stencil reads it (x = 2 or 4, rows 1..3) has v NaN -> cap
    for y in (1, 2, 3):
        for x in (2, 4):
            assert P[y, x] == cap, (y, x)
    # +inf at (4, 5): x = 4 reads it as I[x+1] (v = +inf -> 2 cap) in rows 4 and 5 (row 3 also reads the NaN: cap)
    assert P[3, 4] == cap
    for y in (4, 5):
        assert P[y, 4] == 2 * cap, y
    img2 = np.full((4, 5), 0, np.float32)
    img2[1, 0], img2[1, 2] = np.inf, np.inf             # inf - inf = NaN at (1, 1)
    assert pf(img2, cap)[1, 1] == cap
    img3 = np.zeros((4, 5), np.float32)
    img3[1, 0] = -np.inf                                # 0 - (-inf) = +inf -> 2 cap
    assert pf(img3, cap)[1, 1] == 2 * cap


@pytest.mark.parametrize("cap", [1, 9, 63])
def test_8bit_valued_f32_equals_u8(cap):
    rng = np.random.default_rng(cap)
    for rows, cols in ((17, 33), (16, 40), (1, 5), (2, 2)):
        a = rng.integers(0, 256, (rows, cols)).astype(np.uint8)
        assert np.array_equal(pf(a.astype(np.float32), cap), pf(a, cap)), (rows, cols)


@pytest.mark.parametrize("rows", [1, 2, 3])
@pytest.mark.parametrize("cols", [1, 2, 3])
def test_tiny_shapes(rows, cols):
    cap = 10
    img = (np.arange(rows * cols).reshape(rows, cols) * 37 % 256).astype(np.uint8)
    P = pf(img, cap)
    assert P.shape == (rows, cols) and P.dtype == np.uint8
    if rows == 1 or cols < 3:
        assert (P == cap).all()
        return
    if rows & 1:
        assert (P[-1] == cap).all()
    I = img.astype(np.int64)
    for y in range(rows - (rows & 1)):
        a = y - 1 if y > 0 else 1
        b = y + 1 if y < rows - 1 else rows - 2
        v = (I[a, 2] - I[a, 0]) + 2 * (I[y, 2] - I[y, 0]) + (I[b, 2] - I[b, 0])
        assert P[y, 1] == min(max(v, -cap), cap) + cap, (y, v)


def test_threshold_is_strict():
    cap, R = 5, 1
    P = np.full((5, 5), cap, np.uint8)
    P[2, 2] = cap + 4                                   # one pixel of |P - cap| = 4 in every window that holds (2, 2)
    s = texture_sum(P, cap, R)
    assert s[2, 2] == 4 and s[0, 0] == 0
    assert texture_keep(P, cap, R, 4)[2, 2]             # 4 < 4 is false: kept
    assert not texture_keep(P, cap, R, 5)[2, 2]         # 4 < 5: rejected
    assert not texture_keep(P, cap, R, 1)[0, 0] and texture_keep(P, cap, R, 0).all()


def test_texture_window_clamps_to_the_image():
    cap, R = 3, 2
    P = np.full((4, 6), cap, np.uint8)
    P[0, 0] = cap + 1
    s = texture_sum(P, cap, R)
    # (0, 0) replicated: the window at (0, 0) covers rows / cols -2..2, clamped: row 0 three times, col 0 three times
    assert s[0, 0] == 9
    assert s[3, 5] == 0


def test_invalid_cap_is_rejected():
    for cap in (0, 64, -1):
        with pytest.raises(ValueError):
            pf(np.zeros((3, 3), np.uint8), cap)
