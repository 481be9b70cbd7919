"""Restatement of StereoBM's X-Sobel prefilter and texture threshold (stereo_ctx_set_prefilter) for the tests: numpy on the
host, never part of the product.  pf() is OpenCV's prefilterXSobel (modules/calib3d/src/stereobm.cpp) for u8 images and
the library's stated extension for float32 images; texture_keep() is StereoBM's textureThreshold over the matcher's
replicate-padded window."""
import numpy as np


def pf(img, cap):
    """The prefiltered 8-bit image P of a u8 or float32 image.  Columns 0 and cols - 1, and the whole last row when rows is
    odd, are cap; every other pixel takes rows a = y - 1, b = y + 1 reflected 101-style and
    v = (I[a][x+1] - I[a][x-1]) + 2 (I[y][x+1] - I[y][x-1]) + (I[b][x+1] - I[b][x-1]), P = clip(v, -cap, cap) + cap
    (float32: each difference and sum rounded to float32 in that order, v rounded half to even, P = cap where v is NaN)."""
    img = np.asarray(img)
    if not 1 <= cap <= 63:
        raise ValueError("cap must be in [1, 63]")
    rows, cols = img.shape
    out = np.full((rows, cols), cap, np.uint8)
    n = rows - (rows & 1)                 # rows OpenCV filters (in pairs)
    if n == 0 or cols < 3:
        return out
    y = np.arange(n)
    ya = np.where(y > 0, y - 1, 1)
    yb = np.where(y < rows - 1, y + 1, rows - 2)
    if img.dtype == np.uint8:
        I = img.astype(np.int64)
        d = I[:, 2:] - I[:, :-2]
        v = d[ya] + 2 * d[y] + d[yb]
        out[:n, 1:-1] = (np.clip(v, -cap, cap) + cap).astype(np.uint8)
        return out
    I = img.astype(np.float32)
    with np.errstate(invalid="ignore", over="ignore"):
        d = (I[:, 2:] - I[:, :-2]).astype(np.float32)
        v = ((d[ya] + np.float32(2) * d[y]).astype(np.float32) + d[yb]).astype(np.float32)
        r = np.where(np.isnan(v), 0, np.clip(np.rint(v), -cap, cap))
    out[:n, 1:-1] = (r + cap).astype(np.uint8)
    return out


def texture_sum(P, cap, R):
    """Sum of |P - cap| over the (2R + 1)^2 window centred on each pixel, coordinates clamped to the image (int64)."""
    a = np.abs(np.asarray(P, np.int64) - cap)
    a = np.pad(a, R, mode="edge")
    I = np.zeros((a.shape[0] + 1, a.shape[1] + 1), np.int64)
    I[1:, 1:] = a.cumsum(0).cumsum(1)
    w = 2 * R + 1
    return I[w:, w:] - I[:-w, w:] - I[w:, :-w] + I[:-w, :-w]


def texture_keep(P, cap, R, threshold):
    """Mask of the pixels the texture threshold keeps: window sum >= threshold (a pixel is rejected when it is below)."""
    return texture_sum(P, cap, R) >= threshold
