"""Case builders for the exact-family and kernel-family-bound tests (test_exact_family.py on the GPU, test_exact_cases.py
on the CPU).  numpy only; nothing here calls the library.

The float running-sum family (FAST_F32) takes an SSD problem only when the image pair's value range keeps the 32-bit key
`128 * SSD + position` and the per-element 2^23 mantissa trick exact (classify_images in stereo_b200.cu).  The functions
below restate that rule and build image pairs on both sides of it that drive the keys as close to the top as the rule
allows.  For NCC the same function admits an image only while a DC offset leaves its scores a band the float keys resolve
(ncc_score_band)."""
from __future__ import annotations

import numpy as np

KEY_LIMIT = 2.0 ** 32            # the SSD key 128 * SSD + position is a uint32
MANTISSA_LIMIT = 2.0 ** 23       # round((l - r)^2) + 0.5 is read off the mantissa of a float above 2^23
SSD_NO_CANDIDATE = 99999999      # the reference's initial best cost (DisparitySSD.cpp:37)


def ssd_value_range(lo: float, hi: float) -> float:
    """The range classify_images bounds: blocks without a non-8-bit pixel count as [0, 255], plus a 1e-6 margin."""
    return (max(hi, 255.0) - min(lo, 0.0)) * (1.0 + 1e-6)


def ssd_fast_f32_admits(lo: float, hi: float, R: int) -> bool:
    """True when an SSD problem with window radius R on images whose values lie in [lo, hi] may take FAST_F32."""
    r2 = ssd_value_range(lo, hi) ** 2
    wnd = float(2 * R + 1) ** 2
    return r2 + 1.0 < 8388607.0 and wnd * (r2 + 1.0) < 33554432.0 - 8193.0


def ssd_edge(R: int, step: float = 0.25):
    """(inside, outside): the largest multiple of `step` that FAST_F32 admits as the top of [0, top] at radius R, and the next
    one, which it does not admit."""
    wnd = float(2 * R + 1) ** 2
    r2_max = min(8388607.0 - 1.0, (33554432.0 - 8193.0) / wnd - 1.0)
    top = np.floor(np.sqrt(r2_max) / (1.0 + 1e-6) / step) * step
    while not ssd_fast_f32_admits(0.0, top, R):
        top -= step
    while ssd_fast_f32_admits(0.0, top + step, R):
        top += step
    return float(top), float(top + step)


def ssd_edge_pair(R: int, top: float, rows: int, cols: int, seed: int):
    """A float32 pair with values in [0, top] (both ends present) built to reach the top of the SSD key:
      * rows [0, h): left all 0, right all `top` - every candidate of an inner pixel costs (2R+1)^2 * top^2, so the keys
        tie and only their position bits order them (the first candidate must win);
      * rows [h, 2h): the same with the images swapped;
      * the rest: a textured scene (right = left shifted by 3 columns) on 0.25-steps, every fourth pixel replaced by 0 or
        `top`, and quarter values next to both ends - for R = 0 that puts (l - r)^2 on half-integers (round half away from
        zero) right below 2^23."""
    g = np.random.default_rng(seed)
    h = 2 * R + 3
    L = np.empty((rows, cols), np.float32)
    Rt = np.empty((rows, cols), np.float32)
    L[:h], Rt[:h] = 0.0, top
    L[h:2 * h], Rt[h:2 * h] = top, 0.0
    n = rows - 2 * h
    if n > 0:
        base = np.round(g.uniform(0.0, top, (n, cols + 3)) * 4) / 4
        ends = np.array([0.0, 0.25, 0.5, 0.75, top - 0.75, top - 0.5, top - 0.25, top])
        m = g.random(base.shape) < 0.25
        base[m] = g.choice(ends, int(m.sum()))
        L[2 * h:] = base[:, 3:]
        Rt[2 * h:] = base[:, :cols]
    return L, Rt


def ssd_key_headroom(cost: np.ndarray, disp: np.ndarray, R: int) -> float:
    """Largest 128 * cost + position over the map (position: the winning candidate's column in the padded image), the value
    the float SSD kernels keep in a uint32."""
    cols = cost.shape[1]
    pos = np.arange(cols)[None, :] + R + disp.astype(np.int64)
    return float(np.max(128 * cost.astype(np.int64) + pos))


def max_element(L: np.ndarray, Rt: np.ndarray, dmin: int, dmax: int) -> float:
    """Largest round-free per-element term f32((l - r)^2) + 0.5 any candidate of an R = 0 search reads (the replicate padding
    of R = 0 is empty, and every shift within [dmin, dmax] is tried against the clamped target column)."""
    cols = L.shape[1]
    best = 0.0
    for d in range(dmin, dmax + 1):
        s = np.clip(np.arange(cols) + d, 0, cols - 1)
        q = (L - Rt[:, s]).astype(np.float32)
        best = max(best, float(np.max(q * q)) + 0.5)
    return best


def the_99999999_pair(rows: int, cols: int, seed: int, hot: float = 1500.0):
    """A float32 pair at R = 7 whose SSD lies beyond what FAST_F32 admits: a textured 8-bit scene, and in the left image a
    square of `hot` pixels.  Pixels well inside the square have every candidate at or above 99999999 (225 * (hot - 255)^2),
    so the reference keeps disparity 0 and cost 99999999 there; pixels near its edge do not."""
    g = np.random.default_rng(seed)
    base = g.integers(0, 256, (rows, cols + 8)).astype(np.float32)
    L = base[:, 8:].copy()
    Rt = base[:, :cols].copy()
    y0, x0, s = rows // 4, cols // 3, max(20, rows // 2)
    L[y0:y0 + s, x0:x0 + s] = hot
    return L, Rt


NCC_MIN_SCORE_BAND = 1.0 / 16    # FAST_F32 NCC keeps at least 2^12 of its ~2^16 key steps across the scores' band


def ncc_score_band(lo: float, hi: float) -> float:
    """Width of the band [1 - band, 1] every NCC score of an image with values in [lo, hi] lies in: 1 unless every value has
    one sign, else (hi - lo)^2 / (lo^2 + hi^2) (one minus the least cosine between two windows of the box [lo, hi]^n)."""
    if lo <= 0.0 <= hi:
        return 1.0
    return (hi - lo) ** 2 / (lo * lo + hi * hi)


def ncc_offset_pair(L_u8: np.ndarray, R_u8: np.ndarray, offset: float = 0.0, gain: float = 1.0):
    """A textured 8-bit pair moved to float32 values gain * v + offset (integer-valued while gain and offset are)."""
    f = lambda a: (a.astype(np.float64) * gain + offset).astype(np.float32)
    return f(L_u8), f(R_u8)
