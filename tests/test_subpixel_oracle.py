"""The sub-pixel restatement (subpixel_oracle) on the CPU: the vectorised rule against a literal loop, the offset range and
the integer part, exact parabolas, and the accuracy it buys on a pair shifted by a fraction of a pixel."""
import numpy as np
import pytest
from scipy.ndimage import gaussian_filter

from sgm_oracle import cost_volume, winner
from subpixel_oracle import bm_refine_rows, offset, refine, refine_literal


def _random_case(seed, rows=9, cols=13, D=7, dmin=-6):
    g = np.random.default_rng(seed)
    V = g.integers(0, 60, (rows, cols, D)).astype(np.int64)
    present = g.random((rows, cols, D)) > 0.15
    present[..., D // 2] = True
    d = winner(V, present, dmin)
    sentinel = dmin - 1
    d = np.where(g.random((rows, cols)) < 0.1, sentinel, d)
    return V, present, d, dmin, sentinel


@pytest.mark.parametrize("seed", range(6))
def test_vectorised_rule_equals_the_literal_loop(seed):
    V, present, d, dmin, sentinel = _random_case(seed)
    assert np.array_equal(refine(V, present, d, dmin, sentinel), refine_literal(V, present, d, dmin, sentinel))


def test_offset_truncates_toward_zero():
    assert offset(10, 0, 0) == 8                                    # (160 + 10) / 20 = 8.5 -> 8
    assert offset(0, 0, 10) == -7                                   # (-160 + 10) / 20 = -7.5 -> -7, not -8
    assert offset(0, 0, 0) == 0                                     # den = 1, (0 + 1) / 2 -> 0


@pytest.mark.parametrize("seed", range(4))
def test_offset_range_and_integer_part(seed):
    V, present, d, dmin, sentinel = _random_case(100 + seed, rows=40, cols=50, D=9, dmin=0)
    out = refine(V, present, d, dmin, sentinel)
    off = out - 16 * d
    assert off.min() >= -7 and off.max() <= 8
    assert np.array_equal((out + 7) >> 4, d)                         # the sentinel included
    # brute force over every triple of a first minimum: the offset stays in [-7, 8]
    a = np.arange(0, 40)
    vm, v0, vp = np.meshgrid(a, a, a, indexing="ij")
    first_min = (vm > v0) & (vp >= v0)
    o = offset(vm[first_min], v0[first_min], vp[first_min])
    assert o.min() == -7 and o.max() == 8


@pytest.mark.parametrize("A", [1, 3, 7])
def test_exact_parabolas_are_recovered_within_one_sixteenth(A):
    dv = np.arange(-20, 21)
    for t in range(-300, 301):
        V = A * (16 * dv - t) ** 2
        j = int(np.argmin(V))
        if j == 0 or j == len(dv) - 1:
            continue
        out = refine(V[None, None], np.ones((1, 1, len(dv)), bool), np.array([[dv[j]]]), int(dv[0]), -99)[0, 0]
        assert abs(out - t) <= 1, (A, t, out)


@pytest.mark.parametrize("s", [0.25, 0.5, 0.75])
def test_fractional_shift_is_recovered_to_an_eighth_of_a_pixel(s):
    g = np.random.default_rng(7)
    rows, cols, R, rng, shift = 48, 140, 3, 16, 7 + s
    tex = gaussian_filter(g.random((rows, cols + 32)) * 255.0, 1.5)
    tex = (tex - tex.min()) / (tex.max() - tex.min()) * 255.0
    xs = np.arange(cols)
    left = tex[:, :cols].astype(np.float32)
    i0 = np.floor(xs + shift).astype(int)                            # right(x) = left content at x + 7 + s (linear)
    right = ((1 - (xs + shift - i0)) * tex[:, i0] + (xs + shift - i0) * tex[:, i0 + 1]).astype(np.float32)
    V, present = cost_volume(left, right, R, -rng, 0)                # L->R: left(x) matches right(x + d), d = -(7 + s)
    d = winner(V, present, -rng)
    out = refine(V, present, d, -rng, -(rng + 1))
    inner = (slice(R + 2, rows - R - 2), slice(rng + R + 2, cols - R - 2))
    err_int = np.median(np.abs(d[inner] + shift))
    err_sub = np.median(np.abs(out[inner] / 16.0 + shift))
    assert err_int >= 0.25 and err_sub <= 0.125, (err_int, err_sub)


def test_row_helper_equals_the_full_volume():
    g = np.random.default_rng(3)
    L = g.integers(0, 256, (20, 45)).astype(np.uint8)
    Rt = np.roll(L, -5, axis=1)
    for R, lo, hi in ((2, -12, 0), (3, 0, 12)):
        V, present = cost_volume(L if lo < 0 else Rt, Rt if lo < 0 else L, R, lo, hi)
        d = winner(V, present, lo)
        d[3, 4] = -13                                                 # a sentinel
        want = refine(V, present, d, lo, -13)
        ys = [0, 1, 7, 19]
        got = bm_refine_rows(L if lo < 0 else Rt, Rt if lo < 0 else L, R, d[ys], ys, lo, hi, -13)
        assert np.array_equal(got, want[ys]), (R, lo, hi)
