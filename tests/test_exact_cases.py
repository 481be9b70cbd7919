"""The case builders of test_exact_family.py checked on the CPU: the edge values sit on both sides of the FAST_F32 bound for
SSD, and the inside cases drive the oracle's keys to within 1 % of what the float kernels hold, so the GPU test exercises
the top of the key and not some comfortable middle."""
import numpy as np
import pytest

import oracle
import exact_cases as ec

EDGE_RNG = 24


def _edge_pair(R, side):
    inside, outside = ec.ssd_edge(R)
    return ec.ssd_edge_pair(R, inside if side == "inside" else outside, 2 * (2 * R + 3) + 14, 90, 56000 + R)


def test_edge_values():
    # largest admitted multiple of 0.25 and the next one, per radius (range = top * (1 + 1e-6) with lo = 0):
    #   R = 0: range^2 + 1 < 8388607                      -> 2896.25 in, 2896.5 out
    #   R >= 1: (2R+1)^2 * (range^2 + 1) < 2^25 - 8193   -> R = 1: 1930.5 / 1930.75, R = 3: 827.25 / 827.5,
    #                                                       R = 5: 526.5 / 526.75, R = 7: 386 / 386.25
    want = {0: (2896.25, 2896.5), 1: (1930.5, 1930.75), 3: (827.25, 827.5), 5: (526.5, 526.75), 7: (386.0, 386.25)}
    for R, (inside, outside) in want.items():
        assert ec.ssd_edge(R) == (inside, outside), R
        assert ec.ssd_fast_f32_admits(0.0, inside, R) and not ec.ssd_fast_f32_admits(0.0, outside, R)
    # blocks without a non-8-bit pixel count as [0, 255], so a small range is never below that
    assert ec.ssd_value_range(10.0, 20.0) == pytest.approx(255.0 * (1 + 1e-6))
    assert ec.ssd_value_range(-1.0, 256.0) == pytest.approx(257.0 * (1 + 1e-6))


@pytest.mark.parametrize("R", [1, 3, 5, 7])
def test_inside_cases_reach_the_top_of_the_key(R):
    L, Rt = _edge_pair(R, "inside")
    inside, _ = ec.ssd_edge(R)
    assert L.min() == 0 and max(L.max(), Rt.max()) == np.float32(inside)
    for a, b, dmin, dmax in ((L, Rt, -EDGE_RNG, 0), (Rt, L, 0, EDGE_RNG)):
        d, c = oracle.ssd_fast(a, b, R, dmin, dmax, return_cost=True)
        key = ec.ssd_key_headroom(c, d, R)
        assert 0.99 * ec.KEY_LIMIT <= key < ec.KEY_LIMIT - 1, (R, key)
    # R = 7 at 386: the all-0 window against the all-386 one, 128 * 225 * 386^2 = 4 291 084 800
    if R == 7:
        assert 128 * 225 * int(inside) ** 2 == 4291084800


def test_inside_case_of_r0_reaches_the_top_of_the_mantissa():
    L, Rt = _edge_pair(0, "inside")
    for a, b, dmin, dmax in ((L, Rt, -EDGE_RNG, 0), (Rt, L, 0, EDGE_RNG)):
        top = ec.max_element(a, b, dmin, dmax)
        assert 0.99 * ec.MANTISSA_LIMIT <= top < ec.MANTISSA_LIMIT, top
    # and elements whose float square lands on a half-integer: round half away from zero decides the cost
    q = (L[:, :, None] - Rt[:, None, :]).astype(np.float32) ** 2
    q = q[q > 2.0 ** 22]
    assert np.any(q - np.floor(q) == 0.5)


def test_edge_pairs_stay_where_the_reference_is_defined():
    for R in (0, 1, 3, 5, 7):
        for side in ("inside", "outside"):
            L, Rt = _edge_pair(R, side)
            top = float(max(L.max(), Rt.max()))
            assert top ** 2 < 2.0 ** 31 and (2 * R + 1) ** 2 * top ** 2 < 2.0 ** 31


def test_the_99999999_case_has_pixels_on_both_sides():
    L, Rt = ec.the_99999999_pair(48, 120, 55000)
    d, c = oracle.ssd(L, Rt, 7, -20, 0, return_cost=True)
    hot = (c == ec.SSD_NO_CANDIDATE) & (d == 0)
    assert hot.sum() > 10 and (c < ec.SSD_NO_CANDIDATE).sum() > 10
    assert not ec.ssd_fast_f32_admits(0.0, float(L.max()), 7)
    assert 225 * float(L.max()) ** 2 < 2.0 ** 31


def test_ncc_score_band_separates_the_offsets():
    from introtocomputervision_b200 import synth
    L, Rt, _ = synth.make_pair(24, 160, 41, 61000)
    band = lambda a, b: ec.ncc_score_band(float(min(a.min(), b.min())), float(max(a.max(), b.max())))
    assert band(*ec.ncc_offset_pair(L, Rt, 300.0)) >= ec.NCC_MIN_SCORE_BAND
    for offset in (1e3, 1e4, 1e5, 9.9e5):
        assert band(*ec.ncc_offset_pair(L, Rt, offset)) < ec.NCC_MIN_SCORE_BAND, offset
        assert band(*ec.ncc_offset_pair(L, Rt, -offset - 255)) < ec.NCC_MIN_SCORE_BAND, offset
    assert band(*ec.ncc_offset_pair(L, Rt, gain=np.floor(999000.0 / max(L.max(), Rt.max())))) >= ec.NCC_MIN_SCORE_BAND
    # the reference's own float images: noise sigma 10 on both, x1.1 contrast on the left one
    assert band(synth.noisy_variant(L, 1), synth.noisy_variant(Rt, 2)) >= 0.5
    assert band(synth.contrast_variant(L), Rt.astype(np.float32)) >= 0.5
