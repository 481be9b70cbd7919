"""The numpy restatement of the NCC cost of SGM (sgm_ncc_oracle) against the literal oracle, on the CPU: its scores equal
ncc_check.score_at bit for bit at every present candidate, its first maximum is the oracle's NCC disparity in both pair
directions, and a small case derived by hand fixes C, the rounded product of a non-power-of-two q and the zero-penalty
winner."""
import numpy as np
import pytest

import oracle
from ncc_check import candidate_range, score_at
from sgm_ncc_oracle import cost_volume, quantise, scores, sgm, sgm_pair
from sgm_oracle import aggregate, winner


def _images(seed, rows, cols, kind):
    g = np.random.default_rng(seed)
    if kind == "u8":
        a = g.integers(0, 256, (rows, cols)).astype(np.float32)
        b = np.roll(a, -2, axis=1) + g.integers(-3, 4, (rows, cols))
        b = np.clip(b, 0, 255).astype(np.float32)
    elif kind == "float":
        a = (g.random((rows, cols)) * 255).astype(np.float32)
        b = (np.roll(a, -3, axis=1) * np.float32(1.1) + g.normal(0, 4, (rows, cols))).astype(np.float32)
    else:                                         # mixed-sign floats
        a = g.normal(0, 50, (rows, cols)).astype(np.float32)
        b = (np.roll(a, -1, axis=1) + g.normal(0, 10, (rows, cols))).astype(np.float32)
    # zero-energy windows: a dark block in each image
    a[: rows // 3, : cols // 4] = 0
    b[rows // 2:, cols // 2: cols // 2 + 5] = 0
    return a, b


CASES = [(seed, R, kind) for seed, (R, kind) in enumerate([(0, "u8"), (1, "float"), (2, "mixed"), (3, "u8"), (4, "float"),
                                                           (5, "mixed"), (6, "u8"), (7, "float")])]


@pytest.mark.parametrize("seed,R,kind", CASES)
def test_scores_equal_score_at_bit_for_bit(seed, R, kind):
    g = np.random.default_rng(100 + seed)
    rows, cols = int(g.integers(3, 14)), int(g.integers(5, 30))
    a, b = _images(seed, rows, cols, kind)
    rng = int(g.integers(1, cols + 4))
    for lo, hi in ((-rng, 0), (0, rng)):
        s, present = scores(a, b, R, lo, hi)
        ys, xs, js = np.nonzero(present)
        d = lo + js
        # ncc_check names candidates by the oracle's disparity: d itself in both directions (right-aligned for L->R)
        first, last = candidate_range(cols, R, lo, hi, xs)
        assert ((first <= xs + R + d) & (xs + R + d <= last)).all()
        want = score_at(a, b, R, lo, hi, ys, xs, d)
        got = s[ys, xs, js]
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (seed, R, kind, lo, hi)
        # and every legal candidate is present
        f_all, l_all = candidate_range(cols, R, lo, hi, np.arange(cols))
        assert len(d) == rows * int((l_all - f_all + 1).sum())


@pytest.mark.parametrize("seed,R,kind", CASES)
def test_first_maximum_is_the_oracle_ncc_map(seed, R, kind):
    rows, cols = 9 + seed, 24 + 3 * seed
    a, b = _images(50 + seed, rows, cols, kind)
    for rng in (5, cols + 3):
        for ref, tgt, lo, hi in ((a, b, -rng, 0), (b, a, 0, rng)):
            s, present = scores(ref, tgt, R, lo, hi)
            mine = np.where(present, s, -np.inf).argmax(axis=-1) + lo
            assert np.array_equal(mine, oracle.ncorr(ref, tgt, R, lo, hi)), (seed, R, kind, rng, lo)


def test_hand_derived_case():
    # one row, R = 1: replicate padding makes each window three copies of one padded row segment
    ref = np.array([[0, 3, 4]], np.float32)           # padded row 0 0 3 4 4
    tgt = np.array([[0, 4, 3]], np.float32)           # padded row 0 0 4 3 3
    s, present = scores(ref, tgt, 1, -2, 0)           # L->R over [-2, 0]: j = d + 2
    assert present[0].tolist() == [[False, False, True], [False, True, True], [True, True, True]]
    # x = 1: reference window (0 3 4); d = -1 -> target (0 0 4): 3·16 / sqrt(3·16 · 3·25) = 48/60;
    #        d = 0 -> target (0 4 3): 3·24 / sqrt(3·25 · 3·25) = 72/75
    assert s[0, 1, 1] == np.float32(0.8) and s[0, 1, 2] == np.float32(0.96)
    C, _ = cost_volume(ref, tgt, 1, -2, 0, 1000)
    # q = 1000: fl32(1000 · fl32(0.96)) = fl32(959.99997854...) = 960 (the rounded product, not 959), so C = 40;
    # fl32(1000 · fl32(0.8)) = 800, C = 200
    assert C[0, 1, 1] == 200 and C[0, 1, 2] == 40
    C2, _ = cost_volume(ref, tgt, 1, -2, 0, 1024)
    # q = 1024: exact products 819.2000122 and 983.0399780, floors 819 and 983
    assert C2[0, 1, 1] == 1024 - 819 and C2[0, 1, 2] == 1024 - 983
    # x = 0: only d = 0 (reference window (0 0 3) against target (0 0 4): 3·12 / sqrt(27 · 48) = 1, by division or by the
    # 1.125 rule depending on the rounding of t)
    assert s[0, 0, 2] == np.float32(1.0) and C[0, 0, 2] == 0
    # zero penalties: the first d of the largest floor(fl32(q·s)) at every pixel
    for paths in (4, 8):
        assert sgm(ref, tgt, 1, -2, 0, 1000, paths, 0, 0).tolist() == [[0, 0, 0]]
    # q = 1: every score in [0, 1) quantises to 0, so x = 1 and x = 2 pick their first present candidates
    assert sgm(ref, tgt, 1, -2, 0, 1, 4, 0, 0).tolist() == [[0, -1, -2]]


def test_rounded_product_of_a_non_power_of_two_scale():
    # q = 1000: the float32 product is correctly rounded, never below an integer the exact product reaches (the hand case
    # above has one that rounds up to the next integer)
    a, b = _images(7, 12, 40, "float")
    s, present = scores(a, b, 3, -20, 0)
    q = 1000
    exact = np.floor(np.float64(q) * s.astype(np.float64)).astype(np.int64)
    rounded = quantise(s, q)
    assert (rounded[present] >= exact[present]).all() and (rounded[present] <= exact[present] + 1).all()
    assert np.array_equal(rounded, np.floor((np.float32(q) * s).astype(np.float32)).astype(np.int64))
    # a power-of-two q multiplies exactly
    assert np.array_equal(quantise(s, 1 << 15)[present], np.floor(np.float64(1 << 15) * s[present]).astype(np.int64))


@pytest.mark.parametrize("q", [1, 1000, 1 << 15, 1 << 24])
def test_zero_penalties_pick_the_first_candidate_of_the_winners_quantum(q):
    a, b = _images(3, 11, 30, "float")
    for paths in (4, 8):
        dl, dr = sgm_pair(a, b, 2, 12, q, paths, 0, 0)
        for got, ref, tgt, lo, hi in ((dl, a, b, -12, 0), (dr, b, a, 0, 12)):
            want = oracle.ncorr(ref, tgt, 2, lo, hi)
            ys, xs = np.nonzero(got != want)
            assert (got[ys, xs] < want[ys, xs]).all()
            sg = score_at(ref, tgt, 2, lo, hi, ys, xs, got[ys, xs])
            so = score_at(ref, tgt, 2, lo, hi, ys, xs, want[ys, xs])
            assert np.array_equal(quantise(sg, q), quantise(so, q))
            if q == 1 << 24:
                assert len(ys) < got.size // 20


def test_aggregation_is_sgm_oracles():
    a, b = _images(4, 8, 20, "u8")
    C, present = cost_volume(a, b, 1, -6, 0, 500)
    assert C.min() >= 0 and C.max() <= 1000
    assert np.array_equal(sgm(a, b, 1, -6, 0, 500, 8, 30, 300), winner(aggregate(C, present, 8, 30, 300), present, -6))
