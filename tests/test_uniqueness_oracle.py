"""The uniqueness-ratio restatement (uniqueness_oracle) against a literal per-pixel transcription of OpenCV's StereoSGBM
winner-take-all loop (modules/calib3d/src/stereosgbm.cpp), on random volumes with planted cases.  CPU only."""
import numpy as np
import pytest

from uniqueness_oracle import BM_NO_WINNER, apply, unique


def _literal(V, present, u, block_matcher=False):
    """StereoSGBM's loop, one pixel at a time: minS and bestDisp over the present candidates in ascending d (strict <, so
    the first minimum), then the pixel is rejected when some d has Sp[d] * (100 - u) < minS * 100 and |bestDisp - d| > 1."""
    rows, cols, D = V.shape
    keep = np.ones((rows, cols), bool)
    for y in range(rows):
        for x in range(cols):
            minS, best = None, -1
            for d in range(D):
                if present[y, x, d] and (minS is None or int(V[y, x, d]) < minS):
                    minS, best = int(V[y, x, d]), d
            ok = not (block_matcher and minS >= BM_NO_WINNER)
            for d in range(D):
                if present[y, x, d] and int(V[y, x, d]) * (100 - u) < minS * 100 and abs(best - d) > 1:
                    ok = False
                    break
            keep[y, x] = ok
    return keep


def _volume(rng, rows, cols, D, hi):
    V = rng.integers(0, hi, size=(rows, cols, D), dtype=np.int64)
    present = rng.random((rows, cols, D)) < 0.85
    present[..., rng.integers(0, D)] = True          # every pixel has a candidate
    return V, present


@pytest.mark.parametrize("u", [0, 1, 5, 10, 15, 50, 99])
@pytest.mark.parametrize("seed", range(4))
def test_random_volumes_equal_the_literal_loop(u, seed):
    rng = np.random.default_rng(100 * seed + u)
    V, present = _volume(rng, 9, 11, 13, 60 if seed % 2 else 5000)
    for bm in (False, True):
        assert np.array_equal(unique(V, present, u, bm), _literal(V, present, u, bm)), (u, seed, bm)


def _one(values, present=None):
    V = np.array(values, np.int64)[None, None, :]
    p = np.ones(V.shape, bool) if present is None else np.array(present, bool)[None, None, :]
    return V, p


# values over d, present (None: all), u, kept
PLANTED = {
    "second minimum at distance 1 is ignored": ([50, 10, 11, 90, 90], None, 15, True),
    "second minimum at distance 2 is counted": ([50, 10, 90, 11, 90], None, 15, False),
    "equality at the threshold is kept (strict <)": ([100, 0, 90, 95, 100], [1, 0, 1, 1, 1], 10, True),
    "just below the threshold is rejected": ([100, 0, 90, 95, 99], [1, 0, 1, 1, 1], 10, False),
    "equal minima far apart": ([7, 30, 30, 30, 7], None, 1, False),
    "only one present candidate": ([0, 0, 5, 0, 0], [0, 0, 1, 0, 0], 99, True),
    "absent candidates cheaper than the winner": ([0, 0, 500, 0, 400], [0, 0, 1, 1, 1], 50, True),
    "u = 0 invalidates nothing": ([3, 3, 3, 3, 3], None, 0, True),
}


@pytest.mark.parametrize("case", list(PLANTED))
def test_planted_cases(case):
    values, pres, u, kept = PLANTED[case]
    V, p = _one(values, pres)
    assert bool(unique(V, p, u)[0, 0]) == kept
    assert bool(_literal(V, p, u)[0, 0]) == kept


def test_large_values_take_the_int64_product():
    # V (100 - u) and V* 100 are far beyond 2^31: 32-bit products would wrap and decide wrongly
    big = (1 << 31) - 5
    V, p = _one([big, 2 * 10 ** 9, 1, 2 * 10 ** 9, big])           # winner 2 (value 1), the others far and far larger
    assert unique(V, p, 50)[0, 0] and _literal(V, p, 50)[0, 0]
    V, p = _one([big - 1, 5, big, 2, big - 3])                       # winner 3 (value 2): far candidate 1 has 5 * 1 < 2 * 100
    assert not unique(V, p, 99)[0, 0] and not _literal(V, p, 99)[0, 0]
    V, p = _one([big, 5, big, big - 10, 0xFFFFFFFF])                 # winner 1 (value 5): every far candidate is far larger
    assert unique(V, p, 10)[0, 0] and _literal(V, p, 10)[0, 0]
    V, p = _one([big, big - 1, 3 * 10 ** 9, big, big - 2])
    for u in (1, 50, 99):
        assert unique(V, p, u)[0, 0] == _literal(V, p, u)[0, 0]


def test_block_matcher_pixels_without_an_accepted_candidate():
    V, p = _one([BM_NO_WINNER, BM_NO_WINNER + 5, 2 * BM_NO_WINNER])
    assert not unique(V, p, 0, block_matcher=True)[0, 0]
    assert unique(V, p, 0)[0, 0]
    V, p = _one([BM_NO_WINNER - 1, BM_NO_WINNER + 5, 2 * BM_NO_WINNER])
    assert unique(V, p, 10, block_matcher=True)[0, 0]


def test_zero_ratio_never_fires_on_random_volumes():
    rng = np.random.default_rng(7)
    V, present = _volume(rng, 12, 12, 20, 4)
    assert unique(V, present, 0).all()


def test_apply_writes_the_sentinel_in_the_maps_dtype():
    d = np.array([[1, -2], [3, 4]], np.int8)
    keep = np.array([[True, False], [False, True]])
    out = apply(d, keep, 20)
    assert out.dtype == np.int8 and out.tolist() == [[1, -21], [-21, 4]]
