"""The speckle filter's restatement (speckle_oracle.filter_speckles) against executed cv2.filterSpeckles on int16 and uint8
maps, and against answers derived by hand for int8 and int32 maps, which cv2 does not take.  CPU only."""
import numpy as np
import pytest

from speckle_oracle import filter_speckles


def _cv2():
    return pytest.importorskip("cv2")


def _cv(d, new_val, max_size, max_diff):
    return _cv2().filterSpeckles(d.copy(), new_val, max_size, max_diff)[0]


def _random_map(g, rows, cols, dtype, new_val, smooth):
    """Random blobs: a row-wise random walk (long, thin regions) or uniform noise over a small span, with a tenth of the
    pixels set to new_val."""
    lo, hi = (0, 254) if dtype == np.uint8 else (-40, 40)
    if smooth:
        d = np.clip(np.cumsum(g.integers(-1, 2, (rows, cols)), axis=1) + (lo + hi) // 2, lo, hi)
    else:
        span = int(g.integers(1, 12))
        d = g.integers(0, span + 1, (rows, cols)) + (lo + hi) // 2
    d = d.astype(dtype)
    d[g.random((rows, cols)) < 0.1] = new_val
    return d


@pytest.mark.parametrize("dtype,new_val", [(np.int16, -41), (np.uint8, 255)])
def test_random_maps_equal_cv2(dtype, new_val):
    g = np.random.default_rng(7 if dtype == np.int16 else 8)
    for t in range(150):
        rows, cols = (int(v) for v in g.integers(1, 50, 2))
        d = _random_map(g, rows, cols, dtype, new_val, t % 2 == 1)
        max_size, max_diff = int(g.integers(0, 40)), int(g.integers(0, 3))
        got = filter_speckles(d, new_val, max_size, max_diff)
        assert got.dtype == d.dtype
        assert np.array_equal(got, _cv(d, new_val, max_size, max_diff)), (t, rows, cols, max_size, max_diff)


@pytest.mark.parametrize("shape", [(1, 200), (200, 1), (1, 1)])
@pytest.mark.parametrize("dtype,new_val", [(np.int16, -41), (np.uint8, 255)])
def test_single_row_and_column_equal_cv2(shape, dtype, new_val):
    g = np.random.default_rng(shape[0] * 3 + shape[1])
    d = _random_map(g, *shape, dtype, new_val, True)
    for max_size, max_diff in ((0, 1), (1, 0), (5, 1), (30, 2)):
        assert np.array_equal(filter_speckles(d, new_val, max_size, max_diff), _cv(d, new_val, max_size, max_diff))


@pytest.mark.parametrize("dtype,new_val", [(np.int16, -41), (np.uint8, 255)])
def test_all_sentinel_and_degenerate_settings_equal_cv2(dtype, new_val):
    d = np.full((9, 13), new_val, dtype)
    assert np.array_equal(filter_speckles(d, new_val, 50, 1), d)
    assert np.array_equal(_cv(d, new_val, 50, 1), d)
    g = np.random.default_rng(11)
    d = _random_map(g, 30, 40, dtype, new_val, False)
    assert np.array_equal(filter_speckles(d, new_val, 0, 1), d)                 # max_size 0: nothing is that small
    for max_size in (1, 3, 1000):
        got = filter_speckles(d, new_val, max_size, 0)                          # max_diff 0: equal values only
        assert np.array_equal(got, _cv(d, new_val, max_size, 0)), max_size
    assert (filter_speckles(d, new_val, 30 * 40, 5) == new_val).all()


@pytest.mark.parametrize("dtype,new_val", [(np.int16, -41), (np.uint8, 255)])
def test_size_exactly_max_size_is_removed_one_more_is_kept(dtype, new_val):
    # two plateaus separated by a column of sentinels: 4 x 3 = 12 pixels (left) and 13 pixels (right, one extra pixel)
    d = np.full((5, 9), new_val, dtype)
    d[0:4, 0:3] = 7
    d[0:4, 4:7] = 9
    d[4, 4] = 9
    want = d.copy()
    want[0:4, 0:3] = new_val
    got = filter_speckles(d, new_val, 12, 1)
    assert np.array_equal(got, want)
    assert np.array_equal(_cv(d, new_val, 12, 1), want)


def test_hand_derived_int8():
    nv = -128
    d = np.array([[1, 1, 5, nv, 3],
                  [1, 2, 5, nv, 3],
                  [9, 9, 9, 9, 3]], np.int8)
    # max_diff 1: {1,1,1,2} (4 px), {5,5} (2 px), {9,9,9,9} (4 px), {3,3,3} (3 px); |9 - 3| > 1 keeps 9s and 3s apart
    got = filter_speckles(d, nv, 3, 1)
    want = np.array([[1, 1, nv, nv, nv],
                     [1, 2, nv, nv, nv],
                     [9, 9, 9, 9, nv]], np.int8)
    assert got.dtype == np.int8 and np.array_equal(got, want)
    # max_diff 0: the 2 splits off {1,1,1} (3 px) as a component of its own
    got = filter_speckles(d, nv, 1, 0)
    want = d.copy()
    want[1, 1] = nv
    assert np.array_equal(got, want)
    # the extremes of int8 link when max_diff covers their difference (255), computed without wrapping
    e = np.array([[-127, 127]], np.int8)
    assert np.array_equal(filter_speckles(e, nv, 1, 254), e)             # linked: one component of 2 pixels
    assert (filter_speckles(e, nv, 1, 253) == nv).all()                   # apart: two of 1 pixel each
    assert (filter_speckles(e, nv, 2, 254) == nv).all()


def test_hand_derived_int32_near_the_limits():
    lo, hi = np.iinfo(np.int32).min, np.iinfo(np.int32).max
    nv = 0
    d = np.array([[lo, lo + 1, hi - 1, hi]], np.int32)
    # lo and hi differ by 2^32 - 1: linked only when max_diff reaches that, which a 32-bit difference would wrap
    assert np.array_equal(filter_speckles(d, nv, 2, 1), np.array([[nv, nv, nv, nv]], np.int32))
    assert np.array_equal(filter_speckles(d, nv, 1, 1), d)
    col = np.array([[lo], [hi]], np.int32)
    assert np.array_equal(filter_speckles(col, nv, 1, 2 ** 32 - 1), col)
    assert np.array_equal(filter_speckles(col, nv, 2, 2 ** 32 - 1), np.zeros_like(col))
    assert np.array_equal(filter_speckles(col, nv, 1, 2 ** 32 - 2), np.zeros_like(col))
    # the sentinel itself never joins a component, whatever max_diff
    s = np.array([[5, nv, 5]], np.int32)
    assert np.array_equal(filter_speckles(s, nv, 1, 10), np.array([[nv, nv, nv]], np.int32))
    assert np.array_equal(filter_speckles(s, nv, 0, 10), s)


def test_rejects_bad_arguments():
    with pytest.raises(ValueError):
        filter_speckles(np.zeros((2, 2), np.float32), 0, 1, 1)
    with pytest.raises(ValueError):
        filter_speckles(np.zeros((2, 2), np.int16), 0, -1, 1)
    with pytest.raises(ValueError):
        filter_speckles(np.zeros(4, np.int16), 0, 1, 1)
