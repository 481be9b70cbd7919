"""The left-right consistency check's restatement (lr_oracle.lr_check) against answers derived by hand, and against a plain
numpy loop on random maps.  CPU only."""
import numpy as np
import pytest

from lr_oracle import lr_check


def _loop(dl, dr, rng, max_diff):
    rows, cols = dl.shape
    ol, orr = dl.astype(np.int64), dr.astype(np.int64)
    for y in range(rows):
        for x in range(cols):
            for a, b, out in ((dl, dr, ol), (dr, dl, orr)):
                p = x + int(a[y, x])
                if not (0 <= p < cols and abs(int(a[y, x]) + int(b[y, p])) <= max_diff):
                    out[y, x] = -(rng + 1)
    return ol, orr


def test_constant_shift_loses_the_columns_whose_partner_is_outside():
    s, cols, rng = 3, 10, 5
    dl = np.full((2, cols), -s, np.int16)
    dr = np.full((2, cols), s, np.int16)
    ol, orr = lr_check(dl, dr, rng, 0)
    assert ol.dtype == np.int16 and orr.dtype == np.int16
    want_l = np.where(np.arange(cols) >= s, -s, -(rng + 1))
    want_r = np.where(np.arange(cols) < cols - s, s, -(rng + 1))
    assert np.array_equal(ol, np.broadcast_to(want_l, (2, cols)))
    assert np.array_equal(orr, np.broadcast_to(want_r, (2, cols)))


def test_occluding_step():
    # background at disparity 0, a foreground object at disparity 2 over left columns 3..5 (right columns 1..3): left 1, 2
    # are hidden behind it in the right view, right 4, 5 in the left view
    dl = np.array([[0, 0, 0, -2, -2, -2, 0, 0]], np.int8)
    dr = np.array([[0, 2, 2, 2, 0, 0, 0, 0]], np.int8)
    for m in (0, 1):
        ol, orr = lr_check(dl, dr, 3, m)
        assert ol.tolist() == [[0, -4, -4, -2, -2, -2, 0, 0]], m
        assert orr.tolist() == [[0, 2, 2, 2, -4, -4, 0, 0]], m
    ol, orr = lr_check(dl, dr, 3, 2)
    assert np.array_equal(ol, dl) and np.array_equal(orr, dr)


def test_partners_off_both_edges_fail_whatever_max_diff():
    rng = 4
    dl = np.zeros((1, 6), np.int32)
    dr = np.zeros((1, 6), np.int32)
    dl[0, 0], dl[0, 1] = -1, -2          # partners at -1 and -1
    dr[0, 5], dr[0, 4] = 1, 3            # partners at 6 and 7
    for m in (0, 1, 2 * rng):
        ol, orr = lr_check(dl, dr, rng, m)
        assert ol[0, :2].tolist() == [-5, -5] and orr[0, 4:].tolist() == [-5, -5], m
    # with max_diff = 2 * range nothing else fails
    assert ol[0, 2:].tolist() == [0, 0, 0, 0] and orr[0, :4].tolist() == [0, 0, 0, 0]


def test_max_diff_zero_one_and_twice_the_range():
    rng = 3
    dl = np.array([[0, 0, 0, -1, 0, 0]], np.int16)     # left 3 -> right 2, whose value is 2: |-1 + 2| = 1
    dr = np.array([[0, 0, 2, 0, 0, 0]], np.int16)      # right 2 -> left 4, whose value is 0: |2 + 0| = 2
    ol, orr = lr_check(dl, dr, rng, 0)
    # left 2 -> right 2 (|0 + 2| = 2), left 3 (1); right 2 (2) and right 3 -> left 3 (|0 - 1| = 1)
    assert ol.tolist() == [[0, 0, -4, -4, 0, 0]]
    assert orr.tolist() == [[0, 0, -4, -4, 0, 0]]
    ol, orr = lr_check(dl, dr, rng, 1)
    assert ol.tolist() == [[0, 0, -4, -1, 0, 0]]
    assert orr.tolist() == [[0, 0, -4, 0, 0, 0]]
    ol, orr = lr_check(dl, dr, rng, 2 * rng)
    assert np.array_equal(ol, dl) and np.array_equal(orr, dr)


def test_both_maps_are_read_before_any_pixel_is_invalidated():
    # left 4 (-1 -> right 3, value 3: |2| > 1) fails; right 2 (2 -> left 4, value -1: |1| <= 1) is checked against the -1,
    # not against left 4's sentinel
    dl = np.array([[0, 0, 0, 0, -1, 0, 0]], np.int32)
    dr = np.array([[0, 0, 2, 3, 0, 0, 0]], np.int32)
    ol, orr = lr_check(dl, dr, 3, 1)
    assert ol[0, 4] == -4 and orr[0, 2] == 2


def test_range_zero():
    dl = np.zeros((3, 5), np.int8)
    dr = np.zeros((3, 5), np.int8)
    ol, orr = lr_check(dl, dr, 0, 0)
    assert np.array_equal(ol, dl) and np.array_equal(orr, dr)
    dr[1, 4] = 1                          # partner at column 5: outside, and the sentinel is -1
    ol, orr = lr_check(dl, dr, 0, 0)
    assert orr[1, 4] == -1 and ol[1, 4] == -1 and np.count_nonzero(orr) + np.count_nonzero(ol) == 2


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_random_maps_equal_a_plain_loop(seed):
    g = np.random.default_rng(seed)
    rows, cols, rng = 4, int(g.integers(1, 40)), int(g.integers(0, 20))
    dl = g.integers(-rng, 1, (rows, cols)).astype(np.int32)
    dr = g.integers(0, rng + 1, (rows, cols)).astype(np.int32)
    for m in (0, 1, 3, 2 * rng):
        ol, orr = lr_check(dl, dr, rng, m)
        wl, wr = _loop(dl, dr, rng, m)
        assert np.array_equal(ol, wl) and np.array_equal(orr, wr), (seed, m)


def test_rejects_bad_arguments():
    a = np.zeros((2, 3), np.int32)
    with pytest.raises(ValueError):
        lr_check(a, np.zeros((2, 4), np.int32), 1, 0)
    with pytest.raises(ValueError):
        lr_check(a, a, -1, 0)
    with pytest.raises(ValueError):
        lr_check(a, a, 1, -1)
