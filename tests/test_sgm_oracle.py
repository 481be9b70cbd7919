"""The numpy restatement of semi-global matching (sgm_oracle) on the CPU: its cost volume against the compiled-reference-
pinned oracle.ssd (first minimum = disparity, minimum = cost), the vectorised sweeps against the per-pixel loop of the
definition, one hand-derived case, and the zero-penalty identity with the SSD maps."""
import numpy as np
import pytest

import oracle
import sgm_oracle as so


def _rand(g, rows, cols, levels=256):
    return g.integers(0, levels, (rows, cols)).astype(np.float32)


def _check_cost(ref, tgt, R, dmin, dmax):
    C, present = so.cost_volume(ref, tgt, R, dmin, dmax)
    d, cost = oracle.ssd(ref, tgt, R, dmin, dmax, return_cost=True)
    assert present[..., -dmin].all()                       # d = 0 is always present
    # the present set is contiguous
    assert (np.diff(present.astype(np.int8), axis=-1) != 0).sum(-1).max() <= 2
    masked = np.where(present, C, np.iinfo(np.int64).max)
    assert np.array_equal(masked.argmin(-1) + dmin, d)
    assert np.array_equal(masked.min(-1), cost)


@pytest.mark.parametrize("R", range(8))
def test_cost_volume_equals_the_oracle_random(R):
    g = np.random.default_rng(100 + R)
    rows, cols = 6 + R, 9 + 2 * R
    L, Rt = _rand(g, rows, cols), _rand(g, rows, cols)
    for dmin, dmax in ((-6, 0), (0, 6)):
        _check_cost(L, Rt, R, dmin, dmax)
        _check_cost(Rt, L, R, dmin, dmax)


@pytest.mark.parametrize("shape,R,rng", [((5, 9), 1, 6), ((4, 7), 0, 10), ((6, 8), 2, 4), ((3, 5), 3, 40), ((7, 4), 7, 30)])
def test_cost_volume_equals_the_oracle_ranges_wider_than_the_image(shape, R, rng):
    g = np.random.default_rng(shape[0] * 31 + R)
    L, Rt = _rand(g, *shape), _rand(g, *shape)
    _check_cost(L, Rt, R, -rng, 0)
    _check_cost(Rt, L, R, 0, rng)


def test_cost_volume_equals_the_oracle_float_images():
    g = np.random.default_rng(7)
    L = (g.random((8, 21)) * 300 - 20).astype(np.float32)
    Rt = (L * np.float32(1.1) + g.normal(0, 3, L.shape)).astype(np.float32)
    for R in (0, 2):
        _check_cost(L, Rt, R, -9, 0)
        _check_cost(Rt, L, R, 0, 9)


def test_cost_volume_equals_the_oracle_golden(golden):
    for name, R, a, b in golden.names("ssd")[:6]:
        case = golden.get("ssd", name)
        L, Rt = case["left"].astype(np.float32), case["right"].astype(np.float32)
        if L.size > 20000:
            continue
        _check_cost(L, Rt, R, a, b)


@pytest.mark.parametrize("paths", [4, 8])
@pytest.mark.parametrize("P1,P2", [(0, 0), (1, 5), (7, 7), (30, 400), (0, 100000)])
def test_sweeps_equal_the_literal_loop(paths, P1, P2):
    g = np.random.default_rng(paths * 1000 + P1 * 7 + P2)
    for shape, R, dmin, dmax in (((4, 6), 1, -5, 0), ((5, 5), 0, 0, 7), ((3, 8), 2, -12, 0), ((6, 3), 1, 0, 9)):
        L, Rt = _rand(g, *shape, levels=16), _rand(g, *shape, levels=16)
        C, present = so.cost_volume(L, Rt, R, dmin, dmax)
        # absent candidates at the left edge (dmin < 0) or the right edge (dmax > 0)
        assert not present.all()
        got = so.aggregate(C, present, paths, P1, P2)
        want = so.aggregate_literal(C, present, paths, P1, P2)
        assert np.array_equal(np.where(present, got, 0), want)


def test_hand_derived_one_row():
    # one row, three pixels, candidates d in {0, 1} (the right-referenced direction of a pair): the last pixel has only
    # d = 0.  Path (0, +1), P1 = 2, P2 = 10:
    #   x0: L = C = [4, 9]                                  m = 4
    #   x1: d0: 1 + min(4, 9 + 2, 14) - 4 = 1               d1: 6 + min(9, 4 + 2, 14) - 4 = 8        m = 1
    #   x2: d0: 3 + min(1, 8 + 2, 11) - 1 = 3
    # Path (0, -1): x2: [3, -]  m = 3;  x1: d0: 1 + min(3, 13) - 3 = 1, d1: 6 + min(3 + 2, 13) - 3 = 8;
    #   x0: d0: 4 + min(1, 10, 11) - 1 = 4, d1: 9 + min(8, 3, 11) - 1 = 11
    # S over the two horizontal paths (the vertical ones are L = C on one row): x0 [4+4+4+4, 9+11+9+9] = [16, 38]
    C = np.array([[[4, 9], [1, 6], [3, 0]]], np.int64)
    present = np.array([[[True, True], [True, True], [True, False]]])
    S = so.aggregate(C, present, 4, 2, 10)
    assert S[0, 0].tolist() == [16, 38]
    assert S[0, 1].tolist() == [1 + 1 + 1 + 1, 8 + 8 + 6 + 6]
    assert S[0, 2, 0] == 3 * 4
    assert np.array_equal(np.where(present, S, 0), so.aggregate_literal(C, present, 4, 2, 10))
    assert so.winner(S, present, 0).tolist() == [[0, 0, 0]]


def test_ties_take_the_first_minimum():
    C = np.array([[[5, 5, 5]]], np.int64)
    present = np.ones(C.shape, bool)
    assert so.winner(so.aggregate(C, present, 8, 3, 9), present, -2).tolist() == [[-2]]


@pytest.mark.parametrize("paths", [4, 8])
def test_zero_penalties_give_the_ssd_maps(paths):
    g = np.random.default_rng(paths)
    for shape, R, rng in (((5, 9), 1, 6), ((4, 7), 0, 10), ((6, 8), 2, 4), ((9, 30), 3, 12)):
        L, Rt = _rand(g, *shape), _rand(g, *shape)
        dl, dr = so.sgm_pair(L, Rt, R, rng, paths, 0, 0)
        assert np.array_equal(dl, oracle.ssd(L, Rt, R, -rng, 0))
        assert np.array_equal(dr, oracle.ssd(Rt, L, R, 0, rng))


def test_penalties_smooth_the_map():
    from introtocomputervision_b200 import synth
    L, Rt, _ = synth.make_pair(24, 64, 12, 3)
    L = (L.astype(np.float32) + np.random.default_rng(1).normal(0, 12, L.shape)).astype(np.float32)
    wta = so.sgm(L, Rt, 1, -12, 0, 8, 0, 0)
    smooth = so.sgm(L, Rt, 1, -12, 0, 8, 200, 3000)
    jumps = lambda d: int(np.abs(np.diff(d, axis=1)).sum() + np.abs(np.diff(d, axis=0)).sum())
    assert jumps(smooth) < jumps(wta)
