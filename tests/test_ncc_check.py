"""tests/ncc_check.py against the oracle (CPU only): score_at reproduces the oracle's winning scores bit for bit, and the
per-pixel checker rejects the ways an NCC map can be wrong while the north-star fraction still passes."""
import numpy as np
import pytest

import oracle
import ncc_check as nc
from introtocomputervision_b200 import synth


def _random_case(seed):
    rng = np.random.default_rng(70000 + seed)
    rows, cols = int(rng.integers(2, 24)), int(rng.integers(6, 70))
    R = seed % 8
    kind = seed % 3
    if kind == 0:
        dmin, dmax = -int(rng.integers(0, 2 * cols)), 0                 # right-aligned, up to twice the width
    elif kind == 1:
        dmin, dmax = 0, int(rng.integers(0, 2 * cols))                  # left-aligned
    else:
        dmin, dmax = -int(rng.integers(1, cols)), int(rng.integers(1, cols))   # mixed signs
    # (a range that excludes 0 leaves a border pixel without candidates: the reference throws, the library refuses it)
    L, Rt, _ = synth.make_pair(rows, cols, max(2, min(cols // 2, 20)), 70100 + seed)
    if seed % 3 == 1:
        a, b = synth.noisy_variant(L, seed), synth.noisy_variant(Rt, seed + 1)   # float images: the order of the sums matters
    else:
        a, b = L.astype(np.float32), Rt.astype(np.float32)
    if seed % 5 == 0:                                                     # zero-energy windows (both images)
        a[:, : cols // 3] = 0
        b[rows // 2:, cols // 2:] = 0
    return a, b, R, dmin, dmax


@pytest.mark.parametrize("seed", range(40))
def test_score_at_equals_the_oracles_winning_score(seed):
    a, b, R, dmin, dmax = _random_case(seed)
    try:
        d, s = oracle.ncorr(a, b, R, dmin, dmax, return_score=True)
    except oracle.OracleError:
        pytest.skip("a pixel without candidates (the reference throws)")
    ys, xs = np.indices(d.shape).reshape(2, -1)
    got = nc.score_at(a, b, R, dmin, dmax, ys, xs, d.ravel()).reshape(d.shape)
    assert np.array_equal(got.view(np.uint32), s.view(np.uint32)), (R, dmin, dmax)
    # and the oracle's map passes its own check in every family
    for fam in nc.FAMILIES:
        assert nc.check_ncc_map(d, a, b, R, dmin, dmax, fam, oracle_disp=d)["differ"] == 0


def test_random_cases_cover_what_they_are_for():
    cases = [_random_case(s) for s in range(40)]
    assert {R for _, _, R, _, _ in cases} == set(range(8))
    assert any(dmax == 0 and -dmin > a.shape[1] for a, _, _, dmin, dmax in cases)
    assert any(dmin == 0 and dmax > a.shape[1] for a, _, _, dmin, dmax in cases)
    assert any(dmin < 0 < dmax for *_, dmin, dmax in cases)
    assert any((a == 0).any() for a, *_ in cases)


def test_score_at_against_executed_opencv(golden):
    # the committed fixtures hold executed cv2.matchTemplate scores (tests/golden/make_golden.py); OpenCV's float32 numerator
    # may differ from the exactly rounded one by a few 1e-7 (test_oracle.py)
    for name, R, dmin, dmax in golden.names("ncc"):
        g = golden.get("ncc", name)
        L, Rt = g["left"].astype(np.float32), g["right"].astype(np.float32)
        ys, xs = np.indices(L.shape).reshape(2, -1)
        s = nc.score_at(L, Rt, R, dmin, dmax, ys, xs, g["disp"].astype(np.int64).ravel()).reshape(L.shape)
        np.testing.assert_allclose(s, g["score"], rtol=2e-6, atol=1e-7, err_msg=name)


@pytest.mark.parametrize("R,dmin,dmax", [(2, -9, 0), (1, 0, 7), (3, -4, 5)])
def test_score_at_against_live_opencv(R, dmin, dmax):
    pytest.importorskip("cv2")
    from oracle.ncc_cv2 import ncorr_cv2
    L, Rt, _ = synth.make_pair(6, 24, 8, 71000 + R)
    d, s = ncorr_cv2(L, Rt, R, dmin, dmax)
    ys, xs = np.indices(L.shape).reshape(2, -1)
    got = nc.score_at(L, Rt, R, dmin, dmax, ys, xs, d.ravel()).reshape(L.shape)
    np.testing.assert_allclose(got, s, rtol=2e-6, atol=1e-7)


def test_unwrap_i8_recovers_wide_ranges():
    L, Rt, _ = synth.make_pair(8, 300, 200, 71100)
    a, b = L.astype(np.float32), Rt.astype(np.float32)
    for dmin, dmax in ((-200, 0), (0, 200)):
        d = oracle.ncorr_fast(a, b, 2, dmin, dmax)
        assert np.abs(d).max() > 127
        assert np.array_equal(nc.unwrap_i8(oracle.narrow_i8(d), 300, 2, dmin, dmax), d)


# ---- the checker rejects wrong maps ---------------------------------------------------------------------------------

ROWS, COLS, R_T, D_T = 40, 200, 4, 40


def _textured():
    L, Rt, _ = synth.make_pair(ROWS, COLS, D_T + 1, 71200)
    return L.astype(np.float32), Rt.astype(np.float32)


def _all_scores(a, b, R, dmin, dmax, y, x):
    """Scores of every legal candidate of pixel (y, x), by disparity."""
    first, last = nc.candidate_range(a.shape[1], R, dmin, dmax, np.array([x]))
    n = int(last[0] - first[0])
    ds = np.arange(-n, 1) if (dmin <= 0 and dmax <= 0) else np.arange(0, n + 1)
    return ds, nc.score_at(a, b, R, dmin, dmax, np.full(len(ds), y), np.full(len(ds), x), ds)


@pytest.mark.parametrize("family", nc.FAMILIES)
def test_checker_rejects_a_neighbouring_candidate_beyond_tau(family):
    a, b = _textured()
    if family == "f32":
        a, b = synth.noisy_variant(a.astype(np.uint8), 1), synth.noisy_variant(b.astype(np.uint8), 2)
    d = oracle.ncorr(a, b, R_T, -D_T, 0)
    y, x = ROWS // 2, COLS // 2
    ds, s = _all_scores(a, b, R_T, -D_T, 0, y, x)
    assert d[y, x] == ds[np.argmax(s)]
    bad = d.copy()
    bad[y, x] = d[y, x] - 1 if d[y, x] > -D_T else d[y, x] + 1
    assert s[np.argmax(s)] - s[list(ds).index(bad[y, x])] > 2 ** -12       # far beyond every family's tau here
    nc.check_ncc_map(d, a, b, R_T, -D_T, 0, family, oracle_disp=d)
    with pytest.raises(AssertionError, match="beyond tau"):
        nc.check_ncc_map(bad, a, b, R_T, -D_T, 0, family, oracle_disp=d)
    # one wrong pixel in 8000 keeps the north-star fraction: only the per-pixel check sees it
    assert np.mean(bad == d) >= nc.NCC_DISP_AGREE


def test_checker_rejects_a_disparity_outside_the_candidates():
    a, b = _textured()
    for dmin, dmax in ((-D_T, 0), (0, D_T), (-7, 9)):
        d = oracle.ncorr_fast(a, b, R_T, dmin, dmax)
        first, last = nc.candidate_range(COLS, R_T, dmin, dmax, np.arange(COLS))
        for x, v in ((3, -(last[3] - first[3]) - 1 if dmax <= 0 else last[3] - first[3] + 1), (COLS - 1, 1 if dmax <= 0 else -1)):
            bad = d.copy()
            bad[5, x] = v
            with pytest.raises(AssertionError, match="no legal candidate"):
                nc.check_ncc_map(bad, a, b, R_T, dmin, dmax, "u8_fused", oracle_disp=d)


@pytest.mark.parametrize("shift", [-1, 1])
def test_checker_rejects_the_alignment_rule_off_by_one_at_the_left_border(shift):
    # right-aligned range: at the left border (x < D) the search is clipped and d = i - (ncand - 1); an off-by-one ncand
    # shifts every border disparity by one candidate
    a, b = _textured()
    d = oracle.ncorr_fast(a, b, R_T, -D_T, 0)
    bad = d.copy()
    bad[7, :8] += shift
    assert np.mean(bad == d) >= nc.NCC_DISP_AGREE
    with pytest.raises(AssertionError):
        nc.check_ncc_map(bad, a, b, R_T, -D_T, 0, "u8_fused", oracle_disp=d)


def test_checker_rejects_a_wrapped_int8_map_read_as_is():
    L, Rt, _ = synth.make_pair(8, 300, 200, 71300)
    a, b = L.astype(np.float32), Rt.astype(np.float32)
    d = oracle.ncorr_fast(a, b, 2, -200, 0)
    d8 = oracle.narrow_i8(d)
    nc.check_ncc_map(d8, a, b, 2, -200, 0, "u8_fused", oracle_disp=d)          # int8 maps are unwrapped
    with pytest.raises(AssertionError, match="no legal candidate"):
        nc.check_ncc_map(d8.astype(np.int32), a, b, 2, -200, 0, "u8_fused", oracle_disp=d)


def _near_tie_image():
    # smooth gradients + weak texture (test_ncc_fast_smooth_low_texture): dozens of candidates within a few float32 ulps
    yy, xx = np.mgrid[0:12, 0:160]
    rng = np.random.default_rng(5)
    L = np.clip(60 + 0.3 * xx + 0.2 * yy + rng.integers(-3, 4, xx.shape), 0, 255).astype(np.float32)
    Rt = np.clip(60 + 0.3 * (xx + 7) + 0.2 * yy + rng.integers(-3, 4, xx.shape), 0, 255).astype(np.float32)
    return L, Rt


def test_checker_accepts_a_genuine_near_tie_and_rejects_it_for_the_exact_family():
    L, Rt = _near_tie_image()
    R, dmin, dmax = 4, -40, 0
    d = oracle.ncorr(L, Rt, R, dmin, dmax)
    found = None
    for y in range(2, 10):
        for x in range(45, 160):
            ds, s = _all_scores(L, Rt, R, dmin, dmax, y, x)
            best = int(np.argmax(s))
            gaps = s[best].astype(np.float64) - s.astype(np.float64)
            near = np.nonzero((gaps > 0) & (gaps <= 2 ** -22))[0]
            if len(near):
                found = (y, x, int(ds[near[0]]), float(gaps[near[0]]))
                break
        if found:
            break
    assert found, "no near-tie in the image"
    y, x, alt, gap = found
    tie = d.copy()
    tie[y, x] = alt
    st = nc.check_ncc_map(tie, L, Rt, R, dmin, dmax, "u8_fused", oracle_disp=d)
    assert st["differ"] == 1 and 0 < st["max_gap"] <= 2 ** -22 and st["max_ratio"] <= 0.25
    nc.check_ncc_map(tie, L, Rt, R, dmin, dmax, "u8", oracle_disp=d)
    with pytest.raises(AssertionError, match="beyond tau"):
        nc.check_ncc_map(tie, L, Rt, R, dmin, dmax, "exact", oracle_disp=d)


def test_checker_requires_the_first_candidate_where_the_reference_window_is_dark():
    a, b = _textured()
    a[:, 50:80] = 0                       # EL = 0 for the pixels whose whole window is dark: every score is 0
    d = oracle.ncorr(a, b, R_T, -D_T, 0)
    bad = d.copy()
    bad[10, 65] += 1                      # another candidate of score 0: no gap, but not the first maximum
    with pytest.raises(AssertionError, match="beyond tau"):
        nc.check_ncc_map(bad, a, b, R_T, -D_T, 0, "u8", oracle_disp=d)


def test_tau_of_the_unfused_kernels_widens_next_to_a_bright_window():
    # a dark textured stripe next to a bright one: the unfused kernels' strip scale comes from the bright window, the fused
    # pairs' per-pixel scale does not; far from the bright half both are the plain four key steps
    a, b = _textured()
    a[:, :100] = np.round(a[:, :100] / 32)
    ys, xs = np.array([20, 20, 20]), np.array([90, 40, 150])
    _, el, er = nc.score_at(a, b, R_T, -D_T, 0, ys, xs, np.zeros(3, np.int64), energies=True)
    tau_u8, _ = nc.tolerance("u8", a, b, R_T, ys, xs, el, er, er, ROWS)
    tau_fused, _ = nc.tolerance("u8_fused", a, b, R_T, ys, xs, el, er, er, ROWS)
    full = nc._el_map(a, R_T)
    assert tau_u8[0] == pytest.approx(2 ** -20 * np.sqrt(full[20, 67:114].max() / el[0])) and tau_u8[0] > 16 * 2 ** -20
    assert tau_u8[1] < 2 * 2 ** -20 and tau_u8[2] < 2 * 2 ** -20
    assert np.all(tau_fused == 2 ** -20)
    tau_f32, key_f32 = nc.tolerance("f32", a, b, R_T, ys, xs, el, er, er, ROWS)
    assert np.allclose(key_f32, 2 * tau_u8) and np.all(tau_f32 > key_f32)
    assert np.all(nc.tolerance("exact", a, b, R_T, ys, xs, el, er, er, ROWS)[0] == 0)
