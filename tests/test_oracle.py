"""CPU tests of the parity oracle itself: the C restatement against the golden vectors (which were
produced by the reference's own compiled SSD and by executed OpenCV), and against the reference's own compiled
SSD / NCC loop on random inputs and the pair helpers' ranges - live where oracle/_ref is built from the reference
sources, otherwise against its outputs recorded in tests/golden/ref_cases.npz (tests/golden/make_golden.py)."""
from pathlib import Path

import numpy as np
import pytest

import oracle
from introtocomputervision_b200 import synth

REF_CASES = Path(__file__).resolve().parent / "golden" / "ref_cases.npz"
SSD_PAIR_RANGES = [(14, 300, 2, 127), (9, 96, 3, 127), (8, 130, 1, 127), (10, 97, 2, 63), (7, 160, 5, 63), (6, 40, 4, 255),
                   (12, 320, 0, 127)]
NCC_PAIR_RANGES = [(8, 200, 2, 127), (6, 96, 3, 63), (7, 130, 1, 127), (5, 70, 4, 63)]
NCC_EMPTY_CASE = ((8, 16), 1, 3, 5)          # image shape, R, dmin, dmax: the right-most columns have no window


def _cases(cost):
    from conftest import Golden
    return Golden().names(cost)


def ssd_random_case(seed):
    """(left, right, R, dmin, dmax) of test_ssd_restatement_matches_compiled_reference_random."""
    rng = np.random.default_rng(seed)
    rows, cols = int(rng.integers(6, 28)), int(rng.integers(12, 70))
    R = int(rng.integers(0, 5))
    a, b = sorted(int(v) for v in rng.integers(-14, 15, 2))
    L, Rt, _ = synth.make_pair(rows, cols, 12, 100 + seed)
    if seed % 2:
        L, Rt = synth.noisy_variant(L, seed), synth.contrast_variant(Rt)
    else:
        L, Rt = L.astype(np.float32), Rt.astype(np.float32)
    return L, Rt, R, a, b


def ncc_random_case(seed):
    """(left, right, R, dmin, dmax) of test_ncc_restatement_matches_compiled_reference_random."""
    rng = np.random.default_rng(50 + seed)
    rows, cols = int(rng.integers(5, 20)), int(rng.integers(12, 60))
    R = int(rng.integers(0, 5))
    a, b = [(-14, 0), (0, 14), (-9, 0), (0, 5), (-6, 7), (-3, 0), (0, 21), (-30, 0)][seed]
    L, Rt, _ = synth.make_pair(rows, cols, 8, 300 + seed)
    if seed % 3 == 1:
        L, Rt = synth.noisy_variant(L, seed), synth.contrast_variant(Rt)
    elif seed % 3 == 2:
        L = L.astype(np.float32); L[2:9, 5:30] = 0          # zero-energy templates and windows: score 0, first candidate
        Rt = Rt.astype(np.float32); Rt[0:6, 10:40] = 0
    else:
        L, Rt = L.astype(np.float32), Rt.astype(np.float32)
    return L, Rt, R, a, b


def pair_range_images(rows, cols, rng, seed):
    L, Rt, _ = synth.make_pair(rows, cols, min(rng + 1, 32), seed + rows + cols)
    return L.astype(np.float32), Rt.astype(np.float32)


def _original(key, live, fn, *args):
    """The reference's own compiled code on one input: run live where oracle/_ref is built (and then the recorded output
    must agree with it), else the output recorded under `key` in tests/golden/ref_cases.npz."""
    rec = np.load(REF_CASES)[key]
    if not live:
        return rec
    out = fn(*args)
    assert np.array_equal(out, rec), f"tests/golden/ref_cases.npz [{key}] differs from the compiled reference"
    return out


@pytest.mark.parametrize("name,R,dmin,dmax", _cases("ssd"))
def test_ssd_restatement_matches_reference_golden(golden, name, R, dmin, dmax):
    g = golden.get("ssd", name)
    L, Rt = g["left"].astype(np.float32), g["right"].astype(np.float32)
    d_lit = oracle.ssd(L, Rt, R, dmin, dmax)
    d_fast = oracle.ssd_fast(L, Rt, R, dmin, dmax)
    assert np.array_equal(oracle.narrow_i8(d_lit), g["disp"])
    assert np.array_equal(d_lit, d_fast)


@pytest.mark.parametrize("name,R,dmin,dmax", _cases("ncc"))
def test_ncc_restatement_matches_opencv_golden(golden, name, R, dmin, dmax):
    g = golden.get("ncc", name)
    L, Rt = g["left"].astype(np.float32), g["right"].astype(np.float32)
    d, s = oracle.ncorr(L, Rt, R, dmin, dmax, return_score=True)
    assert np.array_equal(d, g["disp"].astype(np.int32))
    # tolerance: OpenCV's float32 numerator vs our exactly-rounded one (SURVEY.md §8c: <= 4.3e-7)
    np.testing.assert_allclose(s, g["score"], rtol=2e-6, atol=1e-7)


@pytest.mark.parametrize("seed", range(6))
def test_ssd_restatement_matches_compiled_reference_random(seed):
    L, Rt, R, a, b = ssd_random_case(seed)
    ref = _original(f"ssd_random/{seed}", oracle.have_ref(), oracle.ref_ssd, L, Rt, R, a, b)
    lit = oracle.ssd(L, Rt, R, a, b)
    assert np.array_equal(ref, oracle.narrow_i8(lit))
    assert np.array_equal(lit, oracle.ssd_fast(L, Rt, R, a, b))


@pytest.mark.parametrize("seed", range(8))
def test_ncc_restatement_matches_compiled_reference_random(seed):
    """The reference's own DisparityNCorr.cpp loop (compiled in place over the shim's matchTemplate) against the
    C restatement: search-rectangle clamping, result width, the `- (result.cols - 1)` rule of :67 for searches
    that end at the pixel, mixed-sign ranges, the char store."""
    L, Rt, R, a, b = ncc_random_case(seed)
    ref = _original(f"ncc_random/{seed}", oracle.have_ref_ncc(), oracle.ref_ncorr, L, Rt, R, a, b)
    lit = oracle.ncorr(L, Rt, R, a, b)
    assert np.array_equal(ref, oracle.narrow_i8(lit))


@pytest.mark.skipif(not oracle.have_ref_ncc(), reason="oracle/_ref/libref_ncc.so not built")
@pytest.mark.parametrize("name,R,dmin,dmax", _cases("ncc"))
def test_ncc_compiled_reference_matches_opencv_golden(golden, name, R, dmin, dmax):
    """Closes the loop: reference loop + shim arithmetic == the fixtures produced by EXECUTED OpenCV
    (cv2.matchTemplate / cv2.minMaxLoc inside a mirror of the same loop, tests/golden/make_golden.py)."""
    g = golden.get("ncc", name)
    if g["left"].size * (dmax - dmin + 1) > 3_000_000:
        pytest.skip("too large for the O(w^2) reference loop")
    L, Rt = g["left"].astype(np.float32), g["right"].astype(np.float32)
    ref = oracle.ref_ncorr(L, Rt, R, dmin, dmax)
    agree = float(np.mean(ref == oracle.narrow_i8(g["disp"])))
    assert agree >= 0.999, agree      # float32 DFT numerator (OpenCV) vs exactly rounded sum: near-ties may flip


def test_ncc_compiled_reference_throws_where_restatement_rejects():
    shape, R, a, b = NCC_EMPTY_CASE
    img = np.ones(shape, np.float32)
    if oracle.have_ref_ncc():
        with pytest.raises(oracle.OracleError):
            oracle.ref_ncorr(img, img, R, a, b)
    assert np.load(REF_CASES)["ncc_empty/throws"][0] == 1        # recorded: the reference threw on this case
    with pytest.raises(oracle.OracleError):
        oracle.ncorr(img, img, R, a, b)


@pytest.mark.parametrize("rows,cols,R,rng", SSD_PAIR_RANGES)
def test_ssd_restatement_matches_compiled_reference_on_pair_ranges(rows, cols, R, rng):
    """The mirrored ranges of the pair helpers (main.cpp:33,43) at the candidate counts the fused pair kernels take
    (64 / 128 / 256): the fast restatement the GPU tests compare against equals the reference's own compiled code, both
    directions - including the right-referenced map's candidates centred in the right padding (row-wrap reads, §A.1)
    and images narrower than the search range."""
    Lf, Rf = pair_range_images(rows, cols, rng, 400)
    key = f"ssd_pair/{rows}x{cols}_R{R}_{rng}"
    assert np.array_equal(_original(key + "/LR", oracle.have_ref(), oracle.ref_ssd, Lf, Rf, R, -rng, 0),
                          oracle.narrow_i8(oracle.ssd_fast(Lf, Rf, R, -rng, 0)))
    assert np.array_equal(_original(key + "/RL", oracle.have_ref(), oracle.ref_ssd, Rf, Lf, R, 0, rng),
                          oracle.narrow_i8(oracle.ssd_fast(Rf, Lf, R, 0, rng)))


@pytest.mark.parametrize("rows,cols,R,rng", NCC_PAIR_RANGES)
def test_ncc_fast_restatement_matches_compiled_reference_on_pair_ranges(rows, cols, R, rng):
    """The O(rows*cols*D) NCC restatement the GPU tests compare against, on the pair helpers' mirrored ranges, against
    the reference's own compiled loop (both directions; images narrower than the range clip the search strip)."""
    Lf, Rf = pair_range_images(rows, cols, rng, 500)
    key = f"ncc_pair/{rows}x{cols}_R{R}_{rng}"
    assert np.array_equal(_original(key + "/LR", oracle.have_ref_ncc(), oracle.ref_ncorr, Lf, Rf, R, -rng, 0),
                          oracle.narrow_i8(oracle.ncorr_fast(Lf, Rf, R, -rng, 0)))
    assert np.array_equal(_original(key + "/RL", oracle.have_ref_ncc(), oracle.ref_ncorr, Rf, Lf, R, 0, rng),
                          oracle.narrow_i8(oracle.ncorr_fast(Rf, Lf, R, 0, rng)))


def test_ssd_known_answer_shift():
    # right(x) = left(x + k)  =>  interior L->R disparity = -k   (SURVEY.md §8c KAT)
    rng = np.random.default_rng(3)
    left = rng.integers(0, 256, (24, 80)).astype(np.float32)
    k = 4
    right = np.empty_like(left)
    right[:, :-k] = left[:, k:]
    right[:, -k:] = left[:, -1:]
    d = oracle.ssd(left, right, 3, -10, 0)
    assert np.all(d[:, 14:-8] == -k)
    d2 = oracle.ncorr(left, right, 3, -10, 0)
    assert np.all(d2[:, 14:-8] == -k)


def test_ssd_tie_break_first_minimum_and_wrap_quirk():
    flat = np.full((10, 30), 7, np.float32)
    d, c = oracle.ssd(flat, flat, 2, -6, 0, return_cost=True)
    # interior rows: all candidates cost 0 -> the first (most negative) candidate wins (strict <).
    # Candidate centres may sit in the left padding: x + dmin clamped at padded column 0.
    for x in range(30):
        assert d[5, x] == max(-6, -(x + 2))
    assert np.all(c[1:] == 0)
    # row 0, left columns: the wrapped reads leave the buffer (zero guard) -> those candidates cost > 0
    assert d[0, 0] != d[5, 0]
    dr = oracle.ssd(flat, flat, 2, 0, 6)
    assert np.all(dr == 0)


def test_narrow_matches_char_store():
    v = np.array([0, -1, 127, 128, 255, -128, -129, 300], np.int32)
    assert oracle.narrow_i8(v).tolist() == [0, -1, 127, -128, -1, -128, 127, 44]


def test_ncc_rejects_empty_candidate_sets():
    img = np.ones((8, 16), np.float32)
    with pytest.raises(oracle.OracleError):
        oracle.ncorr(img, img, 1, 3, 5)     # right-most columns have no window: the reference would throw


@pytest.mark.parametrize("rows,cols,R,dmin,dmax", [(30, 90, 3, -20, 0), (30, 90, 3, 0, 20), (25, 70, 5, -7, 9),
                                                   (18, 60, 0, -5, 0), (24, 120, 7, -95, 0)])
def test_ncc_fast_restatement_equals_literal(rows, cols, R, dmin, dmax):
    L, Rt, _ = synth.make_pair(rows, cols, 16, rows + cols)
    Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
    d1, s1 = oracle.ncorr(Lf, Rf, R, dmin, dmax, return_score=True)
    d2, s2 = oracle.ncorr_fast(Lf, Rf, R, dmin, dmax, return_score=True)
    assert np.array_equal(d1, d2) and np.array_equal(s1, s2)
