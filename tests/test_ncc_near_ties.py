"""NCC maps checked pixel by pixel against the oracle (tests/ncc_check.py) where no other test reaches: every pair entry point
fused and unfused on 8-bit and float images, the full-size configurations, and images built to stress the key scales (a dark
stripe next to a bright one, mixed-sign values, a DC offset at the edge of the float family's admission band, ranges wider than
the image) and the float running sums (the longest row segment a launch can give a CTA).  Needs a B200.

Every disparity that differs from the oracle's must name a candidate whose oracle score is within the key resolution of the
oracle's winner; the returned score of single-direction calls is the oracle's score of the returned candidate, bit for bit."""
import ctypes as C

import numpy as np
import pytest

import oracle
import ncc_check as nc
import introtocomputervision_b200 as sb
from introtocomputervision_b200 import _capi, synth
from pair_calls import FAMILIES, RANGE_T, _images, _run, _set_fuse

pytestmark = pytest.mark.gpu

ENTRIES = ["pair_host", "pair_device", "batch_device", "batch_host", "band_host", "band_halo_device", "mgpu_batch", "mgpu_bands"]


@pytest.fixture(scope="module")
def mg():
    n = _capi.lib().stereo_device_count()
    with sb.MultiGpu([0, 1] if n >= 2 else [0, 0]) as m:
        yield m


def _plan_segment(rows, cols, R, rng, f32):
    """Longest row segment a CTA walks in the hot-kernel launch of one unfused NCC pair (stereo_launch_plan)."""
    p = _capi.LaunchPlan()
    assert _capi.lib().stereo_launch_plan(sb.COST_NCORR, int(f32), 1, rows, cols, R, rng, 0, 148, C.byref(p)) == 0
    return min(p.rows_per_item, rows)


def _family(kind, fuse, entry):
    if kind == "noisy":
        return "f32"                          # float operands: never fused
    if entry.startswith("mgpu_"):
        return "u8"                           # per-device contexts: the per-strip tolerance covers fused and unfused
    return "u8_fused" if fuse else "u8"


def _check_pair_maps(dl, dr, Ls, Rs, R, rng, family, what):
    for i in range(len(Ls)):
        a, b = Ls[i].astype(np.float32), Rs[i].astype(np.float32)
        nc.check_ncc_map(dl[i], a, b, R, -rng, 0, family, what=f"{what} pair {i} L->R")
        nc.check_ncc_map(dr[i], b, a, R, 0, rng, family, what=f"{what} pair {i} R->L")


# ---- every pair entry point, fused and unfused, 8-bit and float images -------------------------------------------------

@pytest.mark.parametrize("family", list(FAMILIES))
@pytest.mark.parametrize("fuse", [True, False])
@pytest.mark.parametrize("entry", ENTRIES)
def test_every_pair_entry_point_ncc_per_pixel(ctx, mg, entry, fuse, family):
    kind, win, dt = FAMILIES[family]
    if kind != "u8" and entry in ("batch_device", "band_halo_device"):
        pytest.skip("8-bit device entry point")
    if kind == "noisy" and entry == "band_host":
        pytest.skip("the host row-band entry points take 8-bit-valued images only")
    h = mg if entry.startswith("mgpu_") else ctx
    n = 3 if "batch" in entry else 1
    Ls, Rs = _images(kind, n, 800 + 7 * ENTRIES.index(entry))
    _set_fuse(h, fuse)
    try:
        dl, dr = _run(h, entry, sb.COST_NCORR, Ls, Rs, win, RANGE_T, dt)
        if not entry.startswith("mgpu_"):
            want = sb.PATH_EXACT_F32 if win > 7 else sb.PATH_FAST_F32 if kind == "noisy" else sb.PATH_FAST_U8
            assert ctx.last_path == want
            if want == sb.PATH_FAST_U8 and entry not in ("band_host", "band_halo_device"):
                assert (ctx.last_fused_pairs > 0) == fuse
    finally:
        _set_fuse(h, True)
    fam = "exact" if win > 7 else _family(kind, fuse, entry)
    _check_pair_maps(dl, dr, Ls, Rs, win, RANGE_T, fam, f"{entry} fuse={fuse} {family}")


# ---- full size ---------------------------------------------------------------------------------------------------------

def test_config3_single_call_returned_score_and_pair(ctx):
    """1920x1080, 128 disparities, 9x9: the single call's returned score at EVERY pixel is the oracle's score of the
    returned candidate, bit for bit; both maps of the fused pair pixel by pixel."""
    L, Rt, _ = synth.make_pair(1080, 1920, 128, 1001)
    Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
    d_ref = oracle.ncorr_fast(Lf, Rf, 4, -127, 0)
    d, s = ctx.disparity(sb.COST_NCORR, L, Rt, 4, -127, 0, dtype=np.int16, return_best=True)
    assert ctx.last_path == sb.PATH_FAST_U8 and ctx.last_fused_pairs == 0
    st = nc.check_ncc_map(d, Lf, Rf, 4, -127, 0, "u8", oracle_disp=d_ref, what="1080p single")
    print(f"1080p/128 single (u8): {st}")
    nc.check_best(s, d, Lf, Rf, 4, -127, 0, what="1080p single")
    dl, dr = ctx.disparity_pair(sb.COST_NCORR, L, Rt, 4, 127, dtype=np.int16)
    assert ctx.last_fused_pairs >= 1                  # (one per row band of the host pipeline)
    st = nc.check_ncc_map(dl, Lf, Rf, 4, -127, 0, "u8_fused", oracle_disp=d_ref, what="1080p pair L->R")
    print(f"1080p/128 pair L->R (u8_fused): {st}")
    nc.check_ncc_map(dr, Rf, Lf, 4, 0, 127, "u8_fused", what="1080p pair R->L")


def test_config5_shape_batch_of_16(ctx):
    """1280x720, 64 disparities, 9x9, 16 pairs in one device batch (one launch sequence): the first, a middle and the last
    pair pixel by pixel."""
    n = 16
    Ls, Rs = zip(*[synth.make_pair(720, 1280, 64, 2000 + i)[:2] for i in range(n)])
    Ls, Rs = np.stack(Ls), np.stack(Rs)
    dl, dr = _run(ctx, "batch_device", sb.COST_NCORR, Ls, Rs, 4, 63, np.int8)
    assert ctx.last_path == sb.PATH_FAST_U8 and ctx.last_fused_pairs == n
    idx = [0, 7, 15]
    _check_pair_maps(dl[idx], dr[idx], Ls[idx], Rs[idx], 4, 63, "u8_fused", "720p x16")


@pytest.mark.parametrize("rows,rng,seed", [(511, 95, 11), (529, 80, 12)])
def test_reference_problems_clean_noisy_contrast(ctx, rows, rng, seed):
    """The reference's NCC problems (511x640 / 529x640, R = 7, ranges 95 and 80) through the pair call: clean images on the
    fused packed kernels, noise sigma 10 and x1.1 contrast on the float kernels (unfused pairs)."""
    R, cols = 7, 640
    L, Rt, _ = synth.make_pair(rows, cols, rng + 1, seed)
    for name, a, b in (("clean", L.astype(np.float32), Rt.astype(np.float32)),
                       ("noisy", synth.noisy_variant(L, seed + 1), synth.noisy_variant(Rt, seed + 2)),
                       ("contrast", synth.contrast_variant(L), Rt.astype(np.float32))):
        dl, dr = ctx.disparity_pair(sb.COST_NCORR, a, b, R, rng, dtype=np.int16)
        family = nc.family_of(ctx)
        assert family == ("u8_fused" if name == "clean" else "f32"), (name, family)
        seg = _plan_segment(rows, cols, R, rng, family == "f32")
        for got, x, y, lo, hi, side in ((dl, a, b, -rng, 0, "L->R"), (dr, b, a, 0, rng, "R->L")):
            st = nc.check_ncc_map(got, x, y, R, lo, hi, family, seg_rows=seg, what=f"{name} {side}")
            print(f"{rows}x{cols}/{rng} {name} {side} ({family}): {st}")


# ---- adversarial images ------------------------------------------------------------------------------------------------

def _single_and_pairs(ctx, a, b, R, rng, what, seg=None, min_agree=nc.NCC_DISP_AGREE):
    """Single L->R call (with the returned score), then the pair call fused and unfused, all pixel by pixel."""
    af, bf = np.asarray(a, np.float32), np.asarray(b, np.float32)
    d_ref = oracle.ncorr_fast(af, bf, R, -rng, 0)
    r_ref = oracle.ncorr_fast(bf, af, R, 0, rng)
    d, s = ctx.disparity(sb.COST_NCORR, a, b, R, -rng, 0, dtype=np.int16, return_best=True)
    fam = nc.family_of(ctx)
    st = nc.check_ncc_map(d, af, bf, R, -rng, 0, fam, oracle_disp=d_ref, seg_rows=seg, min_agree=min_agree, what=f"{what} single")
    print(f"{what} single ({fam}): {st}")
    nc.check_best(s, d, af, bf, R, -rng, 0, what=f"{what} single")
    try:
        for fuse in (True, False):
            ctx.set_fuse_pairs(fuse)
            dl, dr = ctx.disparity_pair(sb.COST_NCORR, a, b, R, rng, dtype=np.int16)
            fam = nc.family_of(ctx)
            for got, x, y, lo, hi, ref_d, side in ((dl, af, bf, -rng, 0, d_ref, "L->R"), (dr, bf, af, 0, rng, r_ref, "R->L")):
                st = nc.check_ncc_map(got, x, y, R, lo, hi, fam, oracle_disp=ref_d, seg_rows=seg, min_agree=min_agree,
                                      what=f"{what} pair fuse={fuse} {side}")
                print(f"{what} pair fuse={fuse} {side} ({fam}): {st}")
    finally:
        ctx.set_fuse_pairs(True)
    return fam


def test_dark_stripe_next_to_a_bright_one(ctx):
    """Textured rows whose dark stripes (values / 16, 4..40 pixels wide) sit next to bright ones: the unfused kernels' strip
    row shares the bright window's key scale, so the dark pixels' keys hold up to 2^4 fewer value bits."""
    rows, cols, R, rng = 48, 480, 4, 63
    L, Rt, _ = synth.make_pair(rows, cols, 64, 73000)
    L, Rt = L.astype(np.int32), Rt.astype(np.int32)
    x = np.arange(cols)
    dark = ((x // 24) % 3 == 1) & (x % 24 < 4 + (x // 72) % 5 * 5)
    L[:, dark] //= 16
    Rt[:, dark] //= 16
    assert _single_and_pairs(ctx, L.astype(np.uint8), Rt.astype(np.uint8), R, rng, "dark stripes") == "u8"


def test_mixed_sign_float_images(ctx):
    rows, cols, R, rng = 40, 300, 3, 47
    L, Rt, _ = synth.make_pair(rows, cols, 48, 73100)
    a = synth.noisy_variant(L, 1) - np.float32(127.5)
    b = synth.noisy_variant(Rt, 2) - np.float32(127.5)
    assert a.min() < 0 < a.max()
    assert _single_and_pairs(ctx, a, b, R, rng, "mixed sign") == "f32"


def test_offset_just_inside_the_float_admission_band(ctx):
    """A DC offset with (hi - lo)^2 / (lo^2 + hi^2) just above 2^-4 (the least band the float NCC family admits), plus noise:
    every score crowds towards 1 and the candidates' gaps are as small as that family ever sees."""
    rows, cols, R, rng = 36, 260, 3, 40
    L, Rt, _ = synth.make_pair(rows, cols, rng + 1, 73200)
    a0, b0 = synth.noisy_variant(L, 3, sigma=2.0), synth.noisy_variant(Rt, 4, sigma=2.0)
    lo, hi = float(min(a0.min(), b0.min())), float(max(a0.max(), b0.max()))
    # largest offset t with band(lo + t, hi + t) >= 2^-4 (the band shrinks as t grows): bisection
    t0, t1 = 0.0, 1e4
    for _ in range(80):
        tm = 0.5 * (t0 + t1)
        t0, t1 = (tm, t1) if (hi - lo) ** 2 / ((lo + tm) ** 2 + (hi + tm) ** 2) >= 1 / 16 else (t0, tm)
    off = np.float32(t0 * (1 - 1e-4))
    a, b = a0 + off, b0 + off
    band = ((float(max(a.max(), b.max())) - float(min(a.min(), b.min()))) ** 2
            / (float(min(a.min(), b.min())) ** 2 + float(max(a.max(), b.max())) ** 2))
    assert 1 / 16 <= band < 1 / 16 * 1.01, band
    assert _single_and_pairs(ctx, a, b, R, rng, "offset band") == "f32"


@pytest.mark.parametrize("dmin,dmax", [(-300, 0), (0, 300), (-150, 200), (-37, 0), (0, 37), (-9, 5), (-1, 130)])
def test_ranges_at_and_beyond_the_borders(ctx, dmin, dmax):
    """Right-aligned, left-aligned and mixed ranges, some wider than the image: the candidate sets clipped at both borders
    and the alignment rule of DisparityNCorr.cpp:67, on 8-bit and float images."""
    rows, cols, R = 22, 120, 3
    L, Rt, _ = synth.make_pair(rows, cols, 30, 73300 + dmax - dmin)
    for a, b, fam in ((L, Rt, "u8"), (synth.noisy_variant(L, 5), synth.noisy_variant(Rt, 6), "f32")):
        af, bf = np.asarray(a, np.float32), np.asarray(b, np.float32)
        d_ref = oracle.ncorr(af, bf, R, dmin, dmax)
        d, s = ctx.disparity(sb.COST_NCORR, a, b, R, dmin, dmax, dtype=np.int16, return_best=True)
        assert nc.family_of(ctx) == fam
        nc.check_ncc_map(d, af, bf, R, dmin, dmax, fam, oracle_disp=d_ref, what=f"[{dmin}, {dmax}]")
        nc.check_best(s, d, af, bf, R, dmin, dmax, what=f"[{dmin}, {dmax}]")


def test_float_running_sums_over_the_longest_segment(ctx):
    """A noisy float pair whose shape makes the hot kernel walk its longest row segments (stereo_launch_plan: a linear split
    of 64 tiles of 4000 rows; > 1700 rows per CTA without a restart of the float32 column sums).  The per-pixel check holds
    with the drift bound of that segment; the statistics show how far the gaps really get beyond the key term alone."""
    rows, cols, R, rng = 4000, 4096, 7, 31
    seg = _plan_segment(rows, cols, R, rng, True)
    assert seg > 1700, seg
    L, Rt, _ = synth.make_pair(rows, cols, rng + 1, 73400)
    a, b = synth.noisy_variant(L, 7), synth.noisy_variant(Rt, 8)
    dl, dr = _run(ctx, "pair_device", sb.COST_NCORR, a[None], b[None], R, rng, np.int16)
    assert ctx.last_path == sb.PATH_FAST_F32 and ctx.last_fused_pairs == 0
    for got, x, y, lo, hi, side in ((dl[0], a, b, -rng, 0, "L->R"), (dr[0], b, a, 0, rng, "R->L")):
        st = nc.check_ncc_map(got, x, y, R, lo, hi, "f32", seg_rows=seg, what=f"longest segment {side}")
        print(f"{rows}x{cols}/{rng} R={R} noisy, segment {seg} rows, {side} (f32): {st}")
