"""GPU parity tests: the CUDA path, called through the C ABI, against the oracle on the same inputs.

SSD: bit-exact disparities (and costs).  NCC: winning score within 1e-5 relative and disparity equal
on >= 99.9 % of pixels (BASELINE.json north_star); every pixel that differs names a candidate whose oracle score is within
the key resolution of the oracle's winner (tests/ncc_check.py), and the exact path is identical.
"""
import numpy as np
import pytest

import oracle
import ncc_check as nc
import introtocomputervision_b200 as sb
from introtocomputervision_b200 import synth

pytestmark = pytest.mark.gpu

NCC_SCORE_RTOL = 1e-5      # BASELINE.json: "NCC scores must agree within 1e-5 relative"
NCC_DISP_AGREE = 0.999     # "... disparity agreement on >= 99.9 % of pixels"


def _cases(cost):
    from conftest import Golden
    return Golden().names(cost)


def assert_ncc_close(d, s, d_ref, s_ref, ref, tgt, R, dmin, dmax, family, min_agree=NCC_DISP_AGREE):
    """Per-pixel check of the map against the oracle's (ncc_check), the north-star fraction, the scores within 1e-5, and where
    the disparity differs the returned score is the oracle's score of the returned candidate, bit for bit."""
    nc.check_ncc_map(d, ref, tgt, R, dmin, dmax, family, oracle_disp=d_ref, min_agree=min_agree)
    np.testing.assert_allclose(s, s_ref, rtol=NCC_SCORE_RTOL, atol=1e-7)
    nc.check_best(s, d, ref, tgt, R, dmin, dmax, mask=d != d_ref)


# ---- golden vectors (reference-generated) ----------------------------------------------------------

@pytest.mark.parametrize("name,R,dmin,dmax", _cases("ssd"))
def test_ssd_golden(ctx, golden, name, R, dmin, dmax):
    g = golden.get("ssd", name)
    L, Rt = g["left"], g["right"]
    d = ctx.disparity(sb.COST_SSD, L.astype(np.float32), Rt.astype(np.float32), R, dmin, dmax)
    assert d.dtype == np.int8 and np.array_equal(d, g["disp"])
    if L.dtype == np.uint8:
        d8 = ctx.disparity(sb.COST_SSD, L, Rt, R, dmin, dmax)
        assert np.array_equal(d8, g["disp"])


@pytest.mark.parametrize("name,R,dmin,dmax", _cases("ncc"))
def test_ncc_golden(ctx, golden, name, R, dmin, dmax):
    g = golden.get("ncc", name)
    L, Rt = g["left"], g["right"]
    Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
    d, s = ctx.disparity(sb.COST_NCORR, Lf, Rf, R, dmin, dmax, dtype=np.int16, return_best=True)
    assert_ncc_close(d, s, g["disp"], g["score"], Lf, Rf, R, dmin, dmax, nc.family_of(ctx))
    if L.dtype == np.uint8:
        d8, s8 = ctx.disparity(sb.COST_NCORR, L, Rt, R, dmin, dmax, dtype=np.int16, return_best=True)
        assert_ncc_close(d8, s8, g["disp"], g["score"], Lf, Rf, R, dmin, dmax, nc.family_of(ctx))


# ---- seeded random inputs against the oracle ----------------------------------------------------------

@pytest.mark.parametrize("seed", range(10))
def test_ssd_random_vs_oracle(ctx, seed):
    rng = np.random.default_rng(1000 + seed)
    rows, cols = int(rng.integers(5, 70)), int(rng.integers(8, 200))
    R = int(rng.integers(0, 8))
    a, b = sorted(int(v) for v in rng.integers(-40, 41, 2))
    L, Rt, _ = synth.make_pair(rows, cols, 30, seed)
    kind = seed % 3
    if kind == 0:
        Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
    elif kind == 1:
        Lf, Rf = synth.noisy_variant(L, seed), synth.noisy_variant(Rt, seed + 1)
    else:
        Lf, Rf = synth.contrast_variant(L), Rt.astype(np.float32)
    d_ref, c_ref = oracle.ssd(Lf, Rf, R, a, b, return_cost=True)
    d, c = ctx.disparity(sb.COST_SSD, Lf, Rf, R, a, b, dtype=np.int32, return_best=True)
    assert np.array_equal(d, d_ref)
    assert np.array_equal(c, c_ref)
    d8 = ctx.disparity(sb.COST_SSD, Lf, Rf, R, a, b, dtype=np.int8)
    assert np.array_equal(d8, oracle.narrow_i8(d_ref))


@pytest.mark.parametrize("seed", range(6))
def test_ncc_random_vs_oracle(ctx, seed):
    rng = np.random.default_rng(2000 + seed)
    rows, cols = int(rng.integers(5, 40)), int(rng.integers(20, 160))
    R = int(rng.integers(0, 8))
    rng_d = int(rng.integers(0, 40))
    dmin, dmax = (-rng_d, 0) if seed % 2 == 0 else (0, rng_d)
    L, Rt, _ = synth.make_pair(rows, cols, 30, 50 + seed)
    if seed % 3 == 1:
        Lf, Rf = synth.noisy_variant(L, seed), synth.noisy_variant(Rt, seed + 1)
    else:
        Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
    d_ref, s_ref = oracle.ncorr(Lf, Rf, R, dmin, dmax, return_score=True)
    d, s = ctx.disparity(sb.COST_NCORR, Lf, Rf, R, dmin, dmax, dtype=np.int32, return_best=True)
    assert_ncc_close(d, s, d_ref, s_ref, Lf, Rf, R, dmin, dmax, nc.family_of(ctx))


# ---- BASELINE config shapes ------------------------------------------------------------------------------

def test_ssd_pair1_shape_vs_oracle(ctx):
    # config 1/2 stand-in: 511 x 640, R=7, range=95 (config/ps2.yaml:24-26); both directions
    L, Rt, _ = synth.make_pair(511, 640, 96, 11)
    Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
    dl, dr = sb.disparitySSDPair(Lf, Rf, sb.DisparityConfig(7, 95), ctx=ctx)
    assert np.array_equal(dl, oracle.narrow_i8(oracle.ssd_fast(Lf, Rf, 7, -95, 0)))
    assert np.array_equal(dr, oracle.narrow_i8(oracle.ssd_fast(Rf, Lf, 7, 0, 95)))


def test_ssd_noisy_contrast_variants_vs_oracle(ctx):
    # BASELINE config 2 family on a band of the pair1 stand-in: Gaussian noise and x1.1 contrast
    L, Rt, _ = synth.make_pair(96, 640, 96, 11)
    for Lf, Rf in ((synth.noisy_variant(L, 12), synth.noisy_variant(Rt, 13)),
                   (synth.contrast_variant(L), Rt.astype(np.float32))):
        dl, dr = sb.disparitySSDPair(Lf, Rf, sb.DisparityConfig(7, 95), ctx=ctx)
        assert ctx.last_path == sb.PATH_FAST_F32 and ctx.last_fused_pairs == 1
        assert np.array_equal(dl, oracle.narrow_i8(oracle.ssd_fast(Lf, Rf, 7, -95, 0)))
        assert np.array_equal(dr, oracle.narrow_i8(oracle.ssd_fast(Rf, Lf, 7, 0, 95)))


def test_ncc_pair1_band_variants_vs_oracle(ctx):
    L, Rt, _ = synth.make_pair(48, 640, 96, 11)
    for Lf, Rf in ((L.astype(np.float32), Rt.astype(np.float32)),
                   (synth.noisy_variant(L, 12), synth.noisy_variant(Rt, 13)),
                   (synth.contrast_variant(L), Rt.astype(np.float32))):
        for (a, b, dmin, dmax) in ((Lf, Rf, -95, 0), (Rf, Lf, 0, 95)):
            d_ref, s_ref = oracle.ncorr(a, b, 7, dmin, dmax, return_score=True)
            d, s = ctx.disparity(sb.COST_NCORR, a, b, 7, dmin, dmax, dtype=np.int16, return_best=True)
            assert_ncc_close(d, s, d_ref, s_ref, a, b, 7, dmin, dmax, nc.family_of(ctx))


# ---- API behaviour ------------------------------------------------------------------------------------------

def test_pair_equals_two_singles_and_batch_equals_pairs(ctx):
    n = 3
    Ls, Rs = [], []
    for i in range(n):
        L, Rt, _ = synth.make_pair(40, 96, 16, 300 + i)
        Ls.append(L), Rs.append(Rt)
    Ls, Rs = np.stack(Ls), np.stack(Rs)
    for cost in (sb.COST_SSD, sb.COST_NCORR):
        bl, br = ctx.disparity_pair_batch(cost, Ls, Rs, 3, 15)
        for i in range(n):
            dl, dr = ctx.disparity_pair(cost, Ls[i], Rs[i], 3, 15)
            assert np.array_equal(dl, ctx.disparity(cost, Ls[i], Rs[i], 3, -15, 0))
            assert np.array_equal(dr, ctx.disparity(cost, Rs[i], Ls[i], 3, 0, 15))
            assert np.array_equal(bl[i], dl) and np.array_equal(br[i], dr)


@pytest.mark.parametrize("n,rng,R", [(5, 63, 4), (9, 40, 2), (6, 150, 5), (4, 127, 7), (17, 30, 1), (33, 20, 3)])
def test_device_batch_launch_chunks_vs_oracle(ctx, n, rng, R):
    """Device batches share launch sequences (up to 32 directions each): chunk boundaries (16+1, 16+16+1 pairs),
    2-strips-per-warp kernels (<= 64 candidates), one and two 128-disparity groups — all against the oracle."""
    import torch
    from introtocomputervision_b200 import _capi
    import ctypes as C
    rows, cols = 45, 250
    Ls, Rs = [], []
    for i in range(n):
        L, Rt, _ = synth.make_pair(rows, cols, min(64, rng), 900 + 17 * i + n)
        Ls.append(L), Rs.append(Rt)
    Ls, Rs = np.stack(Ls), np.stack(Rs)
    dl_, dr_ = torch.from_numpy(Ls).cuda(), torch.from_numpy(Rs).cuda()
    for cost in (sb.COST_SSD, sb.COST_NCORR):
        ol = torch.zeros((n, rows, cols), dtype=torch.int16, device="cuda")
        orr = torch.zeros_like(ol)
        rc = _capi.lib().stereo_disparity_pair_batch_u8_device(
            ctx.handle, cost, n, dl_.data_ptr(), dr_.data_ptr(), cols, rows * cols, rows, cols, R, rng,
            ol.data_ptr(), orr.data_ptr(), cols * 2, rows * cols * 2, 2, None)
        assert rc == 0, _capi.last_error()
        ctx.synchronize()
        assert ctx.last_path == sb.PATH_FAST_U8
        family = nc.family_of(ctx)
        bl, br = ol.cpu().numpy(), orr.cpu().numpy()
        for i in range(n):
            Lf, Rf = Ls[i].astype(np.float32), Rs[i].astype(np.float32)
            if cost == sb.COST_SSD:
                assert np.array_equal(bl[i], oracle.ssd_fast(Lf, Rf, R, -rng, 0)), f"pair {i} L->R"
                assert np.array_equal(br[i], oracle.ssd_fast(Rf, Lf, R, 0, rng)), f"pair {i} R->L"
            else:
                nc.check_ncc_map(bl[i], Lf, Rf, R, -rng, 0, family, what=f"pair {i} L->R")
                nc.check_ncc_map(br[i], Rf, Lf, R, 0, rng, family, what=f"pair {i} R->L")


def test_config5_shape_batch_pairs_vs_oracle(ctx):
    """BASELINE config 5's shape (1280x720, 64 disparities, 9x9) on a few pairs: the 2-strips-per-warp kernels."""
    n = 3
    Ls, Rs = [], []
    for i in range(n):
        L, Rt, _ = synth.make_pair(720, 1280, 64, 2000 + i)
        Ls.append(L), Rs.append(Rt)
    Ls, Rs = np.stack(Ls), np.stack(Rs)
    bl, br = ctx.disparity_pair_batch(sb.COST_SSD, Ls, Rs, 4, 63)
    for i in range(n):
        Lf, Rf = Ls[i].astype(np.float32), Rs[i].astype(np.float32)
        assert np.array_equal(bl[i], oracle.narrow_i8(oracle.ssd_fast(Lf, Rf, 4, -63, 0)))
        assert np.array_equal(br[i], oracle.narrow_i8(oracle.ssd_fast(Rf, Lf, 4, 0, 63)))
    nl, nr = ctx.disparity_pair_batch(sb.COST_NCORR, Ls[:1], Rs[:1], 4, 63)
    family = nc.family_of(ctx)
    Lf, Rf = Ls[0].astype(np.float32), Rs[0].astype(np.float32)
    nc.check_ncc_map(nl[0], Lf, Rf, 4, -63, 0, family, what="L->R")
    nc.check_ncc_map(nr[0], Rf, Lf, 4, 0, 63, family, what="R->L")


def test_wide_disparity_needs_wide_output(ctx):
    # > 127 disparities: int16 holds the true value, int8 wraps exactly like the reference's char store
    L, Rt, _ = synth.make_pair(16, 400, 200, 77)
    Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
    d_ref = oracle.ssd_fast(Lf, Rf, 2, -200, 0)
    assert d_ref.min() < -128
    assert np.array_equal(ctx.disparity(sb.COST_SSD, Lf, Rf, 2, -200, 0, dtype=np.int16), d_ref.astype(np.int16))
    assert np.array_equal(ctx.disparity(sb.COST_SSD, Lf, Rf, 2, -200, 0, dtype=np.int8), oracle.narrow_i8(d_ref))


def test_error_codes(ctx):
    img = np.zeros((8, 16), np.float32)
    with pytest.raises(sb.StereoError) as e:
        ctx.disparity(sb.COST_SSD, img, img, 1, 3, 1)
    assert e.value.status == -2
    with pytest.raises(sb.StereoError) as e:
        ctx.disparity(sb.COST_NCORR, img, img, 1, 3, 5)      # the reference would throw in cv::Mat(Rect)
    assert e.value.status == -2
    with pytest.raises(sb.StereoError) as e:
        ctx.disparity(sb.COST_SSD, img, img, -1, -3, 0)
    assert e.value.status == -1
    # strided (non-contiguous rows) inputs are honoured
    big = np.random.default_rng(0).integers(0, 255, (12, 64)).astype(np.float32)
    a, b = big[:, 3:43], big[:, 10:50]
    assert np.array_equal(ctx.disparity(sb.COST_SSD, a, b, 2, -5, 0, dtype=np.int32),
                          oracle.ssd(np.ascontiguousarray(a), np.ascontiguousarray(b), 2, -5, 0))


def test_device_pointer_and_band_entry_points(ctx):
    import ctypes as C
    import torch
    from introtocomputervision_b200 import _capi
    lib = _capi.lib()
    L, Rt, _ = synth.make_pair(70, 130, 20, 9)
    dl = torch.from_numpy(L).cuda()
    dr = torch.from_numpy(Rt).cuda()
    full = torch.empty((70, 130), dtype=torch.int16, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    for cost, fn in ((sb.COST_SSD, oracle.ssd), (sb.COST_NCORR, oracle.ncorr)):
        for (a, b, dmin, dmax) in ((dl, dr, -19, 0), (dr, dl, 0, 19)):
            rc = lib.stereo_disparity_u8_device(ctx.handle, cost, a.data_ptr(), 130, b.data_ptr(), 130, 70, 130, 4, dmin, dmax,
                                                full.data_ptr(), 260, 2, None, 0, C.c_void_p(st))
            assert rc == 0, _capi.last_error()
            ctx.synchronize(st)
            ref = fn(a.cpu().numpy().astype(np.float32), b.cpu().numpy().astype(np.float32), 4, dmin, dmax)
            if cost == sb.COST_SSD:
                assert np.array_equal(full.cpu().numpy(), ref.astype(np.int16))
            else:
                nc.check_ncc_map(full.cpu().numpy(), a.cpu().numpy(), b.cpu().numpy(), 4, dmin, dmax, nc.family_of(ctx), oracle_disp=ref)
                ref = full.cpu().numpy().astype(np.int32)        # bands must reproduce the full call exactly
            # row bands (with the R+1 halo the SSD wrap quirk needs) reproduce the same rows
            for (r0, r1) in ((0, 23), (23, 47), (47, 70)):
                band = torch.empty((r1 - r0, 130), dtype=torch.int16, device="cuda")
                rc = lib.stereo_disparity_band_u8_device(ctx.handle, cost, a.data_ptr(), 130, b.data_ptr(), 130, 70, 130, r0, r1,
                                                         4, dmin, dmax, band.data_ptr(), 260, 2, C.c_void_p(st))
                assert rc == 0, _capi.last_error()
                ctx.synchronize(st)
                assert np.array_equal(band.cpu().numpy(), ref[r0:r1].astype(np.int16))


# ---- pipelined host entry points (row bands through upload / compute / download streams) --------------

@pytest.mark.parametrize("bands", [1, 2, 3, 7])
def test_pipelined_host_bands_vs_oracle(ctx, bands):
    L, Rt, _ = synth.make_pair(101, 300, 40, 900 + bands)
    Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
    ref_l = oracle.ssd_fast(Lf, Rf, 5, -39, 0)
    ref_r = oracle.ssd_fast(Rf, Lf, 5, 0, 39)
    try:
        ctx.set_pipe_bands(bands)
        for a, b in ((Lf, Rf), (L, Rt)):                       # CV_32FC1 like the reference, and u8
            dl, dr = ctx.disparity_pair(sb.COST_SSD, a, b, 5, 39, dtype=np.int16)
            assert ctx.last_path == sb.PATH_FAST_U8
            assert np.array_equal(dl, ref_l) and np.array_equal(dr, ref_r)
        # single direction, R->L (the SSD row wrap reads the NEXT row there: band seams need the +1 halo row)
        assert np.array_equal(ctx.disparity(sb.COST_SSD, Rf, Lf, 5, 0, 39, dtype=np.int16), ref_r)
        # NCC: banded result == whole-image result, and close to the oracle
        dn = ctx.disparity(sb.COST_NCORR, Lf, Rf, 5, -39, 0, dtype=np.int16)
        family = nc.family_of(ctx)
        ctx.set_pipe_bands(1)
        assert np.array_equal(dn, ctx.disparity(sb.COST_NCORR, Lf, Rf, 5, -39, 0, dtype=np.int16))
        nc.check_ncc_map(dn, Lf, Rf, 5, -39, 0, family)
    finally:
        ctx.set_pipe_bands(0)


@pytest.mark.parametrize("bands", [0, 2])
def test_pipelined_batch_reuses_device_slots(ctx, bands):
    # 7 pairs through 3 device slots: every slot is overwritten at least once while its predecessor downloads
    n = 7
    Ls, Rs = [], []
    for i in range(n):
        L, Rt, _ = synth.make_pair(45, 150, 24, 700 + i)
        Ls.append(L), Rs.append(Rt)
    Ls, Rs = np.stack(Ls), np.stack(Rs)
    try:
        ctx.set_pipe_bands(bands)
        bl, br = ctx.disparity_pair_batch(sb.COST_SSD, Ls, Rs, 4, 23, dtype=np.int8)
    finally:
        ctx.set_pipe_bands(0)
    for i in range(n):
        Lf, Rf = Ls[i].astype(np.float32), Rs[i].astype(np.float32)
        assert np.array_equal(bl[i], oracle.narrow_i8(oracle.ssd_fast(Lf, Rf, 4, -23, 0))), i
        assert np.array_equal(br[i], oracle.narrow_i8(oracle.ssd_fast(Rf, Lf, 4, 0, 23))), i


@pytest.mark.parametrize("n,kind", [(13, np.float32), (13, np.uint8), (6, np.float32), (2, np.float32)])
def test_host_batch_chunked_items_vs_oracle(ctx, n, kind):
    """Host batches of small images ride several pairs per pipeline item (13 pairs -> items of 4+4+4+1 pairs, 8
    directions per launch sequence; 6 pairs -> items of 2), CV_32FC1 and uint8 inputs, SSD and NCC."""
    rows, cols, R, rng = 37, 130, 3, 21
    Ls, Rs = [], []
    for i in range(n):
        L, Rt, _ = synth.make_pair(rows, cols, 16, 5100 + 3 * i + n)
        Ls.append(L), Rs.append(Rt)
    Ls, Rs = np.stack(Ls).astype(kind), np.stack(Rs).astype(kind)
    for cost in (sb.COST_SSD, sb.COST_NCORR):
        bl, br = ctx.disparity_pair_batch(cost, Ls, Rs, R, rng, dtype=np.int16)
        assert ctx.last_path == sb.PATH_FAST_U8
        family = nc.family_of(ctx)
        for i in range(n):
            Lf, Rf = Ls[i].astype(np.float32), Rs[i].astype(np.float32)
            if cost == sb.COST_SSD:
                assert np.array_equal(bl[i], oracle.ssd_fast(Lf, Rf, R, -rng, 0)), f"pair {i} L->R"
                assert np.array_equal(br[i], oracle.ssd_fast(Rf, Lf, R, 0, rng)), f"pair {i} R->L"
            else:
                nc.check_ncc_map(bl[i], Lf, Rf, R, -rng, 0, family, what=f"pair {i} L->R")
                nc.check_ncc_map(br[i], Rf, Lf, R, 0, rng, family, what=f"pair {i} R->L")


@pytest.mark.parametrize("n,kind", [(3, np.float32), (3, np.uint8), (1, np.float32), (2, np.uint8)])
def test_host_batch_uneven_bands_of_large_images_vs_oracle(ctx, n, kind):
    """4K-sized images (>= 1024 rows, >= 4 Mpix) are cut unevenly by the host pipeline: the call's first item begins and its
    last item ends with an eighth of the image, whole images in between (one pair: five bands), uploads in quarter-image
    chunks.  Every seam against the oracle, CV_32FC1 (host-converted) and uint8 inputs, plus a pixel that is not 8-bit
    inside the LAST band of the last pair (the call must fall back to the float kernels and still be exact)."""
    from introtocomputervision_b200 import _capi
    import ctypes as C
    rows, cols, R, rng = 1100, 3840, 3, 15
    buf = (C.c_int * 16)()
    k = _capi.lib().stereo_host_pipeline_item_bands(n, rows, cols, 0, 0, buf, 16)
    assert list(buf[:k]) == ([0, 137, 411, 689, 963, 1100] if n == 1 else [0, 137, 411, 1100])
    Ls, Rs = [], []
    for i in range(n):
        L, Rt, _ = synth.make_pair(rows, cols, 12, 8100 + 5 * i + n)
        Ls.append(L), Rs.append(Rt)
    Ls, Rs = np.stack(Ls).astype(kind), np.stack(Rs).astype(kind)

    def check(bl, br):
        for i in range(n):
            Lf, Rf = Ls[i].astype(np.float32), Rs[i].astype(np.float32)
            assert np.array_equal(bl[i], oracle.narrow_i8(oracle.ssd_fast(Lf, Rf, R, -rng, 0))), f"pair {i} L->R"
            assert np.array_equal(br[i], oracle.narrow_i8(oracle.ssd_fast(Rf, Lf, R, 0, rng))), f"pair {i} R->L"

    bl, br = ctx.disparity_pair_batch(sb.COST_SSD, Ls, Rs, R, rng, dtype=np.int8)
    assert ctx.last_path == sb.PATH_FAST_U8
    check(bl, br)
    if kind == np.float32:
        Ls[n - 1, rows - 20, 1717] += 0.5
        bl, br = ctx.disparity_pair_batch(sb.COST_SSD, Ls, Rs, R, rng, dtype=np.int8)
        check(bl, br)


def test_host_batch_f32_non_8bit_pair_takes_float_kernels(ctx):
    # one noisy pair in a CV_32FC1 batch: the batch goes pair by pair, the noisy one on the float running-sum kernels
    n, rows, cols, R, rng = 5, 30, 110, 2, 17
    Ls, Rs = [], []
    for i in range(n):
        L, Rt, _ = synth.make_pair(rows, cols, 12, 6100 + i)
        Ls.append(L.astype(np.float32)), Rs.append(Rt.astype(np.float32))
    Ls[3] = synth.noisy_variant(Ls[3].astype(np.uint8), 5)
    Ls, Rs = np.stack(Ls), np.stack(Rs)
    bl, br = ctx.disparity_pair_batch(sb.COST_SSD, Ls, Rs, R, rng, dtype=np.int8)
    for i in range(n):
        assert np.array_equal(bl[i], oracle.narrow_i8(oracle.ssd_fast(Ls[i], Rs[i], R, -rng, 0))), i
        assert np.array_equal(br[i], oracle.narrow_i8(oracle.ssd_fast(Rs[i], Ls[i], R, 0, rng))), i


# ---- fused pair launches: both maps of a pair from one cost volume (SURVEY.md §8 f2) --------------------------

FUSED_SHAPES = [
    # rows, cols, R, range      (range + 1 a multiple of 128)
    (30, 300, 2, 127),          # cols not a multiple of the 24-pixel strip, one disparity group
    (26, 500, 5, 255),          # two groups in one CTA; the last 255 columns see candidates in the right padding
    (40, 96, 3, 127),           # image narrower than the range: every R->L pixel has right-padding candidates
    (19, 700, 0, 127),          # 1x1 window
    (22, 410, 4, 383),          # three groups (gc = 1)
    (64, 1000, 5, 255),
    (9, 130, 1, 127),           # fewer rows than a pipeline stage
    (33, 450, 4, 63),           # 64 candidates: two strips per warp, 16-lane diagonal chains
    (21, 97, 2, 63),
    (50, 1280, 5, 63),          # 5 tiles of 256 columns exactly: the right-padding candidates come from fused_border_kernel
    (25, 320, 3, 127),          # border-kernel mode, one strip per warp, one group per CTA (2 tiles of 160)
    (31, 400, 5, 255),          # border-kernel mode, two groups per CTA (5 tiles of 80), every pixel has padding candidates
    (20, 512, 5, 63),           # border-kernel mode, two strips per warp
    (17, 160, 1, 127),          # border-kernel mode, R = 1
    (12, 320, 0, 127),          # R = 0: no padding at all
]


@pytest.mark.parametrize("rows,cols,R,rng", FUSED_SHAPES)
def test_fused_pair_equals_oracle_and_unfused(ctx, rows, cols, R, rng):
    L, Rt, _ = synth.make_pair(rows, cols, min(rng + 1, 64), 8000 + rows + cols)
    Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
    ref_l, ref_r = oracle.ssd_fast(Lf, Rf, R, -rng, 0), oracle.ssd_fast(Rf, Lf, R, 0, rng)
    try:
        ctx.set_fuse_pairs(True)
        fl, fr = ctx.disparity_pair(sb.COST_SSD, L, Rt, R, rng, dtype=np.int16)
        assert ctx.last_path == sb.PATH_FAST_U8
        assert ctx.last_fused_pairs == 1, "the fused pair launch did not run"
        ctx.set_fuse_pairs(False)
        ul, ur = ctx.disparity_pair(sb.COST_SSD, L, Rt, R, rng, dtype=np.int16)
        assert ctx.last_fused_pairs == 0
    finally:
        ctx.set_fuse_pairs(True)
    assert np.array_equal(ul, ref_l) and np.array_equal(ur, ref_r)
    assert np.array_equal(fl, ref_l), "fused L->R"
    bad = np.argwhere(fr != ref_r)
    assert bad.size == 0, f"fused R->L differs at {bad[:5].tolist()} (of {len(bad)})"


@pytest.mark.parametrize("seed", range(14))
def test_fused_pair_random_shapes(ctx, seed):
    """Seeded random shapes through the fused pair launch: images narrower than a strip or than the search range, a
    single row, every radius 0..5, 64 / 128 / 256 candidates, uint8 and CV_32FC1 inputs."""
    rng = np.random.default_rng(9000 + seed)
    rows = int(rng.integers(1, 48))
    cols = int(rng.choice([3, 17, 40, 95, 129, 257, 600])) + int(rng.integers(0, 7))
    R = int(rng.integers(0, 6))
    r = int(rng.choice([63, 127, 255]))
    L, Rt, _ = synth.make_pair(rows, cols, min(r + 1, max(2, cols // 2)), 9100 + seed)
    if seed % 3 == 0:                       # low-texture image: many exact ties
        L, Rt = (L // 64 * 64).astype(np.uint8), (Rt // 64 * 64).astype(np.uint8)
    Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
    a, b = (Lf, Rf) if seed % 2 else (L, Rt)
    dl, dr = ctx.disparity_pair(sb.COST_SSD, a, b, R, r, dtype=np.int16)
    assert ctx.last_path == sb.PATH_FAST_U8 and ctx.last_fused_pairs >= 1
    assert np.array_equal(dl, oracle.ssd_fast(Lf, Rf, R, -r, 0)), (rows, cols, R, r)
    assert np.array_equal(dr, oracle.ssd_fast(Rf, Lf, R, 0, r)), (rows, cols, R, r)


def test_fused_pair_ties_flat_images(ctx):
    # flat and banded images: every candidate ties; first-minimum order must survive the diagonal minima
    rows, cols, R, rng = 24, 400, 3, 127
    flat = np.full((rows, cols), 9, np.uint8)
    band = np.tile((np.arange(cols) // 37 % 2 * 200).astype(np.uint8), (rows, 1))
    for L, Rt in ((flat, flat), (band, band), (band, flat)):
        Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
        fl, fr = ctx.disparity_pair(sb.COST_SSD, L, Rt, R, rng, dtype=np.int16)
        assert ctx.last_fused_pairs == 1
        assert np.array_equal(fl, oracle.ssd_fast(Lf, Rf, R, -rng, 0))
        assert np.array_equal(fr, oracle.ssd_fast(Rf, Lf, R, 0, rng))


def test_fused_pair_border_kernel_in_bands(ctx):
    # border-kernel mode (1280 columns, 64 candidates) through the banded host pipeline: band seams see the +1 halo row
    rows, cols, R, rng = 90, 1280, 4, 63
    L, Rt, _ = synth.make_pair(rows, cols, 64, 777)
    Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
    ref_l, ref_r = oracle.ssd_fast(Lf, Rf, R, -rng, 0), oracle.ssd_fast(Rf, Lf, R, 0, rng)
    try:
        for bands in (1, 3):
            ctx.set_pipe_bands(bands)
            dl, dr = ctx.disparity_pair(sb.COST_SSD, L, Rt, R, rng, dtype=np.int16)
            assert ctx.last_fused_pairs == bands
            assert np.array_equal(dl, ref_l) and np.array_equal(dr, ref_r), bands
    finally:
        ctx.set_pipe_bands(0)


def test_fused_pair_bands_and_batches(ctx):
    # host pipeline in row bands (seams: the +1 halo row of the SSD row wrap) and a chunked batch of pairs
    rows, cols, R, rng = 150, 520, 5, 127
    L, Rt, _ = synth.make_pair(rows, cols, 64, 4242)
    Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
    ref_l, ref_r = oracle.ssd_fast(Lf, Rf, R, -rng, 0), oracle.ssd_fast(Rf, Lf, R, 0, rng)
    try:
        for bands in (1, 3, 4):
            ctx.set_pipe_bands(bands)
            dl, dr = ctx.disparity_pair(sb.COST_SSD, Lf, Rf, R, rng, dtype=np.int16)
            assert ctx.last_fused_pairs == bands
            assert np.array_equal(dl, ref_l) and np.array_equal(dr, ref_r), bands
    finally:
        ctx.set_pipe_bands(0)
    n = 7
    Ls, Rs = [], []
    for i in range(n):
        a, b, _ = synth.make_pair(33, 330, 64, 7000 + i)
        Ls.append(a), Rs.append(b)
    Ls, Rs = np.stack(Ls), np.stack(Rs)
    for rng in (127, 63):
        bl, br = ctx.disparity_pair_batch(sb.COST_SSD, Ls, Rs, 4, rng, dtype=np.int8)
        assert ctx.last_fused_pairs == n
        for i in range(n):
            a, b = Ls[i].astype(np.float32), Rs[i].astype(np.float32)
            assert np.array_equal(bl[i], oracle.narrow_i8(oracle.ssd_fast(a, b, 4, -rng, 0))), (rng, i)
            assert np.array_equal(br[i], oracle.narrow_i8(oracle.ssd_fast(b, a, 4, 0, rng))), (rng, i)


def test_fused_pair_with_costs_matches_single_calls(ctx):
    rows, cols, R, rng = 28, 280, 2, 127
    L, Rt, _ = synth.make_pair(rows, cols, 48, 99)
    dl, dr = ctx.disparity_pair(sb.COST_SSD, L, Rt, R, rng, dtype=np.int16)
    assert ctx.last_fused_pairs == 1
    sl, cl = ctx.disparity(sb.COST_SSD, L, Rt, R, -rng, 0, dtype=np.int16, return_best=True)
    sr, cr = ctx.disparity(sb.COST_SSD, Rt, L, R, 0, rng, dtype=np.int16, return_best=True)
    assert np.array_equal(dl, sl) and np.array_equal(dr, sr)
    _, ol = oracle.ssd_fast(L.astype(np.float32), Rt.astype(np.float32), R, -rng, 0, return_cost=True)
    assert np.array_equal(cl, ol)


def test_pipelined_host_non_8bit_is_redone_on_float_kernels(ctx):
    # the 8-bit flag is only known after the pipelined pass: a noisy image must be redone by the float kernels
    L, Rt, _ = synth.make_pair(60, 200, 30, 31)
    Lf, Rf = synth.noisy_variant(L, 1), synth.noisy_variant(Rt, 2)
    Lf[-1, -1] += 0.25                                          # ... even when only the very last pixel is non-integer
    try:
        ctx.set_pipe_bands(3)
        dl, dr = sb.disparitySSDPair(Lf, Rf, sb.DisparityConfig(3, 29), ctx=ctx)
        assert ctx.last_path == sb.PATH_FAST_F32
        assert np.array_equal(dl, oracle.narrow_i8(oracle.ssd_fast(Lf, Rf, 3, -29, 0)))
        assert np.array_equal(dr, oracle.narrow_i8(oracle.ssd_fast(Rf, Lf, 3, 0, 29)))
        Li = L.astype(np.float32)
        Li[-1, -2] += 0.5                                       # (not one of the pixels the host samples before the pipeline)
        d = ctx.disparity(sb.COST_SSD, Li, Rt.astype(np.float32), 3, -29, 0, dtype=np.int16)
        assert ctx.last_path == sb.PATH_FAST_F32
        assert np.array_equal(d, oracle.ssd_fast(Li, Rt.astype(np.float32), 3, -29, 0))
    finally:
        ctx.set_pipe_bands(0)


# ---- the packed u8 kernels ------------------------------------------------------------------------------------

FAST_SHAPES = [
    # rows, cols, R, dmin, dmax
    (40, 100, 2, -10, 0),
    (40, 100, 2, 0, 10),
    (64, 200, 5, -63, 0),
    (64, 200, 5, 0, 63),
    (37, 333, 4, -127, 0),      # exactly one 128-disparity group
    (37, 333, 4, 0, 127),
    (50, 300, 3, -255, 0),      # two groups
    (50, 300, 3, 0, 255),
    (33, 500, 7, -95, 0),       # ps2.yaml problem 2 parameters
    (33, 500, 6, 0, 3),         # ps2.yaml problem 1 parameters
    (45, 260, 1, -80, 0),       # 81 candidates: not a multiple of 4
    (45, 260, 0, -17, 9),       # 1x1 window, mixed-sign range
    (21, 50, 5, -300, 300),     # range far wider than the image
    (150, 97, 2, -30, 0),       # tall and narrow: several row segments
    (9, 24, 3, 5, 11),          # positive-only range
    (300, 700, 5, -130, 0),     # 131 candidates: 2 groups, second almost empty
]


@pytest.mark.parametrize("rows,cols,R,dmin,dmax", FAST_SHAPES)
def test_ssd_fast_u8_vs_oracle(ctx, rows, cols, R, dmin, dmax):
    L, Rt, _ = synth.make_pair(rows, cols, max(2, min(64, max(abs(dmin), abs(dmax)))), rows * 1000 + cols)
    d_ref, c_ref = oracle.ssd_fast(L.astype(np.float32), Rt.astype(np.float32), R, dmin, dmax, return_cost=True)
    d, c = ctx.disparity(sb.COST_SSD, L, Rt, R, dmin, dmax, dtype=np.int32, return_best=True)
    assert ctx.last_path == sb.PATH_FAST_U8
    bad = np.argwhere(d != d_ref)
    assert bad.size == 0, f"{len(bad)} mismatching pixels, first {bad[:5].tolist()}"
    assert np.array_equal(c, c_ref)
    # float images holding 8-bit values take the same kernels
    d2 = ctx.disparity(sb.COST_SSD, L.astype(np.float32), Rt.astype(np.float32), R, dmin, dmax, dtype=np.int32)
    assert ctx.last_path == sb.PATH_FAST_U8
    assert np.array_equal(d2, d_ref)


def test_ssd_fast_flat_and_saturated_images(ctx):
    # ties everywhere (first minimum must win), extreme intensities (largest keys)
    for val in (0, 7, 255):
        img = np.full((40, 90), val, np.uint8)
        for (dmin, dmax) in ((-20, 0), (0, 20)):
            d_ref = oracle.ssd_fast(img.astype(np.float32), img.astype(np.float32), 7, dmin, dmax)
            assert np.array_equal(ctx.disparity(sb.COST_SSD, img, img, 7, dmin, dmax, dtype=np.int32), d_ref)
    a = np.zeros((30, 120), np.uint8)
    b = np.full((30, 120), 255, np.uint8)
    d_ref, c_ref = oracle.ssd_fast(a.astype(np.float32), b.astype(np.float32), 7, -100, 0, return_cost=True)
    d, c = ctx.disparity(sb.COST_SSD, a, b, 7, -100, 0, dtype=np.int32, return_best=True)
    assert np.array_equal(d, d_ref) and np.array_equal(c, c_ref)


def test_ssd_fast_equals_exact_path(ctx):
    L, Rt, _ = synth.make_pair(120, 400, 100, 4242)
    try:
        ctx.force_path(sb.PATH_EXACT_F32)
        d_exact = ctx.disparity(sb.COST_SSD, L, Rt, 5, -140, 0, dtype=np.int16)
        assert ctx.last_path == sb.PATH_EXACT_F32
    finally:
        ctx.force_path(0)
    d_fast = ctx.disparity(sb.COST_SSD, L, Rt, 5, -140, 0, dtype=np.int16)
    assert ctx.last_path == sb.PATH_FAST_U8
    assert np.array_equal(d_fast, d_exact)


# ---- the packed u8 NCC kernels -------------------------------------------------------------------------

NCC_FAST_SHAPES = [
    # rows, cols, R, dmin, dmax   (NCC ranges must contain 0 or some border pixel has no candidate)
    (40, 100, 2, -10, 0),
    (40, 100, 2, 0, 10),
    (64, 200, 5, -63, 0),
    (64, 200, 5, 0, 63),
    (37, 333, 4, -127, 0),      # exactly one 128-disparity group
    (37, 333, 4, 0, 127),
    (50, 300, 3, -255, 0),      # two groups
    (50, 300, 3, 0, 255),
    (33, 500, 7, -95, 0),       # ps2.yaml problem 4 parameters (I2F keys: (2R+1)^2*255^2 >= 2^23)
    (33, 500, 7, 0, 80),        # ps2.yaml problem 5 parameters
    (33, 200, 6, -40, 0),
    (45, 260, 1, -80, 0),       # 81 candidates: not a multiple of 4
    (45, 260, 0, -17, 9),       # 1x1 window, mixed-sign range (left-aligned result index)
    (21, 50, 5, -300, 300),     # range far wider than the image
    (150, 97, 2, -30, 0),       # tall and narrow: several row segments
    (300, 700, 5, -130, 0),     # 131 candidates: 2 groups, second almost empty
]


@pytest.mark.parametrize("rows,cols,R,dmin,dmax", NCC_FAST_SHAPES)
def test_ncc_fast_u8_vs_oracle(ctx, rows, cols, R, dmin, dmax):
    L, Rt, _ = synth.make_pair(rows, cols, max(2, min(64, max(abs(dmin), abs(dmax)))), rows * 1000 + cols + 1)
    d_ref, s_ref = oracle.ncorr_fast(L.astype(np.float32), Rt.astype(np.float32), R, dmin, dmax, return_score=True)
    d, s = ctx.disparity(sb.COST_NCORR, L, Rt, R, dmin, dmax, dtype=np.int32, return_best=True)
    assert ctx.last_path == sb.PATH_FAST_U8
    assert_ncc_close(d, s, d_ref, s_ref, L, Rt, R, dmin, dmax, nc.family_of(ctx))
    # where the disparity agrees the recomputed score is the oracle's, bit for bit (elsewhere: assert_ncc_close)
    same = d == d_ref
    assert np.array_equal(s[same], s_ref[same])
    d2 = ctx.disparity(sb.COST_NCORR, L.astype(np.float32), Rt.astype(np.float32), R, dmin, dmax, dtype=np.int32)
    assert ctx.last_path == sb.PATH_FAST_U8
    assert np.array_equal(d2, d)


def test_ncc_fast_flat_dark_and_saturated_images(ctx):
    # exact ties (first maximum must win), zero-energy windows (score 0), extreme intensities
    for val in (0, 1, 255):
        img = np.full((40, 90), val, np.uint8)
        for (dmin, dmax) in ((-20, 0), (0, 20)):
            for R in (2, 7):
                d_ref, s_ref = oracle.ncorr(img.astype(np.float32), img.astype(np.float32), R, dmin, dmax, return_score=True)
                d, s = ctx.disparity(sb.COST_NCORR, img, img, R, dmin, dmax, dtype=np.int32, return_best=True)
                assert ctx.last_path == sb.PATH_FAST_U8
                assert np.array_equal(d, d_ref) and np.array_equal(s, s_ref)
    # half black / half textured: zero-energy candidates next to real ones
    L, Rt, _ = synth.make_pair(30, 160, 16, 5)
    L[:, :60] = 0
    Rt[:, 40:90] = 0
    for (a, b, dmin, dmax) in ((L, Rt, -30, 0), (Rt, L, 0, 30)):
        d_ref, s_ref = oracle.ncorr(a.astype(np.float32), b.astype(np.float32), 3, dmin, dmax, return_score=True)
        d, s = ctx.disparity(sb.COST_NCORR, a, b, 3, dmin, dmax, dtype=np.int32, return_best=True)
        assert_ncc_close(d, s, d_ref, s_ref, a, b, 3, dmin, dmax, nc.family_of(ctx))


def test_ncc_fast_smooth_low_texture(ctx):
    # smooth gradients + weak texture: many near-ties, the hardest case for the 17-bit keys
    yy, xx = np.mgrid[0:60, 0:400]
    rng = np.random.default_rng(5)
    L = np.clip(60 + 0.3 * xx + 0.2 * yy + rng.integers(-3, 4, xx.shape), 0, 255).astype(np.uint8)
    Rt = np.clip(60 + 0.3 * (xx + 7) + 0.2 * yy + rng.integers(-3, 4, xx.shape), 0, 255).astype(np.uint8)
    d_ref, s_ref = oracle.ncorr_fast(L.astype(np.float32), Rt.astype(np.float32), 4, -40, 0, return_score=True)
    d, s = ctx.disparity(sb.COST_NCORR, L, Rt, 4, -40, 0, dtype=np.int32, return_best=True)
    # near-ties within ~2^-22 relative may resolve differently: a lower fraction, but every differing pixel within tau
    assert_ncc_close(d, s, d_ref, s_ref, L, Rt, 4, -40, 0, nc.family_of(ctx), min_agree=0.99)
    # Why not 99.9 % here: this image is built so that dozens of candidates per pixel score within a few float32 ulps of each
    # other (scores ~ 0.99999).  The oracle ranks float32 scores (2^-24 relative near 1); a key holds 23 value bits of
    # C * rs in a power-of-two scale that can be up to twice the score's magnitude (2^-22 relative), so candidates the oracle
    # separates by one or two ulps tie here and the earlier one wins.  Textured images (every other test) have no such runs.
    # The pair call (fused NCC pairs, one scale per PIXEL instead of per strip row) behaves the same on it.
    fl, fr = ctx.disparity_pair(sb.COST_NCORR, L, Rt, 4, 40, dtype=np.int32)
    assert ctx.last_fused_pairs == 1
    nc.check_ncc_map(fl, L, Rt, 4, -40, 0, "u8_fused", oracle_disp=d_ref, min_agree=0.99, what="pair L->R")
    nc.check_ncc_map(fr, Rt, L, 4, 0, 40, "u8_fused", min_agree=0.99, what="pair R->L")


def test_ncc_fast_equals_exact_path(ctx):
    L, Rt, _ = synth.make_pair(60, 300, 100, 4243)
    try:
        ctx.force_path(sb.PATH_EXACT_F32)
        d_exact, s_exact = ctx.disparity(sb.COST_NCORR, L, Rt, 5, -140, 0, dtype=np.int16, return_best=True)
        assert ctx.last_path == sb.PATH_EXACT_F32
    finally:
        ctx.force_path(0)
    d_fast, s_fast = ctx.disparity(sb.COST_NCORR, L, Rt, 5, -140, 0, dtype=np.int16, return_best=True)
    assert ctx.last_path == sb.PATH_FAST_U8
    # the exact path IS the oracle (tau = 0) ...
    Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
    d_ref = oracle.ncorr_fast(Lf, Rf, 5, -140, 0)
    nc.check_ncc_map(d_exact, Lf, Rf, 5, -140, 0, "exact", oracle_disp=d_ref)
    # ... and the packed kernels are within their key resolution of it
    assert_ncc_close(d_fast, s_fast, d_exact, s_exact, Lf, Rf, 5, -140, 0, nc.family_of(ctx))


# ---- BASELINE config 3 at full size: 1920x1080, 128 disparities, 9x9, SSD and NCC ------------------------

def test_config3_full_size_ssd_and_ncc(ctx):
    L, Rt, _ = synth.make_pair(1080, 1920, 128, 1001)
    Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
    dl, dr = ctx.disparity_pair(sb.COST_SSD, L, Rt, 4, 127)
    assert np.array_equal(dl, oracle.narrow_i8(oracle.ssd_fast(Lf, Rf, 4, -127, 0)))
    assert np.array_equal(dr, oracle.narrow_i8(oracle.ssd_fast(Rf, Lf, 4, 0, 127)))
    d_ref, s_ref = oracle.ncorr_fast(Lf, Rf, 4, -127, 0, return_score=True)
    d, s = ctx.disparity(sb.COST_NCORR, L, Rt, 4, -127, 0, dtype=np.int16, return_best=True)
    assert ctx.last_path == sb.PATH_FAST_U8
    assert_ncc_close(d, s, d_ref, s_ref, Lf, Rf, 4, -127, 0, nc.family_of(ctx))


# ---- fused pair launches for any candidate count and every window radius (SURVEY.md §8 f2) ----------------------
# The reference's own problems (config/ps2.yaml:19-41) are R = 6 / 7 with 4, 96 and 81 candidates: none of them is a
# whole number of 128- (64-) disparity groups.  The walked direction's groups are aligned to the top of its range and the
# candidates below -range are masked in both maps; R > 5 takes explicit selects at the image borders.

GENERAL_FUSED_SHAPES = [
    (20, 300, 7, 95), (20, 300, 6, 80), (16, 128, 6, 3), (12, 200, 5, 100), (9, 260, 3, 129), (14, 333, 7, 127),
    (10, 150, 0, 1), (11, 700, 7, 255), (13, 90, 6, 40), (8, 64, 7, 63), (17, 257, 4, 64), (9, 1290, 6, 70),
    (6, 30, 7, 95), (5, 9, 6, 200), (40, 640, 7, 95), (25, 513, 2, 33),
]


@pytest.mark.parametrize("rows,cols,R,rng", GENERAL_FUSED_SHAPES)
def test_fused_pair_any_range_any_radius(ctx, rows, cols, R, rng):
    L, Rt, _ = synth.make_pair(rows, cols, min(rng + 1, max(2, cols // 2)), 31000 + rows * 7 + cols)
    Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
    ref_l, ref_r = oracle.ssd_fast(Lf, Rf, R, -rng, 0), oracle.ssd_fast(Rf, Lf, R, 0, rng)
    fl, fr = ctx.disparity_pair(sb.COST_SSD, L, Rt, R, rng, dtype=np.int16)
    assert ctx.last_path == sb.PATH_FAST_U8 and ctx.last_fused_pairs == 1
    bad = np.argwhere(fl != ref_l)
    assert bad.size == 0, f"fused L->R differs at {bad[:5].tolist()} (of {len(bad)})"
    bad = np.argwhere(fr != ref_r)
    assert bad.size == 0, f"fused R->L differs at {bad[:5].tolist()} (of {len(bad)})"
    ctx.set_fuse_pairs(False)
    try:
        ul, ur = ctx.disparity_pair(sb.COST_SSD, L, Rt, R, rng, dtype=np.int16)
        assert ctx.last_fused_pairs == 0
    finally:
        ctx.set_fuse_pairs(True)
    assert np.array_equal(ul, ref_l) and np.array_equal(ur, ref_r)


@pytest.mark.parametrize("seed", range(16))
def test_fused_pair_random_any_range(ctx, seed):
    rng = np.random.default_rng(12000 + seed)
    rows = int(rng.integers(1, 40))
    cols = int(rng.choice([5, 21, 47, 99, 160, 290, 640])) + int(rng.integers(0, 9))
    R = int(rng.integers(0, 8))
    r = int(rng.integers(1, 300))
    L, Rt, _ = synth.make_pair(rows, cols, min(r + 1, max(2, cols // 2)), 12100 + seed)
    if seed % 4 == 0:                       # low-texture image: many exact ties
        L, Rt = (L // 64 * 64).astype(np.uint8), (Rt // 64 * 64).astype(np.uint8)
    Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
    a, b = (Lf, Rf) if seed % 2 else (L, Rt)
    dl, dr = ctx.disparity_pair(sb.COST_SSD, a, b, R, r, dtype=np.int16)
    assert ctx.last_path == sb.PATH_FAST_U8 and ctx.last_fused_pairs >= 1
    assert np.array_equal(dl, oracle.ssd_fast(Lf, Rf, R, -r, 0)), (rows, cols, R, r)
    assert np.array_equal(dr, oracle.ssd_fast(Rf, Lf, R, 0, r)), (rows, cols, R, r)


def test_fused_pair_any_range_ties_flat_images(ctx):
    rows, cols = 18, 300
    flat = np.full((rows, cols), 200, np.uint8)
    band = np.tile((np.arange(cols) // 29 % 2 * 255).astype(np.uint8), (rows, 1))
    for R, rng in ((7, 95), (6, 3), (5, 80)):
        for L, Rt in ((flat, flat), (band, band), (band, flat)):
            Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
            fl, fr = ctx.disparity_pair(sb.COST_SSD, L, Rt, R, rng, dtype=np.int16)
            assert ctx.last_fused_pairs == 1
            assert np.array_equal(fl, oracle.ssd_fast(Lf, Rf, R, -rng, 0)), (R, rng)
            assert np.array_equal(fr, oracle.ssd_fast(Rf, Lf, R, 0, rng)), (R, rng)


# ---- the configurations the numbers are quoted on, at their real size ---------------------------------------------------

def test_ps2_problem_shapes_full_size_clean(ctx):
    """config/ps2.yaml:19-41 at the logged image sizes (ps2_cpu.log:6,12,49): pair0 128x128 R=6 range=3 SSD, pair1
    511x640 R=7 range=95 SSD and NCC, pair2 529x640 R=7 range=80 NCC; synthetic stand-ins for the LFS-stubbed pixels."""
    for rows, cols, R, rng, seed in ((128, 128, 6, 3, 10), (511, 640, 7, 95, 11)):
        L, Rt, _ = synth.make_pair(rows, cols, rng + 1, seed)
        Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
        dl, dr = sb.disparitySSDPair(Lf, Rf, sb.DisparityConfig(R, rng), ctx=ctx)
        assert ctx.last_path == sb.PATH_FAST_U8 and ctx.last_fused_pairs == 1
        assert np.array_equal(dl, oracle.narrow_i8(oracle.ssd_fast(Lf, Rf, R, -rng, 0))), (rows, cols)
        assert np.array_equal(dr, oracle.narrow_i8(oracle.ssd_fast(Rf, Lf, R, 0, rng))), (rows, cols)
    for rows, cols, R, rng, seed in ((511, 640, 7, 95, 11), (529, 640, 7, 80, 12)):
        L, Rt, _ = synth.make_pair(rows, cols, rng + 1, seed)
        Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
        for ref, tgt, lo, hi in ((Lf, Rf, -rng, 0), (Rf, Lf, 0, rng)):
            d_ref, s_ref = oracle.ncorr_fast(ref, tgt, R, lo, hi, return_score=True)
            d, s = ctx.disparity(sb.COST_NCORR, ref, tgt, R, lo, hi, dtype=np.int16, return_best=True)
            assert ctx.last_path == sb.PATH_FAST_U8
            assert_ncc_close(d, s, d_ref, s_ref, ref, tgt, R, lo, hi, nc.family_of(ctx))


def test_config4_full_size_fused_pair_and_ncc(ctx):
    """BASELINE config 4's shape on ONE GPU, the configuration the headline number is quoted on: 3840x2160, 256
    disparities, 11x11.  SSD: both maps of the fused pair launch bit-exact against the oracle.  NCC: L->R within the
    north-star tolerance."""
    L, Rt, _ = synth.make_pair(2160, 3840, 256, 1002)
    Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
    dl, dr = ctx.disparity_pair(sb.COST_SSD, L, Rt, 5, 255, dtype=np.int16)
    assert ctx.last_path == sb.PATH_FAST_U8 and ctx.last_fused_pairs >= 1
    ref_l = oracle.ssd_fast(Lf, Rf, 5, -255, 0)
    bad = np.argwhere(dl != ref_l)
    assert bad.size == 0, f"4K fused L->R differs at {bad[:5].tolist()} (of {len(bad)})"
    ref_r = oracle.ssd_fast(Rf, Lf, 5, 0, 255)
    bad = np.argwhere(dr != ref_r)
    assert bad.size == 0, f"4K fused R->L differs at {bad[:5].tolist()} (of {len(bad)})"
    d_ref, s_ref = oracle.ncorr_fast(Lf, Rf, 5, -255, 0, return_score=True)
    d, s = ctx.disparity(sb.COST_NCORR, L, Rt, 5, -255, 0, dtype=np.int16, return_best=True)
    assert ctx.last_path == sb.PATH_FAST_U8
    assert_ncc_close(d, s, d_ref, s_ref, Lf, Rf, 5, -255, 0, nc.family_of(ctx))


# ---- the float running-sum kernels (general float32 images; VERDICT r1 row g1) ------------------------------------------
# SSD: q = (int)round(f32((l - r)^2)) per element (DisparitySSD.cpp:49-51) is an int, so int32 column / horizontal running
# sums are exact: bit-exact disparities AND costs.  NCC: float32 running sums, north-star tolerance.

def _float_variants(L, Rt, seed):
    """The three input families of the ps2 executable: noise on both images (main.cpp:140-153), contrast on the left
    image only (main.cpp:191-193), and both."""
    yield "noisy", synth.noisy_variant(L, seed), synth.noisy_variant(Rt, seed + 1)
    yield "contrast", synth.contrast_variant(L), Rt.astype(np.float32)
    yield "noisy+contrast", synth.noisy_variant(L, seed) * np.float32(1.1), synth.noisy_variant(Rt, seed + 1)


F32_SHAPES = [
    # rows, cols, R, dmin, dmax
    (24, 140, 7, -95, 0), (24, 140, 7, 0, 95), (30, 200, 6, -80, 0), (17, 90, 5, -20, 15), (40, 333, 4, -127, 0),
    (12, 64, 0, 0, 7), (9, 300, 3, 0, 200), (21, 77, 2, -300, -100), (15, 500, 1, -130, 0), (33, 129, 7, 5, 40),
]


@pytest.mark.parametrize("rows,cols,R,dmin,dmax", F32_SHAPES)
def test_ssd_float_kernels_vs_oracle(ctx, rows, cols, R, dmin, dmax):
    L, Rt, _ = synth.make_pair(rows, cols, max(2, min(abs(dmin), abs(dmax), cols // 2)), 41000 + rows + cols)
    for name, Lf, Rf in _float_variants(L, Rt, rows):
        d_ref, c_ref = oracle.ssd_fast(Lf, Rf, R, dmin, dmax, return_cost=True)
        d, c = ctx.disparity(sb.COST_SSD, Lf, Rf, R, dmin, dmax, dtype=np.int32, return_best=True)
        assert ctx.last_path == sb.PATH_FAST_F32, name
        bad = np.argwhere(d != d_ref)
        assert bad.size == 0, f"{name}: disparity differs at {bad[:5].tolist()} (of {len(bad)})"
        assert np.array_equal(c, c_ref), name


@pytest.mark.parametrize("rows,cols,R,rng", [(24, 140, 7, 95), (30, 200, 6, 80), (16, 128, 6, 3), (19, 260, 5, 127),
                                               (11, 90, 3, 40), (14, 700, 4, 255), (8, 40, 7, 95), (27, 641, 2, 63)])
def test_ssd_float_fused_pairs_vs_oracle(ctx, rows, cols, R, rng):
    L, Rt, _ = synth.make_pair(rows, cols, min(rng + 1, max(2, cols // 2)), 42000 + rows + cols)
    for name, Lf, Rf in _float_variants(L, Rt, cols):
        ref_l, ref_r = oracle.ssd_fast(Lf, Rf, R, -rng, 0), oracle.ssd_fast(Rf, Lf, R, 0, rng)
        fl, fr = ctx.disparity_pair(sb.COST_SSD, Lf, Rf, R, rng, dtype=np.int16)
        assert ctx.last_path == sb.PATH_FAST_F32 and ctx.last_fused_pairs == 1, name
        bad = np.argwhere(fl != ref_l)
        assert bad.size == 0, f"{name}: fused L->R differs at {bad[:5].tolist()} (of {len(bad)})"
        bad = np.argwhere(fr != ref_r)
        assert bad.size == 0, f"{name}: fused R->L differs at {bad[:5].tolist()} (of {len(bad)})"
        ctx.set_fuse_pairs(False)
        try:
            ul, ur = ctx.disparity_pair(sb.COST_SSD, Lf, Rf, R, rng, dtype=np.int16)
            assert ctx.last_path == sb.PATH_FAST_F32 and ctx.last_fused_pairs == 0
        finally:
            ctx.set_fuse_pairs(True)
        assert np.array_equal(ul, ref_l) and np.array_equal(ur, ref_r), name


@pytest.mark.parametrize("seed", range(12))
def test_ssd_float_kernels_random(ctx, seed):
    rng = np.random.default_rng(43000 + seed)
    rows, cols = int(rng.integers(1, 50)), int(rng.integers(4, 400))
    R = int(rng.integers(0, 8))
    a, b = sorted(int(v) for v in rng.integers(-150, 151, 2))
    L, Rt, _ = synth.make_pair(rows, cols, 30, 43100 + seed)
    gain = np.float32(rng.choice([1.0, 1.1, 0.37]))
    Lf = (synth.noisy_variant(L, seed, sigma=float(rng.choice([0.3, 10.0, 25.0]))) * gain).astype(np.float32)
    Rf = synth.noisy_variant(Rt, seed + 1)
    if seed % 4 == 0:                         # half-integer pixel values: round-half-away ties in every element
        Lf, Rf = np.round(Lf * 2) / np.float32(2), np.round(Rf * 2) / np.float32(2)
    d_ref, c_ref = (oracle.ssd if seed < 4 else oracle.ssd_fast)(Lf, Rf, R, a, b, return_cost=True)
    d, c = ctx.disparity(sb.COST_SSD, Lf, Rf, R, a, b, dtype=np.int32, return_best=True)
    assert ctx.last_path == sb.PATH_FAST_F32
    assert np.array_equal(d, d_ref), (rows, cols, R, a, b)
    assert np.array_equal(c, c_ref), (rows, cols, R, a, b)


def test_float_kernels_on_8bit_images_equal_packed_kernels(ctx):
    # the same 8-bit-valued CV_32FC1 pair through both running-sum families
    L, Rt, _ = synth.make_pair(40, 300, 64, 77)
    Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
    dl8, dr8 = ctx.disparity_pair(sb.COST_SSD, Lf, Rf, 5, 100, dtype=np.int16)
    assert ctx.last_path == sb.PATH_FAST_U8
    n8, s8 = ctx.disparity(sb.COST_NCORR, Lf, Rf, 5, -100, 0, dtype=np.int16, return_best=True)
    try:
        ctx.force_path(sb.PATH_FAST_F32)
        dlf, drf = ctx.disparity_pair(sb.COST_SSD, Lf, Rf, 5, 100, dtype=np.int16)
        assert ctx.last_path == sb.PATH_FAST_F32
        nf, sf = ctx.disparity(sb.COST_NCORR, Lf, Rf, 5, -100, 0, dtype=np.int16, return_best=True)
        assert ctx.last_path == sb.PATH_FAST_F32
    finally:
        ctx.force_path(0)
    assert np.array_equal(dl8, dlf) and np.array_equal(dr8, drf)
    # both families against the oracle, each within its own key resolution
    n_ref, s_ref = oracle.ncorr_fast(Lf, Rf, 5, -100, 0, return_score=True)
    assert_ncc_close(n8, s8, n_ref, s_ref, Lf, Rf, 5, -100, 0, "u8")
    assert_ncc_close(nf, sf, n_ref, s_ref, Lf, Rf, 5, -100, 0, "f32")


def test_float_kernels_hand_wide_value_ranges_to_the_exact_path(ctx):
    # pixel ranges beyond what the 32-bit keys / the 2^23 mantissa trick hold: exact per-element kernels, same results
    L, Rt, _ = synth.make_pair(14, 80, 12, 5)
    Lf, Rf = synth.noisy_variant(L, 1) * np.float32(40), synth.noisy_variant(Rt, 2) * np.float32(40)
    d = ctx.disparity(sb.COST_SSD, Lf, Rf, 7, -20, 0, dtype=np.int16)
    assert ctx.last_path == sb.PATH_EXACT_F32
    assert np.array_equal(d, oracle.ssd(Lf, Rf, 7, -20, 0))
    Lf[3, 3] = np.inf
    d = ctx.disparity(sb.COST_NCORR, Lf, Rf, 2, -20, 0, dtype=np.int16)
    assert ctx.last_path == sb.PATH_EXACT_F32


@pytest.mark.parametrize("rows,cols,R,dmin,dmax", [(24, 140, 7, -95, 0), (24, 140, 7, 0, 95), (30, 200, 6, 0, 80),
                                                    (17, 90, 5, -20, 15), (20, 333, 4, -127, 0), (9, 300, 3, 0, 200)])
def test_ncc_float_kernels_vs_oracle(ctx, rows, cols, R, dmin, dmax):
    L, Rt, _ = synth.make_pair(rows, cols, max(2, min(abs(dmin) + abs(dmax), cols // 2)), 44000 + rows + cols)
    for name, Lf, Rf in _float_variants(L, Rt, rows):
        d_ref, s_ref = oracle.ncorr_fast(Lf, Rf, R, dmin, dmax, return_score=True)
        d, s = ctx.disparity(sb.COST_NCORR, Lf, Rf, R, dmin, dmax, dtype=np.int32, return_best=True)
        assert ctx.last_path == sb.PATH_FAST_F32, name
        assert_ncc_close(d, s, d_ref, s_ref, Lf, Rf, R, dmin, dmax, "f32")


def test_ps2_problem_shapes_full_size_noisy_and_contrast(ctx):
    """Problems 3 and 4 of the reference executable at their real size (config/ps2.yaml:29-36, main.cpp:140-153,191-193):
    511x640, R = 7, range 95; Gaussian noise sigma 10 on both images, x1.1 contrast on the left one."""
    L, Rt, _ = synth.make_pair(511, 640, 96, 11)
    for name, Lf, Rf in (("noisy", synth.noisy_variant(L, 12), synth.noisy_variant(Rt, 13)),
                         ("contrast", synth.contrast_variant(L), Rt.astype(np.float32))):
        dl, dr = sb.disparitySSDPair(Lf, Rf, sb.DisparityConfig(7, 95), ctx=ctx)
        assert ctx.last_path == sb.PATH_FAST_F32 and ctx.last_fused_pairs == 1, name
        assert np.array_equal(dl, oracle.narrow_i8(oracle.ssd_fast(Lf, Rf, 7, -95, 0))), name
        assert np.array_equal(dr, oracle.narrow_i8(oracle.ssd_fast(Rf, Lf, 7, 0, 95))), name
        for ref, tgt, lo, hi in ((Lf, Rf, -95, 0), (Rf, Lf, 0, 95)):
            d_ref, s_ref = oracle.ncorr_fast(ref, tgt, 7, lo, hi, return_score=True)
            d, s = ctx.disparity(sb.COST_NCORR, ref, tgt, 7, lo, hi, dtype=np.int16, return_best=True)
            assert ctx.last_path == sb.PATH_FAST_F32, name
            assert_ncc_close(d, s, d_ref, s_ref, ref, tgt, 7, lo, hi, "f32")


# ---- host-side packing of CV_32FC1 images (stereo_ctx_set_host_threads) ---------------------------------------------------

@pytest.mark.parametrize("threads", [-1, 1, 3, 16])
def test_host_packing_gives_the_same_maps(ctx, threads):
    """CV_32FC1 host images converted to u8 by host threads (1 byte per pixel over the link) or uploaded as floats and
    converted on the device: identical maps, single pairs in bands and batches; a pixel that is not 8-bit anywhere in the
    image hands the call to the float kernels."""
    L, Rt, _ = synth.make_pair(150, 520, 64, 4242)
    Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
    ref_l, ref_r = oracle.ssd_fast(Lf, Rf, 5, -127, 0), oracle.ssd_fast(Rf, Lf, 5, 0, 127)
    n = 7
    Ls, Rs = zip(*[synth.make_pair(33, 330, 64, 7000 + i)[:2] for i in range(n)])
    Ls, Rs = np.stack(Ls).astype(np.float32), np.stack(Rs).astype(np.float32)
    try:
        ctx.set_host_threads(threads)
        assert ctx.host_threads == threads
        for bands in (1, 3):
            ctx.set_pipe_bands(bands)
            dl, dr = ctx.disparity_pair(sb.COST_SSD, Lf, Rf, 5, 127, dtype=np.int16)
            assert ctx.last_path == sb.PATH_FAST_U8
            assert np.array_equal(dl, ref_l) and np.array_equal(dr, ref_r), (threads, bands)
        ctx.set_pipe_bands(0)
        bl, br = ctx.disparity_pair_batch(sb.COST_SSD, Ls, Rs, 4, 63, dtype=np.int8)
        for i in range(n):
            assert np.array_equal(bl[i], oracle.narrow_i8(oracle.ssd_fast(Ls[i], Rs[i], 4, -63, 0))), (threads, i)
            assert np.array_equal(br[i], oracle.narrow_i8(oracle.ssd_fast(Rs[i], Ls[i], 4, 0, 63))), (threads, i)
        Lbad = Lf.copy()
        Lbad[77, 301] += 0.5                                    # found by the host threads (or the device flag) mid-pipeline
        ctx.set_pipe_bands(3)
        dl, dr = ctx.disparity_pair(sb.COST_SSD, Lbad, Rf, 5, 127, dtype=np.int16)
        assert ctx.last_path == sb.PATH_FAST_F32
        assert np.array_equal(dl, oracle.ssd_fast(Lbad, Rf, 5, -127, 0)) and np.array_equal(dr, oracle.ssd_fast(Rf, Lbad, 5, 0, 127))
    finally:
        ctx.set_pipe_bands(0)
        ctx.set_host_threads(0)


# ---- NCC pairs from one cost volume (SURVEY.md §8 f2) ----------------------------------------------------------------------
# Both maps come out of the same cross terms; every key is scaled per PIXEL from the other direction's window energies.

NCC_PAIR_SHAPES = [(24, 300, 5, 127), (20, 300, 7, 95), (18, 260, 6, 80), (30, 128, 4, 63), (16, 700, 5, 255), (12, 200, 3, 100),
                   (9, 90, 2, 40), (25, 640, 7, 95), (14, 150, 0, 31), (21, 333, 1, 129)]


def _ncc_pair_refs(Lf, Rf, R, rng):
    return (oracle.ncorr_fast(Lf, Rf, R, -rng, 0, return_score=True), oracle.ncorr_fast(Rf, Lf, R, 0, rng, return_score=True))


@pytest.mark.parametrize("rows,cols,R,rng", NCC_PAIR_SHAPES)
def test_ncc_fused_pairs_vs_oracle(ctx, rows, cols, R, rng):
    L, Rt, _ = synth.make_pair(rows, cols, min(rng + 1, max(2, cols // 2)), 46000 + rows + cols)
    Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
    (ref_l, _), (ref_r, _) = _ncc_pair_refs(Lf, Rf, R, rng)
    fl, fr = ctx.disparity_pair(sb.COST_NCORR, L, Rt, R, rng, dtype=np.int16)
    assert ctx.last_path == sb.PATH_FAST_U8 and ctx.last_fused_pairs == 1
    ctx.set_fuse_pairs(False)
    try:
        ul, ur = ctx.disparity_pair(sb.COST_NCORR, L, Rt, R, rng, dtype=np.int16)
        assert ctx.last_fused_pairs == 0
    finally:
        ctx.set_fuse_pairs(True)
    # wherever a map differs from the oracle's, the candidate it chose scores like the oracle's winner (within the key
    # resolution of the family), and the north-star fraction holds
    for got, ref_d, family, (a, b, lo, hi) in ((fl, ref_l, "u8_fused", (Lf, Rf, -rng, 0)), (fr, ref_r, "u8_fused", (Rf, Lf, 0, rng)),
                                               (ul, ref_l, "u8", (Lf, Rf, -rng, 0)), (ur, ref_r, "u8", (Rf, Lf, 0, rng))):
        nc.check_ncc_map(got, a, b, R, lo, hi, family, oracle_disp=ref_d)


def test_ncc_fused_pairs_low_texture_and_flat_images(ctx):
    """Per-pixel key scales: a dark window next to a bright one keeps its mantissa bits (the unfused kernels share one scale
    per strip row and lose bits there); flat / dark / saturated images tie everywhere and must resolve to the first maximum."""
    rows, cols, R, rng = 40, 400, 4, 127
    x = np.arange(cols)
    smooth = np.clip(8 + 3 * np.sin(x / 23.0)[None, :] + np.linspace(0, 240, cols)[None, :] * (np.arange(rows)[:, None] % 2), 0, 255).astype(np.uint8)
    L = smooth
    Rt = np.roll(smooth, 9, axis=1)
    for need, a, b in ((0.95, L, Rt), (NCC_DISP_AGREE, np.full((rows, cols), 7, np.uint8), np.full((rows, cols), 7, np.uint8)),
                       (NCC_DISP_AGREE, np.zeros((rows, cols), np.uint8), np.zeros((rows, cols), np.uint8)),
                       (NCC_DISP_AGREE, np.full((rows, cols), 255, np.uint8), np.full((rows, cols), 255, np.uint8))):
        af, bf = a.astype(np.float32), b.astype(np.float32)
        (ref_l, _), (ref_r, _) = _ncc_pair_refs(af, bf, R, rng)
        fl, fr = ctx.disparity_pair(sb.COST_NCORR, a, b, R, rng, dtype=np.int16)
        assert ctx.last_fused_pairs == 1
        # (the gradient image is full of near-ties at float32 level, see test_ncc_fast_smooth_low_texture; the flat images tie
        # exactly everywhere and must come out as the oracle's first maximum)
        nc.check_ncc_map(fl, af, bf, R, -rng, 0, "u8_fused", oracle_disp=ref_l, min_agree=need, what="L->R")
        nc.check_ncc_map(fr, bf, af, R, 0, rng, "u8_fused", oracle_disp=ref_r, min_agree=need, what="R->L")


def test_ncc_fused_pairs_full_size_and_batches(ctx):
    # the reference's own NCC problems at their real size (config/ps2.yaml:34-41) through the pair call, and a chunked batch
    for rows, cols, R, rng, seed in ((511, 640, 7, 95, 11), (529, 640, 7, 80, 12)):
        L, Rt, _ = synth.make_pair(rows, cols, rng + 1, seed)
        Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
        (ref_l, _), (ref_r, _) = _ncc_pair_refs(Lf, Rf, R, rng)
        dl, dr = sb.disparityNCorrPair(Lf, Rf, sb.DisparityConfig(R, rng), ctx=ctx)
        assert ctx.last_path == sb.PATH_FAST_U8 and ctx.last_fused_pairs == 1
        nc.check_ncc_map(dl, Lf, Rf, R, -rng, 0, "u8_fused", oracle_disp=ref_l, what="L->R")
        nc.check_ncc_map(dr, Rf, Lf, R, 0, rng, "u8_fused", oracle_disp=ref_r, what="R->L")
    n = 6
    Ls, Rs = zip(*[synth.make_pair(33, 330, 64, 7100 + i)[:2] for i in range(n)])
    Ls, Rs = np.stack(Ls), np.stack(Rs)
    bl, br = ctx.disparity_pair_batch(sb.COST_NCORR, Ls, Rs, 4, 63, dtype=np.int8)
    assert ctx.last_fused_pairs == n
    for i in range(n):
        a, b = Ls[i].astype(np.float32), Rs[i].astype(np.float32)
        nc.check_ncc_map(bl[i], a, b, 4, -63, 0, "u8_fused", what=f"pair {i} L->R")
        nc.check_ncc_map(br[i], b, a, 4, 0, 63, "u8_fused", what=f"pair {i} R->L")


def test_config4_full_size_ncc_pair_and_noisy_float_pair(ctx):
    """3840x2160, 256 disparities, 11x11 at full size through the two kernel families added in round 2: the NCC pair from one
    cost volume (both maps within the north-star tolerance) and a noisy CV_32FC1 SSD pair on the float running-sum kernels
    (both maps bit-exact)."""
    L, Rt, _ = synth.make_pair(2160, 3840, 256, 1002)
    Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
    dl, dr = ctx.disparity_pair(sb.COST_NCORR, L, Rt, 5, 255, dtype=np.int16)
    assert ctx.last_path == sb.PATH_FAST_U8 and ctx.last_fused_pairs >= 1
    nc.check_ncc_map(dl, Lf, Rf, 5, -255, 0, "u8_fused", what="4K L->R")
    nc.check_ncc_map(dr, Rf, Lf, 5, 0, 255, "u8_fused", what="4K R->L")
    Ln, Rn = synth.noisy_variant(L, 21), synth.noisy_variant(Rt, 22)
    fl, fr = ctx.disparity_pair(sb.COST_SSD, Ln, Rn, 5, 255, dtype=np.int16)
    assert ctx.last_path == sb.PATH_FAST_F32 and ctx.last_fused_pairs >= 1
    bad = np.argwhere(fl != oracle.ssd_fast(Ln, Rn, 5, -255, 0))
    assert bad.size == 0, f"4K noisy fused L->R differs at {bad[:5].tolist()} (of {len(bad)})"
    bad = np.argwhere(fr != oracle.ssd_fast(Rn, Ln, 5, 0, 255))
    assert bad.size == 0, f"4K noisy fused R->L differs at {bad[:5].tolist()} (of {len(bad)})"


# ---- size-independent properties at the full BASELINE sizes --------------------------------------------------------------------

@pytest.mark.parametrize("rows,cols,nd,R", [(2160, 3840, 256, 5), (1080, 1920, 128, 4), (720, 1280, 64, 4)])
def test_known_shift_at_full_size(ctx, rows, cols, nd, R):
    """right(x) = left(x + k): away from the borders every window has an exact match at disparity -k (L->R) / +k (R->L), for SSD
    and NCC, whatever the image size (SURVEY.md §8c's behavioural known-answer test, at configs 3, 4 and 5's sizes)."""
    rng = np.random.default_rng(rows + nd)
    left = rng.integers(1, 256, (rows, cols + nd), dtype=np.uint8)
    k = nd // 3 + 1
    L, Rt = np.ascontiguousarray(left[:, :cols]), np.ascontiguousarray(left[:, k:k + cols])
    dt = np.int16 if nd > 128 else np.int8
    for cost in (sb.COST_SSD, sb.COST_NCORR):
        dl, dr = ctx.disparity_pair(cost, L, Rt, R, nd - 1, dtype=dt)
        assert ctx.last_fused_pairs >= 1
        # L->R: pixel x of the left image shows up at x - k in the right one; R->L the other way round
        assert np.all(dl[R:-R, k + R + 1:-R - 1] == -k), (cost, "L->R")
        assert np.all(dr[R:-R, R + 1:cols - k - R - 1] == k), (cost, "R->L")
    # idempotence of the pair call and agreement of the u8 and the CV_32FC1 entry points on the same data
    d2l, d2r = ctx.disparity_pair(sb.COST_SSD, L.astype(np.float32), Rt.astype(np.float32), R, nd - 1, dtype=dt)
    d3l, d3r = ctx.disparity_pair(sb.COST_SSD, L, Rt, R, nd - 1, dtype=dt)
    assert np.array_equal(d2l, d3l) and np.array_equal(d2r, d3r)
