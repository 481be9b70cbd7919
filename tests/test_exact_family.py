"""The exact kernel family (EXACT_F32, exact.cuh) against the oracle where only it can go, and the rules that route work
to it: R > 7, more than 4096 candidates, the FAST_F32 value-range bound for SSD at its edge, the classification of single
edge values, and the float NCC family across DC offsets.

SSD: bit-exact disparities and costs against oracle.ssd / oracle.ssd_fast.  NCC: against the literal oracle.ncorr, the exact
family identical (tests/ncc_check.py, tau = 0), the fast families within their key resolution at every pixel, plus the BASELINE
contract (>= 99.9 % equal disparities, scores within 1e-5).  Every value stays where the reference is defined: per
element (l - r)^2 < 2^31 and window sums within int32."""
import ctypes as C

import numpy as np
import pytest

import oracle
import exact_cases as ec
import ncc_check as nc
from lr_oracle import lr_check
from speckle_oracle import filter_speckles
import introtocomputervision_b200 as sb
from introtocomputervision_b200 import _capi, synth
from pair_calls import _ok, _torch

pytestmark = pytest.mark.gpu

NCC_SCORE_RTOL = 1e-5
UNSUP, RANGE = _capi.ERR_UNSUPPORTED, _capi.ERR_INVALID_RANGE


def _tdt(dt):
    t = _torch()
    return {1: t.int8, 2: t.int16, 4: t.int32}[np.dtype(dt).itemsize]


def assert_ncc_close(d, s, d_ref, s_ref, ref, tgt, R, dmin, dmax, family):
    nc.check_ncc_map(d, ref, tgt, R, dmin, dmax, family, oracle_disp=d_ref)
    np.testing.assert_allclose(s, s_ref, rtol=NCC_SCORE_RTOL, atol=1e-7)
    nc.check_best(s, d, ref, tgt, R, dmin, dmax, mask=d != d_ref)


def _mgpu_devices():
    return [0, 1] if _capi.lib().stereo_device_count() >= 2 else [0, 0]


# ---- 1. the exact family where only it can go ---------------------------------------------------------------------------

EXACT_SHAPES = [
    # rows, cols, R, dmin, dmax, output dtype
    (1, 60, 8, -20, 0, np.int32),          # one row
    (1, 75, 11, 0, 30, np.int32),
    (40, 1, 9, -3, 3, np.int32),           # one column
    (12, 10, 8, -6, 6, np.int32),          # cols < 2R + 1
    (7, 50, 10, -15, 0, np.int32),         # rows < 2R + 1
    (9, 33, 15, -12, 12, np.int16),        # both
    (10, 30, 8, 40, 60, np.int32),         # range wholly right of the image
    (10, 30, 8, -70, -45, np.int32),       # range wholly left of the image
    (20, 64, 12, 0, 40, np.int32),         # right-referenced: the last columns read across the row end (zero guard at the end)
    (16, 90, 14, -25, 30, np.int32),       # mixed-sign range
    (6, 300, 8, -200, 0, np.int8),         # D > 127 into int8 (the reference's char store wraps)
    (6, 300, 8, -200, 0, np.int16),
    (5, 260, 13, 0, 180, np.int16),
]


def _check_map(d, d32, dt):
    if np.dtype(dt) == np.int8:
        assert np.array_equal(d, oracle.narrow_i8(d32))
    else:
        assert np.array_equal(d, d32.astype(dt))


@pytest.mark.parametrize("rows,cols,R,dmin,dmax,dt", EXACT_SHAPES)
def test_exact_shapes_ssd_vs_oracle(ctx, rows, cols, R, dmin, dmax, dt):
    L, Rt, _ = synth.make_pair(rows, cols, max(2, min(cols, 40)), 50000 + rows * 31 + cols + R)
    for name, a, b in (("u8", L, Rt), ("noisy", synth.noisy_variant(L, rows), synth.noisy_variant(Rt, cols))):
        af, bf = a.astype(np.float32), b.astype(np.float32)
        d_ref, c_ref = oracle.ssd(af, bf, R, dmin, dmax, return_cost=True)
        d, c = ctx.disparity(sb.COST_SSD, a, b, R, dmin, dmax, dtype=np.int32, return_best=True)
        assert ctx.last_path == sb.PATH_EXACT_F32, name
        bad = np.argwhere(d != d_ref)
        assert bad.size == 0, f"{name}: disparity differs at {bad[:5].tolist()} (of {len(bad)})"
        assert np.array_equal(c, c_ref), name
        if np.dtype(dt) != np.int32:
            _check_map(ctx.disparity(sb.COST_SSD, a, b, R, dmin, dmax, dtype=dt), d_ref, dt)
            assert ctx.last_path == sb.PATH_EXACT_F32, name


@pytest.mark.parametrize("rows,cols,R,dmin,dmax,dt", EXACT_SHAPES)
def test_exact_shapes_ncc_vs_oracle(ctx, rows, cols, R, dmin, dmax, dt):
    L, Rt, _ = synth.make_pair(rows, cols, max(2, min(cols, 40)), 51000 + rows * 31 + cols + R)
    for name, a, b in (("u8", L, Rt), ("noisy", synth.noisy_variant(L, rows), synth.noisy_variant(Rt, cols))):
        af, bf = a.astype(np.float32), b.astype(np.float32)
        try:
            d_ref, s_ref = oracle.ncorr(af, bf, R, dmin, dmax, return_score=True)
        except oracle.OracleError:
            # some pixel has no candidate window: the reference throws inside cv::Mat(Rect), the library refuses the range
            with pytest.raises(sb.StereoError) as e:
                ctx.disparity(sb.COST_NCORR, a, b, R, dmin, dmax, dtype=dt)
            assert e.value.status == RANGE, name
            continue
        d, s = ctx.disparity(sb.COST_NCORR, a, b, R, dmin, dmax, dtype=np.int32, return_best=True)
        assert ctx.last_path == sb.PATH_EXACT_F32, name
        assert_ncc_close(d, s, d_ref, s_ref, af, bf, R, dmin, dmax, "exact")
        if np.dtype(dt) != np.int32:
            _check_map(ctx.disparity(sb.COST_NCORR, a, b, R, dmin, dmax, dtype=dt), d, dt)


def test_exact_shapes_include_an_ncc_refusal_and_a_wrapping_int8_map():
    # (guards the table above against edits that would drop the cases it exists for)
    assert any(dmin > 0 or dmax < 0 for _, _, _, dmin, dmax, _ in EXACT_SHAPES)
    assert any(dmax - dmin > 127 and np.dtype(dt) == np.int8 for *_, dmin, dmax, dt in EXACT_SHAPES)


def test_4096_candidates_fast_4097_exact(ctx):
    rows, cols, R = 4, 6000, 2
    L, Rt, _ = synth.make_pair(rows, cols, 600, 52000)
    Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
    for dmin, path in ((-4095, sb.PATH_FAST_U8), (-4096, sb.PATH_EXACT_F32)):
        d_ref, c_ref = oracle.ssd_fast(Lf, Rf, R, dmin, 0, return_cost=True)
        d, c = ctx.disparity(sb.COST_SSD, L, Rt, R, dmin, 0, dtype=np.int16, return_best=True)
        assert ctx.last_path == path, dmin
        assert np.array_equal(d, d_ref.astype(np.int16)), dmin
        assert np.array_equal(c, c_ref), dmin
        rng = -dmin
        ref_r = oracle.ssd_fast(Rf, Lf, R, 0, rng)
        dl, dr = ctx.disparity_pair(sb.COST_SSD, L, Rt, R, rng, dtype=np.int16)
        assert ctx.last_path == path, rng
        assert np.array_equal(dl, d_ref.astype(np.int16)) and np.array_equal(dr, ref_r.astype(np.int16)), rng


# ---- every entry point that can reach the exact family, at one R > 7 shape ----------------------------------------------

EP_ROWS, EP_COLS, EP_R, EP_RNG = 30, 80, 9, 24
EP_BANDS = ((0, 10), (10, 20), (20, 30))
EP_DT = np.int16


def _ep_images():
    Ls, Rs = zip(*[synth.make_pair(EP_ROWS, EP_COLS, EP_RNG + 1, 53000 + i)[:2] for i in range(3)])
    Ls, Rs = np.stack(Ls), np.stack(Rs)
    Ln = np.stack([synth.noisy_variant(Ls[i], 2 * i) for i in range(3)])
    Rn = np.stack([synth.noisy_variant(Rs[i], 2 * i + 1) for i in range(3)])
    return {"u8": (Ls, Rs), "f32": (Ln, Rn)}


_EP_CACHE = {}


def _ep_refs(cost, kind):
    key = (cost, kind)
    if key not in _EP_CACHE:
        Ls, Rs = _ep_images()[kind]
        fn = oracle.ssd_fast if cost == sb.COST_SSD else oracle.ncorr
        out = []
        for i in range(3):
            a, b = Ls[i].astype(np.float32), Rs[i].astype(np.float32)
            out.append((fn(a, b, EP_R, -EP_RNG, 0), fn(b, a, EP_R, 0, EP_RNG)))
        _EP_CACHE[key] = (Ls, Rs, out)
    return _EP_CACHE[key]


def _same(cost, got, want, ncc=None):
    """SSD: identical maps.  NCC: ncc = (ref, tgt, R, dmin, dmax, family) of the map, checked pixel by pixel (ncc_check)."""
    if cost == sb.COST_SSD:
        bad = np.argwhere(got != want.astype(got.dtype))
        assert bad.size == 0, f"differs at {bad[:5].tolist()} (of {len(bad)})"
    else:
        ref, tgt, R, dmin, dmax, family = ncc
        nc.check_ncc_map(got, ref, tgt, R, dmin, dmax, family, oracle_disp=want)


def _ep(a, b, side):
    """The NCC check arguments of the EP shape's L->R (side 0) or R->L (side 1) map of images a, b (EXACT_F32: R > 7)."""
    a, b = a.astype(np.float32), b.astype(np.float32)
    return (a, b, EP_R, -EP_RNG, 0, "exact") if side == 0 else (b, a, EP_R, 0, EP_RNG, "exact")


def _single_device(ctx, cost, a, b, dmin, dmax, f32):
    torch = _torch()
    ta, tb = torch.from_numpy(np.ascontiguousarray(a)).cuda(), torch.from_numpy(np.ascontiguousarray(b)).cuda()
    out = torch.zeros((EP_ROWS, EP_COLS), dtype=_tdt(EP_DT), device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    fn = _capi.lib().stereo_disparity_f32_device if f32 else _capi.lib().stereo_disparity_u8_device
    step = EP_COLS * a.itemsize
    _ok(fn(ctx.handle, cost, ta.data_ptr(), step, tb.data_ptr(), step, EP_ROWS, EP_COLS, EP_R, dmin, dmax, out.data_ptr(),
           EP_COLS * 2, 2, None, 0, C.c_void_p(st)), "single device")
    ctx.synchronize(st)
    return out.cpu().numpy()


def _pair_entry(ctx, entry, cost, L, Rt):
    """Both maps of one pair (L, Rt of shape (rows, cols)) from `entry`."""
    torch = _torch()
    lib = _capi.lib()
    f32 = L.dtype == np.float32
    step, ostep = EP_COLS * L.itemsize, EP_COLS * 2
    if entry == "pair_host":
        return ctx.disparity_pair(cost, L, Rt, EP_R, EP_RNG, dtype=EP_DT)
    if entry == "band_host":
        dl, dr = np.zeros((EP_ROWS, EP_COLS), EP_DT), np.zeros((EP_ROWS, EP_COLS), EP_DT)
        fn = lib.stereo_disparity_pair_band_f32_host if f32 else lib.stereo_disparity_pair_band_u8_host
        for r0, r1 in EP_BANDS:
            _ok(fn(ctx.handle, cost, L.ctypes.data, step, Rt.ctypes.data, step, EP_ROWS, EP_COLS, r0, r1, EP_R, EP_RNG,
                   dl[r0:].ctypes.data, dr[r0:].ctypes.data, ostep, 2), entry)
        return dl, dr
    tl, tr = torch.from_numpy(np.ascontiguousarray(L)).cuda(), torch.from_numpy(np.ascontiguousarray(Rt)).cuda()
    ol = torch.zeros((EP_ROWS, EP_COLS), dtype=_tdt(EP_DT), device="cuda")
    orr = torch.zeros_like(ol)
    st = torch.cuda.current_stream().cuda_stream
    if entry == "pair_device":
        fn = lib.stereo_disparity_pair_f32_device if f32 else lib.stereo_disparity_pair_u8_device
        _ok(fn(ctx.handle, cost, tl.data_ptr(), step, tr.data_ptr(), step, EP_ROWS, EP_COLS, EP_R, EP_RNG, ol.data_ptr(),
               orr.data_ptr(), ostep, 2, C.c_void_p(st)), entry)
    elif entry == "pair_band_halo_device":
        for r0, r1 in EP_BANDS:
            h0, h1 = C.c_int(), C.c_int()
            _ok(lib.stereo_band_halo_rows(EP_ROWS, r0, r1, EP_R, C.byref(h0), C.byref(h1)))
            _ok(lib.stereo_disparity_pair_band_halo_u8_device(
                ctx.handle, cost, tl[h0.value].data_ptr(), step, tr[h0.value].data_ptr(), step, EP_ROWS, EP_COLS, r0, r1,
                h0.value, h1.value, EP_R, EP_RNG, ol[r0].data_ptr(), orr[r0].data_ptr(), ostep, 2, C.c_void_p(st)), entry)
            assert ctx.last_path == sb.PATH_EXACT_F32
    elif entry in ("band_device", "band_halo_device"):
        for out, a, b, dmin, dmax in ((ol, tl, tr, -EP_RNG, 0), (orr, tr, tl, 0, EP_RNG)):
            for r0, r1 in EP_BANDS:
                if entry == "band_device":
                    _ok(lib.stereo_disparity_band_u8_device(ctx.handle, cost, a.data_ptr(), step, b.data_ptr(), step, EP_ROWS,
                                                            EP_COLS, r0, r1, EP_R, dmin, dmax, out[r0].data_ptr(), ostep, 2,
                                                            C.c_void_p(st)), entry)
                else:
                    h0, h1 = C.c_int(), C.c_int()
                    _ok(lib.stereo_band_halo_rows(EP_ROWS, r0, r1, EP_R, C.byref(h0), C.byref(h1)))
                    _ok(lib.stereo_disparity_band_halo_u8_device(
                        ctx.handle, cost, a[h0.value].data_ptr(), step, b[h0.value].data_ptr(), step, EP_ROWS, EP_COLS, r0, r1,
                        h0.value, h1.value, EP_R, dmin, dmax, out[r0].data_ptr(), ostep, 2, C.c_void_p(st)), entry)
                assert ctx.last_path == sb.PATH_EXACT_F32
    else:
        raise AssertionError(entry)
    ctx.synchronize(st)
    return ol.cpu().numpy(), orr.cpu().numpy()


PAIR_ENTRIES = [("pair_host", "u8"), ("pair_host", "f32"), ("pair_device", "u8"), ("pair_device", "f32"),
                ("band_host", "u8"), ("band_device", "u8"), ("band_halo_device", "u8"), ("pair_band_halo_device", "u8")]


@pytest.mark.parametrize("cost", [sb.COST_SSD, sb.COST_NCORR])
@pytest.mark.parametrize("entry,kind", PAIR_ENTRIES)
def test_every_pair_entry_point_reaches_the_exact_family(ctx, cost, entry, kind):
    Ls, Rs, refs = _ep_refs(cost, kind)
    dl, dr = _pair_entry(ctx, entry, cost, Ls[0], Rs[0])
    assert ctx.last_path == sb.PATH_EXACT_F32
    _same(cost, dl, refs[0][0], _ep(Ls[0], Rs[0], 0))
    _same(cost, dr, refs[0][1], _ep(Ls[0], Rs[0], 1))


@pytest.mark.parametrize("cost", [sb.COST_SSD, sb.COST_NCORR])
@pytest.mark.parametrize("kind", ["u8", "f32"])
def test_single_host_and_device_reach_the_exact_family(ctx, cost, kind):
    Ls, Rs, refs = _ep_refs(cost, kind)
    for side, (a, b, dmin, dmax, want) in enumerate(((Ls[0], Rs[0], -EP_RNG, 0, refs[0][0]), (Rs[0], Ls[0], 0, EP_RNG, refs[0][1]))):
        _same(cost, ctx.disparity(cost, a, b, EP_R, dmin, dmax, dtype=EP_DT), want, _ep(Ls[0], Rs[0], side))
        assert ctx.last_path == sb.PATH_EXACT_F32
        _same(cost, _single_device(ctx, cost, a, b, dmin, dmax, kind == "f32"), want, _ep(Ls[0], Rs[0], side))
        assert ctx.last_path == sb.PATH_EXACT_F32


@pytest.mark.parametrize("cost", [sb.COST_SSD, sb.COST_NCORR])
@pytest.mark.parametrize("entry,kind", [("batch_host", "u8"), ("batch_host", "f32"), ("batch_device", "u8"),
                                        ("mgpu_batch", "u8"), ("mgpu_batch", "f32"), ("mgpu_bands", "u8"), ("mgpu_bands", "f32")])
def test_batch_and_multi_gpu_entry_points_reach_the_exact_family(ctx, cost, entry, kind):
    Ls, Rs, refs = _ep_refs(cost, kind)
    n = len(Ls)
    if entry == "batch_host":
        bl, br = ctx.disparity_pair_batch(cost, Ls, Rs, EP_R, EP_RNG, dtype=EP_DT)
        assert ctx.last_path == sb.PATH_EXACT_F32
    elif entry == "batch_device":
        torch = _torch()
        tl, tr = torch.from_numpy(Ls).cuda(), torch.from_numpy(Rs).cuda()
        ol = torch.zeros((n, EP_ROWS, EP_COLS), dtype=torch.int16, device="cuda")
        orr = torch.zeros_like(ol)
        st = torch.cuda.current_stream().cuda_stream
        _ok(_capi.lib().stereo_disparity_pair_batch_u8_device(
            ctx.handle, cost, n, tl.data_ptr(), tr.data_ptr(), EP_COLS, EP_ROWS * EP_COLS, EP_ROWS, EP_COLS, EP_R, EP_RNG,
            ol.data_ptr(), orr.data_ptr(), EP_COLS * 2, EP_ROWS * EP_COLS * 2, 2, C.c_void_p(st)), entry)
        ctx.synchronize(st)
        assert ctx.last_path == sb.PATH_EXACT_F32
        bl, br = ol.cpu().numpy(), orr.cpu().numpy()
    else:
        with sb.MultiGpu(_mgpu_devices()) as mg:
            if entry == "mgpu_batch":
                bl, br = mg.disparity_pair_batch(cost, Ls, Rs, EP_R, EP_RNG, dtype=EP_DT)
            else:
                pairs = [mg.disparity_pair_bands(cost, Ls[i], Rs[i], EP_R, EP_RNG, dtype=EP_DT) for i in range(n)]
                bl, br = np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs])
    for i in range(n):
        _same(cost, bl[i], refs[i][0], _ep(Ls[i], Rs[i], 0))
        _same(cost, br[i], refs[i][1], _ep(Ls[i], Rs[i], 1))


def test_pair_band_f32_host_refuses_images_that_are_not_8bit(ctx):
    Ls, Rs, _ = _ep_refs(sb.COST_SSD, "f32")
    dl, dr = np.zeros((EP_ROWS, EP_COLS), EP_DT), np.zeros((EP_ROWS, EP_COLS), EP_DT)
    rc = _capi.lib().stereo_disparity_pair_band_f32_host(
        ctx.handle, sb.COST_SSD, Ls[0].ctypes.data, EP_COLS * 4, Rs[0].ctypes.data, EP_COLS * 4, EP_ROWS, EP_COLS, 0, 10, EP_R,
        EP_RNG, dl.ctypes.data, dr.ctypes.data, EP_COLS * 2, 2)
    assert rc == UNSUP
    # the same entry point on 8-bit-valued CV_32FC1 images takes the exact family band by band
    Lu, Ru, refs = _ep_refs(sb.COST_SSD, "u8")
    gl, gr = _pair_entry(ctx, "band_host", sb.COST_SSD, Lu[0].astype(np.float32), Ru[0].astype(np.float32))
    assert ctx.last_path == sb.PATH_EXACT_F32
    _same(sb.COST_SSD, gl, refs[0][0])
    _same(sb.COST_SSD, gr, refs[0][1])


@pytest.mark.parametrize("fuse", [True, False])
def test_exact_pair_with_lr_check_and_speckle_filter(ctx, fuse):
    rows, cols, R, rng, lr_diff, spk_size, spk_diff = 40, 120, 9, 24, 1, 30, 1
    L, Rt, _ = synth.make_pair(rows, cols, rng + 1, 54000)
    Lf, Rf = synth.noisy_variant(L, 3, sigma=6.0), synth.noisy_variant(Rt, 4, sigma=6.0)
    ref_l, ref_r = oracle.ssd_fast(Lf, Rf, R, -rng, 0), oracle.ssd_fast(Rf, Lf, R, 0, rng)
    cl, cr = lr_check(ref_l.astype(np.int16), ref_r.astype(np.int16), rng, lr_diff)
    sentinel = -(rng + 1)
    want_l, want_r = filter_speckles(cl, sentinel, spk_size, spk_diff), filter_speckles(cr, sentinel, spk_size, spk_diff)
    assert (want_l == sentinel).any() and (want_l != sentinel).any()
    try:
        ctx.set_fuse_pairs(fuse)
        ctx.set_lr_check(lr_diff)
        ctx.set_speckle_filter(spk_size, spk_diff)
        dl, dr = ctx.disparity_pair(sb.COST_SSD, Lf, Rf, R, rng, dtype=np.int16)
        assert ctx.last_path == sb.PATH_EXACT_F32
    finally:
        ctx.set_speckle_filter(None)
        ctx.set_lr_check(None)
        ctx.set_fuse_pairs(True)
    assert np.array_equal(dl, want_l) and np.array_equal(dr, want_r)


def test_all_candidates_at_or_above_99999999_keep_disparity_0(ctx):
    rows, cols, R, dmin = 48, 120, 7, -20
    L, Rt = ec.the_99999999_pair(rows, cols, 55000)
    assert not ec.ssd_fast_f32_admits(float(min(L.min(), Rt.min())), float(max(L.max(), Rt.max())), R)
    d_ref, c_ref = oracle.ssd_fast(L, Rt, R, dmin, 0, return_cost=True)
    hot = (c_ref == ec.SSD_NO_CANDIDATE) & (d_ref == 0)
    cool = c_ref < ec.SSD_NO_CANDIDATE
    assert (hot[:, :-1] & cool[:, 1:]).any() or (hot[:, 1:] & cool[:, :-1]).any(), "no pixel at the threshold next to one below"
    d, c = ctx.disparity(sb.COST_SSD, L, Rt, R, dmin, 0, dtype=np.int32, return_best=True)
    assert ctx.last_path == sb.PATH_EXACT_F32
    assert np.array_equal(d, d_ref) and np.array_equal(c, c_ref)
    assert np.array_equal((c == ec.SSD_NO_CANDIDATE) & (d == 0), hot)
    dl, dr = ctx.disparity_pair(sb.COST_SSD, L, Rt, R, -dmin, dtype=np.int16)
    assert ctx.last_path == sb.PATH_EXACT_F32
    assert np.array_equal(dl, d_ref.astype(np.int16))
    assert np.array_equal(dr, oracle.ssd_fast(Rt, L, R, 0, -dmin).astype(np.int16))


# ---- 2. the FAST_F32 / EXACT_F32 line for SSD -------------------------------------------------------------------------

EDGE_RADII = [0, 1, 3, 5, 7]
EDGE_RNG = 24


def _edge_pair(R, side):
    inside, outside = ec.ssd_edge(R)
    top = inside if side == "inside" else outside
    return ec.ssd_edge_pair(R, top, 2 * (2 * R + 3) + 14, 90, 56000 + R)


@pytest.mark.parametrize("side", ["inside", "outside"])
@pytest.mark.parametrize("R", EDGE_RADII)
def test_ssd_float_family_bound_at_its_edge(ctx, R, side):
    L, Rt = _edge_pair(R, side)
    path = sb.PATH_FAST_F32 if side == "inside" else sb.PATH_EXACT_F32
    ref_l, cost_l = oracle.ssd_fast(L, Rt, R, -EDGE_RNG, 0, return_cost=True)
    ref_r, cost_r = oracle.ssd_fast(Rt, L, R, 0, EDGE_RNG, return_cost=True)
    # single calls, both directions, with costs
    for a, b, dmin, dmax, d_ref, c_ref in ((L, Rt, -EDGE_RNG, 0, ref_l, cost_l), (Rt, L, 0, EDGE_RNG, ref_r, cost_r)):
        d, c = ctx.disparity(sb.COST_SSD, a, b, R, dmin, dmax, dtype=np.int32, return_best=True)
        assert ctx.last_path == path
        bad = np.argwhere(d != d_ref)
        assert bad.size == 0, f"disparity differs at {bad[:5].tolist()} (of {len(bad)})"
        bad = np.argwhere(c != c_ref)
        assert bad.size == 0, f"cost differs at {bad[:5].tolist()} (of {len(bad)})"
        torch = _torch()
        ta, tb = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
        od = torch.zeros(a.shape, dtype=torch.int32, device="cuda")
        oc = torch.zeros(a.shape, dtype=torch.int32, device="cuda")
        st = torch.cuda.current_stream().cuda_stream
        cols = a.shape[1]
        _ok(_capi.lib().stereo_disparity_f32_device(ctx.handle, sb.COST_SSD, ta.data_ptr(), cols * 4, tb.data_ptr(), cols * 4,
                                                    a.shape[0], cols, R, dmin, dmax, od.data_ptr(), cols * 4, 4, oc.data_ptr(),
                                                    cols * 4, C.c_void_p(st)), "stereo_disparity_f32_device")
        ctx.synchronize(st)
        assert ctx.last_path == path
        assert np.array_equal(od.cpu().numpy(), d_ref) and np.array_equal(oc.cpu().numpy(), c_ref)
    # pair calls, fused and unfused, host and device
    try:
        for fuse in (True, False):
            ctx.set_fuse_pairs(fuse)
            dl, dr = ctx.disparity_pair(sb.COST_SSD, L, Rt, R, EDGE_RNG, dtype=np.int16)
            assert ctx.last_path == path
            if side == "inside":
                assert ctx.last_fused_pairs == int(fuse)
            assert np.array_equal(dl, ref_l.astype(np.int16)) and np.array_equal(dr, ref_r.astype(np.int16)), fuse
            torch = _torch()
            tl, tr = torch.from_numpy(L).cuda(), torch.from_numpy(Rt).cuda()
            ol = torch.zeros(L.shape, dtype=torch.int16, device="cuda")
            orr = torch.zeros_like(ol)
            st = torch.cuda.current_stream().cuda_stream
            cols = L.shape[1]
            _ok(_capi.lib().stereo_disparity_pair_f32_device(ctx.handle, sb.COST_SSD, tl.data_ptr(), cols * 4, tr.data_ptr(),
                                                             cols * 4, L.shape[0], cols, R, EDGE_RNG, ol.data_ptr(),
                                                             orr.data_ptr(), cols * 2, 2, C.c_void_p(st)), "pair f32 device")
            ctx.synchronize(st)
            assert ctx.last_path == path
            assert np.array_equal(ol.cpu().numpy(), ref_l.astype(np.int16)), fuse
            assert np.array_equal(orr.cpu().numpy(), ref_r.astype(np.int16)), fuse
    finally:
        ctx.set_fuse_pairs(True)
    # forcing the float family onto images beyond its bound is refused, not answered with a wrapped map
    try:
        ctx.force_path(sb.PATH_FAST_F32)
        if side == "inside":
            d = ctx.disparity(sb.COST_SSD, L, Rt, R, -EDGE_RNG, 0, dtype=np.int32)
            assert ctx.last_path == sb.PATH_FAST_F32 and np.array_equal(d, ref_l)
        else:
            with pytest.raises(sb.StereoError) as e:
                ctx.disparity(sb.COST_SSD, L, Rt, R, -EDGE_RNG, 0, dtype=np.int32)
            assert e.value.status == UNSUP
            with pytest.raises(sb.StereoError) as e:
                ctx.disparity_pair(sb.COST_SSD, L, Rt, R, EDGE_RNG, dtype=np.int16)
            assert e.value.status == UNSUP
    finally:
        ctx.force_path(0)


# ---- 3. classification edge values ------------------------------------------------------------------------------------

CLS_SHAPES = [(21, 45), (13, 70)]          # neither a multiple of the 32 x 8 classification block
CLS_R, CLS_DMIN = 2, -10


def _positions(rows, cols):
    # the first block, the last block (partial in both dimensions) and a block partial in its columns only
    return [(0, 0), (rows - 1, cols - 1), (rows // 2, cols - 2)]


CLS_VALUES = [(-0.0, sb.PATH_FAST_U8), (255.0, sb.PATH_FAST_U8), (np.nextafter(np.float32(255), np.float32(256)), sb.PATH_FAST_F32),
              (256.0, sb.PATH_FAST_F32), (-1.0, sb.PATH_FAST_F32), (np.float32(1e-45), sb.PATH_FAST_F32)]


@pytest.mark.parametrize("rows,cols", CLS_SHAPES)
@pytest.mark.parametrize("value,path", CLS_VALUES, ids=["-0", "255", "255+ulp", "256", "-1", "denormal"])
def test_single_edge_value_classifies_and_matches_the_oracle(ctx, rows, cols, value, path):
    L, Rt, _ = synth.make_pair(rows, cols, 12, 57000 + rows + cols)
    for k, (y, x) in enumerate(_positions(rows, cols)):
        Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
        (Lf if k % 2 == 0 else Rf)[y, x] = np.float32(value)
        d_ref, c_ref = oracle.ssd(Lf, Rf, CLS_R, CLS_DMIN, 0, return_cost=True)
        d, c = ctx.disparity(sb.COST_SSD, Lf, Rf, CLS_R, CLS_DMIN, 0, dtype=np.int32, return_best=True)
        assert ctx.last_path == path, (y, x)
        assert np.array_equal(d, d_ref) and np.array_equal(c, c_ref), (y, x)
        dl, dr = ctx.disparity_pair(sb.COST_SSD, Lf, Rf, CLS_R, -CLS_DMIN, dtype=np.int16)
        assert ctx.last_path == path, (y, x)
        assert np.array_equal(dl, d_ref.astype(np.int16)), (y, x)
        assert np.array_equal(dr, oracle.ssd(Rf, Lf, CLS_R, 0, -CLS_DMIN).astype(np.int16)), (y, x)
        n_ref, s_ref = oracle.ncorr(Lf, Rf, CLS_R, CLS_DMIN, 0, return_score=True)
        n, s = ctx.disparity(sb.COST_NCORR, Lf, Rf, CLS_R, CLS_DMIN, 0, dtype=np.int32, return_best=True)
        assert ctx.last_path == path, (y, x)
        assert_ncc_close(n, s, n_ref, s_ref, Lf, Rf, CLS_R, CLS_DMIN, 0, nc.family_of(ctx))


@pytest.mark.parametrize("rows,cols", CLS_SHAPES)
def test_edge_value_in_a_partial_block_decides_the_family(ctx, rows, cols):
    # one pixel at the SSD bound of R = 7, alone in a block the image only partly covers: the block's range must count
    R = 7
    inside, outside = ec.ssd_edge(R)
    L, Rt, _ = synth.make_pair(rows, cols, 12, 58000 + rows + cols)
    for y, x in _positions(rows, cols)[1:]:
        for v, path in ((inside, sb.PATH_FAST_F32), (outside, sb.PATH_EXACT_F32)):
            Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
            Rf[y, x] = v
            d_ref, c_ref = oracle.ssd(Lf, Rf, R, -8, 0, return_cost=True)
            d, c = ctx.disparity(sb.COST_SSD, Lf, Rf, R, -8, 0, dtype=np.int32, return_best=True)
            assert ctx.last_path == path, (y, x, v)
            assert np.array_equal(d, d_ref) and np.array_equal(c, c_ref), (y, x, v)


@pytest.mark.parametrize("rows,cols", CLS_SHAPES)
@pytest.mark.parametrize("value", [np.inf, -np.inf, np.nan], ids=["+inf", "-inf", "nan"])
def test_non_finite_pixel_routes_to_the_exact_family(ctx, rows, cols, value):
    L, Rt, _ = synth.make_pair(rows, cols, 12, 59000 + rows + cols)
    for k, (y, x) in enumerate(_positions(rows, cols)):
        Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
        (Lf if k % 2 == 0 else Rf)[y, x] = np.float32(value)
        # rows whose windows (and the SSD's reads across the row end) cannot reach row y: there the reference is defined
        clean = np.abs(np.arange(rows) - y) > CLS_R + 1
        assert clean.any()
        d_ref, c_ref = oracle.ssd(Lf, Rf, CLS_R, CLS_DMIN, 0, return_cost=True)
        d, c = ctx.disparity(sb.COST_SSD, Lf, Rf, CLS_R, CLS_DMIN, 0, dtype=np.int32, return_best=True)
        assert ctx.last_path == sb.PATH_EXACT_F32, (y, x)
        assert np.array_equal(d[clean], d_ref[clean]) and np.array_equal(c[clean], c_ref[clean]), (y, x)
        dl, dr = ctx.disparity_pair(sb.COST_SSD, Lf, Rf, CLS_R, -CLS_DMIN, dtype=np.int16)
        assert ctx.last_path == sb.PATH_EXACT_F32, (y, x)
        assert np.array_equal(dl[clean], d_ref[clean].astype(np.int16)), (y, x)
        n_ref, s_ref = oracle.ncorr(Lf, Rf, CLS_R, CLS_DMIN, 0, return_score=True)
        n, s = ctx.disparity(sb.COST_NCORR, Lf, Rf, CLS_R, CLS_DMIN, 0, dtype=np.int32, return_best=True)
        assert ctx.last_path == sb.PATH_EXACT_F32, (y, x)
        # (the exact kernels ARE the literal oracle: identical wherever the reference is defined)
        assert np.array_equal(n[clean], n_ref[clean]), (y, x)
        assert np.array_equal(s[clean].view(np.uint32), s_ref[clean].view(np.uint32)), (y, x)


@pytest.mark.parametrize("cost", [sb.COST_SSD, sb.COST_NCORR])
def test_host_f32_batch_with_one_exact_pair(ctx, cost):
    n, rows, cols, R, rng = 5, 30, 110, 3, 17
    Ls, Rs = zip(*[synth.make_pair(rows, cols, 12, 60000 + i)[:2] for i in range(n)])
    Ls, Rs = np.stack(Ls).astype(np.float32), np.stack(Rs).astype(np.float32)
    Ls[2] *= np.float32(5.0)                           # beyond the FAST_F32 bound of R = 3 (827.25)
    assert not ec.ssd_fast_f32_admits(0.0, float(Ls[2].max()), R)
    bl, br = ctx.disparity_pair_batch(cost, Ls, Rs, R, rng, dtype=np.int16)
    fn = oracle.ssd_fast if cost == sb.COST_SSD else oracle.ncorr
    for i in range(n):
        want_l, want_r = fn(Ls[i], Rs[i], R, -rng, 0), fn(Rs[i], Ls[i], R, 0, rng)
        # NCC: pair 2 (x5, not 8-bit) takes the float kernels, the others the packed ones, fused or not ("u8" covers both)
        family = "f32" if i == 2 else "u8"
        _same(cost, bl[i], want_l, (Ls[i], Rs[i], R, -rng, 0, family))
        _same(cost, br[i], want_r, (Rs[i], Ls[i], R, 0, rng, family))
    dl, _ = ctx.disparity_pair(cost, Ls[2], Rs[2], R, rng, dtype=np.int16)
    assert ctx.last_path == (sb.PATH_EXACT_F32 if cost == sb.COST_SSD else sb.PATH_FAST_F32)
    assert np.array_equal(dl, bl[2])


# ---- 4. the float NCC family across value offsets ---------------------------------------------------------------------

NCC_OFFSETS = [0.0, 300.0, 1e3, 1e4, 1e5, 9.9e5]
NCC_SHAPE = (24, 160, 3, 40)                # rows, cols, R, D


def _ncc_case(offset=0.0, gain=1.0):
    rows, cols, R, D = NCC_SHAPE
    L, Rt, _ = synth.make_pair(rows, cols, D + 1, 61000)
    return ec.ncc_offset_pair(L, Rt, offset, gain)


def _ncc_agreement(ctx, Lf, Rf):
    """(agreement of the single call, of the pair call's two maps) with the literal oracle; asserts the contract."""
    _, _, R, D = NCC_SHAPE
    d_ref, s_ref = oracle.ncorr(Lf, Rf, R, -D, 0, return_score=True)
    r_ref = oracle.ncorr(Rf, Lf, R, 0, D)
    d, s = ctx.disparity(sb.COST_NCORR, Lf, Rf, R, -D, 0, dtype=np.int32, return_best=True)
    path, family = ctx.last_path, nc.family_of(ctx)
    dl, dr = ctx.disparity_pair(sb.COST_NCORR, Lf, Rf, R, D, dtype=np.int16)
    assert ctx.last_path == path
    pair_family = nc.family_of(ctx)
    agree = (float(np.mean(d == d_ref)), float(np.mean(dl == d_ref)), float(np.mean(dr == r_ref)))
    print(f"NCC agreement path={path} single={agree[0]:.5f} pair L->R={agree[1]:.5f} R->L={agree[2]:.5f}")
    assert_ncc_close(d, s, d_ref, s_ref, Lf, Rf, R, -D, 0, family)
    nc.check_ncc_map(dl, Lf, Rf, R, -D, 0, pair_family, oracle_disp=d_ref, what="pair L->R")
    nc.check_ncc_map(dr, Rf, Lf, R, 0, D, pair_family, oracle_disp=r_ref, what="pair R->L")
    return path


@pytest.mark.parametrize("offset", NCC_OFFSETS)
def test_ncc_float_family_across_offsets(ctx, offset):
    # an offset crowds every score towards 1: from ~1e3 up the float keys no longer resolve the oracle's first maximum on
    # >= 99.9 % of the pixels, so those images go to the exact kernels (ec.ncc_score_band)
    Lf, Rf = _ncc_case(offset)
    band = ec.ncc_score_band(float(min(Lf.min(), Rf.min())), float(max(Lf.max(), Rf.max())))
    want = sb.PATH_FAST_U8 if offset == 0 else sb.PATH_FAST_F32 if band >= ec.NCC_MIN_SCORE_BAND else sb.PATH_EXACT_F32
    if offset == 300:
        assert want == sb.PATH_FAST_F32
    if offset >= 1e3:
        assert want == sb.PATH_EXACT_F32
    assert _ncc_agreement(ctx, Lf, Rf) == want


def test_ncc_float_family_at_a_gain_that_reaches_1e6(ctx):
    top = float(max(_ncc_case()[0].max(), _ncc_case()[1].max()))
    Lf, Rf = _ncc_case(gain=float(np.floor(999000.0 / top)))
    assert 0.99e6 < max(Lf.max(), Rf.max()) < 1e6
    assert _ncc_agreement(ctx, Lf, Rf) == sb.PATH_FAST_F32


def test_reference_noise_and_contrast_variants_stay_on_the_float_family(ctx):
    rows, cols, R, D = NCC_SHAPE
    L, Rt, _ = synth.make_pair(rows, cols, D + 1, 62000)
    for name, Lf, Rf in (("noisy", synth.noisy_variant(L, 1), synth.noisy_variant(Rt, 2)),
                         ("contrast", synth.contrast_variant(L), Rt.astype(np.float32)),
                         ("noisy+contrast", synth.noisy_variant(L, 1) * np.float32(1.1), synth.noisy_variant(Rt, 2))):
        for cost in (sb.COST_SSD, sb.COST_NCORR):
            ctx.disparity(cost, Lf, Rf, R, -D, 0, dtype=np.int16)
            assert ctx.last_path == sb.PATH_FAST_F32, (name, cost)
            ctx.disparity_pair(cost, Lf, Rf, R, D, dtype=np.int16)
            assert ctx.last_path == sb.PATH_FAST_F32, (name, cost)
