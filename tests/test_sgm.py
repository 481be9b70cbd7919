"""Semi-global matching on the B200 (stereo_ctx_set_sgm): every pair entry point against the numpy restatement
(sgm_oracle), alone and followed by the left-right check and the speckle filter; the zero-penalty identity with the
block matcher's maps on every kernel family and at 4K / 256; a full-size 720p case; the rejections, which write nothing;
the setting and its default and off states; and a CUDA graph replay of a device pair call."""
import ctypes as C

import numpy as np
import pytest

import introtocomputervision_b200 as sb
from introtocomputervision_b200 import _capi, synth
from lr_oracle import lr_check
from sgm_oracle import sgm_pair
from speckle_oracle import filter_speckles
from pair_calls import FAMILIES, RANGE_T, _device_batch, _images, _run

pytestmark = pytest.mark.gpu

ARG, UNSUP = _capi.ERR_INVALID_ARG, _capi.ERR_UNSUPPORTED
ENTRIES = ["pair_host", "pair_device", "batch_device", "batch_host", "band_host", "band_halo_device", "mgpu_batch"]


def _torch():
    import torch
    return torch


def _ok(rc, where=""):
    assert rc == _capi.STEREO_OK, f"{where}: {rc} ({_capi.last_error()})"


@pytest.fixture(scope="module")
def gctx():
    c = sb.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def mg():
    m = sb.MultiGpu([0, 0])
    yield m
    m.close()


def _kind_images(kind, n, seed):
    if kind == "contrast":
        Ls, Rs = _images("f32", n, seed)
        return (Ls * np.float32(1.1)).astype(np.float32), Rs
    return _images(kind, n, seed)


def _expected(Ls, Rs, R, rng, dt, paths, p1, p2, lr, spk):
    out = []
    for L, Rt in zip(Ls, Rs):
        dl, dr = (d.astype(dt) for d in sgm_pair(L, Rt, R, rng, paths, p1, p2))
        if lr:
            dl, dr = lr_check(dl, dr, rng, 1)
        if spk:
            dl, dr = filter_speckles(dl, -(rng + 1), 20, 1), filter_speckles(dr, -(rng + 1), 20, 1)
        out.append((np.asarray(dl, dt), np.asarray(dr, dt)))
    return out


def _set(h, paths, p1, p2, lr, spk):
    h.set_sgm(paths, p1, p2)
    h.set_lr_check(1 if lr else None)
    h.set_speckle_filter(20 if spk else None, 1)


def _reset(h):
    h.set_sgm(None)
    h.set_lr_check(None)
    h.set_speckle_filter(None)


# paths, P1, P2, R, range, map type, left-right check, speckle filter
CONFIGS = [(4, 3, 40, 0, RANGE_T, np.int8, False, False),
           (8, 10, 120, 1, RANGE_T, np.int16, True, False),
           (8, 5, 5, 3, 140, np.int16, False, True),
           (4, 0, 300, 7, RANGE_T, np.int32, True, True)]


# ---- 1. every pair entry point against the restatement ----------------------------------------------------------------

@pytest.mark.parametrize("kind", ["u8", "f32", "noisy", "contrast"])
@pytest.mark.parametrize("entry", ENTRIES)
def test_every_pair_entry_point_equals_the_restatement(gctx, mg, entry, kind):
    if kind != "u8" and entry in ("batch_device", "band_halo_device"):
        pytest.skip("8-bit device entry point")
    if kind in ("noisy", "contrast") and entry == "band_host":
        pytest.skip("the host row-band entry points take 8-bit-valued images only")
    h = mg if entry.startswith("mgpu_") else gctx
    n = 3 if "batch" in entry else 1
    Ls, Rs = _kind_images(kind, n, 700 + 7 * ENTRIES.index(entry))
    for paths, p1, p2, R, rng, dt, lr, spk in CONFIGS:
        _set(h, paths, p1, p2, lr, spk)
        try:
            on = _run(h, entry, sb.COST_SSD, Ls, Rs, R, rng, dt, bands=[(0, Ls.shape[1])])
        finally:
            _reset(h)
        want = _expected(Ls, Rs, R, rng, dt, paths, p1, p2, lr, spk)
        for i in range(n):
            for side in (0, 1):
                bad = np.argwhere(on[side][i] != want[i][side])
                assert bad.size == 0, f"{entry} {kind} {paths}/{p1}/{p2} R{R} rng{rng} pair {i} map {side}: {bad[:5].tolist()} of {len(bad)}"
        if not isinstance(h, sb.MultiGpu):
            assert h.last_path == sb.PATH_SGM


@pytest.mark.parametrize("entry", ["pair_device", "pair_host", "batch_device"])
def test_a_range_wider_than_the_image(gctx, entry):
    L, Rt, _ = synth.make_pair(12, 40, 10, 91)
    for paths, p1, p2, R in ((4, 2, 30, 1), (8, 9, 70, 3)):
        rng = 60
        gctx.set_sgm(paths, p1, p2)
        try:
            on = _run(gctx, entry, sb.COST_SSD, L[None], Rt[None], R, rng, np.int16)
        finally:
            gctx.set_sgm(None)
        dl, dr = sgm_pair(L, Rt, R, rng, paths, p1, p2)
        assert np.array_equal(on[0][0], dl) and np.array_equal(on[1][0], dr), (entry, paths, R)


# rows, cols, R, range, paths, P1, P2: widths that leave a partial last cost block (x0 > 0) and 6, 7, 10 and 16 candidates
# per lane of the path kernels
ODD_SHAPES = [(24, 300, 2, 200, 4, 5, 60), (20, 1000, 1, 300, 8, 7, 90), (12, 600, 3, 511, 4, 3, 50), (30, 333, 0, 170, 8, 2, 20)]


@pytest.mark.parametrize("entry", ["pair_device", "pair_host"])
@pytest.mark.parametrize("shape", ODD_SHAPES)
def test_odd_widths_and_wide_ranges_equal_the_restatement(gctx, shape, entry):
    rows, cols, R, rng, paths, p1, p2 = shape
    L, Rt, _ = synth.make_pair(rows, cols, min(rng, 60), 600 + cols)
    if entry == "pair_host":
        L, Rt = L.astype(np.float32), (Rt.astype(np.float32) * np.float32(1.1)).astype(np.float32)
    gctx.set_sgm(paths, p1, p2)
    try:
        on = _run(gctx, entry, sb.COST_SSD, L[None], Rt[None], R, rng, np.int16)
        assert gctx.last_path == sb.PATH_SGM
    finally:
        gctx.set_sgm(None)
    dl, dr = sgm_pair(L, Rt, R, rng, paths, p1, p2)
    for got, want, side in ((on[0][0], dl, "left"), (on[1][0], dr, "right")):
        bad = np.argwhere(got != want)
        assert bad.size == 0, f"{shape} {entry} {side}: {bad[:5].tolist()} of {len(bad)}"


# ---- 2. zero penalties: the block matcher's maps -----------------------------------------------------------------------

@pytest.mark.parametrize("paths", [4, 8])
@pytest.mark.parametrize("family", list(FAMILIES))
@pytest.mark.parametrize("entry", ["pair_device", "pair_host", "batch_device", "batch_host"])
def test_zero_penalties_equal_the_maps_without_sgm(gctx, entry, family, paths):
    kind, win, dt = FAMILIES[family]
    if kind != "u8" and entry == "batch_device":
        pytest.skip("8-bit device entry point")
    n = 3 if "batch" in entry else 1
    Ls, Rs = _images(kind, n, 40 + paths)
    off = _run(gctx, entry, sb.COST_SSD, Ls, Rs, win, RANGE_T, dt)
    gctx.set_sgm(paths, 0, 0)
    try:
        on = _run(gctx, entry, sb.COST_SSD, Ls, Rs, win, RANGE_T, dt)
    finally:
        gctx.set_sgm(None)
    assert np.array_equal(on[0], off[0]) and np.array_equal(on[1], off[1])


def test_zero_penalties_equal_the_maps_without_sgm_4k(gctx):
    rows, cols, nd, win = 2160, 3840, 256, 5
    L, Rt, _ = synth.make_pair(rows, cols, nd, 4096)
    off = gctx.disparity_pair(sb.COST_SSD, L, Rt, win, nd - 1, dtype=np.int16)
    gctx.set_sgm(8, 0, 0)
    try:
        on = gctx.disparity_pair(sb.COST_SSD, L, Rt, win, nd - 1, dtype=np.int16)
    finally:
        gctx.set_sgm(None)
    assert np.array_equal(on[0], off[0]) and np.array_equal(on[1], off[1])


# ---- 3. full size ------------------------------------------------------------------------------------------------------

def test_full_size_720p_batch_equals_the_restatement(gctx):
    rows, cols, nd, win, paths, p1, p2 = 720, 1280, 64, 4, 8, 10, 150
    pairs = [synth.make_pair(rows, cols, nd, 70 + i)[:2] for i in range(2)]
    Ls, Rs = np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs])
    gctx.set_sgm(paths, p1, p2)
    try:
        on = _device_batch(gctx, Ls, Rs, win, nd, 1)
    finally:
        gctx.set_sgm(None)
    for i in range(2):
        dl, dr = sgm_pair(Ls[i], Rs[i], win, nd, paths, p1, p2)
        assert np.array_equal(on[0, i], dl.astype(np.int8)) and np.array_equal(on[1, i], dr.astype(np.int8)), i


# ---- 4. rejections -----------------------------------------------------------------------------------------------------

def _untouched_call(h, entry, Ls, Rs, R, rng, cost=sb.COST_SSD, dt=np.int16):
    """Calls the entry point on outputs filled with 0x3C; returns (status, outputs untouched)."""
    torch = _torch()
    lib = _capi.lib()
    n, rows, cols = Ls.shape
    elem = np.dtype(dt).itemsize
    f32 = Ls.dtype == np.float32
    step = cols * Ls.itemsize
    if entry in ("pair_device", "batch_device"):
        tl, tr = torch.from_numpy(Ls).cuda(), torch.from_numpy(Rs).cuda()
        out = torch.full((2, n, rows, cols * elem), 0x3C, dtype=torch.uint8, device="cuda")
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        if entry == "pair_device":
            fn = lib.stereo_disparity_pair_f32_device if f32 else lib.stereo_disparity_pair_u8_device
            rc = fn(h.handle, cost, tl.data_ptr(), step, tr.data_ptr(), step, rows, cols, R, rng, out[0].data_ptr(), out[1].data_ptr(),
                    cols * elem, elem, st)
        else:
            rc = lib.stereo_disparity_pair_batch_u8_device(h.handle, cost, n, tl.data_ptr(), tr.data_ptr(), cols, rows * cols, rows, cols,
                                                           R, rng, out[0].data_ptr(), out[1].data_ptr(), cols * elem, rows * cols * elem,
                                                           elem, st)
        torch.cuda.synchronize()
        return rc, bool((out == 0x3C).all().item())
    out = np.full((2, n, rows, cols * elem), 0x3C, np.uint8)
    handle = h._h if isinstance(h, sb.MultiGpu) else h.handle
    if entry == "pair_host":
        fn = lib.stereo_disparity_pair_f32_host if f32 else lib.stereo_disparity_pair_u8_host
        rc = fn(handle, cost, Ls.ctypes.data, step, Rs.ctypes.data, step, rows, cols, R, rng, out[0].ctypes.data, out[1].ctypes.data,
                cols * elem, elem)
    else:
        prefix = "stereo_mgpu_" if entry == "mgpu_batch" else "stereo_"
        fn = getattr(lib, prefix + ("disparity_pair_batch_f32_host" if f32 else "disparity_pair_batch_u8_host"))
        rc = fn(handle, cost, n, Ls.ctypes.data, Rs.ctypes.data, step, rows * step, rows, cols, R, rng, out[0].ctypes.data,
                out[1].ctypes.data, cols * elem, rows * cols * elem, elem)
    return rc, bool((out == 0x3C).all())


HOST_ENTRIES = ["pair_host", "batch_host", "mgpu_batch"]


@pytest.mark.parametrize("entry", ["pair_device", "batch_device"] + HOST_ENTRIES)
def test_ncc_is_rejected_and_writes_nothing(gctx, mg, entry):
    h = mg if entry.startswith("mgpu_") else gctx
    Ls, Rs = _images("u8", 2, 5)
    h.set_sgm(4, 1, 10)
    try:
        rc, untouched = _untouched_call(h, entry, Ls, Rs, 3, RANGE_T, cost=sb.COST_NCORR)
        assert rc == UNSUP and untouched, (entry, rc)
        assert "SSD" in _capi.last_error()
        rc, untouched = _untouched_call(h, entry, Ls, Rs, 3, RANGE_T)            # SSD is served
        _ok(rc, entry)
        assert not untouched
    finally:
        h.set_sgm(None)


@pytest.mark.parametrize("paths", [4, 8])
def test_the_int32_bound_is_exact_for_8bit_images(gctx, paths):
    Ls, Rs = _images("u8", 1, 9)
    Ls, Rs = Ls[:, :20, :90].copy(), Rs[:, :20, :90].copy()
    for R in (20, 31):
        w2 = (2 * R + 1) ** 2
        p2 = (2 ** 31 - 1) // paths - w2 * 255 ** 2
        if p2 < 0:
            continue
        for entry in ("pair_device", "batch_device", "pair_host"):
            gctx.set_sgm(paths, 0, p2)
            try:
                rc, _ = _untouched_call(gctx, entry, Ls, Rs, R, 10)
                _ok(rc, f"{entry} at the bound")
                gctx.set_sgm(paths, 0, p2 + 1)
                rc, untouched = _untouched_call(gctx, entry, Ls, Rs, R, 10)
                assert rc == UNSUP and untouched, (entry, R, rc)
            finally:
                gctx.set_sgm(None)
    gctx.set_sgm(paths, 0, 0)
    try:
        rc, untouched = _untouched_call(gctx, "pair_device", Ls, Rs, 46, 10)     # (93^2 * 255^2 * 4 > 2^31)
        assert rc == UNSUP and untouched
    finally:
        gctx.set_sgm(None)


@pytest.mark.parametrize("entry", ["pair_device"] + HOST_ENTRIES)
def test_float_bound_and_non_finite_images_are_rejected(gctx, mg, entry):
    h = mg if entry.startswith("mgpu_") else gctx
    Ls, Rs = _images("f32", 2, 11)
    h.set_sgm(8, 2, 20)
    try:
        big = (Ls * np.float32(1000)).astype(np.float32)            # (hi - lo)^2 ~ 6.5e10: over the bound at any radius
        rc, untouched = _untouched_call(h, entry, big, Rs, 0, RANGE_T)
        assert rc == UNSUP and untouched, (entry, "bound", rc)
        for bad in (np.nan, np.inf, -np.inf):
            L2 = Ls.copy()
            L2[:, 7, 11] = bad
            rc, untouched = _untouched_call(h, entry, L2, Rs, 1, RANGE_T)
            assert rc == UNSUP and untouched, (entry, bad, rc)
        rc, untouched = _untouched_call(h, entry, Ls, Rs, 1, RANGE_T)
        _ok(rc, entry)
    finally:
        h.set_sgm(None)


def test_too_many_candidates_are_rejected(gctx):
    g = np.random.default_rng(3)
    Ls = g.integers(0, 256, (1, 8, 1000)).astype(np.uint8)
    Rs = g.integers(0, 256, (1, 8, 1000)).astype(np.uint8)
    gctx.set_sgm(4, 1, 10)
    try:
        rc, untouched = _untouched_call(gctx, "pair_device", Ls, Rs, 1, 600)
        assert rc == UNSUP and untouched and "candidates" in _capi.last_error()
        rc, _ = _untouched_call(gctx, "pair_device", Ls, Rs, 1, 511)               # 512 candidates: served
        _ok(rc)
    finally:
        gctx.set_sgm(None)


def _fill(dev, shape, value):
    a = np.full(shape, value, np.uint8)
    return _torch().from_numpy(a).cuda() if dev else a


def test_partial_bands_and_mgpu_bands_are_rejected(gctx, mg):
    torch = _torch()
    lib = _capi.lib()
    rows, cols, win, rng = 48, 96, 3, 16
    L, Rt, _ = synth.make_pair(rows, cols, rng + 4, 88)
    Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
    gctx.set_sgm(4, 2, 20)
    mg.set_sgm(4, 2, 20)
    try:
        for r0, r1 in ((0, 24), (24, 48), (10, 20)):
            for fn, a, b in ((lib.stereo_disparity_pair_band_u8_host, L, Rt), (lib.stereo_disparity_pair_band_f32_host, Lf, Rf)):
                ol, orr = _fill(False, (rows, cols * 2), 0x3C), _fill(False, (rows, cols * 2), 0x3C)
                rc = fn(gctx.handle, sb.COST_SSD, a.ctypes.data, a.strides[0], b.ctypes.data, b.strides[0], rows, cols, r0, r1, win, rng,
                        ol[r0:].ctypes.data, orr[r0:].ctypes.data, cols * 2, 2)
                assert rc == UNSUP and (ol == 0x3C).all() and (orr == 0x3C).all(), (fn.__name__, r0, r1, rc)
            h0, h1 = C.c_int(), C.c_int()
            _ok(lib.stereo_band_halo_rows(rows, r0, r1, win, C.byref(h0), C.byref(h1)))
            tl, tr = torch.from_numpy(L).cuda(), torch.from_numpy(Rt).cuda()
            ol, orr = _fill(True, (rows, cols * 2), 0x3C), _fill(True, (rows, cols * 2), 0x3C)
            rc = lib.stereo_disparity_pair_band_halo_u8_device(gctx.handle, sb.COST_SSD, tl[h0.value].data_ptr(), cols, tr[h0.value].data_ptr(),
                                                               cols, rows, cols, r0, r1, h0.value, h1.value, win, rng, ol[r0].data_ptr(),
                                                               orr[r0].data_ptr(), cols * 2, 2, None)
            torch.cuda.synchronize()
            assert rc == UNSUP and (ol == 0x3C).all().item() and (orr == 0x3C).all().item(), ("band_halo", r0, r1, rc)
        for fn, a, b in ((lib.stereo_mgpu_disparity_pair_bands_u8_host, L, Rt), (lib.stereo_mgpu_disparity_pair_bands_f32_host, Lf, Rf)):
            ol, orr = _fill(False, (rows, cols * 2), 0x3C), _fill(False, (rows, cols * 2), 0x3C)
            rc = fn(mg._h, sb.COST_SSD, a.ctypes.data, a.strides[0], b.ctypes.data, b.strides[0], rows, cols, win, rng,
                    ol.ctypes.data, orr.ctypes.data, cols * 2, 2)
            assert rc == UNSUP and (ol == 0x3C).all() and (orr == 0x3C).all(), (fn.__name__, rc)
    finally:
        gctx.set_sgm(None)
        mg.set_sgm(None)
    dl, dr = mg.disparity_pair_bands(sb.COST_SSD, L, Rt, win, rng, dtype=np.int16)      # off again: served
    assert dl.shape == (rows, cols)


# ---- 5. the setting and its state --------------------------------------------------------------------------------------

def test_setter_checks_and_default_state(mg):
    lib = _capi.lib()
    fresh = sb.Context(0)
    try:
        assert fresh.sgm is None
        assert lib.stereo_ctx_set_sgm(None, 4, 1, 2) == ARG
        assert lib.stereo_mgpu_set_sgm(None, 4, 1, 2) == ARG
        fresh.set_sgm(8, 3, 30)
        for bad in ((1, 1, 2), (2, 1, 2), (5, 1, 2), (16, 1, 2), (-4, 1, 2), (4, -1, 2), (4, 3, 2), (0, 5, 1)):
            assert lib.stereo_ctx_set_sgm(fresh.handle, *bad) == ARG, bad
            assert fresh.sgm == (8, 3, 30), bad                      # the old setting stays
        fresh.set_sgm(4, 7, 7)
        assert fresh.sgm == (4, 7, 7)
        fresh.set_sgm(4)
        assert fresh.sgm == (4, 0, 0)
        fresh.set_sgm(0, 1, 2)
        assert fresh.sgm is None
        fresh.set_sgm(8, 1, 2)
        fresh.set_sgm(None)
        assert fresh.sgm is None
        paths, p1, p2 = C.c_int(), C.c_int(), C.c_int()
        assert lib.stereo_ctx_sgm(None, C.byref(paths), C.byref(p1), C.byref(p2)) == ARG
        with pytest.raises(sb.StereoError):
            mg.set_sgm(4, 5, 1)
        mg.set_sgm(8, 2, 9)
        for i in range(mg.device_count):
            _ok(lib.stereo_ctx_sgm(lib.stereo_mgpu_ctx(mg._h, i), C.byref(paths), C.byref(p1), C.byref(p2)))
            assert (paths.value, p1.value, p2.value) == (8, 2, 9)
    finally:
        fresh.close()
        mg.set_sgm(None)


def test_off_again_is_byte_identical_to_a_fresh_context(gctx):
    Ls, Rs = _images("u8", 3, 79)
    fresh = sb.Context(0)
    try:
        for entry in ("pair_host", "pair_device", "batch_device", "batch_host"):
            for cost in (sb.COST_SSD, sb.COST_NCORR):
                want = _run(fresh, entry, cost, Ls, Rs, 3, RANGE_T, np.int16)
                if cost == sb.COST_SSD:
                    gctx.set_sgm(8, 10, 200)
                    on = _run(gctx, entry, cost, Ls, Rs, 3, RANGE_T, np.int16)
                    assert (on[0] != want[0]).any()
                gctx.set_sgm(0)
                got = _run(gctx, entry, cost, Ls, Rs, 3, RANGE_T, np.int16)
                assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), (entry, cost)
                assert gctx.last_path != sb.PATH_SGM
    finally:
        fresh.close()
        gctx.set_sgm(None)


def test_single_direction_and_refgpu_calls_ignore_the_setting(gctx):
    L, Rt, _ = synth.make_pair(48, 160, 24, 517)
    Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)

    def singles(c):
        return [c.disparity(sb.COST_SSD, Lf, Rf, 3, -20, 0, dtype=np.int16), c.disparity(sb.COST_SSD, L, Rt, 3, -20, 0),
                c.disparity(sb.COST_NCORR, L, Rt, 3, 0, 20), c.disparity_refgpu(sb.COST_SSD, Lf, Rf, 3, -20, 0)]

    fresh = sb.Context(0)
    try:
        want = singles(fresh)
        gctx.set_sgm(8, 10, 200)
        got = singles(gctx)
        assert gctx.last_path == sb.PATH_REFGPU
    finally:
        fresh.close()
        gctx.set_sgm(None)
    for a, b in zip(got, want):
        assert np.array_equal(a, b)


def test_state_reported_for_sgm_calls(gctx):
    Ls, Rs = _images("u8", 1, 80)
    gctx.set_sgm(4, 3, 30)
    try:
        for entry in ("pair_device", "pair_host", "batch_device"):
            _run(gctx, entry, sb.COST_SSD, Ls, Rs, 3, RANGE_T, np.int16)
            assert gctx.last_path == sb.PATH_SGM
            assert gctx.last_fused_pairs == 0
            assert gctx.last_hot_kernel_ms()[0] < 0
            assert gctx.last_launches >= 2 * (3 + 4)
    finally:
        gctx.set_sgm(None)


# ---- 6. graph capture --------------------------------------------------------------------------------------------------

def test_device_pair_call_with_sgm_replays_in_a_cuda_graph(gctx):
    torch = _torch()
    rows, cols, win, rng, paths, p1, p2 = 96, 200, 3, 30, 8, 8, 90
    inputs = [synth.make_pair(rows, cols, rng + 4, 3130 + k)[:2] for k in range(3)]
    s = torch.cuda.Stream()
    tl = torch.from_numpy(inputs[0][0]).cuda()
    tr = torch.from_numpy(inputs[0][1]).cuda()
    out = torch.full((2, rows, cols), 99, dtype=torch.int16, device="cuda")
    s.wait_stream(torch.cuda.current_stream())

    def call():
        _ok(_capi.lib().stereo_disparity_pair_u8_device(gctx.handle, sb.COST_SSD, tl.data_ptr(), cols, tr.data_ptr(), cols, rows, cols,
                                                        win, rng, out[0].data_ptr(), out[1].data_ptr(), cols * 2, 2, C.c_void_p(s.cuda_stream)))

    gctx.set_sgm(paths, p1, p2)
    try:
        with torch.cuda.stream(s):
            call()                                       # warm-up: sizes the scratch arena
        s.synchronize()
        g = torch.cuda.CUDAGraph()
        out.fill_(99)
        torch.cuda.synchronize()
        with torch.cuda.graph(g, stream=s, capture_error_mode="thread_local"):
            call()
        assert (out == 99).all().item()                  # captured, not run
        for L, Rt in inputs[1:]:
            tl.copy_(torch.from_numpy(L))
            tr.copy_(torch.from_numpy(Rt))
            torch.cuda.synchronize()
            g.replay()
            torch.cuda.synchronize()
            got = out.cpu().numpy()
            dl, dr = sgm_pair(L, Rt, win, rng, paths, p1, p2)
            assert np.array_equal(got[0], dl) and np.array_equal(got[1], dr)
    finally:
        gctx.set_sgm(None)
