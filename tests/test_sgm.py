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
from pair_calls import FAMILIES, RANGE_T, _device_batch, _images, _ok, _run, _torch, _untouched, gctx, mg

pytestmark = pytest.mark.gpu

ARG, UNSUP = _capi.ERR_INVALID_ARG, _capi.ERR_UNSUPPORTED
ENTRIES = ["pair_host", "pair_device", "batch_device", "batch_host", "band_host", "band_halo_device", "mgpu_batch"]


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

HOST_ENTRIES = ["pair_host", "batch_host", "mgpu_batch"]


@pytest.mark.parametrize("entry", ["pair_device", "batch_device"] + HOST_ENTRIES)
def test_ncc_is_rejected_and_writes_nothing(gctx, mg, entry):
    h = mg if entry.startswith("mgpu_") else gctx
    Ls, Rs = _images("u8", 2, 5)
    h.set_sgm(4, 1, 10)
    try:
        rc, untouched = _untouched(h, entry, Ls, Rs, 3, RANGE_T, cost=sb.COST_NCORR)
        assert rc == UNSUP and untouched, (entry, rc)
        assert "SSD" in _capi.last_error()
        rc, untouched = _untouched(h, entry, Ls, Rs, 3, RANGE_T)            # SSD is served
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
                rc, _ = _untouched(gctx, entry, Ls, Rs, R, 10)
                _ok(rc, f"{entry} at the bound")
                gctx.set_sgm(paths, 0, p2 + 1)
                rc, untouched = _untouched(gctx, entry, Ls, Rs, R, 10)
                assert rc == UNSUP and untouched, (entry, R, rc)
            finally:
                gctx.set_sgm(None)
    gctx.set_sgm(paths, 0, 0)
    try:
        rc, untouched = _untouched(gctx, "pair_device", Ls, Rs, 46, 10)     # (93^2 * 255^2 * 4 > 2^31)
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
        rc, untouched = _untouched(h, entry, big, Rs, 0, RANGE_T)
        assert rc == UNSUP and untouched, (entry, "bound", rc)
        for bad in (np.nan, np.inf, -np.inf):
            L2 = Ls.copy()
            L2[:, 7, 11] = bad
            rc, untouched = _untouched(h, entry, L2, Rs, 1, RANGE_T)
            assert rc == UNSUP and untouched, (entry, bad, rc)
        rc, untouched = _untouched(h, entry, Ls, Rs, 1, RANGE_T)
        _ok(rc, entry)
    finally:
        h.set_sgm(None)


def test_too_many_candidates_are_rejected(gctx):
    g = np.random.default_rng(3)
    Ls = g.integers(0, 256, (1, 8, 1000)).astype(np.uint8)
    Rs = g.integers(0, 256, (1, 8, 1000)).astype(np.uint8)
    gctx.set_sgm(4, 1, 10)
    try:
        rc, untouched = _untouched(gctx, "pair_device", Ls, Rs, 1, 600)
        assert rc == UNSUP and untouched and "candidates" in _capi.last_error()
        rc, _ = _untouched(gctx, "pair_device", Ls, Rs, 1, 511)               # 512 candidates: served
        _ok(rc)
    finally:
        gctx.set_sgm(None)


# ---- 5. the state of SGM calls -----------------------------------------------------------------------------------------

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
