"""StereoBM's X-Sobel prefilter and texture threshold on the B200 (stereo_ctx_set_prefilter): the standalone prefilter calls
against the restatement (prefilter_oracle); every pair entry point and kernel family, SSD and NCC, fused and unfused, with
and without the texture threshold, against the oracle run on the restated prefiltered images; SGM (SSD and NCC) and the
uniqueness ratio, left-right check and speckle filter on top; the exact offset invariance; band-sharded equivalence through
the standalone call; the refusals, which write nothing; the setting; CUDA graph replays; and full-size cases."""
import ctypes as C

import numpy as np
import pytest

import introtocomputervision_b200 as sb
import oracle
from introtocomputervision_b200 import _capi, synth
from lr_oracle import lr_check
from ncc_check import check_ncc_map
from pair_calls import FAMILIES, RANGE_T, _device_batch, _images, _ok, _run, _set_fuse, _torch, gctx, mg
from prefilter_oracle import pf, texture_keep, texture_sum
from sgm_ncc_oracle import sgm_pair as sgm_ncc_pair
from sgm_oracle import cost_volume, sgm_pair
from speckle_oracle import filter_speckles
from uniqueness_oracle import apply, unique

pytestmark = pytest.mark.gpu

ARG, UNSUP = _capi.ERR_INVALID_ARG, _capi.ERR_UNSUPPORTED
ENTRIES = ["pair_host", "pair_device", "batch_device", "batch_host", "band_host", "band_halo_device", "mgpu_batch"]
NCC_AGREE = 0.99        # clipped responses form plateaus: more near-ties than raw images (each one is checked against tau)


def _threshold(img, cap, R, q=0.2):
    """A texture threshold that rejects about a fraction q of the pixels of img (the synthetic pairs are richly textured)."""
    return int(np.quantile(texture_sum(pf(img, cap), cap, R), q)) + 1


def _narrow(d, dt):
    return np.asarray(d).astype(np.int64).astype(dt)


def _ssd_expected(L, Rt, R, rng, cap, T, dt):
    """Both block-matcher SSD maps of a pair with the prefilter (and texture threshold T) on, from the oracle."""
    PL, PR = pf(L, cap), pf(Rt, cap)
    out = []
    for ref, tgt, lo, hi in ((PL, PR, -rng, 0), (PR, PL, 0, rng)):
        d = _narrow(oracle.ssd_fast(ref, tgt, R, lo, hi), dt)
        out.append(apply(d, texture_keep(ref, cap, R, T), rng) if T else d)
    return out


# ---- 1. the standalone calls ---------------------------------------------------------------------------------------------

def _standalone(ctx, img, cap, dst_pad=0, src_pad=0):
    """pf(img) through stereo_prefilter_{u8,f32}_device with padded steps; returns (P, the padding bytes of dst)."""
    torch = _torch()
    rows, cols = img.shape
    f32 = img.dtype == np.float32
    src = np.zeros((rows, cols + src_pad), img.dtype)
    src[:, :cols] = img
    ts = torch.from_numpy(src).cuda()
    td = torch.full((rows, cols + dst_pad), 0xAB, dtype=torch.uint8, device="cuda")
    fn = _capi.lib().stereo_prefilter_f32_device if f32 else _capi.lib().stereo_prefilter_u8_device
    _ok(fn(ctx.handle, ts.data_ptr(), src.strides[0], rows, cols, cap, td.data_ptr(), cols + dst_pad,
           C.c_void_p(torch.cuda.current_stream().cuda_stream)), "prefilter")
    torch.cuda.synchronize()
    out = td.cpu().numpy()
    return out[:, :cols], out[:, cols:]


SHAPES = [(1, 1), (1, 7), (2, 2), (3, 3), (2, 17), (3, 40), (40, 150), (41, 150), (37, 1000), (64, 2048), (33, 4099)]


@pytest.mark.parametrize("kind", ["u8", "f32", "noisy", "nonfinite"])
@pytest.mark.parametrize("rows,cols", SHAPES)
def test_standalone_equals_the_restatement(gctx, kind, rows, cols):
    g = np.random.default_rng(rows * 7919 + cols)
    img = g.integers(0, 256, (rows, cols)).astype(np.uint8)
    if kind == "f32":
        img = img.astype(np.float32)
    elif kind == "noisy":
        img = synth.noisy_variant(img, rows + cols)
    elif kind == "nonfinite":
        img = synth.noisy_variant(img, rows + cols) * np.float32(3)
        flat = img.reshape(-1)
        for i, v in enumerate((np.nan, np.inf, -np.inf, np.nan)):
            flat[(i * 7919 + 13) % flat.size] = v
        img[:, ::97] += np.float32(0.5)                     # exact .5 steps next to the rounding
    for cap in (1, 31, 63):
        for pads in ((0, 0), (13, 5), (240, 1)):
            got, tail = _standalone(gctx, img, cap, *pads)
            want = pf(img, cap)
            bad = np.argwhere(got != want)
            assert bad.size == 0, f"{kind} {rows}x{cols} cap={cap} pads={pads}: {bad[:5].tolist()} of {len(bad)}"
            assert (tail == 0xAB).all(), (kind, rows, cols, cap, pads)     # bytes past cols untouched


# ---- 2. every pair entry point and family ------------------------------------------------------------------------------

@pytest.mark.parametrize("fuse", [True, False])
@pytest.mark.parametrize("family", list(FAMILIES))
@pytest.mark.parametrize("entry", ENTRIES)
def test_pair_entry_points_equal_the_oracle(gctx, mg, entry, family, fuse):
    kind, R, dt = FAMILIES[family]
    if kind != "u8" and entry in ("batch_device", "band_halo_device"):
        pytest.skip("8-bit device entry point")
    if kind == "noisy" and entry == "band_host":
        pytest.skip("the host row-band entry points take 8-bit-valued images only")
    h = mg if entry.startswith("mgpu_") else gctx
    n = 2 if "batch" in entry else 1
    Ls, Rs = _images(kind, n, 2100 + 13 * ENTRIES.index(entry))
    whole = [(0, Ls.shape[1])]
    cap = 31
    _set_fuse(h, fuse)
    try:
        for T in (0, _threshold(Ls[0], cap, R)):
            h.set_prefilter(cap, T)
            try:
                ssd = _run(h, entry, sb.COST_SSD, Ls, Rs, R, RANGE_T, dt, bands=whole)
                ncc = _run(h, entry, sb.COST_NCORR, Ls, Rs, R, RANGE_T, dt, bands=whole)
                if entry in ("pair_device", "batch_device"):
                    assert h.last_path == (sb.PATH_EXACT_F32 if R > 7 else sb.PATH_FAST_U8), (entry, family, h.last_path)
                    assert (h.last_fused_pairs > 0) == (fuse and R <= 7), (entry, family, h.last_fused_pairs)
            finally:
                h.set_prefilter(None)
            if T == 0:
                ncc0 = ncc
            for i in range(n):
                want = _ssd_expected(Ls[i], Rs[i], R, RANGE_T, cap, T, dt)
                PL, PR = pf(Ls[i], cap), pf(Rs[i], cap)
                for side, (ref, tgt, lo, hi) in enumerate(((PL, PR, -RANGE_T, 0), (PR, PL, 0, RANGE_T))):
                    bad = np.argwhere(ssd[side][i] != want[side])
                    assert bad.size == 0, f"{entry} {family} fuse={fuse} T={T} SSD pair {i} map {side}: {bad[:5].tolist()} of {len(bad)}"
                    if T == 0:
                        check_ncc_map(ncc[side][i], ref, tgt, R, lo, hi, "exact" if R > 7 else "u8", min_agree=NCC_AGREE,
                                      what=f"{entry} {family} fuse={fuse} NCC pair {i} map {side}")
                    else:
                        keep = texture_keep(ref, cap, R, T)
                        assert 0 < (~keep).sum() < keep.size, (family, side)             # the threshold fires, not everywhere
                        assert np.array_equal(ncc[side][i], apply(ncc0[side][i], keep, RANGE_T)), (entry, family, side)
    finally:
        _set_fuse(h, True)


# ---- 3. SGM, uniqueness ratio, left-right check, speckle filter ----------------------------------------------------------

@pytest.mark.parametrize("cost", ["ssd", "ncc"])
@pytest.mark.parametrize("paths", [4, 8])
@pytest.mark.parametrize("entry", ["pair_device", "pair_host", "batch_device", "batch_host"])
def test_sgm_on_the_prefiltered_images(gctx, entry, paths, cost):
    q = None if cost == "ssd" else 64
    n = 2 if "batch" in entry else 1
    Ls, Rs = _images("u8", n, 2300 + paths)
    if entry == "pair_host":
        Ls, Rs = Ls.astype(np.float32), synth.noisy_variant(Rs[0], 5)[None]
    p1, p2, R, cap = (10, 120, 3, 15) if cost == "ssd" else (2, 24, 2, 15)
    T = _threshold(Ls[0], cap, R)
    gctx.set_sgm(paths, p1, p2)
    gctx.set_sgm_ncc_scale(q or 0)
    gctx.set_prefilter(cap, T)
    try:
        on = _run(gctx, entry, sb.COST_SSD if q is None else sb.COST_NCORR, Ls, Rs, R, RANGE_T, np.int16)
        assert gctx.last_path == sb.PATH_SGM
    finally:
        gctx.set_prefilter(None)
        gctx.set_sgm(None)
        gctx.set_sgm_ncc_scale(0)
    for i in range(n):
        PL, PR = pf(Ls[i], cap), pf(Rs[i], cap)
        want = sgm_pair(PL, PR, R, RANGE_T, paths, p1, p2) if q is None else sgm_ncc_pair(PL, PR, R, RANGE_T, q, paths, p1, p2)
        for side, ref in enumerate((PL, PR)):
            w = apply(_narrow(want[side], np.int16), texture_keep(ref, cap, R, T), RANGE_T)
            bad = np.argwhere(on[side][i] != w)
            assert bad.size == 0, f"{entry} {cost} {paths} pair {i} map {side}: {bad[:5].tolist()} of {len(bad)}"


@pytest.mark.parametrize("entry", ["pair_device", "batch_device", "pair_host", "batch_host"])
def test_with_uniqueness_left_right_check_and_speckle_filter(gctx, entry):
    n = 2 if "batch" in entry else 1
    Ls, Rs = _images("u8", n, 2400)
    if entry == "pair_host":
        Ls, Rs = synth.noisy_variant(Ls[0], 1)[None], synth.noisy_variant(Rs[0], 2)[None]
    R, cap, u = 3, 31, 15
    T = _threshold(Ls[0], cap, R, 0.1)
    gctx.set_prefilter(cap, T)
    gctx.set_uniqueness(u)
    gctx.set_lr_check(1)
    gctx.set_speckle_filter(20, 1)
    try:
        on = _run(gctx, entry, sb.COST_SSD, Ls, Rs, R, RANGE_T, np.int16)
    finally:
        gctx.set_prefilter(None)
        gctx.set_uniqueness(0)
        gctx.set_lr_check(None)
        gctx.set_speckle_filter(None)
    for i in range(n):
        PL, PR = pf(Ls[i], cap), pf(Rs[i], cap)
        maps = []
        for ref, tgt, lo, hi in ((PL, PR, -RANGE_T, 0), (PR, PL, 0, RANGE_T)):
            d = _narrow(oracle.ssd_fast(ref, tgt, R, lo, hi), np.int16)
            d = apply(d, unique(*cost_volume(ref, tgt, R, lo, hi), u, block_matcher=True), RANGE_T)
            maps.append(apply(d, texture_keep(ref, cap, R, T), RANGE_T))
        dl, dr = lr_check(maps[0], maps[1], RANGE_T, 1)
        dl, dr = filter_speckles(dl, -(RANGE_T + 1), 20, 1), filter_speckles(dr, -(RANGE_T + 1), 20, 1)
        assert np.array_equal(on[0][i], dl) and np.array_equal(on[1][i], dr), (entry, i)


# ---- 4. offset invariance -------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("entry", ["pair_device", "pair_host", "batch_device"])
def test_an_additive_offset_cancels_exactly(gctx, entry):
    n = 2 if "batch" in entry else 1
    Ls, Rs = _images("u8", n, 2500)
    Ls, Rs = (Ls.astype(np.int32) * 200 // 255).astype(np.uint8), (Rs.astype(np.int32) * 200 // 255).astype(np.uint8)
    Lc = (Ls.astype(np.int32) + 37).astype(np.uint8)             # <= 237: nothing saturates
    off = [_run(gctx, entry, sb.COST_SSD, a, Rs, 3, RANGE_T, np.int16) for a in (Ls, Lc)]
    assert any((a != b).any() for a, b in zip(off[0], off[1]))       # the offset biases raw matching
    gctx.set_prefilter(31, _threshold(Ls[0], 31, 3))
    try:
        on = [_run(gctx, entry, sb.COST_SSD, a, Rs, 3, RANGE_T, np.int16) for a in (Ls, Lc)]
    finally:
        gctx.set_prefilter(None)
    assert np.array_equal(on[0][0], on[1][0]) and np.array_equal(on[0][1], on[1][1]), entry


# ---- 5. band-sharded callers --------------------------------------------------------------------------------------------

@pytest.mark.parametrize("rows", [48, 49])
def test_prefiltered_bands_equal_the_whole_pair_call(gctx, rows):
    torch = _torch()
    lib = _capi.lib()
    cols, win, rng, cap = 160, 3, 24, 20
    L, Rt, _ = synth.make_pair(rows, cols, rng + 4, 2600 + rows)
    PL, _ = _standalone(gctx, L, cap)
    PR, _ = _standalone(gctx, Rt, cap)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for cost in (sb.COST_SSD, sb.COST_NCORR):
        gctx.set_prefilter(cap, 0)
        try:
            want = gctx.disparity_pair(cost, L, Rt, win, rng, dtype=np.int16)
        finally:
            gctx.set_prefilter(None)
        tl, tr = torch.from_numpy(PL).cuda(), torch.from_numpy(PR).cuda()
        ol = torch.full((rows, cols), 99, dtype=torch.int16, device="cuda")
        orr = torch.full_like(ol, 99)
        for r0, r1 in ((0, 17), (17, 30), (30, rows)):
            h0, h1 = C.c_int(), C.c_int()
            _ok(lib.stereo_band_halo_rows(rows, r0, r1, win, C.byref(h0), C.byref(h1)))
            _ok(lib.stereo_disparity_pair_band_halo_u8_device(gctx.handle, cost, tl[h0.value].data_ptr(), cols, tr[h0.value].data_ptr(),
                                                              cols, rows, cols, r0, r1, h0.value, h1.value, win, rng, ol[r0].data_ptr(),
                                                              orr[r0].data_ptr(), cols * 2, 2, st), "band")
        torch.cuda.synchronize()
        assert np.array_equal(ol.cpu().numpy(), want[0]) and np.array_equal(orr.cpu().numpy(), want[1]), (rows, cost)


# ---- 6. refusals of the standalone calls --------------------------------------------------------------------------------

def test_standalone_refusals(gctx):
    torch = _torch()
    lib = _capi.lib()
    rows, cols = 20, 64
    src = torch.zeros((rows, cols), dtype=torch.uint8, device="cuda")
    srcf = torch.zeros((rows, cols), dtype=torch.float32, device="cuda")
    dst = torch.full((rows, cols), 0x3C, dtype=torch.uint8, device="cuda")
    s, d = src.data_ptr(), dst.data_ptr()
    bad = [
        (lib.stereo_prefilter_u8_device, (gctx.handle, None, cols, rows, cols, 31, d, cols, None)),
        (lib.stereo_prefilter_u8_device, (gctx.handle, s, cols, rows, cols, 31, None, cols, None)),
        (lib.stereo_prefilter_u8_device, (None, s, cols, rows, cols, 31, d, cols, None)),
        (lib.stereo_prefilter_u8_device, (gctx.handle, s, cols, 0, cols, 31, d, cols, None)),
        (lib.stereo_prefilter_u8_device, (gctx.handle, s, cols, rows, -1, 31, d, cols, None)),
        (lib.stereo_prefilter_u8_device, (gctx.handle, s, cols - 1, rows, cols, 31, d, cols, None)),
        (lib.stereo_prefilter_u8_device, (gctx.handle, s, cols, rows, cols, 31, d, cols - 1, None)),
        (lib.stereo_prefilter_u8_device, (gctx.handle, s, cols, rows, cols, 0, d, cols, None)),
        (lib.stereo_prefilter_u8_device, (gctx.handle, s, cols, rows, cols, 64, d, cols, None)),
        (lib.stereo_prefilter_u8_device, (gctx.handle, s, cols, rows, cols, 31, s, cols, None)),                  # in place
        (lib.stereo_prefilter_u8_device, (gctx.handle, s, cols, rows, cols, 31, s + cols * (rows - 1) + 5, cols, None)),   # overlaps
        (lib.stereo_prefilter_f32_device, (gctx.handle, srcf.data_ptr(), cols * 2, rows, cols, 31, d, cols, None)),   # short step
        (lib.stereo_prefilter_f32_device, (gctx.handle, srcf.data_ptr(), cols * 4, rows, cols, 31, srcf.data_ptr() + 8, cols, None)),
    ]
    for fn, args in bad:
        assert fn(*args) == ARG, (fn.__name__, args)
    torch.cuda.synchronize()
    assert (dst == 0x3C).all().item() and (src == 0).all().item() and (srcf == 0).all().item()


# ---- 7. graph capture ----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("f32", [False, True])
def test_device_pair_call_replays_in_a_cuda_graph(f32):
    torch = _torch()
    rows, cols, win, rng, cap = 96, 200, 3, 30, 31
    inputs = [synth.make_pair(rows, cols, rng + 4, 3330 + k)[:2] for k in range(3)]
    if f32:
        inputs = [(synth.noisy_variant(a, k), synth.noisy_variant(b, k + 10)) for k, (a, b) in enumerate(inputs)]
    T = _threshold(inputs[0][0], cap, win)
    s = torch.cuda.Stream()
    tl = torch.from_numpy(inputs[0][0]).cuda()
    tr = torch.from_numpy(inputs[0][1]).cuda()
    out = torch.full((2, rows, cols), 99, dtype=torch.int16, device="cuda")
    step = cols * (4 if f32 else 1)
    s.wait_stream(torch.cuda.current_stream())
    fn = _capi.lib().stereo_disparity_pair_f32_device if f32 else _capi.lib().stereo_disparity_pair_u8_device
    gctx = sb.Context(0)             # its own context: the captured call is this context's last

    def call():
        _ok(fn(gctx.handle, sb.COST_SSD, tl.data_ptr(), step, tr.data_ptr(), step, rows, cols, win, rng, out[0].data_ptr(),
               out[1].data_ptr(), cols * 2, 2, C.c_void_p(s.cuda_stream)))

    gctx.set_prefilter(cap, T)
    try:
        with torch.cuda.stream(s):
            call()                                       # warm-up: sizes the prefilter buffer and the scratch arena
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
            want = _ssd_expected(L, Rt, win, rng, cap, T, np.int16)
            assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
        del g
    finally:
        gctx.close()


# ---- 8. full size -------------------------------------------------------------------------------------------------------

def test_full_size_720p_device_batch(gctx):
    rows, cols, nd, win, n, cap = 720, 1280, 64, 4, 16, 31
    pairs = [synth.make_pair(rows, cols, nd, 370 + i)[:2] for i in range(n)]
    Ls, Rs = np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs])
    T = _threshold(Ls[0], cap, win)
    gctx.set_prefilter(cap, T)
    try:
        on = _device_batch(gctx, Ls, Rs, win, nd, 1)
    finally:
        gctx.set_prefilter(None)
    for i in range(n):
        want = _ssd_expected(Ls[i], Rs[i], win, nd, cap, T, np.int8)
        assert np.array_equal(on[0, i], want[0]) and np.array_equal(on[1, i], want[1]), i


def test_full_size_4k_pair(gctx):
    rows, cols, nd, win, cap = 2160, 3840, 256, 5, 31
    L, Rt, _ = synth.make_pair(rows, cols, nd, 4196)
    Lf = synth.noisy_variant(L, 3)
    T = _threshold(Lf, cap, win)
    gctx.set_prefilter(cap, T)
    try:
        on = gctx.disparity_pair(sb.COST_SSD, Lf, Rt.astype(np.float32), win, nd, dtype=np.int16)
    finally:
        gctx.set_prefilter(None)
    want = _ssd_expected(Lf, Rt, win, nd, cap, T, np.int16)
    for side in (0, 1):
        bad = np.argwhere(on[side] != want[side])
        assert bad.size == 0, f"4K map {side}: {bad[:5].tolist()} of {len(bad)}"
