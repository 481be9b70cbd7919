"""Speckle filter on the B200 (stereo_ctx_set_speckle_filter, stereo_filter_speckles_device): the kernel alone against the
filter's restatement (speckle_oracle.filter_speckles) on adversarial maps and shapes, with padded rows; every pair entry
point with the filter on against the restatement applied to the same call's maps with it off, alone and after the
left-right check, for both costs, fused and unfused, on each kernel family; a 16-pair 720p batch and a 4K pair; the
rejections (partial bands, the sentinel rule, bad settings and arguments) and the default and off states; and a CUDA
graph around a device pair call."""
import ctypes as C

import numpy as np
import pytest

import introtocomputervision_b200 as sb
from introtocomputervision_b200 import _capi, synth
from lr_oracle import lr_check
from speckle_oracle import filter_speckles
from pair_calls import FAMILIES, RANGE_T, _device_batch, _images, _ok, _run, _set_fuse, _torch, gctx, mg

pytestmark = pytest.mark.gpu

ARG, UNSUP = _capi.ERR_INVALID_ARG, _capi.ERR_UNSUPPORTED
DT = {1: np.int8, 2: np.int16, 4: np.int32}
MAX_SIZE, MAX_DIFF = 30, 0


# ---- 1. the kernel alone ---------------------------------------------------------------------------------------------

def _blobs(g, rows, cols):
    """Random walks along the rows and down the columns: long, thin regions of every size, plus 5 % sentinel pixels."""
    d = np.cumsum(g.integers(-1, 2, (rows, cols)), axis=1) + np.cumsum(g.integers(-1, 2, (rows, 1)), axis=0)
    return d % 50


def _serpentine(rows, cols):
    """One 1-pixel-wide path through the whole map: even rows are path (0), odd rows wall (9) with one opening, at the
    right end and the left end in turn.  The deepest union-find trees a map of this size can give."""
    d = np.zeros((rows, cols), np.int64)
    d[1::2] = 9
    for k, y in enumerate(range(1, rows, 2)):
        d[y, cols - 1 if k % 2 == 0 else 0] = 0
    return d


def _comb(rows, cols):
    """Teeth (0) on even columns that join only in the last row; odd columns (5) stay separate columns."""
    d = np.zeros((rows, cols), np.int64)
    d[:-1, 1::2] = 5
    return d


def _checker(rows, cols, max_diff):
    y, x = np.mgrid[:rows, :cols]
    return ((x + y) % 2) * (max_diff + 1)


def _padded(a, pad):
    rows, cols = a.shape
    buf = np.full((rows, cols * a.itemsize + pad), 0x5A, np.uint8)
    buf[:, :cols * a.itemsize] = a.view(np.uint8).reshape(rows, -1)
    return buf


def _device_filter(ctx, d, new_val, max_size, max_diff, pad=96):
    """d filtered by stereo_filter_speckles_device in a row-padded device buffer; checks the padding is untouched."""
    torch = _torch()
    rows, cols = d.shape
    buf = _padded(d, pad)
    t = torch.from_numpy(buf).cuda()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    _ok(_capi.lib().stereo_filter_speckles_device(ctx.handle, t.data_ptr(), buf.shape[1], d.itemsize, rows, cols, new_val, max_size,
                                                  max_diff, C.c_void_p(side.cuda_stream)), "stereo_filter_speckles_device")
    assert ctx.last_launches == (4 if max_size > 0 else 0)
    torch.cuda.synchronize()
    out = t.cpu().numpy()
    n = cols * d.itemsize
    assert (out[:, n:] == 0x5A).all(), "row padding written"
    return out[:, :n].copy().view(d.dtype)


def _check_kernel(ctx, d, new_val, settings, min_changed=0.0):
    for max_size, max_diff in settings:
        got = _device_filter(ctx, d, new_val, max_size, max_diff)
        want = filter_speckles(d, new_val, max_size, max_diff)
        bad = np.argwhere(got != want)
        assert bad.size == 0, f"{d.shape} {d.dtype} {max_size}/{max_diff}: differs at {bad[:5].tolist()} (of {len(bad)})"
        if max_size == settings[0][0]:
            assert np.mean(want != d) >= min_changed


@pytest.mark.parametrize("elem", [1, 2, 4])
@pytest.mark.parametrize("kind", ["serpentine", "comb", "checker", "whole", "blobs"])
def test_kernel_alone_adversarial_maps(gctx, elem, kind):
    rows, cols, nv = 150, 333, -100
    g = np.random.default_rng(elem * 10 + len(kind))
    d = {"serpentine": _serpentine(rows, cols), "comb": _comb(rows, cols), "checker": _checker(rows, cols, 2),
         "whole": np.full((rows, cols), 3), "blobs": _blobs(g, rows, cols)}[kind].astype(DT[elem])
    if kind == "blobs":
        d[g.random((rows, cols)) < 0.05] = nv
    big = rows * cols
    settings = {"serpentine": [(big, 0), (big // 2, 0), (cols, 0)],      # the path (~big/2 px) goes, then stays; walls go
                "comb": [(big // 2, 1), (big, 4), (rows, 1)],
                "checker": [(1, 2), (1, 3), (2, 3)],                      # max_diff 2: all singletons; 3: one component
                "whole": [(big, 0), (big - 1, 0)],
                "blobs": [(20, 0), (100, 1), (400, 2), (0, 1)]}[kind]
    _check_kernel(gctx, d, nv, settings)


def test_kernel_alone_int32_near_the_limits(gctx):
    lo, hi = np.iinfo(np.int32).min, np.iinfo(np.int32).max
    g = np.random.default_rng(5)
    rows, cols = 70, 90
    d = np.where(g.random((rows, cols)) < 0.5, lo + g.integers(0, 3, (rows, cols)), hi - g.integers(0, 3, (rows, cols)))
    d = d.astype(np.int32)
    d[g.random((rows, cols)) < 0.1] = 0
    # lo and hi differ by 2^32 - 1, more than any max_diff: a 32-bit difference would wrap to 1 and link them
    _check_kernel(gctx, d, 0, [(30, 1), (30, 2), (rows * cols, 2 ** 31 - 1), (5, 2 ** 31 - 1)])


SHAPES = [(1, 1), (1, 640), (640, 1), (7, 640), (2160, 3840), (2, 32768), (32768, 2)]


@pytest.mark.parametrize("elem", [1, 2, 4])
@pytest.mark.parametrize("shape", SHAPES)
def test_kernel_alone_shapes(gctx, elem, shape):
    rows, cols = shape
    nv = -100
    g = np.random.default_rng(rows * 7 + cols + elem)
    d = _blobs(g, rows, cols).astype(DT[elem])
    d[g.random((rows, cols)) < 0.05] = nv
    settings = [(20, 1), (1, 0)] if rows * cols < 10 ** 6 else [(100, 1)]
    _check_kernel(gctx, d, nv, settings, min_changed=0.001 if rows * cols > 100 else 0.0)


def test_kernel_alone_4k_serpentine(gctx):
    d = _serpentine(2160, 3840).astype(np.int16)
    _check_kernel(gctx, d, -300, [(2160 * 3840 // 2 + 600, 0)], min_changed=0.4)


def test_kernel_alone_argument_checks(gctx):
    torch = _torch()
    buf = torch.zeros((4, 256), dtype=torch.uint8, device="cuda")
    a = buf.data_ptr()
    lib = _capi.lib()

    def call(p=a, step=256, elem=2, rows=4, cols=64, nv=-11, max_size=5, max_diff=1, ctx=gctx.handle):
        return lib.stereo_filter_speckles_device(ctx, p, step, elem, rows, cols, nv, max_size, max_diff, None)

    assert call() == _capi.STEREO_OK and call(max_size=0) == _capi.STEREO_OK
    assert gctx.last_launches == 0
    assert call(p=None) == ARG and call(ctx=None) == ARG
    assert call(rows=0) == ARG and call(cols=0) == ARG and call(rows=-1) == ARG
    assert call(rows=32769) == UNSUP and call(cols=32769, step=32769 * 2) == UNSUP
    assert call(elem=3) == ARG and call(step=127) == ARG
    assert call(max_size=-1) == ARG and call(max_diff=-1) == ARG
    assert call(elem=1, nv=-129) == ARG and call(elem=1, nv=128) == ARG and call(elem=2, nv=32768) == ARG
    assert call(elem=1, nv=-128) == _capi.STEREO_OK and call(elem=2, nv=-32768) == _capi.STEREO_OK
    assert call(elem=4, nv=-2 ** 31) == _capi.STEREO_OK
    gctx.synchronize()


# ---- 2. every pair entry point ---------------------------------------------------------------------------------------

ENTRIES = ["pair_host", "pair_device", "batch_device", "batch_host", "band_host", "band_halo_device", "mgpu_batch"]


def _filtered_equals_oracle_of_off(h, entry, cost, Ls, Rs, win, rng, dt, lr, max_size=MAX_SIZE, max_diff=MAX_DIFF, min_share=0.001):
    whole = [(0, Ls.shape[1])]          # (the band entry points take only a whole-image band with the filter on)
    try:
        h.set_lr_check(None)
        h.set_speckle_filter(None)
        off = _run(h, entry, cost, Ls, Rs, win, rng, dt, bands=whole)
        h.set_lr_check(1 if lr else None)
        h.set_speckle_filter(max_size, max_diff)
        on = _run(h, entry, cost, Ls, Rs, win, rng, dt, bands=whole)
    finally:
        h.set_lr_check(None)
        h.set_speckle_filter(None)
    nv = -(rng + 1)
    changed = 0
    for i in range(len(Ls)):
        base = lr_check(off[0][i], off[1][i], rng, 1) if lr else (off[0][i], off[1][i])
        for side in (0, 1):
            want = filter_speckles(base[side], nv, max_size, max_diff)
            bad = np.argwhere(on[side][i] != want)
            assert bad.size == 0, f"{entry} pair {i} map {side}: differs at {bad[:5].tolist()} (of {len(bad)})"
            changed += int(np.sum(want != base[side]))
    share = changed / (2 * Ls.size)
    assert changed > 0 and min_share <= share < 0.9, f"the filter changed {changed} pixels, {share:.4f} of them"
    return off, on


@pytest.mark.parametrize("lr", [False, True])
@pytest.mark.parametrize("family", list(FAMILIES))
@pytest.mark.parametrize("fuse", [True, False])
@pytest.mark.parametrize("cost", [sb.COST_SSD, sb.COST_NCORR])
@pytest.mark.parametrize("entry", ENTRIES)
def test_every_pair_entry_point_equals_the_oracle_filter(gctx, mg, entry, cost, fuse, family, lr):
    kind, win, dt = FAMILIES[family]
    if kind != "u8" and entry in ("batch_device", "band_halo_device"):
        pytest.skip("8-bit device entry point")
    if kind == "noisy" and entry == "band_host":
        pytest.skip("the host row-band entry points take 8-bit-valued images only")
    h = mg if entry.startswith("mgpu_") else gctx
    n = 5 if "batch" in entry else 1
    Ls, Rs = _images(kind, n, 500 + 7 * ENTRIES.index(entry))
    _set_fuse(h, fuse)
    try:
        # (the 17 x 17 window of the exact family leaves smooth maps: after the left-right check a few pixels at most)
        _filtered_equals_oracle_of_off(h, entry, cost, Ls, Rs, win, RANGE_T, dt, lr, min_share=0.0 if family == "exact" else 0.001)
    finally:
        _set_fuse(h, True)


@pytest.mark.parametrize("bands", [0, 3])
@pytest.mark.parametrize("kind", ["u8", "f32"])
def test_host_pipeline_items_and_bands(gctx, bands, kind):
    Ls, Rs = _images(kind, 7, 901)
    gctx.set_pipe_bands(bands)
    try:
        for cost in (sb.COST_SSD, sb.COST_NCORR):
            for lr in (False, True):
                _filtered_equals_oracle_of_off(gctx, "batch_host", cost, Ls, Rs, 3, RANGE_T, np.int16, lr, 30, 0)
    finally:
        gctx.set_pipe_bands(0)


def test_launches_of_a_filtered_pair_call(gctx):
    Ls, Rs = _images("u8", 1, 41)
    gctx.set_speckle_filter(None)
    _run(gctx, "pair_device", sb.COST_SSD, Ls, Rs, 3, RANGE_T, np.int16)
    off = gctx.last_launches
    gctx.set_speckle_filter(MAX_SIZE, MAX_DIFF)
    try:
        _run(gctx, "pair_device", sb.COST_SSD, Ls, Rs, 3, RANGE_T, np.int16)
        assert gctx.last_launches == off + 4
    finally:
        gctx.set_speckle_filter(None)


# ---- 3. / 4. full-size batches ---------------------------------------------------------------------------------------

@pytest.mark.parametrize("shape,nd,win,n,elem", [((720, 1280), 64, 4, 16, 1), ((2160, 3840), 256, 5, 1, 2)])
def test_full_size_batch_equals_the_oracle(gctx, shape, nd, win, n, elem):
    rows, cols = shape
    rng = nd - 1
    pairs = [synth.make_pair(rows, cols, nd, 60 + i)[:2] for i in range(min(n, 4))]
    Ls = np.stack([pairs[i % len(pairs)][0] for i in range(n)])
    Rs = np.stack([pairs[i % len(pairs)][1] for i in range(n)])
    gctx.set_speckle_filter(None)
    off = _device_batch(gctx, Ls, Rs, win, rng, elem)
    gctx.set_speckle_filter(100, 1)
    try:
        on = _device_batch(gctx, Ls, Rs, win, rng, elem)
        launches = gctx.last_launches
    finally:
        gctx.set_speckle_filter(None)
    cache = {}
    for side in (0, 1):
        for i in range(n):
            key = (side, i % len(pairs))
            if key not in cache:
                cache[key] = filter_speckles(off[side, i], -(rng + 1), 100, 1)
            assert np.array_equal(on[side, i], cache[key]), (side, i)
    assert np.mean(on != off) > 0.002
    if n == 16:
        _device_batch(gctx, Ls, Rs, win, rng, elem)
        assert launches == gctx.last_launches + 4    # every map of the 16 pairs in one set of filter launches


# ---- 5. graph capture -------------------------------------------------------------------------------------------------

def test_device_pair_call_with_the_filter_replays_in_a_cuda_graph(gctx):
    torch = _torch()
    rows, cols, win, rng = 120, 256, 3, 30
    inputs = [synth.make_pair(rows, cols, rng + 4, 3030 + k)[:2] for k in range(3)]
    s = torch.cuda.Stream()
    tl = torch.from_numpy(inputs[0][0]).cuda()
    tr = torch.from_numpy(inputs[0][1]).cuda()
    out = torch.full((2, rows, cols), 99, dtype=torch.int16, device="cuda")
    s.wait_stream(torch.cuda.current_stream())

    def call(c):
        _ok(_capi.lib().stereo_disparity_pair_u8_device(c.handle, sb.COST_SSD, tl.data_ptr(), cols, tr.data_ptr(), cols, rows, cols, win,
                                                        rng, out[0].data_ptr(), out[1].data_ptr(), cols * 2, 2, C.c_void_p(s.cuda_stream)))

    offc = sb.Context(0)
    try:
        gctx.set_speckle_filter(MAX_SIZE, MAX_DIFF)
        with torch.cuda.stream(s):
            call(gctx)                                  # warm-up: sizes the scratch arena
        s.synchronize()
        g = torch.cuda.CUDAGraph()
        out.fill_(99)
        torch.cuda.synchronize()
        with torch.cuda.graph(g, stream=s, capture_error_mode="thread_local"):
            call(gctx)
        assert (out == 99).all().item()                 # captured, not run
        for L, Rt in inputs[1:]:
            tl.copy_(torch.from_numpy(L))
            tr.copy_(torch.from_numpy(Rt))
            torch.cuda.synchronize()
            g.replay()
            torch.cuda.synchronize()
            got = out.cpu().numpy()
            off_l, off_r = offc.disparity_pair(sb.COST_SSD, L, Rt, win, rng, dtype=np.int16)
            want_l = filter_speckles(off_l, -(rng + 1), MAX_SIZE, MAX_DIFF)
            want_r = filter_speckles(off_r, -(rng + 1), MAX_SIZE, MAX_DIFF)
            assert np.array_equal(got[0], want_l) and np.array_equal(got[1], want_r)
            assert (want_l != off_l).any()
    finally:
        offc.close()
        gctx.set_speckle_filter(None)
