"""Left-right consistency check on the B200 (stereo_ctx_set_lr_check, stereo_lr_check_device): the kernel alone against the
check's restatement (lr_oracle.lr_check) on adversarial maps; every pair entry point with the check on against the
restatement applied to the same call's maps with it off, for both costs, fused and unfused, on each kernel family; the
reference's SSD at the ps2 shape; the default and off states; the sentinel rule; and a CUDA graph around the band-halo
pair call."""
import ctypes as C

import numpy as np
import pytest

import oracle
from lr_oracle import lr_check
import introtocomputervision_b200 as sb
from introtocomputervision_b200 import _capi, synth
from pair_calls import COLS_T, FAMILIES, RANGE_T, _images, _ok, _run, _set_fuse, _torch, gctx, mg

pytestmark = pytest.mark.gpu

ARG, RANGE, UNSUP = _capi.ERR_INVALID_ARG, _capi.ERR_INVALID_RANGE, _capi.ERR_UNSUPPORTED


# ---- 1. the kernel alone ---------------------------------------------------------------------------------------------

def _maps(g, rows, cols, rng, dt):
    """A row-wise constant shift (partners off the left edge of the left map and the right edge of the right map), a
    quarter of the pixels replaced by values around the image width, and both range ends present."""
    near = min(rng, cols + 2)
    s = g.integers(0, min(rng, cols) + 1, (rows, 1))
    dl = np.broadcast_to(-s, (rows, cols)).copy()
    dr = np.broadcast_to(s, (rows, cols)).copy()
    for d, sign in ((dl, -1), (dr, 1)):
        m = g.random((rows, cols)) < 0.25
        d[m] = sign * g.integers(0, near + 1, int(m.sum()))
        d[0, 0] = sign * rng
        d[-1, -1] = sign * rng
    return dl.astype(dt), dr.astype(dt)


def _padded(a, pad):
    rows, cols = a.shape
    buf = np.full((rows, cols * a.itemsize + pad), 0x5A, np.uint8)
    buf[:, :cols * a.itemsize] = a.view(np.uint8).reshape(rows, -1)
    return buf


KERNEL_CASES = [(e, c) for e in (1, 2, 4) for c in (1, 7, 640, 3840)] + [(1, 20480), (2, 20481), (4, 32768), (2, 32768)]


@pytest.mark.parametrize("elem,cols", KERNEL_CASES)
def test_kernel_alone_equals_the_oracle(gctx, elem, cols):
    torch = _torch()
    dt = {1: np.int8, 2: np.int16, 4: np.int32}[elem]
    rng = {1: 127, 2: 32767 if cols == 32768 else 700, 4: 32768 if cols == 32768 else 5000}[elem]
    rows, pad = (2 if cols == 32768 else 5), 96
    g = np.random.default_rng(cols * 10 + elem)
    dl, dr = _maps(g, rows, cols, rng, dt)
    side = torch.cuda.Stream()
    for max_diff in (0, 1, 2 * rng):
        hl, hr = _padded(dl, pad), _padded(dr, pad)
        tl, tr = torch.from_numpy(hl).cuda(), torch.from_numpy(hr).cuda()
        side.wait_stream(torch.cuda.current_stream())
        rc = _capi.lib().stereo_lr_check_device(gctx.handle, tl.data_ptr(), tr.data_ptr(), hl.shape[1], elem, rows, cols, rng,
                                                max_diff, C.c_void_p(side.cuda_stream))
        _ok(rc, "stereo_lr_check_device")
        assert gctx.last_launches == 1
        torch.cuda.synchronize()
        ol, orr = tl.cpu().numpy(), tr.cpu().numpy()
        wl, wr = lr_check(dl, dr, rng, max_diff)
        n = cols * elem
        assert np.array_equal(ol[:, :n].copy().view(dt), wl), (elem, cols, max_diff)
        assert np.array_equal(orr[:, :n].copy().view(dt), wr), (elem, cols, max_diff)
        assert (ol[:, n:] == 0x5A).all() and (orr[:, n:] == 0x5A).all(), "row padding written"
        if cols >= 640 and max_diff == 0:
            kept = float(np.mean(wl == dl))
            assert 0.05 < kept < 0.95, kept


def test_kernel_alone_argument_checks(gctx):
    torch = _torch()
    buf = torch.zeros((2, 4, 256), dtype=torch.uint8, device="cuda")
    a, b = buf[0].data_ptr(), buf[1].data_ptr()
    lib = _capi.lib()

    def call(l=a, r=b, step=256, elem=2, rows=4, cols=64, rng=10, max_diff=1):
        return lib.stereo_lr_check_device(gctx.handle, l, r, step, elem, rows, cols, rng, max_diff, None)

    assert call() == _capi.STEREO_OK
    assert call(l=None) == ARG and call(r=None) == ARG
    assert call(rows=0) == ARG and call(cols=0) == ARG
    assert call(rows=32769) == UNSUP and call(cols=32769, step=32769 * 2) == UNSUP
    assert call(elem=3) == ARG and call(step=127) == ARG
    assert call(rng=-1) == RANGE and call(max_diff=-1) == ARG
    assert call(elem=1, rng=128) == UNSUP and call(elem=2, rng=32768) == UNSUP
    assert call(elem=1, rng=127) == _capi.STEREO_OK and call(elem=4, rng=32768) == _capi.STEREO_OK
    assert lib.stereo_lr_check_device(None, a, b, 256, 2, 4, 64, 10, 1, None) == ARG
    gctx.synchronize()


# ---- 2. every pair entry point ---------------------------------------------------------------------------------------

ENTRIES = ["pair_host", "pair_device", "batch_device", "batch_host", "band_host", "band_halo_device", "mgpu_batch", "mgpu_bands"]
def _on_equals_oracle_of_off(h, entry, cost, Ls, Rs, win, rng, dt, max_diff):
    try:
        h.set_lr_check(None)
        off_l, off_r = _run(h, entry, cost, Ls, Rs, win, rng, dt)
        h.set_lr_check(max_diff)
        on_l, on_r = _run(h, entry, cost, Ls, Rs, win, rng, dt)
    finally:
        h.set_lr_check(None)
    for i in range(len(Ls)):
        wl, wr = lr_check(off_l[i], off_r[i], rng, max_diff)
        bad = np.argwhere(on_l[i] != wl)
        assert bad.size == 0, f"{entry} pair {i}: left map differs at {bad[:5].tolist()} (of {len(bad)})"
        assert np.array_equal(on_r[i], wr), f"{entry} pair {i}: right map differs"
    changed = (on_l != off_l) | (on_r != off_r)
    assert changed.any() and not changed.all()
    return off_l, off_r


@pytest.mark.parametrize("family", list(FAMILIES))
@pytest.mark.parametrize("fuse", [True, False])
@pytest.mark.parametrize("cost", [sb.COST_SSD, sb.COST_NCORR])
@pytest.mark.parametrize("entry", ENTRIES)
def test_every_pair_entry_point_equals_the_oracle_check(gctx, mg, entry, cost, fuse, family):
    kind, win, dt = FAMILIES[family]
    if kind != "u8" and entry in ("batch_device", "band_halo_device"):
        pytest.skip("8-bit device entry point")
    if kind == "noisy" and entry == "band_host":
        pytest.skip("the host row-band entry points take 8-bit-valued images only")
    h = mg if entry.startswith("mgpu_") else gctx
    n = 5 if "batch" in entry else 1
    Ls, Rs = _images(kind, n, 300 + 7 * ENTRIES.index(entry))
    _set_fuse(h, fuse)
    try:
        _on_equals_oracle_of_off(h, entry, cost, Ls, Rs, win, RANGE_T, dt, 1)
    finally:
        _set_fuse(h, True)


@pytest.mark.parametrize("bands", [0, 3])
@pytest.mark.parametrize("kind", ["u8", "f32"])
def test_host_pipeline_items_and_bands(gctx, bands, kind):
    Ls, Rs = _images(kind, 7, 900)
    gctx.set_pipe_bands(bands)
    try:
        for cost in (sb.COST_SSD, sb.COST_NCORR):
            _on_equals_oracle_of_off(gctx, "batch_host", cost, Ls, Rs, 3, RANGE_T, np.int16, 0)
    finally:
        gctx.set_pipe_bands(0)


# ---- 3. against the reference at the ps2 shape ---------------------------------------------------------------------

def test_ps2_shape_ssd_pair_equals_the_reference_checked(gctx):
    L, Rt, _ = synth.make_pair(511, 640, 96, 4242)
    Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
    want_l, want_r = lr_check(oracle.ssd_fast(Lf, Rf, 7, -96, 0), oracle.ssd_fast(Rf, Lf, 7, 0, 96), 96, 1)
    gctx.set_lr_check(1)
    try:
        dl, dr = sb.disparitySSDPair(Lf, Rf, sb.DisparityConfig(7, 96), ctx=gctx)
    finally:
        gctx.set_lr_check(None)
    assert np.array_equal(dl, oracle.narrow_i8(want_l)) and np.array_equal(dr, oracle.narrow_i8(want_r))
    assert 0.01 < float(np.mean(want_l == -97)) < 0.5


# ---- 4. twice the range ---------------------------------------------------------------------------------------------

def test_twice_the_range_only_drops_partners_outside_the_image(gctx):
    Ls, Rs = _images("u8", 1, 31)
    rng, cols = RANGE_T, COLS_T
    off_l, off_r = _on_equals_oracle_of_off(gctx, "pair_host", sb.COST_SSD, Ls, Rs, 3, rng, np.int16, 2 * rng)
    gctx.set_lr_check(2 * rng)
    try:
        on_l, on_r = _run(gctx, "pair_host", sb.COST_SSD, Ls, Rs, 3, rng, np.int16)
    finally:
        gctx.set_lr_check(None)
    x = np.arange(cols)
    n_outside = 0
    for off, on in ((off_l[0], on_l[0]), (off_r[0], on_r[0])):
        p = x + off.astype(np.int64)
        outside = (p < 0) | (p >= cols)
        n_outside += int(outside.sum())
        assert np.array_equal(on, np.where(outside, -(rng + 1), off))
    assert n_outside > 0


# ---- 5. graph capture -------------------------------------------------------------------------------------------------

def test_band_halo_pair_call_with_the_check_replays_in_a_cuda_graph(gctx):
    torch = _torch()
    rows, cols, win, rng, r0, r1 = 64, 200, 4, 30, 16, 48
    L, Rt, _ = synth.make_pair(rows, cols, rng + 4, 2024)
    h0, h1 = C.c_int(), C.c_int()
    _ok(_capi.lib().stereo_band_halo_rows(rows, r0, r1, win, C.byref(h0), C.byref(h1)))
    s = torch.cuda.Stream()
    tl, tr = torch.from_numpy(L).cuda(), torch.from_numpy(Rt).cuda()
    outs = {k: torch.full((2, r1 - r0, cols), 99, dtype=torch.int16, device="cuda") for k in ("off", "eager", "graph")}
    s.wait_stream(torch.cuda.current_stream())

    def call(o):
        _ok(_capi.lib().stereo_disparity_pair_band_halo_u8_device(
            gctx.handle, sb.COST_SSD, tl[h0.value].data_ptr(), cols, tr[h0.value].data_ptr(), cols, rows, cols, r0, r1, h0.value,
            h1.value, win, rng, o[0].data_ptr(), o[1].data_ptr(), cols * 2, 2, C.c_void_p(s.cuda_stream)))

    try:
        with torch.cuda.stream(s):
            call(outs["off"])
            gctx.set_lr_check(1)
            call(outs["eager"])
        s.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s, capture_error_mode="thread_local"):
            call(outs["graph"])
        assert (outs["graph"] == 99).all()            # captured, not run
        g.replay()
        torch.cuda.synchronize()
    finally:
        gctx.set_lr_check(None)
    off, eager, graph = (outs[k].cpu().numpy() for k in ("off", "eager", "graph"))
    assert np.array_equal(graph, eager)
    wl, wr = lr_check(off[0], off[1], rng, 1)
    assert np.array_equal(eager[0], wl) and np.array_equal(eager[1], wr)
    assert (eager != off).any()
