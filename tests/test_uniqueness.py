"""The uniqueness ratio on the B200 (stereo_ctx_set_uniqueness): the block matcher's SSD maps on every pair entry point and
kernel family, fused and unfused, against the restatement (uniqueness_oracle) applied to the same call's maps without it;
SGM maps (SSD and NCC, 4 and 8 paths) against sgm_oracle / sgm_ncc_oracle; the ratio followed by the left-right check and
the speckle filter; full-size cases; the refusals, which write nothing; the setting; and a CUDA graph replay."""
import ctypes as C

import numpy as np
import pytest

import introtocomputervision_b200 as sb
from introtocomputervision_b200 import _capi, synth
from lr_oracle import lr_check
from pair_calls import RANGE_T, _device_batch, _images, _ok, _run, _set_fuse, _torch, _untouched, gctx, mg
from sgm_ncc_oracle import clip_range
from sgm_ncc_oracle import cost_volume as ncc_cost_volume
from sgm_oracle import aggregate, cost_volume, winner
from speckle_oracle import filter_speckles
from uniqueness_oracle import apply, unique

pytestmark = pytest.mark.gpu

ARG, UNSUP = _capi.ERR_INVALID_ARG, _capi.ERR_UNSUPPORTED
ENTRIES = ["pair_host", "pair_device", "batch_device", "batch_host", "band_host", "band_halo_device", "mgpu_batch"]


def _directions(L, Rt, rng):
    """(ref, tgt, dmin, dmax) of both directions of a pair call."""
    return ((L, Rt, -rng, 0), (Rt, L, 0, rng))


def _bm_keep(L, Rt, R, rng, u):
    """The ratio's keep masks of both block-matcher maps of a pair, from the restated SSD cost volumes."""
    return [unique(*cost_volume(a, b, R, lo, hi), u, block_matcher=True) for a, b, lo, hi in _directions(L, Rt, rng)]


# ---- 1. block-matcher SSD maps: every pair entry point and kernel family ---------------------------------------------

KINDS = {                # images, window radius, map type
    "u8": ("u8", 3, np.int8),
    "f32_8bit": ("f32", 3, np.int16),
    "f32_noisy": ("noisy", 3, np.int16),           # the float running-sum kernels (FAST_F32)
    "f32_wide": ("wide", 3, np.int16),             # a value range the running sums do not cover: exact kernels after the classification
    "u8_exact": ("u8", 8, np.int32),               # a radius the running sums do not cover: exact kernels
    "f32_exact": ("f32", 8, np.int32),             # the same for float images, which are then classified for the bound only
}


def _kind_images(kind, n, seed):
    if kind == "wide":
        Ls, Rs = _images("f32", n, seed)
        return (Ls * np.float32(4)).astype(np.float32), (Rs * np.float32(4)).astype(np.float32)
    return _images(kind, n, seed)


@pytest.mark.parametrize("fuse", [True, False])
@pytest.mark.parametrize("family", list(KINDS))
@pytest.mark.parametrize("entry", ENTRIES)
def test_block_matcher_maps_equal_the_restatement(gctx, mg, entry, family, fuse):
    kind, R, dt = KINDS[family]
    if kind != "u8" and entry in ("batch_device", "band_halo_device"):
        pytest.skip("8-bit device entry point")
    if kind in ("noisy", "wide") and entry == "band_host":
        pytest.skip("the host row-band entry points take 8-bit-valued images only")
    h = mg if entry.startswith("mgpu_") else gctx
    n = 2 if "batch" in entry else 1
    Ls, Rs = _kind_images(kind, n, 900 + 11 * ENTRIES.index(entry))
    whole = [(0, Ls.shape[1])]
    _set_fuse(h, fuse)
    try:
        off = _run(h, entry, sb.COST_SSD, Ls, Rs, R, RANGE_T, dt, bands=whole)
        device = entry in ("pair_device", "batch_device", "band_halo_device")       # (host calls with it on are not pipelined)
        state = (h.last_path, h.last_fused_pairs) if device else None
        for u in (10, 40):
            h.set_uniqueness(u)
            try:
                on = _run(h, entry, sb.COST_SSD, Ls, Rs, R, RANGE_T, dt, bands=whole)
                if device:
                    assert (h.last_path, h.last_fused_pairs) == state, entry
            finally:
                h.set_uniqueness(0)
            for i in range(n):
                keeps = _bm_keep(Ls[i], Rs[i], R, RANGE_T, u)
                for side in (0, 1):
                    want = apply(off[side][i], keeps[side], RANGE_T)
                    bad = np.argwhere(on[side][i] != want)
                    assert bad.size == 0, f"{entry} {family} fuse={fuse} u={u} pair {i} map {side}: {bad[:5].tolist()} of {len(bad)}"
                    assert np.array_equal(on[side][i][keeps[side]], off[side][i][keeps[side]])      # kept pixels untouched
                    if u == 40:
                        assert 0 < (~keeps[side]).sum() < keeps[side].size, (family, side)          # the rule fires, not everywhere
    finally:
        _set_fuse(h, True)


# ---- 2. SGM maps --------------------------------------------------------------------------------------------------------

def _sgm_expected(L, Rt, R, rng, paths, p1, p2, u, q=None):
    out = []
    rr = rng if q is None else clip_range(L.shape[1], rng)
    for a, b, lo, hi in _directions(L, Rt, rr):
        Cv, present = cost_volume(a, b, R, lo, hi) if q is None else ncc_cost_volume(a, b, R, lo, hi, q)
        S = aggregate(Cv, present, paths, p1, p2)
        out.append(apply(winner(S, present, lo), unique(S, present, u), rng))
    return out


@pytest.mark.parametrize("cost", ["ssd", "ncc"])
@pytest.mark.parametrize("paths", [4, 8])
@pytest.mark.parametrize("entry", ["pair_device", "pair_host", "batch_device", "batch_host"])
def test_sgm_maps_equal_the_restatement(gctx, entry, paths, cost):
    q = None if cost == "ssd" else 64
    n = 2 if "batch" in entry else 1
    Ls, Rs = _images("u8", n, 1300 + paths)
    if entry == "pair_host":
        Ls, Rs = Ls.astype(np.float32), (Rs.astype(np.float32) * np.float32(1.1)).astype(np.float32)
    p1, p2, R, u = (10, 120, 3, 10) if cost == "ssd" else (2, 24, 2, 10)
    gctx.set_sgm(paths, p1, p2)
    gctx.set_sgm_ncc_scale(q or 0)
    gctx.set_uniqueness(u)
    try:
        on = _run(gctx, entry, sb.COST_SSD if q is None else sb.COST_NCORR, Ls, Rs, R, RANGE_T, np.int16)
        assert gctx.last_path == sb.PATH_SGM
    finally:
        gctx.set_uniqueness(0)
        gctx.set_sgm(None)
        gctx.set_sgm_ncc_scale(0)
    for i in range(n):
        want = _sgm_expected(Ls[i], Rs[i], R, RANGE_T, paths, p1, p2, u, q)
        for side in (0, 1):
            bad = np.argwhere(on[side][i] != want[side])
            assert bad.size == 0, f"{entry} {cost} {paths} pair {i} map {side}: {bad[:5].tolist()} of {len(bad)}"
            assert (want[side] == -(RANGE_T + 1)).any()


# ---- 3. with the left-right check and the speckle filter --------------------------------------------------------------

@pytest.mark.parametrize("sgm", [False, True])
@pytest.mark.parametrize("entry", ["pair_device", "batch_device", "pair_host"])
def test_with_the_left_right_check_and_the_speckle_filter(gctx, entry, sgm):
    n = 2 if "batch" in entry else 1
    Ls, Rs = _images("u8", n, 1400)
    R, u = 3, 15
    off = None if sgm else _run(gctx, entry, sb.COST_SSD, Ls, Rs, R, RANGE_T, np.int16)
    if sgm:
        gctx.set_sgm(8, 10, 120)
    gctx.set_uniqueness(u)
    gctx.set_lr_check(1)
    gctx.set_speckle_filter(20, 1)
    try:
        on = _run(gctx, entry, sb.COST_SSD, Ls, Rs, R, RANGE_T, np.int16)
    finally:
        gctx.set_uniqueness(0)
        gctx.set_lr_check(None)
        gctx.set_speckle_filter(None)
        gctx.set_sgm(None)
    for i in range(n):
        if sgm:
            dl, dr = _sgm_expected(Ls[i], Rs[i], R, RANGE_T, 8, 10, 120, u)
        else:
            kl, kr = _bm_keep(Ls[i], Rs[i], R, RANGE_T, u)
            dl, dr = apply(off[0][i], kl, RANGE_T), apply(off[1][i], kr, RANGE_T)
        dl, dr = lr_check(dl, dr, RANGE_T, 1)
        dl, dr = filter_speckles(dl, -(RANGE_T + 1), 20, 1), filter_speckles(dr, -(RANGE_T + 1), 20, 1)
        assert np.array_equal(on[0][i], dl) and np.array_equal(on[1][i], dr), (entry, sgm, i)


# ---- 4. full size -------------------------------------------------------------------------------------------------------

def test_full_size_720p_device_batch(gctx):
    rows, cols, nd, win, n, u = 720, 1280, 64, 4, 16, 10
    pairs = [synth.make_pair(rows, cols, nd, 170 + i)[:2] for i in range(n)]
    Ls, Rs = np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs])
    off = _device_batch(gctx, Ls, Rs, win, nd, 1)
    gctx.set_uniqueness(u)
    try:
        on = _device_batch(gctx, Ls, Rs, win, nd, 1)
    finally:
        gctx.set_uniqueness(0)
    for i in range(n):
        for side, (a, b, lo, hi) in enumerate(_directions(Ls[i], Rs[i], nd)):
            keep = unique(*cost_volume(a, b, win, lo, hi), u, block_matcher=True)
            assert np.array_equal(on[side, i], apply(off[side, i], keep, nd)), (i, side)


def _rows_cost(ref, tgt, R, dmin, dmax, ys):
    """sgm_oracle.cost_volume restricted to the output rows ys: (len(ys), cols, D) window sums and the present mask."""
    ref = np.asarray(ref, np.float32)
    tgt = np.asarray(tgt, np.float32)
    rows, cols = ref.shape
    Hp, Wp, w = rows + 2 * R, cols + 2 * R, 2 * R + 1
    Lp = np.pad(ref, R, mode="edge")
    flat = np.concatenate([np.pad(tgt, R, mode="edge").reshape(-1), np.zeros(1, np.float32)])     # [-1]: the zero guard
    c = np.arange(Wp)[:, None] + np.arange(dmin, dmax + 1)[None, :]
    out = np.empty((len(ys), cols, dmax - dmin + 1), np.int64)
    for k, y in enumerate(ys):
        acc = np.zeros((Wp, dmax - dmin + 1), np.int64)
        for wy in range(w):
            f = (y + wy) * Wp + c
            f = np.where((f >= 0) & (f < Hp * Wp), f, -1)
            dd = Lp[y + wy][:, None] - flat[f]
            acc += np.floor((dd * dd).astype(np.float32).astype(np.float64) + 0.5).astype(np.int64)
        I = np.concatenate([np.zeros((1, acc.shape[1]), np.int64), acc.cumsum(0)])
        out[k] = I[w:] - I[:-w]
    s = np.arange(cols)[:, None] + R + np.arange(dmin, dmax + 1)[None, :]
    return out, np.broadcast_to(((s >= 0) & (s <= Wp - 1))[None], out.shape)


def test_rows_cost_equals_the_cost_volume():
    L, Rt, _ = synth.make_pair(20, 70, 12, 5)
    full, present = cost_volume(L, Rt, 2, -15, 3)
    ys = [0, 7, 19]
    part, pp = _rows_cost(L, Rt, 2, -15, 3, ys)
    assert np.array_equal(part, full[ys]) and np.array_equal(pp, present[ys])


def test_full_size_4k_pair_on_spread_rows(gctx):
    rows, cols, nd, win, u = 2160, 3840, 256, 5, 10
    L, Rt, _ = synth.make_pair(rows, cols, nd, 4096)
    off = gctx.disparity_pair(sb.COST_SSD, L, Rt, win, nd, dtype=np.int16)
    gctx.set_uniqueness(u)
    try:
        on = gctx.disparity_pair(sb.COST_SSD, L, Rt, win, nd, dtype=np.int16)
    finally:
        gctx.set_uniqueness(0)
    ys = np.linspace(0, rows - 1, 64).round().astype(int)
    for side, (a, b, lo, hi) in enumerate(_directions(L, Rt, nd)):
        keep = unique(*_rows_cost(a, b, win, lo, hi, ys), u, block_matcher=True)
        assert np.array_equal(on[side][ys], apply(off[side][ys], keep, nd)), side
        others = np.setdiff1d(np.arange(rows), ys)
        changed = on[side][others] != off[side][others]
        assert (on[side][others][changed] == -(nd + 1)).all()                  # elsewhere only sentinels are written


# ---- 5. refusals ----------------------------------------------------------------------------------------------------------

REFUSE_ENTRIES = ["pair_device", "batch_device", "pair_host", "batch_host", "mgpu_batch"]


@pytest.mark.parametrize("entry", REFUSE_ENTRIES)
def test_sentinel_ncc_bound_and_candidate_refusals_write_nothing(gctx, mg, entry):
    h = mg if entry.startswith("mgpu_") else gctx
    Ls, Rs = _images("u8", 2, 31)
    h.set_uniqueness(10)
    try:
        rc, untouched = _untouched(h, entry, Ls, Rs, 3, 128, dt=np.int8)            # -(128 + 1) does not fit int8
        assert rc == UNSUP and untouched, (entry, "sentinel", rc)
        rc, untouched = _untouched(h, entry, Ls, Rs, 3, RANGE_T, cost=sb.COST_NCORR)     # NCC block matcher
        assert rc == UNSUP and untouched and "NCC" in _capi.last_error(), (entry, "ncc", rc)
        rc, untouched = _untouched(h, entry, Ls, Rs, 64, RANGE_T)                    # 129^2 * 255^2 >= 2^30
        assert rc == UNSUP and untouched, (entry, "bound", rc)
        rc, _ = _untouched(h, entry, Ls, Rs, 63, RANGE_T)                            # 127^2 * 255^2 < 2^30: served
        _ok(rc, entry)
        g = np.random.default_rng(3)
        Lw = g.integers(0, 256, (2, 6, 1000)).astype(np.uint8)
        Rw = g.integers(0, 256, (2, 6, 1000)).astype(np.uint8)
        rc, untouched = _untouched(h, entry, Lw, Rw, 1, 600, dt=np.int16)           # 601 candidates
        assert rc == UNSUP and untouched and "candidates" in _capi.last_error(), (entry, "candidates", rc)
        rc, _ = _untouched(h, entry, Lw, Rw, 1, 511, dt=np.int16)                    # 512: served
        _ok(rc, entry)
    finally:
        h.set_uniqueness(0)
    rc, untouched = _untouched(h, entry, Ls, Rs, 3, RANGE_T, cost=sb.COST_NCORR)    # off again: NCC served
    _ok(rc, entry)


@pytest.mark.parametrize("entry", ["pair_device", "pair_host", "batch_host", "mgpu_batch"])
def test_float_bound_and_non_finite_images_are_refused(gctx, mg, entry):
    h = mg if entry.startswith("mgpu_") else gctx
    Ls, Rs = _images("f32", 2, 41)
    h.set_uniqueness(10)
    try:
        for R in (3, 8):                                   # classified by the block matcher, and classified for the bound only
            big = (Ls * np.float32(100)).astype(np.float32)          # (hi - lo)^2 ~ 6.5e8: over the bound at any radius
            rc, untouched = _untouched(h, entry, big, Rs, R, RANGE_T)
            assert rc == UNSUP and untouched, (entry, R, "bound", rc)
            for bad in (np.nan, np.inf):
                L2 = Ls.copy()
                L2[:, 7, 11] = bad
                rc, untouched = _untouched(h, entry, L2, Rs, R, RANGE_T)
                assert rc == UNSUP and untouched, (entry, R, bad, rc)
            rc, _ = _untouched(h, entry, Ls, Rs, R, RANGE_T)
            _ok(rc, entry)
    finally:
        h.set_uniqueness(0)


# ---- 6. graph capture ----------------------------------------------------------------------------------------------------

def test_device_pair_call_replays_in_a_cuda_graph(gctx):
    torch = _torch()
    rows, cols, win, rng, u = 96, 200, 3, 30, 15
    inputs = [synth.make_pair(rows, cols, rng + 4, 3230 + k)[:2] for k in range(3)]
    s = torch.cuda.Stream()
    tl = torch.from_numpy(inputs[0][0]).cuda()
    tr = torch.from_numpy(inputs[0][1]).cuda()
    out = torch.full((2, rows, cols), 99, dtype=torch.int16, device="cuda")
    s.wait_stream(torch.cuda.current_stream())

    def call():
        _ok(_capi.lib().stereo_disparity_pair_u8_device(gctx.handle, sb.COST_SSD, tl.data_ptr(), cols, tr.data_ptr(), cols, rows, cols,
                                                        win, rng, out[0].data_ptr(), out[1].data_ptr(), cols * 2, 2, C.c_void_p(s.cuda_stream)))

    fresh = sb.Context(0)
    gctx.set_uniqueness(u)
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
            off = fresh.disparity_pair(sb.COST_SSD, L, Rt, win, rng, dtype=np.int16)
            keeps = _bm_keep(L, Rt, win, rng, u)
            assert np.array_equal(got[0], apply(off[0], keeps[0], rng)) and np.array_equal(got[1], apply(off[1], keeps[1], rng))
        del g
    finally:
        gctx.set_uniqueness(0)
        fresh.close()
