"""Semi-global matching of NCC pair calls on the B200 (stereo_ctx_set_sgm_ncc_scale): every pair entry point against the
numpy restatement (sgm_ncc_oracle) bit for bit, on 8-bit images (sliding cost kernel) and float images that are not
(per-cell cost kernel), alone and followed by the left-right check and the speckle filter; the zero-penalty rule against
the oracle's NCC maps on every kernel family's images, at 4K / 256 and on the reference's x1.1 contrast problem; a range
wider than the image; the rejections, which write nothing; the setting; settings that change nothing; and a CUDA graph
replay of a device NCC pair call."""
import ctypes as C

import numpy as np
import pytest

import introtocomputervision_b200 as sb
import oracle
from introtocomputervision_b200 import _capi, synth
from lr_oracle import lr_check
from ncc_check import score_at
from pair_calls import FAMILIES, RANGE_T, _images, _ok, _run, _torch, _untouched, gctx, mg
from sgm_ncc_oracle import quantise, sgm_pair
from speckle_oracle import filter_speckles

pytestmark = pytest.mark.gpu

ARG, UNSUP = _capi.ERR_INVALID_ARG, _capi.ERR_UNSUPPORTED
ENTRIES = ["pair_host", "pair_device", "batch_device", "batch_host", "band_host", "band_halo_device", "mgpu_batch"]
NCC = sb.COST_NCORR


def _kind_images(kind, n, seed):
    if kind == "contrast":
        Ls, Rs = _images("f32", n, seed)
        return (Ls * np.float32(1.1)).astype(np.float32), Rs
    return _images(kind, n, seed)


def _set(h, q, paths, p1, p2, lr=False, spk=False):
    h.set_sgm_ncc_scale(q)
    h.set_sgm(paths, p1, p2)
    h.set_lr_check(1 if lr else None)
    h.set_speckle_filter(20 if spk else None, 1)


def _reset(h):
    h.set_sgm(None)
    h.set_sgm_ncc_scale(0)
    h.set_lr_check(None)
    h.set_speckle_filter(None)


def _expected(Ls, Rs, R, rng, dt, q, paths, p1, p2, lr, spk):
    out = []
    for L, Rt in zip(Ls, Rs):
        dl, dr = (d.astype(dt) for d in sgm_pair(L, Rt, R, rng, q, paths, p1, p2))
        if lr:
            dl, dr = lr_check(dl, dr, rng, 1)
        if spk:
            dl, dr = filter_speckles(dl, -(rng + 1), 20, 1), filter_speckles(dr, -(rng + 1), 20, 1)
        out.append((np.asarray(dl, dt), np.asarray(dr, dt)))
    return out


def _assert_maps(on, want, n, what):
    for i in range(n):
        for side in (0, 1):
            bad = np.argwhere(on[side][i] != want[i][side])
            assert bad.size == 0, f"{what} pair {i} map {side}: {bad[:5].tolist()} of {len(bad)}"


# paths, P1, P2, R, range, map type, left-right check, speckle filter, q
CONFIGS = [(4, 1, 3, 0, RANGE_T, np.int8, False, False, 1),
           (8, 20, 300, 1, RANGE_T, np.int16, True, False, 1000),
           (8, 600, 6000, 3, 140, np.int16, False, True, 1 << 15),
           (4, 0, 3000000, 7, RANGE_T, np.int32, True, True, 1 << 24)]


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
    Ls, Rs = _kind_images(kind, n, 900 + 7 * ENTRIES.index(entry))
    for paths, p1, p2, R, rng, dt, lr, spk, q in CONFIGS:
        _set(h, q, paths, p1, p2, lr, spk)
        try:
            on = _run(h, entry, NCC, Ls, Rs, R, rng, dt, bands=[(0, Ls.shape[1])])
        finally:
            _reset(h)
        if not isinstance(h, sb.MultiGpu):
            assert h.last_path == sb.PATH_SGM
        _assert_maps(on, _expected(Ls, Rs, R, rng, dt, q, paths, p1, p2, lr, spk), n, f"{entry} {kind} q{q} {paths}/{p1}/{p2} R{R}")


@pytest.mark.parametrize("entry", ["pair_device", "pair_host"])
def test_a_range_wider_than_the_image(gctx, entry):
    L, Rt, _ = synth.make_pair(12, 40, 10, 91)
    if entry == "pair_host":
        L, Rt = (L * np.float32(1.1)).astype(np.float32), Rt.astype(np.float32)
    rng = 60                                                    # clipped to |d| <= 39
    for paths, p1, p2, R, q in ((4, 20, 300, 1, 1000), (8, 90, 700, 3, 1 << 12)):
        _set(gctx, q, paths, p1, p2)
        try:
            on = _run(gctx, entry, NCC, L[None], Rt[None], R, rng, np.int16)
        finally:
            _reset(gctx)
        dl, dr = sgm_pair(L, Rt, R, rng, q, paths, p1, p2)
        assert np.array_equal(on[0][0], dl) and np.array_equal(on[1][0], dr), (entry, paths, R)


# rows, cols, R, range, paths, P1, P2, q: widths that leave a partial last block and 7, 10 and 16 candidates per lane
ODD_SHAPES = [(24, 300, 2, 200, 4, 40, 400, 1000), (20, 1000, 1, 300, 8, 7, 90, 256), (12, 600, 3, 511, 4, 300, 5000, 1 << 15),
              (30, 333, 0, 170, 8, 2, 20, 100)]


@pytest.mark.parametrize("entry", ["pair_device", "pair_host"])
@pytest.mark.parametrize("shape", ODD_SHAPES)
def test_odd_widths_and_wide_ranges_equal_the_restatement(gctx, shape, entry):
    rows, cols, R, rng, paths, p1, p2, q = shape
    L, Rt, _ = synth.make_pair(rows, cols, min(rng, 60), 600 + cols)
    if entry == "pair_host":                                    # float images that are not 8-bit-valued: per-cell kernel
        L, Rt = L.astype(np.float32), (Rt.astype(np.float32) * np.float32(1.1)).astype(np.float32)
    _set(gctx, q, paths, p1, p2)
    try:
        on = _run(gctx, entry, NCC, L[None], Rt[None], R, rng, np.int16)
        assert gctx.last_path == sb.PATH_SGM
    finally:
        _reset(gctx)
    dl, dr = sgm_pair(L, Rt, R, rng, q, paths, p1, p2)
    for got, want, side in ((on[0][0], dl, "left"), (on[1][0], dr, "right")):
        bad = np.argwhere(got != want)
        assert bad.size == 0, f"{shape} {entry} {side}: {bad[:5].tolist()} of {len(bad)}"


# ---- 2. zero penalties: the first candidate of the oracle winner's quantum ---------------------------------------------

def _check_zero_penalty_map(got, ref, tgt, R, lo, hi, q, what, want=None):
    """Where the map differs from the oracle's NCC map, it holds an earlier candidate whose floor(fl32(q·s)) equals the
    oracle winner's (both scores by ncc_check.score_at).  Returns the number of differing pixels."""
    ref, tgt = np.asarray(ref, np.float32), np.asarray(tgt, np.float32)
    if want is None:
        want = oracle.ncorr(ref, tgt, R, lo, hi)
    got = got.astype(np.int64)
    ys, xs = np.nonzero(got != want)
    assert (got[ys, xs] < want[ys, xs]).all(), f"{what}: a later candidate than the oracle's"
    if len(ys):
        sg = score_at(ref, tgt, R, lo, hi, ys, xs, got[ys, xs])
        so = score_at(ref, tgt, R, lo, hi, ys, xs, want[ys, xs])
        bad = np.nonzero(quantise(sg, q) != quantise(so, q))[0]
        assert bad.size == 0, f"{what}: {len(bad)} pixels outside the winner's quantum, first {[(int(ys[i]), int(xs[i])) for i in bad[:5]]}"
    return len(ys)


@pytest.mark.parametrize("q", [1, 1000, 1 << 24])
@pytest.mark.parametrize("family", list(FAMILIES))
@pytest.mark.parametrize("entry", ["pair_device", "pair_host", "batch_device", "batch_host"])
def test_zero_penalties_keep_the_oracle_winners_quantum(gctx, entry, family, q):
    kind, win, dt = FAMILIES[family]
    if kind != "u8" and entry == "batch_device":
        pytest.skip("8-bit device entry point")
    n = 2 if "batch" in entry else 1
    Ls, Rs = _images(kind, n, 40 + q % 7)
    for paths in (4, 8):
        _set(gctx, q, paths, 0, 0)
        try:
            on = _run(gctx, entry, NCC, Ls, Rs, win, RANGE_T, np.int32)
        finally:
            _reset(gctx)
        for i in range(n):
            _check_zero_penalty_map(on[0][i], Ls[i], Rs[i], win, -RANGE_T, 0, q, f"{entry} {family} q{q} L->R")
            _check_zero_penalty_map(on[1][i], Rs[i], Ls[i], win, 0, RANGE_T, q, f"{entry} {family} q{q} R->L")


def test_zero_penalties_at_4k(gctx):
    rows, cols, nd, win, q = 2160, 3840, 256, 5, 1 << 20
    L, Rt, _ = synth.make_pair(rows, cols, nd, 4096)
    _set(gctx, q, 8, 0, 0)
    try:
        dl, dr = gctx.disparity_pair(NCC, L, Rt, win, nd - 1, dtype=np.int16)
    finally:
        _reset(gctx)
    for got, a, b, lo, hi in ((dl, L, Rt, 1 - nd, 0), (dr, Rt, L, 0, nd - 1)):
        differ = _check_zero_penalty_map(got, a, b, win, lo, hi, q, f"4K [{lo}, {hi}]", want=oracle.ncorr_fast(a, b, win, lo, hi))
        print(f"4K/256 q=2^20 [{lo}, {hi}]: {differ} pixels differ from the oracle, all in the winner's quantum")


def test_reference_contrast_problem_at_full_size(gctx):
    """The reference's NCC problem (511x640, R = 7, range 95) at x1.1 contrast: float images, the per-cell cost kernel."""
    rows, cols, R, rng, q = 511, 640, 7, 95, 1 << 16
    L, Rt, _ = synth.make_pair(rows, cols, rng + 1, 11)
    a, b = synth.contrast_variant(L), Rt.astype(np.float32)
    _set(gctx, q, 8, 0, 0)
    try:
        dl, dr = gctx.disparity_pair(NCC, a, b, R, rng, dtype=np.int16)
        assert gctx.last_path == sb.PATH_SGM
    finally:
        _reset(gctx)
    for got, x, y, lo, hi in ((dl, a, b, -rng, 0), (dr, b, a, 0, rng)):
        differ = _check_zero_penalty_map(got, x, y, R, lo, hi, q, f"contrast [{lo}, {hi}]")
        print(f"511x640/95 contrast q=2^16 [{lo}, {hi}]: {differ} pixels differ from the oracle, all in the winner's quantum")


# ---- 3. rejections -----------------------------------------------------------------------------------------------------

HOST_ENTRIES = ["pair_host", "batch_host", "mgpu_batch"]


@pytest.mark.parametrize("entry", ["pair_device", "batch_device"] + HOST_ENTRIES)
def test_scale_zero_still_refuses_ncc(gctx, mg, entry):
    h = mg if entry.startswith("mgpu_") else gctx
    Ls, Rs = _images("u8", 2, 5)
    _set(h, 0, 4, 1, 10)
    try:
        rc, untouched = _untouched(h, entry, Ls, Rs, 3, RANGE_T, cost=NCC)
        assert rc == UNSUP and untouched, (entry, rc)
        assert "SSD" in _capi.last_error()
        h.set_sgm_ncc_scale(100)                                    # the same call with a scale is served
        rc, untouched = _untouched(h, entry, Ls, Rs, 3, RANGE_T, cost=NCC)
        _ok(rc, entry)
        assert not untouched
    finally:
        _reset(h)


@pytest.mark.parametrize("paths", [4, 8])
@pytest.mark.parametrize("q", [1000, 1 << 24])
def test_the_int32_bound_is_exact(gctx, paths, q):
    Ls, Rs = _images("u8", 1, 9)
    Lf = (Ls * np.float32(1.1)).astype(np.float32)
    p2 = (2 ** 31 - 1) // paths - 2 * q                   # the largest P2 with paths (2q + P2) <= 2^31 - 1
    for entry, a, b in (("pair_device", Ls, Rs), ("batch_device", Ls, Rs), ("pair_host", Ls, Rs), ("pair_host", Lf, Rs.astype(np.float32))):
        for R in (0, 7):
            _set(gctx, q, paths, 0, p2)
            try:
                rc, _ = _untouched(gctx, entry, a, b, R, 10, cost=NCC)
                _ok(rc, f"{entry} at the bound")
                gctx.set_sgm(paths, 0, p2 + 1)
                rc, untouched = _untouched(gctx, entry, a, b, R, 10, cost=NCC)
                assert rc == UNSUP and untouched, (entry, R, rc)
            finally:
                _reset(gctx)


@pytest.mark.parametrize("entry", ["pair_device"] + HOST_ENTRIES)
def test_non_finite_images_are_rejected(gctx, mg, entry):
    h = mg if entry.startswith("mgpu_") else gctx
    Ls, Rs = _images("noisy", 2, 11)
    _set(h, 1000, 8, 20, 200)
    try:
        for bad in (np.nan, np.inf, -np.inf):
            L2 = Ls.copy()
            L2[:, 7, 11] = bad
            rc, untouched = _untouched(h, entry, L2, Rs, 1, RANGE_T, cost=NCC)
            assert rc == UNSUP and untouched, (entry, bad, rc)
        rc, untouched = _untouched(h, entry, Ls, Rs, 1, RANGE_T, cost=NCC)
        _ok(rc, entry)
    finally:
        _reset(h)


def test_too_many_candidates_are_rejected(gctx):
    g = np.random.default_rng(3)
    Ls = g.integers(0, 256, (1, 8, 1000)).astype(np.uint8)
    Rs = g.integers(0, 256, (1, 8, 1000)).astype(np.uint8)
    _set(gctx, 1000, 4, 10, 100)
    try:
        rc, untouched = _untouched(gctx, "pair_device", Ls, Rs, 1, 600, cost=NCC)
        assert rc == UNSUP and untouched and "candidates" in _capi.last_error()
        rc, _ = _untouched(gctx, "pair_device", Ls, Rs, 1, 511, cost=NCC)               # 512 candidates: served
        _ok(rc)
    finally:
        _reset(gctx)


# ---- 4. settings that change nothing -----------------------------------------------------------------------------------

def test_settings_that_change_nothing(gctx):
    Ls, Rs = _images("u8", 2, 79)
    Lf, Rf = _images("noisy", 1, 81)
    fresh = sb.Context(0)
    try:
        for entry, a, b in (("pair_host", Ls[:1], Rs[:1]), ("pair_device", Ls[:1], Rs[:1]), ("batch_device", Ls, Rs),
                            ("batch_host", Ls, Rs), ("pair_host", Lf, Rf)):
            # q with SGM off: the NCC maps of a fresh context
            want = _run(fresh, entry, NCC, a, b, 3, RANGE_T, np.int16)
            gctx.set_sgm_ncc_scale(1000)
            got = _run(gctx, entry, NCC, a, b, 3, RANGE_T, np.int16)
            assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), entry
            assert gctx.last_path != sb.PATH_SGM
            # SSD with SGM on: the same maps with q set or not
            gctx.set_sgm(8, 10, 200)
            with_q = _run(gctx, entry, sb.COST_SSD, a, b, 3, RANGE_T, np.int16)
            gctx.set_sgm_ncc_scale(0)
            without = _run(gctx, entry, sb.COST_SSD, a, b, 3, RANGE_T, np.int16)
            assert np.array_equal(with_q[0], without[0]) and np.array_equal(with_q[1], without[1]), entry
            gctx.set_sgm(None)
        fresh.set_sgm_ncc_scale(77)                                    # SGM on and off again: q stays
        fresh.set_sgm(8, 1, 2)
        fresh.set_sgm(None)
        assert fresh.sgm_ncc_scale == 77 and fresh.sgm is None
    finally:
        fresh.close()
        _reset(gctx)


# ---- 5. graph capture --------------------------------------------------------------------------------------------------

def test_device_ncc_pair_call_with_sgm_replays_in_a_cuda_graph(gctx):
    torch = _torch()
    rows, cols, win, rng, paths, p1, p2, q = 96, 200, 3, 30, 8, 40, 400, 1000
    inputs = [synth.make_pair(rows, cols, rng + 4, 3170 + k)[:2] for k in range(3)]
    s = torch.cuda.Stream()
    tl = torch.from_numpy(inputs[0][0]).cuda()
    tr = torch.from_numpy(inputs[0][1]).cuda()
    out = torch.full((2, rows, cols), 99, dtype=torch.int16, device="cuda")
    s.wait_stream(torch.cuda.current_stream())

    def call():
        _ok(_capi.lib().stereo_disparity_pair_u8_device(gctx.handle, NCC, tl.data_ptr(), cols, tr.data_ptr(), cols, rows, cols,
                                                        win, rng, out[0].data_ptr(), out[1].data_ptr(), cols * 2, 2, C.c_void_p(s.cuda_stream)))

    _set(gctx, q, paths, p1, p2)
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
            dl, dr = sgm_pair(L, Rt, win, rng, q, paths, p1, p2)
            assert np.array_equal(got[0], dl) and np.array_equal(got[1], dr)
    finally:
        _reset(gctx)
