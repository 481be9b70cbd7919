"""Sub-pixel disparity on the B200 (stereo_ctx_set_subpixel): every pair entry point and kernel family of the block
matcher, fused and unfused, and SGM (SSD and NCC, 4 and 8 paths), each against the restatement (subpixel_oracle) applied
to the same call's integer maps; the option after the prefilter, texture threshold, uniqueness ratio, left-right check
and speckle filter; a 4K pair; the pair-option contract (setter, off again, single-direction calls, whole maps); the
refusals, which write nothing; and CUDA graph replays."""
import ctypes as C

import numpy as np
import pytest

import introtocomputervision_b200 as sb
import test_pair_options as contract
import test_uniqueness as uq
from introtocomputervision_b200 import _capi, synth
from pair_calls import RANGE_T, _images, _ok, _run, _set_fuse, _torch, _untouched, gctx, mg
from prefilter_oracle import pf
from sgm_ncc_oracle import clip_range
from sgm_ncc_oracle import cost_volume as ncc_cost_volume
from sgm_oracle import aggregate, cost_volume
from subpixel_oracle import bm_refine_rows, refine

pytestmark = pytest.mark.gpu

ARG, UNSUP = _capi.ERR_INVALID_ARG, _capi.ERR_UNSUPPORTED
SSD, NCC = sb.COST_SSD, sb.COST_NCORR
SENT = -(RANGE_T + 1)
ENTRIES = ["pair_host", "pair_device", "batch_device", "batch_host", "mgpu_batch"]


def _directions(L, Rt, rng):
    return ((L, Rt, -rng, 0), (Rt, L, 0, rng))


def _bm_want(off, L, Rt, R, rng):
    """Both refined block-matcher maps of a pair from its integer maps off = (left, right)."""
    return [refine(*cost_volume(a, b, R, lo, hi), off[side], lo, -(rng + 1))
            for side, (a, b, lo, hi) in enumerate(_directions(L, Rt, rng))]


def _check(on, want, what):
    bad = np.argwhere(on != want)
    assert bad.size == 0, f"{what}: {bad[:5].tolist()} of {len(bad)}; got {on[tuple(bad[0])]} want {want[tuple(bad[0])]}"


def _fractional(on):
    return ((np.asarray(on, np.int64) & 15) != 0).mean()


# ---- 1. block-matcher SSD maps: every pair entry point and kernel family ---------------------------------------------

@pytest.mark.parametrize("fuse", [True, False])
@pytest.mark.parametrize("family", list(uq.KINDS))
@pytest.mark.parametrize("entry", ENTRIES)
def test_block_matcher_maps_equal_the_restatement(gctx, mg, entry, family, fuse):
    kind, R, dt = uq.KINDS[family]
    dt = np.int16 if np.dtype(dt).itemsize == 1 else dt             # (1-byte maps are refused)
    if kind != "u8" and entry == "batch_device":
        pytest.skip("8-bit device entry point")
    h = mg if entry.startswith("mgpu_") else gctx
    n = 2 if "batch" in entry else 1
    Ls, Rs = uq._kind_images(kind, n, 1900 + 11 * ENTRIES.index(entry))
    _set_fuse(h, fuse)
    try:
        off = _run(h, entry, SSD, Ls, Rs, R, RANGE_T, dt)
        device = entry in ("pair_device", "batch_device")
        state = (h.last_path, h.last_fused_pairs) if device else None
        h.set_subpixel(True)
        try:
            on = _run(h, entry, SSD, Ls, Rs, R, RANGE_T, dt)
            if device:
                assert (h.last_path, h.last_fused_pairs) == state, entry
        finally:
            h.set_subpixel(False)
    finally:
        _set_fuse(h, True)
    for i in range(n):
        want = _bm_want((off[0][i], off[1][i]), Ls[i], Rs[i], R, RANGE_T)
        for side in (0, 1):
            _check(on[side][i], want[side], f"{entry} {family} fuse={fuse} pair {i} map {side}")
            assert _fractional(on[side][i]) > 0, (family, side)      # the refinement is not a no-op


# ---- 2. SGM maps ----------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("cost", ["ssd", "ncc"])
@pytest.mark.parametrize("paths", [4, 8])
@pytest.mark.parametrize("entry", ["pair_device", "pair_host", "batch_device", "batch_host", "mgpu_batch"])
def test_sgm_maps_equal_the_restatement(gctx, mg, entry, paths, cost):
    q = None if cost == "ssd" else 64
    h = mg if entry.startswith("mgpu_") else gctx
    n = 2 if "batch" in entry else 1
    Ls, Rs = _images("u8", n, 2300 + paths)
    if entry == "pair_host":
        Ls, Rs = Ls.astype(np.float32), (Rs.astype(np.float32) * np.float32(1.1)).astype(np.float32)
    p1, p2, R = (10, 120, 3) if cost == "ssd" else (2, 24, 2)
    c = SSD if q is None else NCC
    h.set_sgm(paths, p1, p2)
    h.set_sgm_ncc_scale(q or 0)
    try:
        off = _run(h, entry, c, Ls, Rs, R, RANGE_T, np.int16)
        h.set_subpixel(True)
        try:
            on = _run(h, entry, c, Ls, Rs, R, RANGE_T, np.int16)
        finally:
            h.set_subpixel(False)
    finally:
        h.set_sgm(None)
        h.set_sgm_ncc_scale(0)
    rr = RANGE_T if q is None else clip_range(Ls.shape[2], RANGE_T)
    for i in range(n):
        for side, (a, b, lo, hi) in enumerate(_directions(Ls[i], Rs[i], rr)):
            Cv, present = cost_volume(a, b, R, lo, hi) if q is None else ncc_cost_volume(a, b, R, lo, hi, q)
            want = refine(aggregate(Cv, present, paths, p1, p2), present, off[side][i], lo, SENT)
            _check(on[side][i], want, f"{entry} {cost} {paths} pair {i} map {side}")
            assert _fractional(on[side][i]) > 0


# ---- 3. after every other step ------------------------------------------------------------------------------------------

COMBOS = {
    "bm_all": dict(sgm=None, uniq=15, lr=1, spk=(20, 1), pf=None),
    "bm_prefilter_texture": dict(sgm=None, uniq=10, lr=1, spk=(20, 1), pf=(31, 150)),
    "sgm_all": dict(sgm=(8, 10, 120), uniq=15, lr=1, spk=(20, 1), pf=None),
    "sgm_prefilter_texture": dict(sgm=(8, 10, 120), uniq=0, lr=1, spk=(20, 1), pf=(31, 150)),
}


def _set_combo(h, c, on):
    h.set_sgm(*c["sgm"]) if on and c["sgm"] else h.set_sgm(None)
    h.set_uniqueness(c["uniq"] if on else 0)
    h.set_lr_check(c["lr"] if on else None)
    h.set_speckle_filter(*c["spk"]) if on else h.set_speckle_filter(None)
    h.set_prefilter(*c["pf"]) if on and c["pf"] else h.set_prefilter(None)


@pytest.mark.parametrize("combo", list(COMBOS))
@pytest.mark.parametrize("entry", ["pair_device", "batch_device", "pair_host"])
def test_after_the_other_options_only_the_refinement_changes(gctx, entry, combo):
    c = COMBOS[combo]
    n = 2 if "batch" in entry else 1
    Ls, Rs = _images("u8", n, 2400)
    R = 3
    _set_combo(gctx, c, True)
    try:
        off = _run(gctx, entry, SSD, Ls, Rs, R, RANGE_T, np.int16)
        gctx.set_subpixel(True)
        try:
            on = _run(gctx, entry, SSD, Ls, Rs, R, RANGE_T, np.int16)
        finally:
            gctx.set_subpixel(False)
    finally:
        _set_combo(gctx, c, False)
    for i in range(n):
        refs = (Ls[i], Rs[i]) if c["pf"] is None else (pf(Ls[i], c["pf"][0]), pf(Rs[i], c["pf"][0]))
        for side, (a, b, lo, hi) in enumerate(_directions(*refs, RANGE_T)):
            d = off[side][i]
            assert (d == SENT).any() and (d != SENT).any(), (combo, side)
            Cv, present = cost_volume(a, b, R, lo, hi)
            V = aggregate(Cv, present, c["sgm"][0], *c["sgm"][1:]) if c["sgm"] else Cv
            _check(on[side][i], refine(V, present, d, lo, SENT), f"{entry} {combo} pair {i} map {side}")
            assert np.array_equal((on[side][i].astype(np.int64) + 7) >> 4, d)      # the sentinel becomes 16x, nothing else


# ---- 4. full size ---------------------------------------------------------------------------------------------------------

def test_full_size_4k_pair_on_a_band_of_rows(gctx):
    rows, cols, nd, win = 2160, 3840, 256, 5
    L, Rt, _ = synth.make_pair(rows, cols, nd, 4097)
    off = gctx.disparity_pair(SSD, L, Rt, win, nd, dtype=np.int16)
    gctx.set_subpixel(True)
    try:
        on = gctx.disparity_pair(SSD, L, Rt, win, nd, dtype=np.int16)
    finally:
        gctx.set_subpixel(False)
    for side, (a, b, lo, hi) in enumerate(_directions(L, Rt, nd)):
        assert np.array_equal((on[side].astype(np.int64) + 7) >> 4, off[side]), side
        for ys in (np.arange(0, 24), np.arange(1068, 1092), np.arange(rows - 24, rows)):
            want = bm_refine_rows(a, b, win, off[side][ys], ys, lo, hi, -(nd + 1))
            _check(on[side][ys], want, f"4K map {side} rows {ys[0]}..{ys[-1]}")


# ---- 5. the pair-option contract ------------------------------------------------------------------------------------------

ROW = contract.Option("subpixel", "subpixel", "subpixel", 0, ARG, [("set_subpixel", (True,))], True, [("set_subpixel", (False,))],
                      False, bad=[(2,), (-1,), (16,)], good=[((True,), True), ((False,), False), ((1,), True), ((None,), False)],
                      c_off=[(0,)], whole=True, sentinel=None, quiet=None, changes=(SSD,))


def test_contract_off_again_is_byte_identical_to_a_fresh_context(gctx):
    contract.test_off_again_is_byte_identical_to_a_fresh_context(opt=ROW, gctx=gctx)


def test_contract_single_direction_and_refgpu_calls_ignore_the_option(gctx):
    contract.test_single_direction_and_refgpu_calls_ignore_the_option(opt=ROW, gctx=gctx)


def test_contract_partial_bands_and_mgpu_bands_are_refused_and_write_nothing(gctx, mg):
    contract.test_partial_bands_and_mgpu_bands_are_refused_and_write_nothing(opt=ROW, gctx=gctx, mg=mg)


def test_setter_and_getter(mg):
    lib = _capi.lib()
    fresh = sb.Context(0)
    try:
        assert fresh.subpixel is False and lib.stereo_ctx_subpixel(fresh.handle) == 0
        assert lib.stereo_ctx_set_subpixel(None, 1) == ARG and lib.stereo_mgpu_set_subpixel(None, 1) == ARG
        assert lib.stereo_ctx_subpixel(None) == ARG
        fresh.set_subpixel(True)
        assert fresh.subpixel is True and lib.stereo_ctx_subpixel(fresh.handle) == 1
        for bad in ROW.bad:
            assert lib.stereo_ctx_set_subpixel(fresh.handle, *bad) == ARG, bad
            assert fresh.subpixel is True, bad                                   # the old setting stays
        with pytest.raises(sb.StereoError):
            fresh.set_subpixel(2)
        for args, value in ROW.good:
            fresh.set_subpixel(*args)
            assert fresh.subpixel is value, args
        _ok(lib.stereo_ctx_set_subpixel(fresh.handle, 0))
        assert fresh.subpixel is False
        assert lib.stereo_mgpu_set_subpixel(mg._h, 2) == ARG
        with pytest.raises(sb.StereoError):
            mg.set_subpixel(3)
        try:
            mg.set_subpixel(True)
            for i in range(mg.device_count):
                assert lib.stereo_ctx_subpixel(lib.stereo_mgpu_ctx(mg._h, i)) == 1, i
        finally:
            mg.set_subpixel(False)
        for i in range(mg.device_count):
            assert lib.stereo_ctx_subpixel(lib.stereo_mgpu_ctx(mg._h, i)) == 0, i
    finally:
        fresh.close()


@pytest.mark.parametrize("entry", ["pair_device", "batch_device", "pair_host", "batch_host", "mgpu_batch"])
def test_maps_that_cannot_hold_it_and_ncc_block_matcher_calls_are_refused(gctx, mg, entry):
    h = mg if entry.startswith("mgpu_") else gctx
    Ls, Rs = _images("u8", 2, 37)
    h.set_subpixel(True)
    try:
        rc, untouched = _untouched(h, entry, Ls, Rs, 3, RANGE_T, dt=np.int8)            # 1-byte maps
        assert rc == UNSUP and untouched and "sub-pixel" in _capi.last_error(), (entry, "int8", rc)
        rc, untouched = _untouched(h, entry, Ls, Rs, 3, 2048, dt=np.int16)             # 16 (2048 + 1) > 32767
        assert rc == UNSUP and untouched and "sub-pixel" in _capi.last_error(), (entry, "int16", rc)
        rc, untouched = _untouched(h, entry, Ls, Rs, 3, RANGE_T, cost=NCC)              # NCC block matcher
        assert rc == UNSUP and untouched and "NCC" in _capi.last_error(), (entry, "ncc", rc)
        rc, _ = _untouched(h, entry, Ls[:, :, :60], Rs[:, :, :60], 1, 2047, dt=np.int16)   # range 2047 fits int16
        _ok(rc, entry)
        rc, _ = _untouched(h, entry, Ls, Rs, 3, RANGE_T, dt=np.int32)
        _ok(rc, entry)
    finally:
        h.set_subpixel(False)
    rc, untouched = _untouched(h, entry, Ls, Rs, 3, RANGE_T, dt=np.int8)                # off again: served
    _ok(rc, entry)


# ---- 6. graph capture -------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("sgm", [False, True])
def test_device_pair_call_replays_in_a_cuda_graph(sgm):
    torch = _torch()
    rows, cols, win, rng = 96, 200, 3, 30
    inputs = [synth.make_pair(rows, cols, rng + 4, 3330 + k)[:2] for k in range(3)]
    s = torch.cuda.Stream()
    tl = torch.from_numpy(inputs[0][0]).cuda()
    tr = torch.from_numpy(inputs[0][1]).cuda()
    out = torch.full((2, rows, cols), 99, dtype=torch.int16, device="cuda")
    s.wait_stream(torch.cuda.current_stream())

    def call():
        _ok(_capi.lib().stereo_disparity_pair_u8_device(cap.handle, SSD, tl.data_ptr(), cols, tr.data_ptr(), cols, rows, cols,
                                                        win, rng, out[0].data_ptr(), out[1].data_ptr(), cols * 2, 2, C.c_void_p(s.cuda_stream)))

    fresh, cap = sb.Context(0), sb.Context(0)          # (cap: a context whose calls all come from this test)
    if sgm:
        fresh.set_sgm(8, 10, 120)
        cap.set_sgm(8, 10, 120)
    cap.set_subpixel(True)
    try:
        with torch.cuda.stream(s):
            call()                                       # warm-up: sizes the scratch arena and the offset buffer
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
            off = fresh.disparity_pair(SSD, L, Rt, win, rng, dtype=np.int16)
            for side, (a, b, lo, hi) in enumerate(_directions(L, Rt, rng)):
                Cv, present = cost_volume(a, b, win, lo, hi)
                V = aggregate(Cv, present, 8, 10, 120) if sgm else Cv
                _check(got[side], refine(V, present, off[side], lo, -(rng + 1)), f"graph sgm={sgm} map {side}")
        del g
    finally:
        fresh.close()
        cap.close()
