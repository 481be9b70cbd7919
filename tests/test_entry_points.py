"""Rejected inputs, entry point by entry point: the status each C ABI disparity entry point returns for one bad argument
in an otherwise valid call.  Host entry points report images over 32768 pixels as INVALID_ARG, the device ones (except the
reference-semantics kernel) as UNSUPPORTED; the host row-band pair reports a negative range as INVALID_ARG."""
import ctypes as C

import numpy as np
import pytest

import introtocomputervision_b200 as sb
from introtocomputervision_b200 import _capi

pytestmark = pytest.mark.gpu

ARG, RANGE, UNSUP = _capi.ERR_INVALID_ARG, _capi.ERR_INVALID_RANGE, _capi.ERR_UNSUPPORTED
ROWS, COLS, PITCH = 16, 32, 128           # PITCH: bytes per row of every buffer (>= COLS * 4)

# one bad argument each; every other argument is that of a valid call
CASES = {
    "null_image": dict(img=False),
    "null_output": dict(out=False),
    "zero_rows": dict(rows=0),
    "over_32768": dict(rows=32769),
    "short_step": dict(short=True),
    "dmin_gt_dmax": dict(dmin=-3, dmax=-5),
    "negative_range": dict(rng=-1),
    "empty_halo": dict(halo=(5, 5)),
    "halo_past_image": dict(halo=(0, ROWS + 1)),
    "no_pairs": dict(n=0),
    "elem_3": dict(elem=3),
}

_SINGLE = dict(null_image=ARG, null_output=ARG, zero_rows=ARG, short_step=ARG, dmin_gt_dmax=RANGE, elem_3=ARG)
_PAIR = dict(null_image=ARG, null_output=ARG, zero_rows=ARG, short_step=ARG, negative_range=RANGE, elem_3=ARG)
_HALO = dict(empty_halo=ARG, halo_past_image=ARG)
_BATCH = dict(no_pairs=ARG)
EXPECTED = {
    "stereo_disparity_f32_host": dict(_SINGLE, over_32768=ARG),
    "stereo_disparity_u8_host": dict(_SINGLE, over_32768=ARG),
    "stereo_disparity_f32_device": dict(_SINGLE, over_32768=UNSUP),
    "stereo_disparity_u8_device": dict(_SINGLE, over_32768=UNSUP),
    "stereo_disparity_band_u8_device": dict(_SINGLE, over_32768=UNSUP),
    "stereo_disparity_band_halo_u8_device": dict(_SINGLE, over_32768=UNSUP, **_HALO),
    "stereo_disparity_refgpu_f32_host": {k: v for k, v in dict(_SINGLE, over_32768=ARG).items() if k != "elem_3"},
    "stereo_disparity_refgpu_f32_device": {k: v for k, v in dict(_SINGLE, over_32768=ARG).items() if k != "elem_3"},
    "stereo_disparity_pair_f32_host": dict(_PAIR, over_32768=ARG),
    "stereo_disparity_pair_u8_host": dict(_PAIR, over_32768=ARG),
    "stereo_disparity_pair_f32_device": dict(_PAIR, over_32768=UNSUP),
    "stereo_disparity_pair_u8_device": dict(_PAIR, over_32768=UNSUP),
    "stereo_disparity_pair_band_halo_u8_device": dict(_PAIR, over_32768=UNSUP, **_HALO),
    "stereo_disparity_pair_band_u8_host": dict(_PAIR, over_32768=ARG, negative_range=ARG),
    "stereo_disparity_pair_band_f32_host": dict(_PAIR, over_32768=ARG, negative_range=ARG),
    "stereo_disparity_pair_batch_u8_device": dict(_PAIR, over_32768=UNSUP, **_BATCH),
    "stereo_disparity_pair_batch_u8_host": dict(_PAIR, over_32768=ARG, **_BATCH),
    "stereo_disparity_pair_batch_f32_host": dict(_PAIR, over_32768=ARG, **_BATCH),
}


@pytest.fixture(scope="module")
def bufs():
    """A context of its own (nothing forced) and two images and two maps of 2 x ROWS x PITCH bytes each, on the host and
    on the device.  No rejected call reads or writes them."""
    import torch
    c = sb.Context(0)
    host = [np.zeros((2, ROWS, PITCH), np.uint8) for _ in range(4)]
    dev = [torch.zeros((2, ROWS, PITCH), dtype=torch.uint8, device="cuda") for _ in range(4)]
    torch.cuda.synchronize()
    yield c, [a.ctypes.data for a in host], [t.data_ptr() for t in dev]
    c.close()


def _args(name, ctx, ptrs, img=True, out=True, rows=ROWS, short=False, dmin=-3, dmax=0, rng=3, halo=(0, ROWS), n=2, elem=1):
    left, right, dl, dr = ptrs
    left = left if img else None
    dl = dl if out else None
    step = COLS * (4 if "f32" in name else 1) - (1 if short else 0)
    R, cost = 1, _capi.COST_SSD
    pair_stride = ROWS * PITCH
    if name in ("stereo_disparity_f32_host", "stereo_disparity_u8_host"):
        return [ctx, cost, left, step, right, step, rows, COLS, R, dmin, dmax, dl, PITCH, elem, None, 0]
    if name in ("stereo_disparity_f32_device", "stereo_disparity_u8_device"):
        return [ctx, cost, left, step, right, step, rows, COLS, R, dmin, dmax, dl, PITCH, elem, None, 0, None]
    if name == "stereo_disparity_band_u8_device":
        return [ctx, cost, left, step, right, step, rows, COLS, 4, 12, R, dmin, dmax, dl, PITCH, elem, None]
    if name == "stereo_disparity_band_halo_u8_device":
        return [ctx, cost, left, step, right, step, rows, COLS, 4, 12, halo[0], halo[1], R, dmin, dmax, dl, PITCH, elem, None]
    if name == "stereo_disparity_refgpu_f32_host":
        return [ctx, cost, left, step, right, step, rows, COLS, R, dmin, dmax, dl, PITCH, None, 0]
    if name == "stereo_disparity_refgpu_f32_device":
        return [ctx, cost, left, step, right, step, rows, COLS, R, dmin, dmax, dl, PITCH, None, 0, None]
    if name in ("stereo_disparity_pair_f32_host", "stereo_disparity_pair_u8_host"):
        return [ctx, cost, left, step, right, step, rows, COLS, R, rng, dl, dr, PITCH, elem]
    if name in ("stereo_disparity_pair_f32_device", "stereo_disparity_pair_u8_device"):
        return [ctx, cost, left, step, right, step, rows, COLS, R, rng, dl, dr, PITCH, elem, None]
    if name == "stereo_disparity_pair_band_halo_u8_device":
        return [ctx, cost, left, step, right, step, rows, COLS, 4, 12, halo[0], halo[1], R, rng, dl, dr, PITCH, elem, None]
    if name in ("stereo_disparity_pair_band_u8_host", "stereo_disparity_pair_band_f32_host"):
        return [ctx, cost, left, step, right, step, rows, COLS, 4, 12, R, rng, dl, dr, PITCH, elem]
    if name.startswith("stereo_disparity_pair_batch_"):
        a = [ctx, cost, n, left, right, step, pair_stride, rows, COLS, R, rng, dl, dr, PITCH, pair_stride, elem]
        return a + [None] if name.endswith("_device") else a
    raise KeyError(name)


@pytest.mark.parametrize("name,case", [(n, c) for n, exp in EXPECTED.items() for c in exp])
def test_rejected_input_status(bufs, name, case):
    ctx, host, dev = bufs
    ptrs = dev if name.endswith("_device") else host
    rc = getattr(_capi.lib(), name)(*_args(name, ctx.handle, ptrs, **CASES[case]))
    assert rc == EXPECTED[name][case], f"{name} / {case}: {rc} ({_capi.last_error()})"


def test_valid_baseline_calls_succeed(bufs):
    """The argument set the table perturbs is itself accepted by every entry point (so each row tests one argument)."""
    ctx, host, dev = bufs
    for name in EXPECTED:
        ptrs = dev if name.endswith("_device") else host
        rc = getattr(_capi.lib(), name)(*_args(name, ctx.handle, ptrs))
        assert rc == _capi.STEREO_OK, f"{name}: {rc} ({_capi.last_error()})"
    assert _capi.lib().stereo_ctx_synchronize(ctx.handle, None) == 0
