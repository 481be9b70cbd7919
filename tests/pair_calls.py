"""Calls of every pair entry point on small synthetic pairs, for the tests of the pair options (the left-right check, the
speckle filter, SGM, the uniqueness ratio, the prefilter): the same images and maps through each entry point's own
interface, calls on outputs that must stay untouched, and the contexts the tests share.  Needs a B200."""
import ctypes as C

import numpy as np
import pytest

import introtocomputervision_b200 as sb
from introtocomputervision_b200 import _capi, synth
from test_entry_points import EXPECTED, ROWS

FAMILIES = {            # images, window radius, output type
    "u8": ("u8", 3, np.int8),
    "f32_8bit": ("f32", 3, np.int16),
    "f32_noisy": ("noisy", 3, np.int16),
    "exact": ("u8", 8, np.int32),
}
ROWS_T, COLS_T, RANGE_T = 40, 150, 20

PAIR_ENTRY_POINTS = [n for n in EXPECTED if n.startswith("stereo_disparity_pair_")]
MGPU_ENTRY_POINTS = {"stereo_mgpu_disparity_pair_batch_u8_host": "stereo_disparity_pair_batch_u8_host",      # (called as)
                     "stereo_mgpu_disparity_pair_batch_f32_host": "stereo_disparity_pair_batch_f32_host",
                     "stereo_mgpu_disparity_pair_bands_u8_host": "stereo_disparity_pair_u8_host",
                     "stereo_mgpu_disparity_pair_bands_f32_host": "stereo_disparity_pair_f32_host"}


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


def _torch():
    import torch
    return torch


def _tdt(dt):
    t = _torch()
    return {1: t.int8, 2: t.int16, 4: t.int32}[np.dtype(dt).itemsize]


def _ok(rc, where=""):
    assert rc == _capi.STEREO_OK, f"{where}: {rc} ({_capi.last_error()})"


def _bands(rows):
    cut = [0, rows // 3 + 1, 2 * rows // 3, rows]
    return list(zip(cut[:-1], cut[1:]))


def _images(kind, n, seed):
    Ls, Rs = zip(*[synth.make_pair(ROWS_T, COLS_T, RANGE_T + 4, seed + i)[:2] for i in range(n)])
    Ls, Rs = np.stack(Ls), np.stack(Rs)
    if kind == "f32":
        return Ls.astype(np.float32), Rs.astype(np.float32)
    if kind == "noisy":
        return (np.stack([synth.noisy_variant(a, seed + 10 + i) for i, a in enumerate(Ls)]),
                np.stack([synth.noisy_variant(b, seed + 20 + i) for i, b in enumerate(Rs)]))
    return Ls, Rs


def _run(h, entry, cost, Ls, Rs, win, rng, dt, bands=None):
    """Both maps of every pair of Ls / Rs ((n, rows, cols)) from one entry point; h is a Context or, for mgpu_*, a MultiGpu.
    The band entry points are called once per row band [r0, r1) of `bands` (default: three bands of about a third)."""
    lib = _capi.lib()
    n, rows, cols = Ls.shape
    dt = np.dtype(dt)
    elem, f32 = dt.itemsize, Ls.dtype == np.float32
    bands = _bands(rows) if bands is None else bands
    if entry in ("batch_host", "mgpu_batch"):
        return h.disparity_pair_batch(cost, Ls, Rs, win, rng, dtype=dt)
    if entry == "batch_device":
        torch = _torch()
        tl, tr = torch.from_numpy(Ls).cuda(), torch.from_numpy(Rs).cuda()
        ol = torch.empty((n, rows, cols), dtype=_tdt(dt), device="cuda")
        orr = torch.empty_like(ol)
        _ok(lib.stereo_disparity_pair_batch_u8_device(h.handle, cost, n, tl.data_ptr(), tr.data_ptr(), cols, rows * cols, rows, cols,
                                                      win, rng, ol.data_ptr(), orr.data_ptr(), cols * elem, rows * cols * elem, elem,
                                                      C.c_void_p(torch.cuda.current_stream().cuda_stream)), entry)
        torch.cuda.synchronize()
        return ol.cpu().numpy(), orr.cpu().numpy()
    out_l, out_r = np.empty((n, rows, cols), dt), np.empty((n, rows, cols), dt)
    for i in range(n):
        L, R, dl, dr = Ls[i], Rs[i], out_l[i], out_r[i]
        if entry == "pair_host":
            dl[:], dr[:] = h.disparity_pair(cost, L, R, win, rng, dtype=dt)
        elif entry == "mgpu_bands":
            dl[:], dr[:] = h.disparity_pair_bands(cost, L, R, win, rng, dtype=dt)
        elif entry == "band_host":
            fn = lib.stereo_disparity_pair_band_f32_host if f32 else lib.stereo_disparity_pair_band_u8_host
            for r0, r1 in bands:
                _ok(fn(h.handle, cost, L.ctypes.data, L.strides[0], R.ctypes.data, R.strides[0], rows, cols, r0, r1, win, rng,
                       dl[r0:].ctypes.data, dr[r0:].ctypes.data, dl.strides[0], elem), entry)
        else:
            torch = _torch()
            st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
            tl, tr = torch.from_numpy(L).cuda(), torch.from_numpy(R).cuda()
            ol = torch.empty((rows, cols), dtype=_tdt(dt), device="cuda")
            orr = torch.empty_like(ol)
            step = cols * L.itemsize
            if entry == "pair_device":
                fn = lib.stereo_disparity_pair_f32_device if f32 else lib.stereo_disparity_pair_u8_device
                _ok(fn(h.handle, cost, tl.data_ptr(), step, tr.data_ptr(), step, rows, cols, win, rng, ol.data_ptr(), orr.data_ptr(),
                       cols * elem, elem, st), entry)
            else:
                assert entry == "band_halo_device"
                for r0, r1 in bands:
                    h0, h1 = C.c_int(), C.c_int()
                    _ok(lib.stereo_band_halo_rows(rows, r0, r1, win, C.byref(h0), C.byref(h1)))
                    _ok(lib.stereo_disparity_pair_band_halo_u8_device(
                        h.handle, cost, tl[h0.value].data_ptr(), step, tr[h0.value].data_ptr(), step, rows, cols, r0, r1, h0.value,
                        h1.value, win, rng, ol[r0].data_ptr(), orr[r0].data_ptr(), cols * elem, elem, st), entry)
            torch.cuda.synchronize()
            dl[:], dr[:] = ol.cpu().numpy(), orr.cpu().numpy()
    return out_l, out_r


def _set_fuse(h, fuse):
    if isinstance(h, sb.MultiGpu):
        for i in range(h.device_count):
            _ok(_capi.lib().stereo_ctx_set_fuse_pairs(_capi.lib().stereo_mgpu_ctx(h._h, i), int(fuse)))
    else:
        h.set_fuse_pairs(fuse)


def _device_batch(ctx, Ls, Rs, win, rng, elem):
    """Both maps of every pair of the u8 images Ls / Rs from one SSD stereo_disparity_pair_batch_u8_device call, as
    (2, n, rows, cols)."""
    torch = _torch()
    n, rows, cols = Ls.shape
    tl, tr = torch.from_numpy(Ls).cuda(), torch.from_numpy(Rs).cuda()
    out = torch.empty((2, n, rows, cols), dtype={1: torch.int8, 2: torch.int16}[elem], device="cuda")
    _ok(_capi.lib().stereo_disparity_pair_batch_u8_device(ctx.handle, sb.COST_SSD, n, tl.data_ptr(), tr.data_ptr(), cols, rows * cols,
                                                          rows, cols, win, rng, out[0].data_ptr(), out[1].data_ptr(), cols * elem,
                                                          rows * cols * elem, elem, C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    return out.cpu().numpy()


def _fill(dev, shape, value):
    a = np.full(shape, value, np.uint8)
    return _torch().from_numpy(a).cuda() if dev else a


def _untouched(h, entry, Ls, Rs, R, rng, cost=sb.COST_SSD, dt=np.int16):
    """Calls the entry point (pair_device, batch_device, pair_host, batch_host or mgpu_batch) on outputs filled with 0x3C;
    returns (status, outputs untouched)."""
    lib = _capi.lib()
    n, rows, cols = Ls.shape
    elem = np.dtype(dt).itemsize
    f32 = Ls.dtype == np.float32
    step = cols * Ls.itemsize
    if entry in ("pair_device", "batch_device"):
        torch = _torch()
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


def _whole_band_args(name, args):
    """test_entry_points._args of a band entry point, with the band [4, 12) widened to the whole image [0, ROWS)."""
    a = list(args)
    i = a.index(4)
    assert a[i + 1] == 12
    a[i], a[i + 1] = 0, ROWS
    if name == "stereo_disparity_pair_band_halo_u8_device":
        a[i + 2], a[i + 3] = 0, ROWS
    return a
