"""Single-process multi-GPU context (stereo_mgpu_*): pair-sharded batches and row-band sharded pairs through the C ABI,
against the oracle.  Uses two different B200s when the box has them, otherwise several contexts on device 0 - the sharding,
the halo slabs and the seams are the same either way."""
import numpy as np
import pytest

import oracle
import ncc_check as nc
import introtocomputervision_b200 as sb
from introtocomputervision_b200 import _capi, synth

pytestmark = pytest.mark.gpu


def _device_lists():
    n = _capi.lib().stereo_device_count()
    return [[0, 1 % max(n, 1)], [0, 0, 0], list(range(min(n, 8))) or [0]]


@pytest.mark.parametrize("which", [0, 1, 2])
def test_mgpu_row_bands_equal_the_oracle(which):
    devices = _device_lists()[which]
    L, Rt, _ = synth.make_pair(301, 700, 128, 5150)
    Lf, Rf = L.astype(np.float32), Rt.astype(np.float32)
    with sb.MultiGpu(devices) as mg:
        assert mg.device_count == len(devices)
        for R, rng in ((5, 127), (7, 95), (2, 200)):
            ref_l, ref_r = oracle.ssd_fast(Lf, Rf, R, -rng, 0), oracle.ssd_fast(Rf, Lf, R, 0, rng)
            for a, b in ((L, Rt), (Lf, Rf)):
                dl, dr = mg.disparity_pair_bands(sb.COST_SSD, a, b, R, rng, dtype=np.int16)
                bad = np.argwhere(dl != ref_l)
                assert bad.size == 0, f"L->R differs at {bad[:5].tolist()} (of {len(bad)}), devices {devices}, R {R}"
                assert np.array_equal(dr, ref_r), (devices, R, rng)
        dl, dr = mg.disparity_pair_bands(sb.COST_NCORR, L, Rt, 4, 63, dtype=np.int16)
        # packed kernels, fused or not per device context: "u8" (the per-strip tolerance) covers both
        nc.check_ncc_map(dl, Lf, Rf, 4, -63, 0, "u8", what="L->R")
        nc.check_ncc_map(dr, Rf, Lf, 4, 0, 63, "u8", what="R->L")
        # float images that are not 8-bit-valued: computed whole on the first device by the float kernels
        Ln, Rn = synth.noisy_variant(L, 1), synth.noisy_variant(Rt, 2)
        dl, dr = mg.disparity_pair_bands(sb.COST_SSD, Ln, Rn, 3, 40, dtype=np.int16)
        assert np.array_equal(dl, oracle.ssd_fast(Ln, Rn, 3, -40, 0)) and np.array_equal(dr, oracle.ssd_fast(Rn, Ln, 3, 0, 40))


@pytest.mark.parametrize("which", [0, 1])
def test_mgpu_pair_batches_equal_the_oracle(which):
    devices = _device_lists()[which]
    n = 7
    Ls, Rs = zip(*[synth.make_pair(40, 330, 64, 8100 + i)[:2] for i in range(n)])
    Ls, Rs = np.stack(Ls), np.stack(Rs)
    with sb.MultiGpu(devices) as mg:
        for kind in (np.uint8, np.float32):
            bl, br = mg.disparity_pair_batch(sb.COST_SSD, Ls.astype(kind), Rs.astype(kind), 4, 63, dtype=np.int8)
            for i in range(n):
                a, b = Ls[i].astype(np.float32), Rs[i].astype(np.float32)
                assert np.array_equal(bl[i], oracle.narrow_i8(oracle.ssd_fast(a, b, 4, -63, 0))), (devices, kind, i)
                assert np.array_equal(br[i], oracle.narrow_i8(oracle.ssd_fast(b, a, 4, 0, 63))), (devices, kind, i)
        # fewer pairs than devices: the empty shares are skipped
        bl, br = mg.disparity_pair_batch(sb.COST_SSD, Ls[:1], Rs[:1], 4, 63, dtype=np.int8)
        assert np.array_equal(bl[0], oracle.narrow_i8(oracle.ssd_fast(Ls[0].astype(np.float32), Rs[0].astype(np.float32), 4, -63, 0)))


def test_mgpu_errors():
    with pytest.raises(sb.StereoError):
        sb.MultiGpu([99])
    with sb.MultiGpu([0]) as mg:
        img = np.zeros((8, 8), np.uint8)
        with pytest.raises(sb.StereoError):
            mg.disparity_pair_bands(sb.COST_SSD, img, img, 1, -5)


def test_band_host_entry_point_equals_full_image(ctx):
    L, Rt, _ = synth.make_pair(97, 410, 64, 616)
    lib = _capi.lib()
    ref_l, ref_r = ctx.disparity_pair(sb.COST_SSD, L, Rt, 5, 127, dtype=np.int16)
    out_l, out_r = np.zeros_like(ref_l), np.zeros_like(ref_r)
    for r0, r1 in ((0, 31), (31, 32), (32, 97)):
        st = lib.stereo_disparity_pair_band_u8_host(ctx.handle, sb.COST_SSD, L.ctypes.data, L.strides[0], Rt.ctypes.data, Rt.strides[0],
                                                    97, 410, r0, r1, 5, 127, out_l[r0:].ctypes.data, out_r[r0:].ctypes.data, out_l.strides[0], 2)
        assert st == 0, _capi.last_error()
    assert np.array_equal(out_l, ref_l) and np.array_equal(out_r, ref_r)
