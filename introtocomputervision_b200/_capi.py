"""ctypes view of include/stereo_b200.h.  The library is required: if it is missing the import of any
compute entry point raises (there is no Python or CPU fallback)."""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import os

# STEREO_B200_LIB overrides the library file (kernel-variant experiments); the default is the in-tree build.
# STEREO_LIB_TAG=<tag> loads an experiment build (libstereo_b200_<tag>.so, see build.py)
_TAG = os.environ.get("STEREO_LIB_TAG", "")
LIB_PATH = Path(os.environ.get("STEREO_B200_LIB") or
                (Path(__file__).resolve().parent / ("libstereo_b200" + (f"_{_TAG}" if _TAG else "") + ".so")))

STEREO_OK = 0
ERR_INVALID_ARG, ERR_INVALID_RANGE, ERR_NO_DEVICE, ERR_CUDA, ERR_ALLOC, ERR_UNSUPPORTED = -1, -2, -3, -4, -5, -6
COST_SSD, COST_NCORR = 0, 1
PATH_NONE, PATH_EXACT_F32, PATH_FAST_U8, PATH_FAST_F32, PATH_REFGPU, PATH_SGM = 0, 1, 2, 3, 4, 5

_vp, _sz, _i = C.c_void_p, C.c_size_t, C.c_int

# name -> (restype, argtypes); mirrors include/stereo_b200.h one to one
_SINGLE_HOST = [_vp, _i, _vp, _sz, _vp, _sz, _i, _i, _i, _i, _i, _vp, _sz, _i, _vp, _sz]
_SINGLE_DEV = _SINGLE_HOST + [_vp]
_PAIR_HOST = [_vp, _i, _vp, _sz, _vp, _sz, _i, _i, _i, _i, _vp, _vp, _sz, _i]
SIGNATURES = {
    "stereo_abi_version": (_i, []),
    "stereo_last_error": (C.c_char_p, []),
    "stereo_status_string": (C.c_char_p, [_i]),
    "stereo_device_count": (_i, []),
    "stereo_ctx_create": (_i, [_i, C.POINTER(_vp)]),
    "stereo_ctx_destroy": (None, [_vp]),
    "stereo_ctx_last_path": (_i, [_vp]),
    "stereo_ctx_last_kernel_ms": (C.c_float, [_vp]),
    "stereo_ctx_last_launches": (_i, [_vp]),
    "stereo_ctx_last_hot_kernel_ms": (C.c_float, [_vp, C.POINTER(_i)]),
    "stereo_ctx_last_hot_jobs": (_i, [_vp]),
    "stereo_ctx_force_path": (_i, [_vp, _i]),
    "stereo_ctx_set_pipe_bands": (_i, [_vp, _i]),
    "stereo_host_pipeline_plan": (_i, [_i, _i, _i, _i, C.POINTER(_i), C.POINTER(_i)]),
    "stereo_host_pipeline_item_bands": (_i, [_i, _i, _i, _i, _i, C.POINTER(_i), _i]),
    "stereo_ctx_set_fuse_pairs": (_i, [_vp, _i]),
    "stereo_host_pool_selftest": (_i, [_i, _i]),
    "stereo_ctx_set_host_threads": (_i, [_vp, _i]),
    "stereo_ctx_host_threads": (_i, [_vp]),
    "stereo_launch_plan": (_i, [_i, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "stereo_host_pack_f32_u8": (_i, [_vp, _sz, _vp, _sz, _i, _i, _i, C.POINTER(_i)]),
    "stereo_ctx_last_fused_pairs": (_i, [_vp]),
    "stereo_ctx_set_lr_check": (_i, [_vp, _i]),
    "stereo_ctx_lr_check": (_i, [_vp]),
    "stereo_lr_check_device": (_i, [_vp, _vp, _vp, _sz, _i, _i, _i, _i, _i, _vp]),
    "stereo_mgpu_set_lr_check": (_i, [_vp, _i]),
    "stereo_ctx_set_speckle_filter": (_i, [_vp, _i, _i]),
    "stereo_ctx_speckle_filter": (_i, [_vp, C.POINTER(_i), C.POINTER(_i)]),
    "stereo_filter_speckles_device": (_i, [_vp, _vp, _sz, _i, _i, _i, _i, _i, _i, _vp]),
    "stereo_mgpu_set_speckle_filter": (_i, [_vp, _i, _i]),
    "stereo_ctx_set_sgm": (_i, [_vp, _i, _i, _i]),
    "stereo_ctx_sgm": (_i, [_vp, C.POINTER(_i), C.POINTER(_i), C.POINTER(_i)]),
    "stereo_mgpu_set_sgm": (_i, [_vp, _i, _i, _i]),
    "stereo_ctx_set_sgm_ncc_scale": (_i, [_vp, _i]),
    "stereo_ctx_sgm_ncc_scale": (_i, [_vp]),
    "stereo_mgpu_set_sgm_ncc_scale": (_i, [_vp, _i]),
    "stereo_ctx_set_uniqueness": (_i, [_vp, _i]),
    "stereo_ctx_uniqueness": (_i, [_vp]),
    "stereo_mgpu_set_uniqueness": (_i, [_vp, _i]),
    "stereo_ctx_set_prefilter": (_i, [_vp, _i, _i]),
    "stereo_ctx_prefilter": (_i, [_vp, C.POINTER(_i), C.POINTER(_i)]),
    "stereo_mgpu_set_prefilter": (_i, [_vp, _i, _i]),
    "stereo_ctx_set_subpixel": (_i, [_vp, _i]),
    "stereo_ctx_subpixel": (_i, [_vp]),
    "stereo_mgpu_set_subpixel": (_i, [_vp, _i]),
    "stereo_prefilter_u8_device": (_i, [_vp, _vp, _sz, _i, _i, _i, _vp, _sz, _vp]),
    "stereo_prefilter_f32_device": (_i, [_vp, _vp, _sz, _i, _i, _i, _vp, _sz, _vp]),
    "stereo_ctx_synchronize": (_i, [_vp, _vp]),
    "stereo_disparity_f32_host": (_i, _SINGLE_HOST),
    "stereo_disparity_u8_host": (_i, _SINGLE_HOST),
    "stereo_disparity_f32_device": (_i, _SINGLE_DEV),
    "stereo_disparity_u8_device": (_i, _SINGLE_DEV),
    "stereo_disparity_pair_f32_host": (_i, _PAIR_HOST),
    "stereo_disparity_pair_u8_host": (_i, _PAIR_HOST),
    "stereo_disparity_pair_u8_device": (_i, _PAIR_HOST + [_vp]),
    "stereo_disparity_pair_f32_device": (_i, _PAIR_HOST + [_vp]),
    "stereo_disparity_pair_batch_u8_device": (_i, [_vp, _i, _i, _vp, _vp, _sz, _sz, _i, _i, _i, _i, _vp, _vp, _sz, _sz, _i, _vp]),
    "stereo_disparity_pair_batch_u8_host": (_i, [_vp, _i, _i, _vp, _vp, _sz, _sz, _i, _i, _i, _i, _vp, _vp, _sz, _sz, _i]),
    "stereo_disparity_pair_batch_f32_host": (_i, [_vp, _i, _i, _vp, _vp, _sz, _sz, _i, _i, _i, _i, _vp, _vp, _sz, _sz, _i]),
    "stereo_disparity_band_halo_u8_device": (_i, [_vp, _i, _vp, _sz, _vp, _sz, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _sz, _i, _vp]),
    "stereo_disparity_pair_band_halo_u8_device": (_i, [_vp, _i, _vp, _sz, _vp, _sz, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _sz, _i, _vp]),
    "stereo_band_halo_rows": (_i, [_i, _i, _i, _i, C.POINTER(_i), C.POINTER(_i)]),
    "stereo_peer_buffer_create": (_i, [_vp, _sz, C.POINTER(_vp), _vp]),
    "stereo_peer_buffer_open": (_i, [_vp, _vp, C.POINTER(_vp)]),
    "stereo_peer_buffer_close": (_i, [_vp, _vp]),
    "stereo_peer_buffer_destroy": (_i, [_vp, _vp]),
    "stereo_peer_push": (_i, [_vp, C.POINTER(_vp), _i, _sz, _vp, _sz, _vp]),
    "stereo_peer_mark": (_i, [_vp, C.POINTER(_i)]),
    "stereo_peer_wait": (_i, [_vp, _i, _vp]),
    "stereo_dev_alloc": (_i, [_vp, _sz, C.POINTER(_vp)]),
    "stereo_dev_free": (_i, [_vp, _vp]),
    "stereo_dev_upload": (_i, [_vp, _vp, _sz, _vp, _sz, _sz, _i]),
    "stereo_dev_download": (_i, [_vp, _vp, _sz, _vp, _sz, _sz, _i]),
    "stereo_image_gray_f32_device": (_i, [_vp, _vp, _sz, _i, _i, _i, _i, _vp, _sz, _vp]),
    "stereo_image_scale_add_f32_device": (_i, [_vp, _vp, _sz, _vp, _sz, C.c_float, _i, _i, _vp, _sz, _vp]),
    "stereo_disparity_refgpu_f32_host": (_i, [_vp, _i, _vp, _sz, _vp, _sz, _i, _i, _i, _i, _i, _vp, _sz, _vp, _sz]),
    "stereo_disparity_refgpu_f32_device": (_i, [_vp, _i, _vp, _sz, _vp, _sz, _i, _i, _i, _i, _i, _vp, _sz, _vp, _sz, _vp]),
    "stereo_disparity_pair_band_u8_host": (_i, [_vp, _i, _vp, _sz, _vp, _sz, _i, _i, _i, _i, _i, _i, _vp, _vp, _sz, _i]),
    "stereo_disparity_pair_band_f32_host": (_i, [_vp, _i, _vp, _sz, _vp, _sz, _i, _i, _i, _i, _i, _i, _vp, _vp, _sz, _i]),
    "stereo_mgpu_create": (_i, [C.POINTER(_i), _i, C.POINTER(_vp)]),
    "stereo_mgpu_destroy": (None, [_vp]),
    "stereo_mgpu_device_count": (_i, [_vp]),
    "stereo_mgpu_ctx": (_vp, [_vp, _i]),
    "stereo_mgpu_disparity_pair_batch_u8_host": (_i, [_vp, _i, _i, _vp, _vp, _sz, _sz, _i, _i, _i, _i, _vp, _vp, _sz, _sz, _i]),
    "stereo_mgpu_disparity_pair_batch_f32_host": (_i, [_vp, _i, _i, _vp, _vp, _sz, _sz, _i, _i, _i, _i, _vp, _vp, _sz, _sz, _i]),
    "stereo_mgpu_disparity_pair_bands_u8_host": (_i, _PAIR_HOST),
    "stereo_mgpu_disparity_pair_bands_f32_host": (_i, _PAIR_HOST),
    "stereo_disparity_band_u8_device": (_i, [_vp, _i, _vp, _sz, _vp, _sz, _i, _i, _i, _i, _i, _i, _i, _vp, _sz, _i, _vp]),
}

class LaunchPlan(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("fused", "strip_px", "strips_per_warp", "groups", "tile_px", "tiles", "ctas", "schedule",
                                       "rows_per_item", "bands", "stages", "smem_bytes", "border_kernel")]


_lib = None


class StereoLibraryMissing(ImportError):
    pass


def lib() -> C.CDLL:
    """Load libstereo_b200.so (built in-tree by ``introtocomputervision_b200.build``)."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise StereoLibraryMissing(
                f"{LIB_PATH} is missing: build it with `python -m introtocomputervision_b200.build` "
                "(nvcc, sm_100a).  There is no CPU fallback.")
        handle = C.CDLL(str(LIB_PATH))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)   # AttributeError here = header/library mismatch
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def last_error() -> str:
    return lib().stereo_last_error().decode("utf-8", "replace")
