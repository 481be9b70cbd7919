"""Host-side mirror of the reference's ps2 disparity interface on top of the C ABI.

Reference surface reproduced (names, argument meaning, error behaviour):

* ``cuda::disparitySSD(left, right, windowRad, minDisparity, maxDisparity, disparity)``
  — ProblemSets/ps2_cpp/include/DisparitySSD.h:18-23
* ``cuda::disparityNCorr(...)`` — ProblemSets/ps2_cpp/include/DisparityNCorr.h:19-24
* ``disparitySSDPair`` / ``disparityNCorrPair`` — ProblemSets/ps2_cpp/src/main.cpp:21-48, 51-78
* ``Config::DisparitySSD{_windowRadius, _disparityRange}`` — ProblemSets/ps2_cpp/include/Config.h:40-46

Inputs are numpy arrays (the stand-in for ``cv::Mat``): float32 ``CV_32FC1`` like the reference
asserts (DisparitySSD.cu:150), or uint8.  The returned disparity is int8 (``CV_8SC1``) by default,
exactly like the reference; pass ``dtype=np.int16``/``np.int32`` for searches beyond 127.
All computation happens in libstereo_b200.so on a B200; nothing here computes on the CPU.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Tuple

import numpy as np

from . import _capi
from ._capi import COST_NCORR, COST_SSD


class StereoError(RuntimeError):
    def __init__(self, status: int, where: str):
        self.status = status
        msg = _capi.last_error()
        name = _capi.lib().stereo_status_string(status).decode()
        super().__init__(f"{where}: {name} ({status}): {msg}")


def _check(status: int, where: str) -> None:
    if status != _capi.STEREO_OK:
        raise StereoError(status, where)


@dataclass
class DisparityConfig:
    """``Config::DisparitySSD`` (include/Config.h:40-46): YAML keys ``window_radius``, ``disparity_range``."""
    window_radius: int
    disparity_range: int


_ELEM = {np.dtype(np.int8): 1, np.dtype(np.int16): 2, np.dtype(np.int32): 4}


class Context:
    """Owns the device-side state for one GPU (``stereo_ctx``)."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        _check(_capi.lib().stereo_ctx_create(int(device), C.byref(self._h)), "stereo_ctx_create")
        self.device = int(device)

    def close(self) -> None:
        if self._h:
            _capi.lib().stereo_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- introspection -------------------------------------------------------------------------
    @property
    def handle(self) -> C.c_void_p:
        return self._h

    @property
    def last_path(self) -> int:
        return int(_capi.lib().stereo_ctx_last_path(self._h))

    @property
    def last_kernel_ms(self) -> float:
        return float(_capi.lib().stereo_ctx_last_kernel_ms(self._h))

    @property
    def last_launches(self) -> int:
        return int(_capi.lib().stereo_ctx_last_launches(self._h))

    def last_hot_kernel_ms(self):
        """(milliseconds, launches measured) of the last call's hot kernels; (-1, 0) if none ran."""
        n = C.c_int(0)
        ms = float(_capi.lib().stereo_ctx_last_hot_kernel_ms(self._h, C.byref(n)))
        return ms, int(n.value)

    @property
    def last_hot_jobs(self) -> int:
        """Directions (one disparity map each) the measured hot launches of the last call covered."""
        return int(_capi.lib().stereo_ctx_last_hot_jobs(self._h))

    def force_path(self, path: int) -> None:
        _check(_capi.lib().stereo_ctx_force_path(self._h, int(path)), "stereo_ctx_force_path")

    def set_pipe_bands(self, bands: int) -> None:
        """Row bands per image pair in the pipelined host entry points (0 = automatic)."""
        _check(_capi.lib().stereo_ctx_set_pipe_bands(self._h, int(bands)), "stereo_ctx_set_pipe_bands")

    @property
    def last_fused_pairs(self) -> int:
        """Image pairs of the last call whose two maps came out of one cost volume."""
        return int(_capi.lib().stereo_ctx_last_fused_pairs(self._h))

    def set_fuse_pairs(self, on: bool) -> None:
        """Pair calls: both maps from one cost volume where possible (default on; results identical either way)."""
        _check(_capi.lib().stereo_ctx_set_fuse_pairs(self._h, int(bool(on))), "stereo_ctx_set_fuse_pairs")

    def set_lr_check(self, max_diff: Optional[int]) -> None:
        """Pair calls: left-right consistency check (``disp12MaxDiff``).  Pixels whose partner in the other map is outside
        the image or differs by more than ``max_diff`` get ``-(disparity_range + 1)`` in both maps.  ``None`` or a negative
        value switches it off (the default)."""
        v = -1 if max_diff is None or max_diff < 0 else int(max_diff)
        _check(_capi.lib().stereo_ctx_set_lr_check(self._h, v), "stereo_ctx_set_lr_check")

    @property
    def lr_check(self) -> Optional[int]:
        """The left-right check's ``max_diff``, or None when the check is off."""
        v = int(_capi.lib().stereo_ctx_lr_check(self._h))
        return None if v < 0 else v

    def set_speckle_filter(self, max_size: Optional[int], max_diff: int = 1) -> None:
        """Pair calls: speckle filter (``cv::filterSpeckles``), after the left-right check when both are on.  In each map,
        connected regions of at most ``max_size`` pixels whose 4-neighbours differ by at most ``max_diff`` get
        ``-(disparity_range + 1)``.  ``None`` or a value <= 0 switches it off (the default)."""
        v = 0 if max_size is None or max_size <= 0 else int(max_size)
        _check(_capi.lib().stereo_ctx_set_speckle_filter(self._h, v, int(max_diff)), "stereo_ctx_set_speckle_filter")

    @property
    def speckle_filter(self) -> Optional[Tuple[int, int]]:
        """``(max_size, max_diff)`` of the speckle filter, or None when it is off."""
        size, diff = C.c_int(), C.c_int()
        _check(_capi.lib().stereo_ctx_speckle_filter(self._h, C.byref(size), C.byref(diff)), "stereo_ctx_speckle_filter")
        return None if size.value <= 0 else (size.value, diff.value)

    def set_sgm(self, paths: Optional[int], p1: int = 0, p2: int = 0) -> None:
        """Pair calls: semi-global matching over ``paths`` (4 or 8) scanline directions with penalties
        ``0 <= p1 <= p2``, before the left-right check and the speckle filter.  ``None`` or 0 switches it off (the
        default).  NCC pair calls are served only while an NCC scale is set (:meth:`set_sgm_ncc_scale`)."""
        v = 0 if paths is None else int(paths)
        _check(_capi.lib().stereo_ctx_set_sgm(self._h, v, int(p1), int(p2)), "stereo_ctx_set_sgm")

    @property
    def sgm(self) -> Optional[Tuple[int, int, int]]:
        """``(paths, p1, p2)`` of semi-global matching, or None when it is off."""
        paths, p1, p2 = C.c_int(), C.c_int(), C.c_int()
        _check(_capi.lib().stereo_ctx_sgm(self._h, C.byref(paths), C.byref(p1), C.byref(p2)), "stereo_ctx_sgm")
        return None if paths.value <= 0 else (paths.value, p1.value, p2.value)

    def set_sgm_ncc_scale(self, q: int) -> None:
        """Integer scale ``q`` (1 .. 2**24) of the NCC matching cost for SGM; 0 (the default) makes SGM refuse NCC pair
        calls.  A candidate d is present at (y, x) when ``0 <= x + d <= cols - 1``; its cost is
        ``C = q - floor(float32(q * s))`` in [0, 2q], with s the candidate's float32 TM_CCORR_NORMED score in the
        reference's arithmetic.  Independent of :meth:`set_sgm`: switching SGM off keeps q, and q alone changes
        nothing.  ``paths * (2q + p2)`` must not exceed 2**31 - 1."""
        _check(_capi.lib().stereo_ctx_set_sgm_ncc_scale(self._h, int(q)), "stereo_ctx_set_sgm_ncc_scale")

    @property
    def sgm_ncc_scale(self) -> int:
        """The NCC cost scale q of SGM (0: NCC pair calls refused while SGM is on)."""
        return int(_capi.lib().stereo_ctx_sgm_ncc_scale(self._h))

    def set_uniqueness(self, ratio: Optional[int]) -> None:
        """Pair calls: StereoSGBM's uniqueness ratio u (1 .. 99), before the left-right check and the speckle filter.  In
        each map a pixel gets ``-(disparity_range + 1)`` when a present candidate more than one disparity away from the
        winner has ``V(d) * (100 - u) < V* * 100``, V the SGM sum or, with SGM off, the SSD window cost (NCC needs SGM).
        ``None`` or 0 switches it off (the default)."""
        v = 0 if ratio is None else int(ratio)
        _check(_capi.lib().stereo_ctx_set_uniqueness(self._h, v), "stereo_ctx_set_uniqueness")

    @property
    def uniqueness(self) -> int:
        """The uniqueness ratio of pair calls (0: off)."""
        return int(_capi.lib().stereo_ctx_uniqueness(self._h))

    def set_prefilter(self, cap: Optional[int], texture_threshold: int = 0) -> None:
        """Pair calls: StereoBM's X-Sobel prefilter with ``preFilterCap`` = ``cap`` (1 .. 63): both maps of a pair match
        the clipped horizontal Sobel responses of the images (8-bit, in [0, 2 cap]) instead of their intensities.
        ``texture_threshold`` > 0 adds StereoBM's ``textureThreshold``: a pixel whose window holds a sum of
        ``|P - cap|`` below it gets ``-(disparity_range + 1)``, before the left-right check and the speckle filter.
        ``None`` or 0 switches both off (the default)."""
        v = 0 if cap is None else int(cap)
        _check(_capi.lib().stereo_ctx_set_prefilter(self._h, v, int(texture_threshold)), "stereo_ctx_set_prefilter")

    @property
    def prefilter(self) -> Optional[Tuple[int, int]]:
        """``(cap, texture_threshold)`` of the prefilter, or None when it is off."""
        cap, tex = C.c_int(), C.c_int()
        _check(_capi.lib().stereo_ctx_prefilter(self._h, C.byref(cap), C.byref(tex)), "stereo_ctx_prefilter")
        return None if cap.value <= 0 else (cap.value, tex.value)

    def set_subpixel(self, on: Optional[bool]) -> None:
        """Pair calls: StereoSGBM's sub-pixel disparity, the last step after the speckle filter.  Every map then holds
        ``16 d + offset`` (1/16 pixel, the sentinel becomes ``16 * sentinel``), the offset from the parabola through the
        costs of d - 1, d and d + 1 (SGM sums or, with SGM off, SSD window costs; NCC needs SGM).  Needs 2-byte maps
        (range <= 2047) or 4-byte maps.  ``True`` switches it on, ``False`` or ``None`` off (the default)."""
        v = 0 if on is None else int(on)
        _check(_capi.lib().stereo_ctx_set_subpixel(self._h, v), "stereo_ctx_set_subpixel")

    @property
    def subpixel(self) -> bool:
        """Whether pair calls write sub-pixel maps."""
        return bool(_capi.lib().stereo_ctx_subpixel(self._h))

    def set_host_threads(self, threads: int) -> None:
        """Host threads that convert CV_32FC1 host images to u8 before the upload (0 = automatic, -1 = off)."""
        _check(_capi.lib().stereo_ctx_set_host_threads(self._h, int(threads)), "stereo_ctx_set_host_threads")

    @property
    def host_threads(self) -> int:
        return int(_capi.lib().stereo_ctx_host_threads(self._h))

    def synchronize(self, stream: int = 0) -> None:
        _check(_capi.lib().stereo_ctx_synchronize(self._h, C.c_void_p(stream)), "stereo_ctx_synchronize")

    # -- host-buffer entry points ----------------------------------------------------------------
    def disparity(self, cost: int, ref: np.ndarray, tgt: np.ndarray, window_rad: int, min_disp: int, max_disp: int,
                  dtype=np.int8, return_best: bool = False):
        ref, tgt, fn = _prep_pair(ref, tgt, "stereo_disparity_f32_host", "stereo_disparity_u8_host")
        rows, cols = ref.shape
        dt = np.dtype(dtype)
        disp = np.empty((rows, cols), dt)
        best = np.empty((rows, cols), np.int32 if cost == COST_SSD else np.float32) if return_best else None
        st = fn(self._h, int(cost), ref.ctypes.data, ref.strides[0], tgt.ctypes.data, tgt.strides[0], rows, cols,
                int(window_rad), int(min_disp), int(max_disp), disp.ctypes.data, disp.strides[0], _ELEM[dt],
                best.ctypes.data if return_best else None, best.strides[0] if return_best else 0)
        _check(st, fn.__name__)
        return (disp, best) if return_best else disp

    def disparity_refgpu(self, cost: int, ref: np.ndarray, tgt: np.ndarray, window_rad: int, min_disp: int, max_disp: int,
                         return_best: bool = False):
        """The function the reference's GPU kernels compute (``stereo_disparity_refgpu_f32_host``; SURVEY.md A.3): int8 map,
        -1 where no candidate passed the kernels' threshold."""
        ref, tgt = np.ascontiguousarray(ref, np.float32), np.ascontiguousarray(tgt, np.float32)
        if ref.ndim != 2 or ref.shape != tgt.shape:
            raise ValueError("left/right must be 2-D arrays of equal shape")
        rows, cols = ref.shape
        disp = np.empty((rows, cols), np.int8)
        best = np.empty((rows, cols), np.float32) if return_best else None
        st = _capi.lib().stereo_disparity_refgpu_f32_host(
            self._h, int(cost), ref.ctypes.data, ref.strides[0], tgt.ctypes.data, tgt.strides[0], rows, cols, int(window_rad),
            int(min_disp), int(max_disp), disp.ctypes.data, disp.strides[0], best.ctypes.data if return_best else None,
            best.strides[0] if return_best else 0)
        _check(st, "stereo_disparity_refgpu_f32_host")
        return (disp, best) if return_best else disp

    def disparity_pair(self, cost: int, left: np.ndarray, right: np.ndarray, window_rad: int, disparity_range: int,
                       dtype=np.int8) -> Tuple[np.ndarray, np.ndarray]:
        left, right, fn = _prep_pair(left, right, "stereo_disparity_pair_f32_host", "stereo_disparity_pair_u8_host")
        rows, cols = left.shape
        dt = np.dtype(dtype)
        dl = np.empty((rows, cols), dt)
        dr = np.empty((rows, cols), dt)
        st = fn(self._h, int(cost), left.ctypes.data, left.strides[0], right.ctypes.data, right.strides[0], rows, cols,
                int(window_rad), int(disparity_range), dl.ctypes.data, dr.ctypes.data, dl.strides[0], _ELEM[dt])
        _check(st, fn.__name__)
        return dl, dr

    def disparity_pair_batch(self, cost: int, left: np.ndarray, right: np.ndarray, window_rad: int,
                             disparity_range: int, dtype=np.int8) -> Tuple[np.ndarray, np.ndarray]:
        """left/right: arrays of shape (n_pairs, rows, cols), both uint8 or both float32 (CV_32FC1 images, the
        type the reference's entry points take): a batch of ``disparitySSDPair`` / ``disparityNCorrPair`` calls."""
        left, right = np.asarray(left), np.asarray(right)
        if left.dtype == np.float32 and right.dtype == np.float32:
            kind, name = np.float32, "stereo_disparity_pair_batch_f32_host"
        elif left.dtype == np.uint8 and right.dtype == np.uint8:
            kind, name = np.uint8, "stereo_disparity_pair_batch_u8_host"
        else:
            raise TypeError("batch images must both be float32 (CV_32FC1) or both uint8")
        left = np.ascontiguousarray(left, kind)
        right = np.ascontiguousarray(right, kind)
        if left.ndim != 3 or left.shape != right.shape:
            raise ValueError("batch inputs must be (n, rows, cols) arrays of equal shape")
        n, rows, cols = left.shape
        dt = np.dtype(dtype)
        dl = np.empty((n, rows, cols), dt)
        dr = np.empty((n, rows, cols), dt)
        st = getattr(_capi.lib(), name)(
            self._h, int(cost), n, left.ctypes.data, right.ctypes.data, left.strides[1], left.strides[0], rows, cols,
            int(window_rad), int(disparity_range), dl.ctypes.data, dr.ctypes.data, dl.strides[1], dl.strides[0], _ELEM[dt])
        _check(st, name)
        return dl, dr


def _prep_pair(a: np.ndarray, b: np.ndarray, f32_name: str, u8_name: str):
    a = np.asarray(a)
    b = np.asarray(b)
    if a.ndim != 2 or a.shape != b.shape:
        # the reference asserts equal sizes in its callers (main.cpp:28)
        raise ValueError("left/right must be 2-D arrays of equal shape")
    if a.dtype == np.uint8 and b.dtype == np.uint8:
        kind, name = np.uint8, u8_name
    elif a.dtype == np.float32 and b.dtype == np.float32:
        kind, name = np.float32, f32_name
    else:
        # the reference: assert(left.type() == CV_32FC1 && right.type() == CV_32FC1) (DisparitySSD.cu:150)
        raise TypeError("images must both be float32 (CV_32FC1) or both uint8")
    # cv::Mat layout only: unit column stride and a non-negative row step of at least one row (views such as
    # img[::-1] or img[:, ::2] are copied; a negative step would wrap in the C ABI's size_t)
    def _mat(v):
        ok = v.strides[1] == v.itemsize and v.strides[0] >= v.shape[1] * v.itemsize
        return v if ok else np.ascontiguousarray(v, kind)
    a, b = _mat(a), _mat(b)
    return a, b, getattr(_capi.lib(), name)


class MultiGpu:
    """Several B200s in one process (``stereo_mgpu_*``): batches sharded by pair, one pair by row bands; host arrays in,
    host arrays out.  ``devices=None``: every visible sm_100 device; an ordinal may repeat (several contexts on one GPU)."""

    def __init__(self, devices=None):
        self._h = C.c_void_p()
        if devices is None:
            st = _capi.lib().stereo_mgpu_create(None, 0, C.byref(self._h))
        else:
            arr = (C.c_int * len(devices))(*[int(d) for d in devices])
            st = _capi.lib().stereo_mgpu_create(arr, len(devices), C.byref(self._h))
        _check(st, "stereo_mgpu_create")

    @property
    def device_count(self) -> int:
        return int(_capi.lib().stereo_mgpu_device_count(self._h))

    def close(self) -> None:
        if self._h:
            _capi.lib().stereo_mgpu_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def set_lr_check(self, max_diff: Optional[int]) -> None:
        """:meth:`Context.set_lr_check` on every device's context."""
        v = -1 if max_diff is None or max_diff < 0 else int(max_diff)
        _check(_capi.lib().stereo_mgpu_set_lr_check(self._h, v), "stereo_mgpu_set_lr_check")

    def set_speckle_filter(self, max_size: Optional[int], max_diff: int = 1) -> None:
        """:meth:`Context.set_speckle_filter` on every device's context (row-band sharded pairs refuse while it is on)."""
        v = 0 if max_size is None or max_size <= 0 else int(max_size)
        _check(_capi.lib().stereo_mgpu_set_speckle_filter(self._h, v, int(max_diff)), "stereo_mgpu_set_speckle_filter")

    def set_sgm(self, paths: Optional[int], p1: int = 0, p2: int = 0) -> None:
        """:meth:`Context.set_sgm` on every device's context (row-band sharded pairs refuse while it is on)."""
        v = 0 if paths is None else int(paths)
        _check(_capi.lib().stereo_mgpu_set_sgm(self._h, v, int(p1), int(p2)), "stereo_mgpu_set_sgm")

    def set_sgm_ncc_scale(self, q: int) -> None:
        """:meth:`Context.set_sgm_ncc_scale` on every device's context: ``C = q - floor(float32(q * s))`` of the NCC
        score s, 0 refuses NCC pair calls while SGM is on."""
        _check(_capi.lib().stereo_mgpu_set_sgm_ncc_scale(self._h, int(q)), "stereo_mgpu_set_sgm_ncc_scale")

    def set_uniqueness(self, ratio: Optional[int]) -> None:
        """:meth:`Context.set_uniqueness` on every device's context (row-band sharded pairs refuse while it is on)."""
        v = 0 if ratio is None else int(ratio)
        _check(_capi.lib().stereo_mgpu_set_uniqueness(self._h, v), "stereo_mgpu_set_uniqueness")

    def set_prefilter(self, cap: Optional[int], texture_threshold: int = 0) -> None:
        """:meth:`Context.set_prefilter` on every device's context (row-band sharded pairs refuse while it is on)."""
        v = 0 if cap is None else int(cap)
        _check(_capi.lib().stereo_mgpu_set_prefilter(self._h, v, int(texture_threshold)), "stereo_mgpu_set_prefilter")

    def set_subpixel(self, on: Optional[bool]) -> None:
        """:meth:`Context.set_subpixel` on every device's context (row-band sharded pairs refuse while it is on)."""
        v = 0 if on is None else int(on)
        _check(_capi.lib().stereo_mgpu_set_subpixel(self._h, v), "stereo_mgpu_set_subpixel")

    def disparity_pair_bands(self, cost: int, left: np.ndarray, right: np.ndarray, window_rad: int, disparity_range: int,
                             dtype=np.int8) -> Tuple[np.ndarray, np.ndarray]:
        left, right, fn = _prep_pair(left, right, "stereo_mgpu_disparity_pair_bands_f32_host", "stereo_mgpu_disparity_pair_bands_u8_host")
        rows, cols = left.shape
        dt = np.dtype(dtype)
        dl, dr = np.empty((rows, cols), dt), np.empty((rows, cols), dt)
        st = fn(self._h, int(cost), left.ctypes.data, left.strides[0], right.ctypes.data, right.strides[0], rows, cols,
                int(window_rad), int(disparity_range), dl.ctypes.data, dr.ctypes.data, dl.strides[0], _ELEM[dt])
        _check(st, fn.__name__)
        return dl, dr

    def disparity_pair_batch(self, cost: int, left: np.ndarray, right: np.ndarray, window_rad: int, disparity_range: int,
                             dtype=np.int8) -> Tuple[np.ndarray, np.ndarray]:
        left, right = np.asarray(left), np.asarray(right)
        if left.dtype == np.float32 and right.dtype == np.float32:
            kind, name = np.float32, "stereo_mgpu_disparity_pair_batch_f32_host"
        elif left.dtype == np.uint8 and right.dtype == np.uint8:
            kind, name = np.uint8, "stereo_mgpu_disparity_pair_batch_u8_host"
        else:
            raise TypeError("batch images must both be float32 (CV_32FC1) or both uint8")
        left, right = np.ascontiguousarray(left, kind), np.ascontiguousarray(right, kind)
        if left.ndim != 3 or left.shape != right.shape:
            raise ValueError("batch inputs must be (n, rows, cols) arrays of equal shape")
        n, rows, cols = left.shape
        dt = np.dtype(dtype)
        dl, dr = np.empty((n, rows, cols), dt), np.empty((n, rows, cols), dt)
        st = getattr(_capi.lib(), name)(
            self._h, int(cost), n, left.ctypes.data, right.ctypes.data, left.strides[1], left.strides[0], rows, cols,
            int(window_rad), int(disparity_range), dl.ctypes.data, dr.ctypes.data, dl.strides[1], dl.strides[0], _ELEM[dt])
        _check(st, name)
        return dl, dr


_default: Optional[Context] = None


def default_context() -> Context:
    global _default
    if _default is None:
        _default = Context(0)
    return _default


# ---- the reference's four free functions ------------------------------------------------------------

def disparitySSD(left, right, windowRad: int, minDisparity: int, maxDisparity: int, dtype=np.int8,
                 ctx: Optional[Context] = None) -> np.ndarray:
    """``cuda::disparitySSD`` (DisparitySSD.h:18-23).  ``left`` is the reference image."""
    return (ctx or default_context()).disparity(COST_SSD, left, right, windowRad, minDisparity, maxDisparity, dtype)


def disparityNCorr(left, right, windowRad: int, minDisparity: int, maxDisparity: int, dtype=np.int8,
                   ctx: Optional[Context] = None) -> np.ndarray:
    """``cuda::disparityNCorr`` (DisparityNCorr.h:19-24)."""
    return (ctx or default_context()).disparity(COST_NCORR, left, right, windowRad, minDisparity, maxDisparity, dtype)


def disparitySSDPair(left, right, config: DisparityConfig, dtype=np.int8, ctx: Optional[Context] = None):
    """``disparitySSDPair`` (main.cpp:21-48): (left-referenced map, right-referenced map)."""
    return (ctx or default_context()).disparity_pair(COST_SSD, left, right, config.window_radius,
                                                     config.disparity_range, dtype)


def disparityNCorrPair(left, right, config: DisparityConfig, dtype=np.int8, ctx: Optional[Context] = None):
    """``disparityNCorrPair`` (main.cpp:51-78)."""
    return (ctx or default_context()).disparity_pair(COST_NCORR, left, right, config.window_radius,
                                                     config.disparity_range, dtype)
