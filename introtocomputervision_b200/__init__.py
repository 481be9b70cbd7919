"""B200-native (sm_100a) dense stereo block matcher — the Problem Set 2 hot path of
tanmaniac/IntroToComputerVision behind the reference's own entry points.

The compute lives in ``libstereo_b200.so`` (hand-written CUDA behind the C ABI declared in
``include/stereo_b200.h``); this package is the thin host-side mirror used by tests and the bench.
"""
from ._capi import (COST_NCORR, COST_SSD, PATH_EXACT_F32, PATH_FAST_F32, PATH_FAST_U8, PATH_NONE, PATH_REFGPU,  # noqa: F401
                    PATH_SGM,
                    StereoLibraryMissing)
from .stereo import (Context, DisparityConfig, MultiGpu, StereoError, default_context, disparityNCorr,  # noqa: F401
                     disparityNCorrPair, disparitySSD, disparitySSDPair)

__all__ = [
    "COST_SSD", "COST_NCORR", "PATH_NONE", "PATH_EXACT_F32", "PATH_FAST_U8", "PATH_FAST_F32", "PATH_REFGPU", "PATH_SGM", "Context", "MultiGpu", "DisparityConfig",
    "StereoError", "StereoLibraryMissing", "default_context", "disparitySSD", "disparityNCorr",
    "disparitySSDPair", "disparityNCorrPair",
]
