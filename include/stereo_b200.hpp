// stereo_b200.hpp — C++ drop-in for the reference's ps2 disparity entry points, on top of the C ABI.
//
// Reproduces, signature for signature, what ProblemSets/ps2_cpp/include/DisparitySSD.h:18-23 and
// include/DisparityNCorr.h:19-24 declare in namespace cuda:: —
//
//     void cuda::disparitySSD  (const Mat& left, const Mat& right, const size_t windowRad,
//                               const int minDisparity, const int maxDisparity, Mat& disparity);
//     void cuda::disparityNCorr(... same ...);
//
// `left` is the reference image, `right` the one searched (main.cpp:33,43).  Inputs must be CV_32FC1
// (the reference asserts it, DisparitySSD.cu:150) or CV_8UC1; the callee (re)allocates `disparity` as
// CV_8SC1 exactly like the reference (DisparitySSD.cu:160) and stores the reference's `char`-narrowed
// value.  sb::disparity*Wide return int16 for searches beyond 127 disparities.
//
// With OpenCV headers present the functions take cv::Mat; without them (this repo's build image has no
// OpenCV C++) they take sb::Mat, a minimal owning matrix with the same members the reference touches
// (rows, cols, step, data, type(), create()).  Header-only; link with -lstereo_b200.
//
// Error behaviour: the reference prints and exit(-1)s on any CUDA error (common/CudaCommon.cuh:11-22).
// Here a failure throws sb::Error carrying the stereo_status and stereo_last_error() text; define
// STEREO_B200_EXIT_ON_ERROR to get the reference's print-and-exit instead.
#ifndef STEREO_B200_HPP_
#define STEREO_B200_HPP_

#include "stereo_b200.h"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>

#if defined(__has_include)
#if __has_include(<opencv2/core.hpp>) && !defined(STEREO_B200_NO_OPENCV)
#include <opencv2/core.hpp>
#define STEREO_B200_HAVE_OPENCV 1
#endif
#endif

namespace sb {

struct Error : std::runtime_error {
    int status;
    Error(int st, const std::string& where)
        : std::runtime_error(where + ": " + stereo_status_string(st) + ": " + stereo_last_error()), status(st) {}
};

inline void check(int st, const char* where) {
    if (st == STEREO_OK) return;
#ifdef STEREO_B200_EXIT_ON_ERROR
    std::fprintf(stderr, "CUDA error at: %s\n%s %s\n", where, stereo_status_string(st), stereo_last_error());
    std::exit(-1);   // common/CudaCommon.cuh:13-21
#else
    throw Error(st, where);
#endif
}

// OpenCV's type codes for the three element types this path uses (opencv2/core/hal/interface.h).
enum : int { U8C1 = 0, S8C1 = 1, S16C1 = 3, F32C1 = 5 };

#ifndef STEREO_B200_HAVE_OPENCV
// Minimal stand-in for cv::Mat: owning, row-major, single channel.
class Mat {
public:
    int rows = 0, cols = 0;
    size_t step = 0;            // bytes per row
    unsigned char* data = nullptr;

    Mat() = default;
    Mat(int r, int c, int type) { create(r, c, type); }
    int type() const { return type_; }
    bool empty() const { return data == nullptr || rows == 0 || cols == 0; }
    size_t elemSize() const { return elem_size(type_); }
    void create(int r, int c, int type) {
        if (r == rows && c == cols && type == type_ && data) return;
        type_ = type; rows = r; cols = c; step = size_t(c) * elem_size(type);
        buf_.assign(size_t(r) * step, 0);
        data = buf_.data();
    }
    template <typename T> T& at(int r, int c) { return reinterpret_cast<T*>(data + size_t(r) * step)[c]; }
    template <typename T> const T& at(int r, int c) const { return reinterpret_cast<const T*>(data + size_t(r) * step)[c]; }
    template <typename T> T* ptr(int r) { return reinterpret_cast<T*>(data + size_t(r) * step); }
    template <typename T> const T* ptr(int r) const { return reinterpret_cast<const T*>(data + size_t(r) * step); }
    Mat(const Mat& o) { *this = o; }
    Mat& operator=(const Mat& o) {
        if (this != &o) { rows = o.rows; cols = o.cols; step = o.step; type_ = o.type_; buf_ = o.buf_; data = buf_.empty() ? nullptr : buf_.data(); }
        return *this;
    }
    static size_t elem_size(int type) { return type == F32C1 ? 4 : (type == S16C1 ? 2 : 1); }

private:
    int type_ = U8C1;
    std::vector<unsigned char> buf_;
};
using MatT = Mat;
#else
using MatT = cv::Mat;
#endif

// Process-wide context on device 0 (the reference has no notion of a device either); created on
// first use — this is also where common::warmup() (CudaWarmup.cu:14-19) is absorbed.
inline stereo_ctx* default_ctx() {
    static stereo_ctx* ctx = [] {
        stereo_ctx* c = nullptr;
        const char* dev = std::getenv("STEREO_B200_DEVICE");
        check(stereo_ctx_create(dev ? std::atoi(dev) : 0, &c), "stereo_ctx_create");
        return c;
    }();
    return ctx;
}

namespace detail {
inline void run(int cost, const MatT& left, const MatT& right, size_t windowRad, int minDisparity, int maxDisparity,
                MatT& disparity, int out_type, stereo_ctx* ctx) {
    if (left.rows != right.rows || left.cols != right.cols || left.type() != right.type())
        check(STEREO_ERR_INVALID_ARG, "disparity: left/right differ in size or type (main.cpp:27-28)");
    if (!ctx) ctx = default_ctx();
    disparity.create(left.rows, left.cols, out_type);          // DisparitySSD.cu:160
    const int elem = out_type == S16C1 ? 2 : 1;
    int st;
    if (left.type() == F32C1)
        st = stereo_disparity_f32_host(ctx, cost, reinterpret_cast<const float*>(left.data), left.step,
                                       reinterpret_cast<const float*>(right.data), right.step, left.rows, left.cols,
                                       int(windowRad), minDisparity, maxDisparity, disparity.data, disparity.step, elem,
                                       nullptr, 0);
    else if (left.type() == U8C1)
        st = stereo_disparity_u8_host(ctx, cost, left.data, left.step, right.data, right.step, left.rows, left.cols,
                                      int(windowRad), minDisparity, maxDisparity, disparity.data, disparity.step, elem,
                                      nullptr, 0);
    else
        st = STEREO_ERR_INVALID_ARG;                           // the reference: assert(type == CV_32FC1)
    check(st, cost == STEREO_COST_SSD ? "disparitySSD" : "disparityNCorr");
}
} // namespace detail

// Both maps of a pair in ONE call: what the reference's disparitySSDPair / disparityNCorrPair (src/main.cpp:21-78)
// do with two calls — left-referenced map over [-range, 0], then the images swapped and [0, +range].  SSD pairs come
// out of one cost volume where the library can fuse them (stereo_ctx_set_fuse_pairs); results are the two calls'.
inline void run_pair(int cost, const MatT& left, const MatT& right, size_t windowRad, int disparityRange,
                     MatT& disparityLeft, MatT& disparityRight, int out_type, stereo_ctx* ctx) {
    if (left.rows != right.rows || left.cols != right.cols || left.type() != right.type())
        check(STEREO_ERR_INVALID_ARG, "disparity pair: left/right differ in size or type (main.cpp:27-28)");
    if (!ctx) ctx = default_ctx();
    disparityLeft.create(left.rows, left.cols, out_type);
    disparityRight.create(left.rows, left.cols, out_type);
    const int elem = out_type == S16C1 ? 2 : 1;
    int st;
    if (left.type() == F32C1)
        st = stereo_disparity_pair_f32_host(ctx, cost, reinterpret_cast<const float*>(left.data), left.step,
                                            reinterpret_cast<const float*>(right.data), right.step, left.rows, left.cols,
                                            int(windowRad), disparityRange, disparityLeft.data, disparityRight.data,
                                            disparityLeft.step, elem);
    else if (left.type() == U8C1)
        st = stereo_disparity_pair_u8_host(ctx, cost, left.data, left.step, right.data, right.step, left.rows, left.cols,
                                           int(windowRad), disparityRange, disparityLeft.data, disparityRight.data,
                                           disparityLeft.step, elem);
    else
        st = STEREO_ERR_INVALID_ARG;
    check(st, cost == STEREO_COST_SSD ? "disparitySSDPair" : "disparityNCorrPair");
}
inline void disparitySSDPair(const MatT& l, const MatT& r, size_t rad, int range, MatT& dl, MatT& dr, bool wide = false, stereo_ctx* ctx = nullptr) {
    run_pair(STEREO_COST_SSD, l, r, rad, range, dl, dr, wide ? S16C1 : S8C1, ctx);
}
inline void disparityNCorrPair(const MatT& l, const MatT& r, size_t rad, int range, MatT& dl, MatT& dr, bool wide = false, stereo_ctx* ctx = nullptr) {
    run_pair(STEREO_COST_NCORR, l, r, rad, range, dl, dr, wide ? S16C1 : S8C1, ctx);
}

// int16 outputs for > 127 disparities (the reference's CV_8SC1 wraps, SURVEY.md §0.8)
inline void disparitySSDWide(const MatT& l, const MatT& r, size_t rad, int dmin, int dmax, MatT& d, stereo_ctx* ctx = nullptr) {
    detail::run(STEREO_COST_SSD, l, r, rad, dmin, dmax, d, S16C1, ctx);
}
inline void disparityNCorrWide(const MatT& l, const MatT& r, size_t rad, int dmin, int dmax, MatT& d, stereo_ctx* ctx = nullptr) {
    detail::run(STEREO_COST_NCORR, l, r, rad, dmin, dmax, d, S16C1, ctx);
}

// Left-right consistency check of the pair calls on `ctx` (default: the default context): maxDiff >= 0 switches it on,
// < 0 off (stereo_ctx_set_lr_check).
inline void setLrCheck(int maxDiff, stereo_ctx* ctx = nullptr) {
    check(stereo_ctx_set_lr_check(ctx ? ctx : default_ctx(), maxDiff), "stereo_ctx_set_lr_check");
}

// Speckle filter of the pair calls on `ctx` (default: the default context): maxSize > 0 switches it on, <= 0 off
// (stereo_ctx_set_speckle_filter).
inline void setSpeckleFilter(int maxSize, int maxDiff, stereo_ctx* ctx = nullptr) {
    check(stereo_ctx_set_speckle_filter(ctx ? ctx : default_ctx(), maxSize, maxDiff), "stereo_ctx_set_speckle_filter");
}

// Semi-global matching of the pair calls on `ctx` (default: the default context): paths 4 or 8 switch it on, 0 off
// (stereo_ctx_set_sgm).
inline void setSgm(int paths, int p1 = 0, int p2 = 0, stereo_ctx* ctx = nullptr) {
    check(stereo_ctx_set_sgm(ctx ? ctx : default_ctx(), paths, p1, p2), "stereo_ctx_set_sgm");
}

// Integer scale q (1 .. 2^24) of the NCC cost C = q - floor(fl32(q * score)) that lets SGM serve NCC pair calls; 0 (the
// default) refuses them (stereo_ctx_set_sgm_ncc_scale).
inline void setSgmNccScale(int q, stereo_ctx* ctx = nullptr) {
    check(stereo_ctx_set_sgm_ncc_scale(ctx ? ctx : default_ctx(), q), "stereo_ctx_set_sgm_ncc_scale");
}

// Uniqueness ratio (StereoSGBM's uniquenessRatio, 1 .. 99) of the pair calls on `ctx` (default: the default context); 0
// switches it off (stereo_ctx_set_uniqueness).
inline void setUniqueness(int uniquenessRatio, stereo_ctx* ctx = nullptr) {
    check(stereo_ctx_set_uniqueness(ctx ? ctx : default_ctx(), uniquenessRatio), "stereo_ctx_set_uniqueness");
}

// Sub-pixel disparity (StereoSGBM's 1/16-pixel fixed point) of the pair calls on `ctx` (default: the default context): true
// writes 16 d + offset, false switches it off (stereo_ctx_set_subpixel).
inline void setSubpixel(bool on, stereo_ctx* ctx = nullptr) {
    check(stereo_ctx_set_subpixel(ctx ? ctx : default_ctx(), on ? 1 : 0), "stereo_ctx_set_subpixel");
}

// StereoBM's X-Sobel prefilter (preFilterCap, 1 .. 63) and texture threshold (textureThreshold, >= 0) of the pair calls on
// `ctx` (default: the default context); cap 0 (with threshold 0) switches both off (stereo_ctx_set_prefilter).
inline void setPrefilter(int cap, int textureThreshold = 0, stereo_ctx* ctx = nullptr) {
    check(stereo_ctx_set_prefilter(ctx ? ctx : default_ctx(), cap, textureThreshold), "stereo_ctx_set_prefilter");
}

// Kernel time of the last call on the default context, the quantity the reference logs as
// "disparitySSDKernel execution took {} ms" (DisparitySSD.cu:203).
inline float lastKernelMs() { return stereo_ctx_last_kernel_ms(default_ctx()); }

} // namespace sb

// ---- the reference's names -------------------------------------------------------------------------
namespace cuda {
inline void disparitySSD(const sb::MatT& left, const sb::MatT& right, const size_t windowRad, const int minDisparity,
                         const int maxDisparity, sb::MatT& disparity) {
    sb::detail::run(STEREO_COST_SSD, left, right, windowRad, minDisparity, maxDisparity, disparity, sb::S8C1, nullptr);
}
inline void disparityNCorr(const sb::MatT& left, const sb::MatT& right, const size_t windowRad, const int minDisparity,
                           const int maxDisparity, sb::MatT& disparity) {
    sb::detail::run(STEREO_COST_NCORR, left, right, windowRad, minDisparity, maxDisparity, disparity, sb::S8C1, nullptr);
}
} // namespace cuda

// The reference's CPU twins (DisparitySSD.h:38-43, DisparityNCorr.h:39-44; selected by `use_gpu_disparity: false`,
// main.cpp:31-37).  Their results are this library's parity target, so the same GPU path serves both names.
namespace serial {
inline void disparitySSD(const sb::MatT& left, const sb::MatT& right, const size_t windowRad, const int minDisparity,
                         const int maxDisparity, sb::MatT& disparity) {
    cuda::disparitySSD(left, right, windowRad, minDisparity, maxDisparity, disparity);
}
inline void disparityNCorr(const sb::MatT& left, const sb::MatT& right, const size_t windowRad, const int minDisparity,
                           const int maxDisparity, sb::MatT& disparity) {
    cuda::disparityNCorr(left, right, windowRad, minDisparity, maxDisparity, disparity);
}
} // namespace serial

namespace sb {

// Several B200s in one process (stereo_mgpu_*): one pair in row bands with halo, batches by pair.
class MultiGpu {
public:
    explicit MultiGpu(const std::vector<int>& devices = {}) {
        check(stereo_mgpu_create(devices.empty() ? nullptr : devices.data(), int(devices.size()), &mg_), "stereo_mgpu_create");
    }
    ~MultiGpu() { stereo_mgpu_destroy(mg_); }
    MultiGpu(const MultiGpu&) = delete;
    MultiGpu& operator=(const MultiGpu&) = delete;
    int deviceCount() const { return stereo_mgpu_device_count(mg_); }
    stereo_mgpu* handle() { return mg_; }
    void setLrCheck(int maxDiff) { check(stereo_mgpu_set_lr_check(mg_, maxDiff), "stereo_mgpu_set_lr_check"); }
    void setSpeckleFilter(int maxSize, int maxDiff) {
        check(stereo_mgpu_set_speckle_filter(mg_, maxSize, maxDiff), "stereo_mgpu_set_speckle_filter");
    }
    void setSgm(int paths, int p1 = 0, int p2 = 0) { check(stereo_mgpu_set_sgm(mg_, paths, p1, p2), "stereo_mgpu_set_sgm"); }
    void setSgmNccScale(int q) { check(stereo_mgpu_set_sgm_ncc_scale(mg_, q), "stereo_mgpu_set_sgm_ncc_scale"); }
    void setUniqueness(int uniquenessRatio) {
        check(stereo_mgpu_set_uniqueness(mg_, uniquenessRatio), "stereo_mgpu_set_uniqueness");
    }
    void setPrefilter(int cap, int textureThreshold = 0) {
        check(stereo_mgpu_set_prefilter(mg_, cap, textureThreshold), "stereo_mgpu_set_prefilter");
    }
    void setSubpixel(bool on) { check(stereo_mgpu_set_subpixel(mg_, on ? 1 : 0), "stereo_mgpu_set_subpixel"); }

    // disparitySSDPair / disparityNCorrPair (main.cpp:21-78) with the output rows sharded over the devices
    void disparityPairBands(int cost, const MatT& left, const MatT& right, size_t windowRad, int disparityRange, MatT& disparityLeft,
                            MatT& disparityRight, bool wide = false) {
        if (left.rows != right.rows || left.cols != right.cols || left.type() != right.type())
            check(STEREO_ERR_INVALID_ARG, "disparity pair: left/right differ in size or type (main.cpp:27-28)");
        const int out_type = wide ? S16C1 : S8C1, elem = wide ? 2 : 1;
        disparityLeft.create(left.rows, left.cols, out_type);
        disparityRight.create(left.rows, left.cols, out_type);
        int st;
        if (left.type() == F32C1)
            st = stereo_mgpu_disparity_pair_bands_f32_host(mg_, cost, reinterpret_cast<const float*>(left.data), left.step,
                                                           reinterpret_cast<const float*>(right.data), right.step, left.rows, left.cols,
                                                           int(windowRad), disparityRange, disparityLeft.data, disparityRight.data,
                                                           disparityLeft.step, elem);
        else if (left.type() == U8C1)
            st = stereo_mgpu_disparity_pair_bands_u8_host(mg_, cost, left.data, left.step, right.data, right.step, left.rows, left.cols,
                                                          int(windowRad), disparityRange, disparityLeft.data, disparityRight.data,
                                                          disparityLeft.step, elem);
        else
            st = STEREO_ERR_INVALID_ARG;
        check(st, "MultiGpu::disparityPairBands");
    }

private:
    stereo_mgpu* mg_ = nullptr;
};

} // namespace sb

#endif // STEREO_B200_HPP_
