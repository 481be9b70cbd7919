// Exact general path: float (or u8) images of any content, any window radius / disparity range.
// Per-element reference arithmetic, one thread per output pixel, no running sums — this is the
// semantic anchor of the library (bit-exact SSD incl. the reference's row-wrap reads, NCC in
// double arithmetic like OpenCV's normalisation) and the fallback for what the packed u8 kernels do not cover.
//   SSD : serial::disparitySSD   ProblemSets/ps2_cpp/lib/DisparitySSD.cpp:35-59
//   NCC : serial::disparityNCorr ProblemSets/ps2_cpp/lib/DisparityNCorr.cpp:44-69 (+ TM_CCORR_NORMED)
#pragma once
#include "common.cuh"
#include <cfloat>

namespace sb {


// cv::copyMakeBorder(..., BORDER_REPLICATE) (DisparitySSD.cpp:20-23) into a contiguous float image.
template <typename T>
__global__ void pad_replicate_kernel(const T* __restrict__ img, size_t step, int rows, int cols, int R,
                                     float* __restrict__ out, int Hp, int Wp, int ar0, int ar1) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= Wp || y >= Hp) return;
    const T* row = reinterpret_cast<const T*>(reinterpret_cast<const char*>(img) + size_t(clampi(clampi(y - R, 0, rows - 1), ar0, ar1 - 1)) * step);
    out[size_t(y) * Wp + x] = float(row[clampi(x - R, 0, cols - 1)]);
}

// One window element, DisparitySSD.cpp:49-51: float subtract, float multiply (never fused),
// round half away from zero, int accumulate.  For q >= 0: trunc(q + 0.5 rounded toward zero).
__device__ __forceinline__ int ssd_elem(float a, float b) {
    const float d = __fsub_rn(a, b);
    const float q = __fmul_rn(d, d);
    return __float2int_rz(__fadd_rz(q, 0.5f));
}

// Lp/Rp: padded images (origin pointers; Rp is followed/preceded by a zeroed guard so that the
// reference's out-of-row reads are reproduced: flat index, SURVEY.md §A.1).
__global__ void __launch_bounds__(128)
ssd_exact_kernel(const float* __restrict__ Lp, const float* __restrict__ Rp, int rows, int cols, int R,
                 int dmin, int dmax, int row_begin, int32_t* __restrict__ disp, int32_t* __restrict__ cost,
                 int x_begin, int x_count) {
    const int xi = blockIdx.x * blockDim.x + threadIdx.x;
    if (xi >= x_count) return;
    const int xu = x_begin + xi;
    const int yu = row_begin + blockIdx.y;
    const int Wp = cols + 2 * R;
    const int x = xu + R, y = yu + R;
    int s = max(0, x + dmin);
    const int smax = min(Wp - 1, x + dmax);
    int bestCost = 99999999, bestDisp = 0;
    for (; s <= smax; ++s) {
        int sum = 0;
        for (int wy = -R; wy <= R; ++wy) {
            const float* lrow = Lp + ptrdiff_t(y + wy) * Wp + x;
            const float* rrow = Rp + ptrdiff_t(y + wy) * Wp + s;
            for (int wx = -R; wx <= R; ++wx) sum += ssd_elem(__ldg(lrow + wx), __ldg(rrow + wx));
        }
        if (sum < bestCost) { bestCost = sum; bestDisp = s - x; }
    }
    const size_t o = size_t(blockIdx.y) * cols + xu;
    disp[o] = bestDisp;
    cost[o] = bestCost;
}

// TM_CCORR_NORMED's normalisation of one candidate (opencv/modules/imgproc/src/templmatch.cpp common_matchTemplate), in
// two halves: the target window's norm from its double energy wnd - 0 below the zero-energy threshold - and the float32
// score of the double numerator acc against t = ncc_target_norm(wnd) * sqrt(reference energy).
__device__ __forceinline__ double ncc_target_norm(double wnd) {
    const double diff2 = wnd > 0 ? wnd : 0;
    const double lim = fmin(0.5, 10 * double(FLT_EPSILON) * wnd);
    return diff2 <= lim ? 0 : sqrt(diff2);
}
__device__ __forceinline__ float ncc_normalise(double acc, double t) {
    double num = double(float(acc));
    if (fabs(num) < t) num /= t;
    else if (fabs(num) < t * 1.125) num = num > 0 ? 1 : -1;
    else num = 0;
    return float(num);
}

// NCC with TM_CCORR_NORMED's arithmetic (float32 numerator, double energies and normalisation,
// float32 result; opencv/modules/imgproc/src/templmatch.cpp common_matchTemplate).
__global__ void __launch_bounds__(128)
ncorr_exact_kernel(const float* __restrict__ Lp, const float* __restrict__ Rp, int rows, int cols, int R,
                   int dmin, int dmax, int row_begin, int32_t* __restrict__ disp, float* __restrict__ score) {
    const int xu = blockIdx.x * blockDim.x + threadIdx.x;
    if (xu >= cols) return;
    const int yu = row_begin + blockIdx.y;
    const int Wp = cols + 2 * R, w = 2 * R + 1;
    const int x = xu + R, y = yu + R;
    double t2 = 0;
    for (int wy = -R; wy <= R; ++wy) {
        const float* lrow = Lp + size_t(y + wy) * Wp + (x - R);
        for (int i = 0; i < w; ++i) { const double v = __ldg(lrow + i); t2 += v * v; }
    }
    const double templNorm = sqrt(t2);
    int startX = x + dmin - R; if (startX < 0) startX = 0;
    int endX = x + dmax + 1 + R; if (endX > Wp) endX = Wp;
    const int ncand = endX - startX - w + 1;
    float bestScore = 0.f; int bestI = -1;
    for (int i = 0; i < ncand; ++i) {
        const int e = startX + i;
        double acc = 0, wnd = 0;
        for (int wy = -R; wy <= R; ++wy) {
            const float* lrow = Lp + size_t(y + wy) * Wp + (x - R);
            const float* rrow = Rp + size_t(y + wy) * Wp + e;
            for (int k = 0; k < w; ++k) {
                const double a = __ldg(lrow + k), b = __ldg(rrow + k);
                acc += a * b;     // float x float products are exact in double: fma == mul+add
                wnd += b * b;
            }
        }
        const float sc = ncc_normalise(acc, ncc_target_norm(wnd) * templNorm);
        if (bestI < 0 || sc > bestScore) { bestScore = sc; bestI = i; }
    }
    const bool right_aligned = (dmin <= 0 && dmax <= 0);
    const size_t o = size_t(blockIdx.y) * cols + xu;
    disp[o] = bestI - (right_aligned ? ncand - 1 : 0);
    score[o] = bestScore;
}

// int32 disparity (+ optional 4-byte best map) -> caller's layout.  elem 1 reproduces the
// reference's `disparity.at<char>() = int` narrowing (DisparitySSD.cpp:59).
__global__ void store_output_kernel(const int32_t* __restrict__ disp, const uint32_t* __restrict__ best,
                                    int band_rows, int cols, void* out, size_t out_step, int elem,
                                    void* best_out, size_t best_step) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y;
    if (x >= cols || y >= band_rows) return;
    const int32_t d = disp[size_t(y) * cols + x];
    char* row = reinterpret_cast<char*>(out) + size_t(y) * out_step;
    if (elem == 1) reinterpret_cast<int8_t*>(row)[x] = int8_t(uint8_t(uint32_t(d) & 0xFFu));
    else if (elem == 2) reinterpret_cast<int16_t*>(row)[x] = int16_t(d);
    else reinterpret_cast<int32_t*>(row)[x] = d;
    if (best_out) {
        char* brow = reinterpret_cast<char*>(best_out) + size_t(y) * best_step;
        reinterpret_cast<uint32_t*>(brow)[x] = best[size_t(y) * cols + x];
    }
}

// Is a float image exactly 8-bit (integral, 0..255)?  Writes the u8 copy and ORs 1 into flag[0] if any pixel is not
// (2 as well if a pixel is not finite).  (convertTo(CV_32FC1) without scaling, main.cpp:87-88, produces such images;
// addNoise / *1.1f, main.cpp:140-153,191-193, do not.)
// Blocks that hold a non-8-bit pixel also fold their pixel range into flag[1] (largest -v) and flag[2] (largest v), in an
// order-preserving unsigned encoding whose zero is "nothing seen": together with [0, 255] for the clean blocks that bounds
// the value range of the image, which decides whether the float running-sum kernels apply (fast.cuh).
__device__ __forceinline__ unsigned f32_ordered(float f) {
    const unsigned b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
static inline float f32_from_ordered(unsigned u) {
    const unsigned b = (u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u;
    float f; memcpy(&f, &b, 4); return f;
}
// blockIdx.z selects the image: both images of a pair go through one launch.
__global__ void classify_convert_kernel(const float* __restrict__ img0, size_t step0, uint8_t* __restrict__ out0,
                                        const float* __restrict__ img1, size_t step1, uint8_t* __restrict__ out1,
                                        int rows, int cols, size_t out_step, int* flag) {
    const float* __restrict__ img = blockIdx.z ? img1 : img0;
    const size_t step = blockIdx.z ? step1 : step0;
    uint8_t* __restrict__ out = blockIdx.z ? out1 : out0;
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    bool bad = false, nonfinite = false;
    float v = 0.f;
    if (x < cols && y < rows) {
        v = reinterpret_cast<const float*>(reinterpret_cast<const char*>(img) + size_t(y) * step)[x];
        const float f = floorf(v);
        bad = !(v >= 0.f && v <= 255.f && f == v);
        nonfinite = !(fabsf(v) <= 3.0e38f);
        out[size_t(y) * out_step + x] = bad ? 0 : uint8_t(int(v));
    }
    if (__syncthreads_or(bad)) {
        __shared__ unsigned smax[2][8];
        // threads outside the image and non-finite pixels track nothing: the range is that of the block's finite pixels
        const bool track = x < cols && y < rows && !nonfinite;
        const unsigned hi = __reduce_max_sync(0xffffffffu, track ? f32_ordered(v) : 0u);
        const unsigned lo = __reduce_max_sync(0xffffffffu, track ? f32_ordered(-v) : 0u);
        const int tid = threadIdx.y * blockDim.x + threadIdx.x, warp = tid >> 5;
        if ((tid & 31) == 0) { smax[0][warp] = lo; smax[1][warp] = hi; }
        const int anynf = __syncthreads_or(nonfinite);
        if (tid == 0) {
            unsigned l = 0, h = 0;
            const int nwarps = (blockDim.x * blockDim.y + 31) >> 5;
            for (int i = 0; i < nwarps && i < 8; ++i) { l = max(l, smax[0][i]); h = max(h, smax[1][i]); }
            atomicOr(flag, anynf ? 3 : 1);
            atomicMax(reinterpret_cast<unsigned*>(flag) + 1, l);
            atomicMax(reinterpret_cast<unsigned*>(flag) + 2, h);
        }
    }
}

} // namespace sb
