// Sub-pixel disparity of the maps of a pair call (stereo_ctx_set_subpixel): StereoSGBM's parabola through the costs of the
// winner and its two neighbours, in 1/16-pixel fixed point, after every integer step (uniqueness, texture, check, filter).
//   out = 16 sentinel                                     where the map holds the sentinel,
//   out = 16 d + subpix_offset(V(d-1), V(d), V(d+1))     where d - 1 and d + 1 are both present,
//   out = 16 d                                            otherwise.
// SGM maps: the last sgm_path_kernel stores the offset of its winner as one signed byte per pixel (SgmOut::subpix) and
// subpix_apply_kernel applies it.  Block-matcher SSD maps: subpix_pad_kernel pads each image of the launch sequence once
// (the single-direction call's replicate padding and zero guards, so that its flat-index row-wrap reads are reproduced),
// then subpix_bm_kernel recomputes V(d - 1), V(d), V(d + 1) of each pixel's final d and writes the result in place.
#pragma once
#include "common.cuh"
#include "exact.cuh"
#include <type_traits>

namespace sb {

constexpr int SP_MAXMAPS = 32;     // maps of one launch (>= FMAXJOBS)
constexpr int SP_THREADS = 128;    // columns of one block
constexpr int SP_RUN = 16;         // rows one thread of subpix_bm_kernel walks down its column

// StereoSGBM's offset ("do subpixel quadratic interpolation", stereosgbm.cpp) in 64-bit with C division: in [-7, 8] when V(d)
// is the first minimum of the three.
__host__ __device__ __forceinline__ int subpix_offset(long long vm, long long v0, long long vp) {
    long long den = vm + vp - 2 * v0;
    if (den < 1) den = 1;
    return int(((vm - vp) * 16 + den) / (2 * den));
}

struct SpMap {
    void* disp; size_t step;       // the map, whole image, refined in place
    const float* Lp; const float* Rp;   // block matcher: the padded reference and target (first pixel; guards around)
    const int8_t* off;             // SGM: rows x cols offsets of the last path kernel
    int dmin, dmax;                // the direction's candidate range
};
struct SpParams { SpMap map[SP_MAXMAPS]; int rows, cols, R, sentinel; };

template <typename T>
__device__ __forceinline__ T* sp_row(const SpMap& m, int y) {
    return reinterpret_cast<T*>(static_cast<char*>(m.disp) + size_t(y) * m.step);
}

// SGM maps: one thread per pixel, blockIdx.z the map.
template <typename T>
__global__ void __launch_bounds__(SP_THREADS) subpix_apply_kernel(SpParams P) {
    const SpMap& m = P.map[blockIdx.z];
    const int x = blockIdx.x * SP_THREADS + threadIdx.x, y = blockIdx.y;
    if (x >= P.cols) return;
    T* row = sp_row<T>(m, y);
    const int d = row[x];
    row[x] = T(d == P.sentinel ? 16 * d : 16 * d + m.off[size_t(y) * P.cols + x]);
}

// One image of a pair, padded like pad_images (replicate border, R + 64 zero guard floats on both sides), for each image
// blockIdx.z of P.  The whole buffer - guards included - is written, so every image may serve as either direction's target.
struct SpImage { const void* src; size_t step; float* dst; };
struct SpPadParams { SpImage img[SP_MAXMAPS]; int rows, cols, R; };

template <typename Px>
__global__ void __launch_bounds__(256) subpix_pad_kernel(SpPadParams P) {
    const SpImage& im = P.img[blockIdx.z];
    const int Wp = P.cols + 2 * P.R;
    const long long guard = P.R + 64, n = (long long)(P.rows + 2 * P.R) * Wp;
    const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
    if (i >= n + 2 * guard) return;
    const long long f = i - guard;
    float v = 0.f;
    if (f >= 0 && f < n) {
        const int r = int(f / Wp), c = int(f - (long long)r * Wp);
        const Px* row = reinterpret_cast<const Px*>(static_cast<const char*>(im.src) + size_t(clampi(r - P.R, 0, P.rows - 1)) * im.step);
        v = float(row[clampi(c - P.R, 0, P.cols - 1)]);
    }
    im.dst[f] = v;
}

// Adds (add) or removes (!add) padded row r of the three window sums V(d - 1), V(d), V(d + 1) of the pixel whose
// window starts at padded column x: reference Lp[r][x + k], target Rp_flat[r Wp + x + d + k + delta], k in [0, 2R].
//   U8: 8-bit-valued images with R <= 7.  Every term (l - r)^2 <= 255^2 is exact in float32, and so is every partial sum:
//       V + one row <= 16 * 15 * 255^2 < 2^24.  One subtract and one fused multiply-add per term.
//   otherwise: exact.cuh's ssd_elem, summed in int32 with wrap-around as the single-direction call sums it.
template <bool U8>
struct SpAcc {
    using A = typename std::conditional<U8, float, unsigned>::type;
    A m = 0, z = 0, p = 0;
    __device__ __forceinline__ void row(const float* lrow, const float* rrow, int w, bool add) {
        float rprev = __ldg(rrow - 1), rcur = __ldg(rrow);
        for (int k = 0; k < w; ++k) {
            const float rnext = __ldg(rrow + k + 1), l = __ldg(lrow + k);
            if (U8) {
                const float a = __fsub_rn(l, rprev), b = __fsub_rn(l, rcur), c = __fsub_rn(l, rnext);
                if (add) { m = __fmaf_rn(a, a, m); z = __fmaf_rn(b, b, z); p = __fmaf_rn(c, c, p); }
                else { m = __fmaf_rn(-a, a, m); z = __fmaf_rn(-b, b, z); p = __fmaf_rn(-c, c, p); }
            } else {
                const unsigned a = unsigned(ssd_elem(l, rprev)), b = unsigned(ssd_elem(l, rcur)), c = unsigned(ssd_elem(l, rnext));
                if (add) { m += a; z += b; p += c; }
                else { m -= a; z -= b; p -= c; }
            }
            rprev = rcur;
            rcur = rnext;
        }
    }
    __device__ __forceinline__ long long v(A a) const { return U8 ? (long long)a : (long long)int(a); }
};

// Block-matcher SSD maps: thread (x, y0) refines rows [y0, y0 + SP_RUN) of column x of map blockIdx.z.  Consecutive rows with
// the same d slide the three window sums down by one row (add the row entering the window, remove the one leaving it);
// any other pixel sums its windows afresh.
template <typename T, bool U8>
__global__ void __launch_bounds__(SP_THREADS) subpix_bm_kernel(SpParams P) {
    const SpMap& m = P.map[blockIdx.z];
    const int x = blockIdx.x * SP_THREADS + threadIdx.x;
    if (x >= P.cols) return;
    const int R = P.R, w = 2 * R + 1, Wp = P.cols + 2 * R;
    const int y0 = blockIdx.y * SP_RUN, y1 = min(P.rows, y0 + SP_RUN);
    SpAcc<U8> acc;
    bool have = false;              // acc holds the window sums of (y - 1, x) for candidate dprev
    int dprev = 0;
    for (int y = y0; y < y1; ++y) {
        T* row = sp_row<T>(m, y);
        const int d = row[x];
        const int s = x + R + d;    // padded target column of the window centre
        if (d == P.sentinel || d - 1 < m.dmin || d + 1 > m.dmax || s - 1 < 0 || s + 1 > Wp - 1) {
            row[x] = T(16 * d);     // (the sentinel, a range edge or an absent neighbour)
            have = false;
            continue;
        }
        const float* L = m.Lp + x;
        const float* Rt = m.Rp + (x + d);
        if (have && d == dprev) {
            acc.row(L + ptrdiff_t(y + w - 1) * Wp, Rt + ptrdiff_t(y + w - 1) * Wp, w, true);
            acc.row(L + ptrdiff_t(y - 1) * Wp, Rt + ptrdiff_t(y - 1) * Wp, w, false);
        } else {
            acc = SpAcc<U8>();
            for (int wy = 0; wy < w; ++wy) acc.row(L + ptrdiff_t(y + wy) * Wp, Rt + ptrdiff_t(y + wy) * Wp, w, true);
        }
        have = true;
        dprev = d;
        row[x] = T(16 * d + subpix_offset(acc.v(acc.m), acc.v(acc.z), acc.v(acc.p)));
    }
}

static inline int subpix_apply_launch(const SpParams& P, int n, int elem, cudaStream_t st) {
    const dim3 g(div_round_up(P.cols, SP_THREADS), P.rows, n);
    if (elem == 2) subpix_apply_kernel<int16_t><<<g, SP_THREADS, 0, st>>>(P);
    else subpix_apply_kernel<int32_t><<<g, SP_THREADS, 0, st>>>(P);
    return cudaGetLastError() == cudaSuccess ? STEREO_OK : STEREO_ERR_CUDA;
}

// Pads the n_img images of Q, then refines the n maps of P from them.  u8: the images are 8-bit (and R <= 7 for the float form).
static inline int subpix_bm_launch(const SpPadParams& Q, int n_img, const SpParams& P, int n, int elem, bool u8, cudaStream_t st) {
    const long long total = (long long)(Q.rows + 2 * Q.R) * (Q.cols + 2 * Q.R) + 2 * (Q.R + 64);
    const dim3 pg(div_round_up(total, 256), 1, n_img);
    if (u8) subpix_pad_kernel<uint8_t><<<pg, 256, 0, st>>>(Q);
    else subpix_pad_kernel<float><<<pg, 256, 0, st>>>(Q);
    const bool fma_form = u8 && P.R <= 7;
    const dim3 g(div_round_up(P.cols, SP_THREADS), div_round_up(P.rows, SP_RUN), n);
    if (elem == 2) {
        if (fma_form) subpix_bm_kernel<int16_t, true><<<g, SP_THREADS, 0, st>>>(P);
        else subpix_bm_kernel<int16_t, false><<<g, SP_THREADS, 0, st>>>(P);
    } else {
        if (fma_form) subpix_bm_kernel<int32_t, true><<<g, SP_THREADS, 0, st>>>(P);
        else subpix_bm_kernel<int32_t, false><<<g, SP_THREADS, 0, st>>>(P);
    }
    return cudaGetLastError() == cudaSuccess ? STEREO_OK : STEREO_ERR_CUDA;
}

} // namespace sb
