// Left-right consistency check of a pair's two maps (OpenCV's disp12MaxDiff filter), in place.
//   left pixel x, value dL:  consistent when xr = x + dL lies in [0, cols) and |dL + dR(xr)| <= max_diff
//   right pixel x, value dR: consistent when xl = x + dR lies in [0, cols) and |dR + dL(xl)| <= max_diff
// Both tests read the maps as they were before any pixel was invalidated; an inconsistent pixel gets `sentinel`
// (-(range + 1), below every valid disparity of either map), every other pixel keeps its value.
#pragma once
#include "common.cuh"

namespace sb {

constexpr int LR_MAXPAIRS = 16;
constexpr int LR_MAXCOLS = 32768;
constexpr int LR_BOTH_MAXCOLS = 20480;     // rows up to this width are staged together: 2 x 80 KB of int32
constexpr int LR_COLS_PER_THREAD = 32;     // wider rows: a thread's left-pixel verdicts are the bits of one register

struct LrMaps { void* left; void* right; size_t left_step, right_step; };     // each at its first row
struct LrParams {
    LrMaps pair[LR_MAXPAIRS];
    int cols, max_diff, sentinel;
};

// Branch-free: a partner outside the row reads the pixel's own column instead (always staged) and fails anyway.
__device__ __forceinline__ bool lr_consistent(int x, int d, const int32_t* partner_row, int cols, int max_diff) {
    const unsigned p = unsigned(x) + unsigned(d);          // >= cols exactly when x + d lies outside [0, cols)
    const bool inside = p < unsigned(cols);
    const long long s = (long long)d + partner_row[inside ? int(p) : x];
    return inside && (unsigned long long)(s + max_diff) <= 2ull * unsigned(max_diff);
}

// NR map rows into shared memory as int32.  Where every row start allows it, 16-byte loads, up to 4 per row and thread
// issued before any of them is stored (plain loads - the kernel writes these rows later, so not through the read-only
// path); element loads for the rest.
template <class T, int NR>
__device__ __forceinline__ void lr_stage(const T* const (&src)[NR], int32_t* const (&dst)[NR], int cols) {
    constexpr int V = 16 / sizeof(T), U = 4;
    bool vec = true;
    #pragma unroll
    for (int r = 0; r < NR; ++r) vec = vec && (reinterpret_cast<uintptr_t>(src[r]) & 15) == 0;
    int done = 0;
    if (vec) {
        const int nv = cols / V;
        for (int i0 = threadIdx.x; i0 < nv; i0 += U * blockDim.x) {
            int4 v[NR][U];
            #pragma unroll
            for (int u = 0; u < U; ++u)
                #pragma unroll
                for (int r = 0; r < NR; ++r)
                    if (i0 + u * int(blockDim.x) < nv) v[r][u] = reinterpret_cast<const int4*>(src[r])[i0 + u * blockDim.x];
            #pragma unroll
            for (int u = 0; u < U; ++u) {
                const int i = i0 + u * blockDim.x;
                if (i >= nv) break;
                #pragma unroll
                for (int r = 0; r < NR; ++r) {
                    const T* e = reinterpret_cast<const T*>(&v[r][u]);
                    #pragma unroll
                    for (int k = 0; k < V; k += 4)
                        *reinterpret_cast<int4*>(dst[r] + i * V + k) = make_int4(e[k], e[k + 1], e[k + 2], e[k + 3]);
                }
            }
        }
        done = nv * V;
    }
    for (int x = done + threadIdx.x; x < cols; x += blockDim.x)
        #pragma unroll
        for (int r = 0; r < NR; ++r) dst[r][x] = src[r][x];
}

// One CTA per (row, pair): grid (rows, pairs).  Rows are staged as int32 whatever the element type, so any int32 map is
// checked exactly.  Every global read of a row happens before the barrier that precedes the first write to it, which is
// what makes the check in place.
//   BOTH (cols <= LR_BOTH_MAXCOLS): stage both rows, then test every pixel of both and invalidate where it fails.
//   otherwise two int32 rows of up to 32768 pixels (256 KB) would not fit a CTA's shared memory, so they take turns in
//   one buffer (128 KB at most):
//     1. stage the right row; test every left pixel, keep its verdict in a register bit
//     2. stage the left row (nothing has been written yet); test every right pixel and invalidate it at once
//     3. invalidate the left pixels that failed in step 1
template <class T, bool BOTH>
__global__ void __launch_bounds__(BOTH ? 256 : 1024, BOTH ? 4 : 1) lr_check_kernel(const __grid_constant__ LrParams P) {
    extern __shared__ __align__(16) int32_t lr_rows[];
    const LrMaps& m = P.pair[blockIdx.y];
    T* L = reinterpret_cast<T*>(static_cast<char*>(m.left) + size_t(blockIdx.x) * m.left_step);
    T* R = reinterpret_cast<T*>(static_cast<char*>(m.right) + size_t(blockIdx.x) * m.right_step);
    const int cols = P.cols, bd = blockDim.x;
    if constexpr (BOTH) {
        int32_t* sl = lr_rows;
        int32_t* sr = lr_rows + ((cols + 3) & ~3);
        lr_stage<T, 2>({L, R}, {sl, sr}, cols);
        __syncthreads();
        // four columns a thread per round, strided by the block so that the partner reads of a warp stay conflict-free
        for (int x0 = threadIdx.x; x0 < cols; x0 += 4 * bd) {
            bool fl[4], fr[4];
            #pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int x = min(x0 + k * bd, cols - 1);
                fl[k] = !lr_consistent(x, sl[x], sr, cols, P.max_diff);
                fr[k] = !lr_consistent(x, sr[x], sl, cols, P.max_diff);
            }
            #pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int x = x0 + k * bd;
                if (x < cols && fl[k]) L[x] = T(P.sentinel);
                if (x < cols && fr[k]) R[x] = T(P.sentinel);
            }
        }
    } else {
        lr_stage<T, 1>({R}, {lr_rows}, cols);
        __syncthreads();
        uint32_t left_fail = 0;
        for (int x = threadIdx.x, k = 0; x < cols; x += bd, ++k)
            if (!lr_consistent(x, L[x], lr_rows, cols, P.max_diff)) left_fail |= 1u << k;
        __syncthreads();
        lr_stage<T, 1>({L}, {lr_rows}, cols);
        __syncthreads();
        for (int x = threadIdx.x; x < cols; x += bd)
            if (!lr_consistent(x, R[x], lr_rows, cols, P.max_diff)) R[x] = T(P.sentinel);
        for (int x = threadIdx.x, k = 0; x < cols; x += bd, ++k)
            if (left_fail >> k & 1u) L[x] = T(P.sentinel);
    }
}

template <class T>
static inline int lr_check_init_one() {
    SB_CUDA(cudaFuncSetAttribute(reinterpret_cast<const void*>(lr_check_kernel<T, true>), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 LR_BOTH_MAXCOLS * 8));
    SB_CUDA(cudaFuncSetAttribute(reinterpret_cast<const void*>(lr_check_kernel<T, false>), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 LR_MAXCOLS * 4));
    return STEREO_OK;
}

static inline int lr_check_init() {
    int rc = lr_check_init_one<int8_t>();
    if (rc == STEREO_OK) rc = lr_check_init_one<int16_t>();
    return rc == STEREO_OK ? lr_check_init_one<int32_t>() : rc;
}

template <class T>
static inline void lr_check_launch_t(const LrParams& P, dim3 grid, cudaStream_t st) {
    const bool both = P.cols <= LR_BOTH_MAXCOLS;
    // at least 256 threads where the row has that many pixels; the two-turn form at most LR_COLS_PER_THREAD columns a thread
    int bd = P.cols < 256 ? P.cols : 256;
    const int need = (P.cols + LR_COLS_PER_THREAD - 1) / LR_COLS_PER_THREAD;
    if (!both && need > bd) bd = need;
    bd = (bd + 31) & ~31;
    if (both) lr_check_kernel<T, true><<<grid, bd, size_t((P.cols + 3) & ~3) * 8, st>>>(P);
    else lr_check_kernel<T, false><<<grid, bd, size_t(P.cols) * 4, st>>>(P);
}

// Rows [0, rows) of the maps of `npairs` pairs whose elements are `elem` bytes.
static inline int lr_check_launch(const LrParams& P, int rows, int npairs, int elem, cudaStream_t st) {
    const dim3 grid(rows, npairs);
    if (elem == 1) lr_check_launch_t<int8_t>(P, grid, st);
    else if (elem == 2) lr_check_launch_t<int16_t>(P, grid, st);
    else lr_check_launch_t<int32_t>(P, grid, st);
    SB_CUDA(cudaGetLastError());
    return STEREO_OK;
}

} // namespace sb
