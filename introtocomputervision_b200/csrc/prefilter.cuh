// StereoBM's X-Sobel prefilter (OpenCV prefilterXSobel, modules/calib3d/src/stereobm.cpp) and its texture threshold.
//   P = pf(I, cap): columns 0 and cols - 1, and the whole last row when rows is odd, get cap; every other pixel
//     v = (I[a][x+1] - I[a][x-1]) + 2 (I[y][x+1] - I[y][x-1]) + (I[b][x+1] - I[b][x-1]),  a = y - 1, b = y + 1 reflected
//     101-style (-1 -> 1, rows -> rows - 2), and P = min(max(v, -cap), cap) + cap.  Float images: each difference and sum
//     rounded to float32 in that order, v rounded half to even, P = cap where v is NaN.
//   texture: a map pixel gets `sentinel` when the sum of |P - cap| over its (2R + 1)^2 window (coordinates clamped to the
//     image, the matcher's replicate padding) is below the threshold.
#pragma once
#include "common.cuh"

namespace sb {

constexpr int PF_MAXIMGS = 32;       // two images per pair of a launch sequence (FMAXJOBS directions)
constexpr int PF_X = 16;             // output bytes per thread: one 16-byte store
constexpr int PF_THREADS = 128;

struct PfImage { const void* src; uint8_t* dst; size_t src_step, dst_step; };
struct PfParams {
    PfImage img[PF_MAXIMGS];
    int rows, cols, cap;
};

// PF_X + 2 consecutive elements of one row starting at column x0 - 1; columns outside the row read a clamped column
// (only border outputs, which become cap, and outputs past cols, which are not stored, read those).
template <class T>
__device__ __forceinline__ void pf_load_row(const T* __restrict__ row, int x0, int cols, T (&v)[PF_X + 2]) {
    constexpr int V = 16 / sizeof(T);
    if (x0 + PF_X <= cols && (reinterpret_cast<uintptr_t>(row + x0) & 15) == 0) {
        #pragma unroll
        for (int i = 0; i < PF_X / V; ++i) {
            const uint4 q = __ldg(reinterpret_cast<const uint4*>(row + x0) + i);
            const T* e = reinterpret_cast<const T*>(&q);
            #pragma unroll
            for (int k = 0; k < V; ++k) v[1 + i * V + k] = e[k];
        }
    } else {
        #pragma unroll
        for (int k = 0; k < PF_X; ++k) v[1 + k] = __ldg(row + min(x0 + k, cols - 1));
    }
    v[0] = __ldg(row + max(x0 - 1, 0));
    v[PF_X + 1] = __ldg(row + min(x0 + PF_X, cols - 1));
}

__device__ __forceinline__ int pf_clip(int d0, int d1, int d2, int cap) { return min(max(d0 + 2 * d1 + d2, -cap), cap) + cap; }

__device__ __forceinline__ int pf_clip(float d0, float d1, float d2, int cap) {
    const float v = __fadd_rn(__fadd_rn(d0, __fmul_rn(2.f, d1)), d2);
    const float c = float(cap);
    return v != v ? cap : cap + int(fminf(fmaxf(rintf(v), -c), c));
}

__device__ __forceinline__ int pf_diff(uint8_t a, uint8_t b) { return int(a) - int(b); }
__device__ __forceinline__ float pf_diff(float a, float b) { return __fsub_rn(a, b); }

// One launch over every image of a call: grid (ceil(cols / (PF_THREADS PF_X)), rows, images).  A thread writes PF_X
// consecutive bytes of one output row (one 16-byte store where the row allows it; bytes past cols are never written).
template <class T>
__global__ void __launch_bounds__(PF_THREADS) prefilter_kernel(const __grid_constant__ PfParams P) {
    const PfImage& im = P.img[blockIdx.z];
    const int y = blockIdx.y, rows = P.rows, cols = P.cols, cap = P.cap;
    const int x0 = (blockIdx.x * PF_THREADS + threadIdx.x) * PF_X;
    if (x0 >= cols) return;
    alignas(16) uint8_t out[PF_X];
    if ((rows & 1) && y == rows - 1) {           // OpenCV filters rows in pairs: an odd last row (rows == 1 too) is cap
        #pragma unroll
        for (int k = 0; k < PF_X; ++k) out[k] = uint8_t(cap);
    } else {
        const int ya = y > 0 ? y - 1 : 1, yb = y < rows - 1 ? y + 1 : rows - 2;      // (rows >= 2 here)
        const char* base = static_cast<const char*>(im.src);
        T a[PF_X + 2], c[PF_X + 2], b[PF_X + 2];
        pf_load_row(reinterpret_cast<const T*>(base + size_t(ya) * im.src_step), x0, cols, a);
        pf_load_row(reinterpret_cast<const T*>(base + size_t(y) * im.src_step), x0, cols, c);
        pf_load_row(reinterpret_cast<const T*>(base + size_t(yb) * im.src_step), x0, cols, b);
        #pragma unroll
        for (int k = 0; k < PF_X; ++k) {
            const int x = x0 + k;
            const int v = pf_clip(pf_diff(a[k + 2], a[k]), pf_diff(c[k + 2], c[k]), pf_diff(b[k + 2], b[k]), cap);
            out[k] = uint8_t(x == 0 || x >= cols - 1 ? cap : v);
        }
    }
    uint8_t* drow = im.dst + size_t(y) * im.dst_step + x0;
    if (x0 + PF_X <= cols && (reinterpret_cast<uintptr_t>(drow) & 15) == 0) {
        *reinterpret_cast<uint4*>(drow) = *reinterpret_cast<const uint4*>(out);
    } else {
        #pragma unroll
        for (int k = 0; k < PF_X; ++k)
            if (x0 + k < cols) drow[k] = out[k];
    }
}

// `n` images of P (element type from `f32`).
static inline int prefilter_launch(const PfParams& P, int n, bool f32, cudaStream_t st) {
    const dim3 grid(div_round_up(P.cols, PF_THREADS * PF_X), unsigned(P.rows), unsigned(n));
    if (f32) prefilter_kernel<float><<<grid, PF_THREADS, 0, st>>>(P);
    else prefilter_kernel<uint8_t><<<grid, PF_THREADS, 0, st>>>(P);
    SB_CUDA(cudaGetLastError());
    return STEREO_OK;
}

// ---- texture threshold ----------------------------------------------------------------------------------------------

constexpr int TX_MAXMAPS = 32;
constexpr int TX_TW = 128, TX_TH = 32;   // output tile
constexpr int TX_THREADS = 256;
constexpr int TX_MAXR = 64;

struct TxMap { const uint8_t* pf; size_t pf_step; void* disp; size_t disp_step; };     // each at row 0
struct TxParams {
    TxMap map[TX_MAXMAPS];
    int rows, cols, R, cap, threshold, sentinel;
};

static inline size_t texture_smem_bytes(int R) {
    const size_t W = TX_TW + 2 * R;
    return size_t(TX_TH) * W * 4 + size_t(TX_TH + 2 * R) * W;
}

// One launch over every map of a call: grid (ceil(cols / TX_TW), ceil(rows / TX_TH), maps).  A tile stages |P - cap| of
// its outputs and their R halo (clamped coordinates) in shared memory; thread c of the W = TX_TW + 2R columns stages
// column c and keeps its running (2R + 1)-row sum (int32: at most 129^2 x 63); then each thread slides a (2R + 1)-column
// sum along 16 outputs of one row and writes the sentinel where it is below the threshold.  The map is written, never read.
template <class T>
__global__ void __launch_bounds__(TX_THREADS) texture_kernel(const __grid_constant__ TxParams P) {
    extern __shared__ __align__(16) unsigned char tx_smem[];
    const TxMap& m = P.map[blockIdx.z];
    const int R = P.R, w = 2 * R + 1, W = TX_TW + 2 * R, H = TX_TH + 2 * R;
    const int x0 = blockIdx.x * TX_TW, y0 = blockIdx.y * TX_TH;
    int32_t* vs = reinterpret_cast<int32_t*>(tx_smem);                  // TX_TH x W column sums
    uint8_t* a = tx_smem + size_t(TX_TH) * W * 4;                        // H x W of |P - cap|
    if (int(threadIdx.x) < W) {
        const int c = threadIdx.x;
        const uint8_t* col = m.pf + clampi(x0 - R + c, 0, P.cols - 1);
        int s = 0;
        for (int r = 0; r < H; ++r) {
            const int v = abs(int(col[size_t(clampi(y0 - R + r, 0, P.rows - 1)) * m.pf_step]) - P.cap);
            a[r * W + c] = uint8_t(v);
            s += v;
            if (r >= w) s -= a[(r - w) * W + c];
            if (r >= w - 1) vs[(r - w + 1) * W + c] = s;
        }
    }
    __syncthreads();
    constexpr int SEG = TX_TW / (TX_THREADS / TX_TH);                    // 16 outputs per thread
    const int r = threadIdx.x % TX_TH, c0 = (threadIdx.x / TX_TH) * SEG, y = y0 + r;
    if (y >= P.rows) return;
    const int32_t* row = vs + r * W;
    int s = 0;
    for (int k = 0; k < w; ++k) s += row[c0 + k];
    T* drow = reinterpret_cast<T*>(static_cast<char*>(m.disp) + size_t(y) * m.disp_step);
    #pragma unroll
    for (int k = 0; k < SEG; ++k) {
        const int x = x0 + c0 + k;
        if (x >= P.cols) break;
        if (s < P.threshold) drow[x] = T(P.sentinel);
        if (k + 1 < SEG) s += row[c0 + k + w] - row[c0 + k];
    }
}

template <class T>
static inline int texture_init_one() {
    SB_CUDA(cudaFuncSetAttribute(reinterpret_cast<const void*>(texture_kernel<T>), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 int(texture_smem_bytes(TX_MAXR))));
    return STEREO_OK;
}

static inline int texture_init() {
    int rc = texture_init_one<int8_t>();
    if (rc == STEREO_OK) rc = texture_init_one<int16_t>();
    return rc == STEREO_OK ? texture_init_one<int32_t>() : rc;
}

// The `n` maps of P, whose elements are `elem` bytes.
static inline int texture_launch(const TxParams& P, int n, int elem, cudaStream_t st) {
    const dim3 grid(div_round_up(P.cols, TX_TW), div_round_up(P.rows, TX_TH), unsigned(n));
    const size_t smem = texture_smem_bytes(P.R);
    if (elem == 1) texture_kernel<int8_t><<<grid, TX_THREADS, smem, st>>>(P);
    else if (elem == 2) texture_kernel<int16_t><<<grid, TX_THREADS, smem, st>>>(P);
    else texture_kernel<int32_t><<<grid, TX_THREADS, smem, st>>>(P);
    SB_CUDA(cudaGetLastError());
    return STEREO_OK;
}

} // namespace sb
