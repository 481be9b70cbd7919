// Speckle filter (OpenCV's cv::filterSpeckles) of disparity maps, in place.
//   Two 4-neighbours are connected when neither equals new_val and |a - b| <= max_diff (in 64 bits).  Every pixel of a
//   connected component of at most max_size pixels becomes new_val; every other pixel keeps its value.
// Connected components by block-based union-find in four launches, each over every map of the call, none of which reads
// anything back to the host (the call stays asynchronous and capturable in a CUDA graph):
//   1. speckle_local_kernel    union-find inside a 32 x 16 tile in shared memory (horizontal runs by warp ballot, unions
//                              between runs); every pixel's label becomes the flat index of its tile root (the smallest
//                              index of its tile-local component), and the tile root's count the size of that component
//                              (0 for every other pixel)
//   2. speckle_merge_kernel    unions across tile borders in global memory: atomicMin links the larger root under the
//                              smaller, so every label only ever decreases and the root of a component is its smallest
//                              index.  Along a border, only the first of a stretch of linked pixels makes the union.
//   3. speckle_resolve_kernel  every tile root finds its component's root, points straight at it and adds its count to the
//                              root's (one global atomic per tile-local component, not per pixel)
//   4. speckle_write_kernel    pixel -> tile root -> root (two loads); new_val where the root's count <= max_size
// Only tile roots are ever parents (unions link roots, path halving writes grandparents), which is what makes step 4's two
// loads reach the root.  Scratch: label and count, 4 bytes each per pixel and map.
#pragma once
#include "common.cuh"

namespace sb {

constexpr int SPK_MAXMAPS = 32;           // both maps of up to 16 pairs (FMAXJOBS directions)
constexpr int SPK_MAXDIM = 32768;         // rows, cols: flat pixel indices fit in int32
constexpr int SPK_TW = 32, SPK_TH = 16;   // tile of the shared-memory pass, one pixel a thread
constexpr int SPK_THREADS = 256;          // passes 3 and 4: one pixel a thread

struct SpeckleMap { void* disp; size_t step; int32_t* label; int32_t* count; };     // label / count: rows * cols each
struct SpeckleParams {
    SpeckleMap map[SPK_MAXMAPS];
    int rows, cols, new_val, max_size, max_diff;
};

template <class T>
__device__ __forceinline__ T* spk_row(const SpeckleMap& m, int y) {
    return reinterpret_cast<T*>(static_cast<char*>(m.disp) + size_t(y) * m.step);
}

__device__ __forceinline__ bool spk_linked(int a, int b, const SpeckleParams& P) {
    const long long d = (long long)a - b;
    return a != P.new_val && b != P.new_val && (d < 0 ? -d : d) <= P.max_diff;
}

// Labels other threads are rewriting are read with relaxed loads at GPU scope, never through the L1.
__device__ __forceinline__ int spk_ld(const int32_t* p) {
    int v;
    asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// Root of x in the global forest, halving the path on the way: x is pointed at its grandparent, an ancestor and so a
// smaller label (atomicMin keeps whichever of two concurrent rewrites is smaller; both are in x's component).
__device__ __forceinline__ int spk_find(int32_t* L, int x) {
    for (;;) {
        const int p = spk_ld(L + x);
        if (p == x) return x;
        const int g = spk_ld(L + p);
        if (g == p) return p;
        atomicMin(L + x, g);
        x = g;
    }
}

// Joins the trees of a and b: the larger root is linked under the smaller.  A root that stopped being one between the
// find and the atomicMin hands back its new parent, and the union goes on from there.
__device__ __forceinline__ void spk_union(int32_t* L, int a, int b) {
    for (;;) {
        a = spk_find(L, a);
        b = spk_find(L, b);
        if (a == b) return;
        if (a < b) { const int old = atomicMin(L + b, a); if (old == b) return; b = old; }
        else { const int old = atomicMin(L + a, b); if (old == a) return; a = old; }
    }
}

__device__ __forceinline__ int spk_find_shared(volatile int* L, int x) {
    int p;
    while ((p = L[x]) != x) x = p;
    return x;
}

__device__ __forceinline__ void spk_union_shared(int* L, int a, int b) {
    for (;;) {
        a = spk_find_shared(L, a);
        b = spk_find_shared(L, b);
        if (a == b) return;
        if (a < b) { const int old = atomicMin(L + b, a); if (old == b) return; b = old; }
        else { const int old = atomicMin(L + a, b); if (old == a) return; a = old; }
    }
}

// grid (tiles across, tiles down, maps), block SPK_TW x SPK_TH: one warp a tile row.  Slots outside the map hold new_val
// and so link to nothing.  A row's horizontal runs are labelled by a ballot (every pixel points at its run's first pixel),
// so the shared-memory unions are only the vertical ones, one per contact of two runs.
template <class T>
__global__ void __launch_bounds__(SPK_TW * SPK_TH) speckle_local_kernel(const __grid_constant__ SpeckleParams P) {
    static_assert(SPK_TW == 32, "a tile row is one warp");
    __shared__ int s_val[SPK_TH * SPK_TW], s_run[SPK_TH * SPK_TW], s_lab[SPK_TH * SPK_TW], s_cnt[SPK_TH * SPK_TW];
    const SpeckleMap& m = P.map[blockIdx.z];
    const int lx = threadIdx.x, ly = threadIdx.y, li = ly * SPK_TW + lx;
    const int x = blockIdx.x * SPK_TW + lx, y = blockIdx.y * SPK_TH + ly;
    const bool in = x < P.cols && y < P.rows;
    const int v = in ? int(spk_row<T>(m, y)[x]) : P.new_val;
    s_val[li] = v;
    s_cnt[li] = 0;
    __syncthreads();
    const bool left = lx > 0 && spk_linked(v, s_val[li - 1], P);
    const unsigned starts = __ballot_sync(0xffffffffu, !left);
    const int run = ly * SPK_TW + 31 - __clz(starts & (0xffffffffu >> (31 - lx)));
    s_run[li] = run;
    s_lab[li] = run;
    __syncthreads();
    // the left neighbour already joined the same two runs when it is in this pixel's run, linked upwards too, and the
    // pixel above it is in the run above this one
    const bool up = ly > 0 && spk_linked(v, s_val[li - SPK_TW], P);
    const unsigned ups = __ballot_sync(0xffffffffu, up);
    const bool again = left && (ups >> (lx - 1) & 1u) && s_run[li - SPK_TW - 1] == s_run[li - SPK_TW];
    if (up && !again) spk_union_shared(s_lab, run, s_run[li - SPK_TW]);
    __syncthreads();
    const int r = spk_find_shared(s_lab, run);
    if (in) atomicAdd(&s_cnt[r], 1);
    __syncthreads();
    if (in) {
        // tile-local indices and flat map indices are both row-major, so the tile's smallest index stays its smallest
        const int i = y * P.cols + x;
        m.label[i] = (blockIdx.y * SPK_TH + r / SPK_TW) * P.cols + blockIdx.x * SPK_TW + r % SPK_TW;
        m.count[i] = s_cnt[li];
    }
}

// grid (tiles across, tiles down, maps), block 64: warp 0 joins the tile's top row to the row above, lanes [0, SPK_TH) of
// warp 1 its left column to the column on the left.  A border pixel skips the union its predecessor along the border
// already made: both pairs linked, and the predecessor linked to the pixel on both sides of the border.
template <class T>
__global__ void __launch_bounds__(64) speckle_merge_kernel(const __grid_constant__ SpeckleParams P) {
    const SpeckleMap& m = P.map[blockIdx.z];
    const int t = threadIdx.x, lane = t & 31;
    const bool top = t < 32;
    int x, y, nx, ny;
    if (top) { x = blockIdx.x * SPK_TW + t; y = blockIdx.y * SPK_TH; nx = x; ny = y - 1; }
    else { x = blockIdx.x * SPK_TW; y = blockIdx.y * SPK_TH + lane; nx = x - 1; ny = y; }
    const bool ok = (top || lane < SPK_TH) && x < P.cols && y < P.rows && nx >= 0 && ny >= 0;
    int a = P.new_val, b = P.new_val;
    if (ok) { a = int(spk_row<T>(m, y)[x]); b = int(spk_row<T>(m, ny)[nx]); }
    const bool link = spk_linked(a, b, P);
    const int pa = __shfl_up_sync(0xffffffffu, a, 1), pb = __shfl_up_sync(0xffffffffu, b, 1);
    const bool plink = __shfl_up_sync(0xffffffffu, int(link), 1) != 0;
    const bool again = lane > 0 && plink && spk_linked(pa, a, P) && spk_linked(pb, b, P);
    if (link && !again) spk_union(m.label, y * P.cols + x, ny * P.cols + nx);
}

// grid (pixel blocks, maps).  Tile roots are the pixels with a count; a root's own count only ever grows.
__global__ void __launch_bounds__(SPK_THREADS) speckle_resolve_kernel(const __grid_constant__ SpeckleParams P) {
    const SpeckleMap& m = P.map[blockIdx.y];
    const int i = blockIdx.x * SPK_THREADS + threadIdx.x;
    if (i >= P.rows * P.cols) return;
    const int c = spk_ld(m.count + i);
    if (c == 0) return;
    const int r = spk_find(m.label, i);
    if (r == i) return;
    atomicMin(m.label + i, r);
    atomicAdd(m.count + r, c);
}

// grid (pixel blocks, maps)
template <class T>
__global__ void __launch_bounds__(SPK_THREADS) speckle_write_kernel(const __grid_constant__ SpeckleParams P) {
    const SpeckleMap& m = P.map[blockIdx.y];
    const int i = blockIdx.x * SPK_THREADS + threadIdx.x;
    if (i >= P.rows * P.cols) return;
    const int y = i / P.cols, x = i - y * P.cols;
    T* row = spk_row<T>(m, y);
    if (int(row[x]) == P.new_val) return;
    const int r = __ldg(m.label + __ldg(m.label + i));
    if (__ldg(m.count + r) <= P.max_size) row[x] = T(P.new_val);
}

// Device bytes of the label and count arrays of `maps` rows x cols maps.
static inline size_t speckle_scratch_bytes(int maps, int rows, int cols) {
    const size_t one = (size_t(rows) * cols * 4 + 255) & ~size_t(255);
    return size_t(maps) * 2 * one + 256;
}

// Points map k's label and count arrays at its share of `scratch` (speckle_scratch_bytes(maps, rows, cols) bytes).
static inline void speckle_bind_scratch(SpeckleParams& P, int maps, void* scratch) {
    const size_t one = (size_t(P.rows) * P.cols * 4 + 255) & ~size_t(255);
    char* s = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(scratch) + 255) & ~uintptr_t(255));
    for (int k = 0; k < maps; ++k) {
        P.map[k].label = reinterpret_cast<int32_t*>(s + size_t(2 * k) * one);
        P.map[k].count = reinterpret_cast<int32_t*>(s + size_t(2 * k + 1) * one);
    }
}

template <class T>
static inline void speckle_launch_t(const SpeckleParams& P, int maps, cudaStream_t st) {
    const dim3 tiles(div_round_up(P.cols, SPK_TW), div_round_up(P.rows, SPK_TH), maps);
    const dim3 px(div_round_up((long long)P.rows * P.cols, SPK_THREADS), maps);
    speckle_local_kernel<T><<<tiles, dim3(SPK_TW, SPK_TH), 0, st>>>(P);
    speckle_merge_kernel<T><<<tiles, 64, 0, st>>>(P);
    speckle_resolve_kernel<<<px, SPK_THREADS, 0, st>>>(P);
    speckle_write_kernel<T><<<px, SPK_THREADS, 0, st>>>(P);
}

constexpr int SPK_LAUNCHES = 4;

// The filter over `maps` maps of P (scratch bound) whose elements are `elem` bytes; max_size must be > 0.
static inline int speckle_launch(const SpeckleParams& P, int maps, int elem, cudaStream_t st) {
    if (elem == 1) speckle_launch_t<int8_t>(P, maps, st);
    else if (elem == 2) speckle_launch_t<int16_t>(P, maps, st);
    else speckle_launch_t<int32_t>(P, maps, st);
    SB_CUDA(cudaGetLastError());
    return STEREO_OK;
}

} // namespace sb
