// Semi-global matching (path aggregation of the matching cost along scanlines) for one direction of a pair.
//   C(y, x, d)  SSD: the reference's SSD window sum of candidate d (exact.cuh's ssd_elem per element, the flat-index
//               row-wrap reads included), for the present candidates: those with s = x + R + d in [0, Wp - 1].
//               NCC: q - floor(fl32(q s)) of the candidate's float32 TM_CCORR_NORMED score s (exact.cuh's ncorr_exact_kernel
//               arithmetic), for the present candidates: those with x + d in [0, cols - 1].
//   L_r(p, d) = C(p, d) + min(L_r(q, d), L_r(q, d -+ 1) + P1, m(q) + P2) - m(q),  q = p - r,  m(q) = min_e L_r(q, e);
//               L_r(p, d) = C(p, d) where q lies outside the image.  Terms of candidates absent at q are left out.
//   S(p, d)   = sum over the 4 or 8 paths r of L_r(p, d);  disparity = the first minimum of S over the present candidates.
// Launches per direction: two replicate pads (exact.cuh), [NCC: sgm_ncc_norm_kernel,] the cost kernel - sgm_cost_kernel, or
// sgm_ncc_cell_kernel for NCC on float images that are not 8-bit-valued - then one sgm_path_kernel per path in stream
// order; the first path writes S, the later ones read-add-write it, the last one also writes the winner-take-all map.
// The uniqueness pass over a block matcher's SSD map reuses the pads, sgm_cost_kernel<false> and one path kernel with
// P1 = P2 = 0 (so L_r = C), S not stored and only the sentinel written (SgmOut::only_invalid).
// Layout: candidate index j = d - dlo innermost, padded to Dp = 32 K (K candidates per lane of the path kernels).  Absent
// and padding candidates hold SGM_ABSENT in C and L; S of an absent candidate is 0xFFFFFFFF, above every present sum as
// an unsigned value.  With paths * (C_max + P2) <= 2^31 - 1 (checked by the caller), every present L is below 2^29, m(q)
// + P2 below 2^30 = SGM_ABSENT, and SGM_ABSENT + P1 below 2^31: absent terms never win a minimum and nothing overflows.
#pragma once
#include "common.cuh"
#include "exact.cuh"
#include "subpixel.cuh"

namespace sb {

constexpr int SGM_ABSENT = 1 << 30;
constexpr int SGM_MAXK = 16;               // candidates per lane (one instantiation each): at most 512 per pixel
constexpr int SGM_XT = 256;                // output columns of one cost block
constexpr int SGM_COST_THREADS = 256;      // 8 warps, SGM_XT / 8 consecutive columns each
constexpr int SGM_PATH_WARPS = 4;          // scanlines (one warp each) per path block

// The NCC cost's per-pixel window norms (sgm_ncc_norm_kernel, rows x cols each) and its scale q.
struct SgmNcc { const double* nref; const double* ntgt; int q; };

// C of a present NCC candidate d at (y, x) from its double numerator acc: q - floor(fl32(q s)), in [0, 2q].
__device__ __forceinline__ int32_t sgm_ncc_cost(double acc, const SgmNcc& n, int cols, int y, int x, int d) {
    const size_t o = size_t(y) * cols + x;
    const float s = ncc_normalise(acc, n.ntgt[o + d] * n.nref[o]);
    return n.q - int(floorf(__fmul_rn(float(n.q), s)));
}

// Window norms of one direction's padded images at every (y, x): the double window energy E in the oracle's (wy, k)
// order, then nref = sqrt(E) of the reference (blockIdx.z 0) and ntgt = ncc_target_norm(E) of the target (blockIdx.z 1),
// so that ntgt(y, x + d) * nref(y, x) is ncorr_exact_kernel's t of candidate d bit for bit.
__global__ void __launch_bounds__(128)
sgm_ncc_norm_kernel(const float* __restrict__ Lp, const float* __restrict__ Rp, int cols, int R, double* __restrict__ nref,
                    double* __restrict__ ntgt) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= cols) return;
    const int Wp = cols + 2 * R, w = 2 * R + 1;
    const float* img = blockIdx.z ? Rp : Lp;
    double e = 0;
    for (int wy = 0; wy < w; ++wy) {
        const float* row = img + size_t(y + wy) * Wp + x;
        for (int k = 0; k < w; ++k) { const double v = __ldg(row + k); e += v * v; }
    }
    const size_t o = size_t(y) * cols + x;
    if (blockIdx.z) ntgt[o] = ncc_target_norm(e);
    else nref[o] = sqrt(e);
}

// C for output rows [y0, y0 + rows_per_block) x columns [x0, x0 + SGM_XT) x candidates [j0, j0 + 32) of one block.
// Vertical window sums V(c, d) of the element image E(r, c, d) are kept in shared memory for the block's columns and
// slide down one row at a time (E is recomputed for the row that leaves); each warp then slides the horizontal window
// along its 32 columns with the candidate in the lane, so every row of C is written as 128-byte lines.
//   SSD: E = ssd_elem(Lp[r][c], Rp_flat[r Wp + c + d]); reads outside [-R, Hp Wp + R) - only ever of absent or padding
//        candidates - count as 0.
//   NCC (8-bit-valued images only): E = Lp[r][c] Rp[r][c + d], 0 where c + d leaves the padded row (again only absent or
//        padding candidates).  The products are integers, so the int32 window sum - below (2R + 1)^2 255^2 < 2^31 - is
//        the oracle's double numerator exactly, whatever the order; the epilogue normalises it (sgm_ncc_cost).
template <bool NCC>
__global__ void __launch_bounds__(SGM_COST_THREADS)
sgm_cost_kernel(const float* __restrict__ Lp, const float* __restrict__ Rp, int rows, int cols, int R, int dlo, int D, int Dp,
                int rows_per_block, SgmNcc ncc, int32_t* __restrict__ C) {
    extern __shared__ int32_t V[];                       // [(SGM_XT + 2R) columns][32 candidates]
    const int Wp = cols + 2 * R, w = 2 * R + 1, nc = SGM_XT + 2 * R;
    const long long flat_lo = -R, flat_hi = (long long)(rows + 2 * R) * Wp + R;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int x0 = blockIdx.x * SGM_XT, y0 = blockIdx.y * rows_per_block, j = blockIdx.z * 32 + lane;
    const int d = dlo + j;
    const int y1 = min(rows, y0 + rows_per_block);
    auto E = [&](int r, int c) -> int {                  // r, c: padded coordinates
        if (NCC) {
            if (c >= Wp || c + d < 0 || c + d >= Wp) return 0;
            return int(__ldg(Lp + (long long)r * Wp + c)) * int(__ldg(Rp + (long long)r * Wp + c + d));
        }
        const long long f = (long long)r * Wp + c + d;
        if (c >= Wp || f < flat_lo || f >= flat_hi) return 0;
        return ssd_elem(__ldg(Lp + (long long)r * Wp + c), __ldg(Rp + f));
    };
    for (int ci = warp; ci < nc; ci += SGM_COST_THREADS / 32) {
        int v = 0;
        for (int r = y0; r < y0 + w; ++r) v += E(r, x0 + ci);
        V[ci * 32 + lane] = v;
    }
    constexpr int SEG = SGM_XT / (SGM_COST_THREADS / 32);
    const int xs = x0 + warp * SEG;
    for (int y = y0;;) {
        __syncthreads();
        if (xs < cols) {
            int h = 0;
            for (int k = 0; k < w; ++k) h += V[(warp * SEG + k) * 32 + lane];
            int32_t* out = C + ((size_t)y * cols + xs) * Dp + j;
            const int xe = min(cols, xs + SEG);
            for (int x = xs; x < xe; ++x, out += Dp) {
                if (NCC) *out = (j < D && x + d >= 0 && x + d < cols) ? sgm_ncc_cost(double(h), ncc, cols, y, x, d) : SGM_ABSENT;
                else *out = (j < D && x + R + d >= 0 && x + R + d < Wp) ? h : SGM_ABSENT;
                const int ci = x - x0;
                if (x + 1 < xe) h += V[(ci + w) * 32 + lane] - V[ci * 32 + lane];
            }
        }
        if (++y >= y1) break;
        __syncthreads();
        for (int ci = warp; ci < nc; ci += SGM_COST_THREADS / 32)
            V[ci * 32 + lane] += E(y - 1 + w, x0 + ci) - E(y - 1, x0 + ci);
    }
}

// C of the NCC cost for float images that are not 8-bit-valued: their products round in double, so each cell's numerator
// is summed on its own in the oracle's (wy, k) order.  One block: row y, columns [x0, x0 + SGM_CELL_XT), candidates
// [j0, j0 + 32) with the candidate in the lane; each warp holds SGM_CELL_XT / 8 consecutive pixels' numerators.  Window
// row by window row, the block stages the reference's and the targets' padded row segments in shared memory (0 outside
// the row: only absent and padding candidates read there); the reference value is a broadcast, the target values are
// consecutive across the lanes, and every row of C is written as 128-byte lines.
constexpr int SGM_CELL_XT = 64;
__global__ void __launch_bounds__(SGM_COST_THREADS)
sgm_ncc_cell_kernel(const float* __restrict__ Lp, const float* __restrict__ Rp, int cols, int R, int dlo, int D, int Dp, SgmNcc ncc,
                    int32_t* __restrict__ C) {
    extern __shared__ float sh[];                        // reference [SGM_CELL_XT + 2R], target [SGM_CELL_XT + 31 + 2R]
    constexpr int PX = SGM_CELL_XT / (SGM_COST_THREADS / 32);
    const int Wp = cols + 2 * R, w = 2 * R + 1, nl = SGM_CELL_XT + 2 * R, nt = nl + 31;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int x0 = blockIdx.x * SGM_CELL_XT, y = blockIdx.y, j = blockIdx.z * 32 + lane, d = dlo + j;
    const int t0 = x0 + dlo + blockIdx.z * 32;            // padded target column of the target segment's first value
    float* Ls = sh;
    float* Ts = sh + nl;
    double acc[PX];
#pragma unroll
    for (int u = 0; u < PX; ++u) acc[u] = 0;
    for (int wy = 0; wy < w; ++wy) {
        const float* lrow = Lp + size_t(y + wy) * Wp;
        const float* rrow = Rp + size_t(y + wy) * Wp;
        for (int i = threadIdx.x; i < nl; i += SGM_COST_THREADS) Ls[i] = x0 + i < Wp ? __ldg(lrow + x0 + i) : 0.f;
        for (int i = threadIdx.x; i < nt; i += SGM_COST_THREADS) Ts[i] = t0 + i >= 0 && t0 + i < Wp ? __ldg(rrow + t0 + i) : 0.f;
        __syncthreads();
#pragma unroll
        for (int u = 0; u < PX; ++u) {
            const int xi = warp * PX + u;
            for (int k = 0; k < w; ++k) acc[u] += double(Ls[xi + k]) * double(Ts[xi + lane + k]);     // (exact products)
        }
        __syncthreads();
    }
#pragma unroll
    for (int u = 0; u < PX; ++u) {
        const int x = x0 + warp * PX + u;
        if (x < cols)
            C[(size_t(y) * cols + x) * Dp + j] = (j < D && x + d >= 0 && x + d < cols) ? sgm_ncc_cost(acc[u], ncc, cols, y, x, d) : SGM_ABSENT;
    }
}

// Scanlines of direction (dy, dx): every pixel whose predecessor p - r lies outside the image starts one.
__host__ __device__ inline int sgm_lines(int rows, int cols, int dy, int dx) {
    return (dy ? cols : 0) + (dx ? (dy ? rows - 1 : rows) : 0);
}

// The map the last path writes (ptr == nullptr: none).  uniq: the uniqueness ratio (0: off), whose rejected pixels get
// `sentinel`.  only_invalid: the block matcher's map is already there; store only the sentinel, also at pixels whose every
// present V is >= 99999999 (the reference's initial best cost, so its map holds the default 0 there).  subpix (nullptr:
// off): rows x cols bytes that receive each pixel's sub-pixel offset of the winner (subpixel.cuh's subpix_offset of S(j* - 1),
// S(j*), S(j* + 1); 0 where a neighbour is absent).
struct SgmOut { void* ptr; size_t step; int elem; int dlo; int uniq; int sentinel; int only_invalid; int8_t* subpix; };

constexpr unsigned SGM_BM_NO_WINNER = 99999999u;

// Winner-take-all of one pixel's V across the warp, lane l holding candidates [l K, l K + K) (absent: 0xFFFFFFFF).
// Returns j*, the first minimum, in every lane, and its V* in *vbest.  *unique is false when uniq > 0 and some present j with
// |j - j*| > 1 has V(j) (100 - uniq) < V* 100 (StereoSGBM's uniquenessRatio rule, in 64-bit); true otherwise, also when every
// other candidate is absent.
template <int K>
__device__ __forceinline__ int sgm_winner(const unsigned (&v)[K], int lane, int uniq, unsigned* vbest, bool* unique) {
    unsigned best = 0xFFFFFFFFu; int bi = 0;
#pragma unroll
    for (int i = K - 1; i >= 0; --i) if (v[i] <= best) { best = v[i]; bi = i; }
    const unsigned wmin = __reduce_min_sync(0xffffffffu, best);
    const unsigned ball = __ballot_sync(0xffffffffu, best == wmin);
    const int src = __ffs(ball) - 1;
    const int jw = __shfl_sync(0xffffffffu, lane * K + bi, src);
    *vbest = wmin;
    *unique = true;
    if (uniq) {
        unsigned far = 0xFFFFFFFFu;
#pragma unroll
        for (int i = 0; i < K; ++i) if (abs(lane * K + i - jw) > 1) far = min(far, v[i]);
        far = __reduce_min_sync(0xffffffffu, far);
        *unique = far == 0xFFFFFFFFu || (unsigned long long)far * unsigned(100 - uniq) >= (unsigned long long)wmin * 100u;
    }
    return jw;
}

// One path direction, one warp per scanline, lane l holding candidates [l K, l K + K) (Dp = 32 K).  The previous pixel's L_r stays in
// registers; d -+ 1 across lanes come through shuffles and m(q) is one warp minimum.  first: S = L; otherwise S += L; S ==
// nullptr (only with first): S is not stored.  With out.ptr, the winner-take-all of the final S (first minimum, unsigned,
// with out.uniq the uniqueness ratio: sgm_winner) is stored in out's element type.
template <int K>
__global__ void __launch_bounds__(SGM_PATH_WARPS * 32)
sgm_path_kernel(const int32_t* __restrict__ C, int32_t* __restrict__ S, int rows, int cols, int dy, int dx, int P1, int P2,
                int first, SgmOut out) {
    constexpr int Dp = 32 * K;
    const int lane = threadIdx.x & 31;
    const int line = blockIdx.x * SGM_PATH_WARPS + (threadIdx.x >> 5);
    if (line >= sgm_lines(rows, cols, dy, dx)) return;
    int y, x;
    if (dy && line < cols) { y = dy > 0 ? 0 : rows - 1; x = line; }
    else {
        const int t = dy ? line - cols : line;
        x = dx > 0 ? 0 : cols - 1;
        y = (dy > 0) ? t + 1 : t;
    }
    const int steps = min(dy > 0 ? rows - y : dy < 0 ? y + 1 : 0x7FFFFFFF, dx > 0 ? cols - x : dx < 0 ? x + 1 : 0x7FFFFFFF);
    const long long stride = ((long long)dy * cols + dx) * Dp;
    long long base = ((long long)y * cols + x) * Dp + lane * K;
    // C and S of the next PF pixels are in flight while this one is computed (S of a pixel is only ever touched by the one
    // warp whose scanline crosses it, and by earlier launches)
    constexpr int PF = K <= 3 ? 4 : K <= 8 ? 2 : 1;
    int Lq[K], cq[PF][K], sq[PF][K];
#pragma unroll
    for (int u = 0; u < PF; ++u)
#pragma unroll
        for (int i = 0; i < K; ++i) {
            cq[u][i] = u < steps ? __ldg(C + base + u * stride + i) : SGM_ABSENT;
            sq[u][i] = u < steps && !first ? S[base + u * stride + i] : 0;
        }
#pragma unroll
    for (int i = 0; i < K; ++i) Lq[i] = SGM_ABSENT;
    int mq = 0;
    for (int s0 = 0; s0 < steps; s0 += PF) {
#pragma unroll
    for (int u = 0; u < PF; ++u) {
        const int st = s0 + u;
        if (st >= steps) break;
        int c[K], so[K];
#pragma unroll
        for (int i = 0; i < K; ++i) { c[i] = cq[u][i]; so[i] = sq[u][i]; }
        if (st + PF < steps) {
#pragma unroll
            for (int i = 0; i < K; ++i) {
                cq[u][i] = __ldg(C + base + PF * stride + i);
                sq[u][i] = first ? 0 : S[base + PF * stride + i];
            }
        }
        // neighbours across lanes: the last candidate of lane - 1 and the first of lane + 1
        int lm = __shfl_up_sync(0xffffffffu, Lq[K - 1], 1);
        int rp = __shfl_down_sync(0xffffffffu, Lq[0], 1);
        if (lane == 0) lm = SGM_ABSENT;
        if (lane == 31) rp = SGM_ABSENT;
        int L[K];
        int lmin = SGM_ABSENT;
#pragma unroll
        for (int i = 0; i < K; ++i) {
            if (st == 0 || c[i] == SGM_ABSENT) L[i] = c[i];
            else {
                const int a = i == 0 ? lm : Lq[i > 0 ? i - 1 : 0];           // (indices stay constant and in range)
                const int b = i + 1 < K ? Lq[i + 1 < K ? i + 1 : i] : rp;
                L[i] = c[i] + min(min(Lq[i], min(a, b) + P1), mq + P2) - mq;
            }
            lmin = min(lmin, L[i]);
        }
        mq = __reduce_min_sync(0xffffffffu, lmin);
        unsigned sn[K];
#pragma unroll
        for (int i = 0; i < K; ++i) {
            Lq[i] = L[i];
            sn[i] = c[i] == SGM_ABSENT ? 0xFFFFFFFFu : unsigned(first ? L[i] : so[i] + L[i]);
            if (S) S[base + i] = int(sn[i]);
        }
        if (out.ptr) {
            unsigned vbest;
            bool unique;
            const int jw = sgm_winner<K>(sn, lane, out.uniq, &vbest, &unique);
            const bool invalid = !unique || (out.only_invalid && vbest >= SGM_BM_NO_WINNER);
            int off = 0;
            if (out.subpix) {
                // S(j* - 1) and S(j* + 1) from the lanes that hold them, by selects over constant register indices
                unsigned vm = 0xFFFFFFFFu, vp = 0xFFFFFFFFu;
#pragma unroll
                for (int i = 0; i < K; ++i) {
                    if (lane * K + i == jw - 1) vm = sn[i];
                    if (lane * K + i == jw + 1) vp = sn[i];
                }
                vm = __reduce_min_sync(0xffffffffu, vm);
                vp = __reduce_min_sync(0xffffffffu, vp);
                if (vm != 0xFFFFFFFFu && vp != 0xFFFFFFFFu) off = subpix_offset(vm, vbest, vp);
            }
            if (lane == 0 && (invalid || !out.only_invalid)) {
                const long long pix = base / Dp;
                const int py = int(pix / cols), px = int(pix - (long long)py * cols);
                char* row = static_cast<char*>(out.ptr) + size_t(py) * out.step;
                const int dv = invalid ? out.sentinel : out.dlo + jw;
                if (out.elem == 1) reinterpret_cast<int8_t*>(row)[px] = int8_t(uint8_t(uint32_t(dv) & 0xFFu));
                else if (out.elem == 2) reinterpret_cast<int16_t*>(row)[px] = int16_t(dv);
                else reinterpret_cast<int32_t*>(row)[px] = dv;
                if (out.subpix) out.subpix[size_t(py) * cols + px] = int8_t(off);
            }
        }
        base += stride;
    }
    }
}

} // namespace sb
