// The hot kernels of the library (sm_100a): packed 8-bit operands (below) and float operands (OPF, see fast_row).
//
// For images that are exactly 8-bit the window cost is an integer and
//     SSD(x,d) = EL(x) + ER(x+d) - 2*C(x,d),   C = sum over the window of l*r,
//     NCC(x,d) = C(x,d) / sqrt(EL(x) * ER(x+d)),
// so the per-disparity work is ONE box-filtered cross term C; the energies are box sums computed
// once per image, not per disparity (north-star item (b)).  The kernel computes C with separable
// running sums held entirely in registers:
//
//   * vertical:   col[m][c] += l_new*r_new - l_old*r_old      ONE IDP.2A (dp2a, s16 x u8) per unit
//                 (the new and the leaving row are packed into one operand pair by the prep kernels)
//   * horizontal: s[m] += col[m][c+2R+1] - col[m][c]          ONE IADD3 per unit
//   * WTA:        key = E2[pos] + 256*s (cost*128 + position) ONE IMAD/LEA, then VIMNMX3 in-thread
//                 and REDUX.MIN across the 32 lanes of the warp (lanes = disparities)
//
// The cost volume never exists in memory: a thread owns K=24 pixels x M=4 disparities, a warp
// 24 pixels x 128 disparities, and only the winning key per pixel and 128-disparity group leaves
// the SM.  Operand rows are staged in shared memory with TMA bulk copies (cp.async.bulk, SASS
// UBLKCP) through a ring of up to 8 stages of 8 rows (full / empty mbarriers); all warps of a CTA share
// the staged rows.
//
// Pair launches (FUSED): the same cross terms also give the map of the OTHER direction of the image pair
// (C(x, d) is candidate -d of the partner pixel x + d), kept as running minima along the diagonals of the
// (x, x + d) plane - see fast_row.  Strips are 20 (16) pixels wide there instead of 24.  SSD for any candidate count, every
// radius up to 7 and either operand type; NCC (diagonal maxima, per-pixel key scales) for packed operands.
//
// Float operands (OPF): general float32 images (noise / contrast variants) on the same running sums - SSD with the
// per-element round((l-r)^2) as exact int32 sums, NCC in float32 - from rows of the padded float images themselves.
//
// Reference semantics reproduced (SURVEY.md Appendix A): replicate padding, the clamped candidate
// range in padded coordinates, the flat-index row wrap of the SSD target reads (realised by building
// the target operand rows from an "extended" image whose out-of-row columns come from the
// neighbouring padded row / zero guard), first-minimum (SSD) and first-maximum (NCC) tie-breaks.
#pragma once
#include "common.cuh"
#include <climits>
#include <cstdlib>

namespace sb {

#ifndef SB_FK_DEFAULT
#define SB_FK_DEFAULT 24
#endif
constexpr int FK_DEFAULT = SB_FK_DEFAULT;  // pixels per thread (strip width); template parameter K of the kernels
// Strip width of the fused pair kernels.  Their 8 extra live registers per thread make 24-pixel strips spill (ncu: 2.07 ms
// vs 1.82 ms per two 4K/256 pairs).  One strip per warp: 20 pixels (255 registers, no spills for R = 5, 24 bytes for R = 4);
// two strips per warp: 16 pixels (20 spills there; 0.150 vs 0.167 ms per four 720p/64 pairs).
#ifndef SB_FK_FUSED
#define SB_FK_FUSED 20
#endif
#ifndef SB_FK_FUSED2
#define SB_FK_FUSED2 16
#endif
constexpr int FK_FUSED = SB_FK_FUSED, FK_FUSED2 = SB_FK_FUSED2;
// Wide windows (R = 6, 7; the reference's own config/ps2.yaml:19-41 uses nothing else): a thread keeps K + 2R column sums
// per disparity, so the strips narrow by 4 pixels to stay inside the register file (K = 24 spilled 100-136 bytes there).
#ifndef SB_FK_WIDE
#define SB_FK_WIDE 20
#endif
#ifndef SB_FK_FUSED_WIDE
#define SB_FK_FUSED_WIDE 16
#endif
constexpr int FK_WIDE_R = 6;    // first radius that takes the narrower strips
#ifndef SB_FK_FUSED_NCC
#define SB_FK_FUSED_NCC 16
#endif
constexpr int FK_FUSED_NCC = SB_FK_FUSED_NCC;   // fused NCC pairs: the per-position scales take the registers four more pixels would
// float-operand kernels (OPF): K + 2R <= 30 column sums per disparity next to the operand words in flight
__host__ __device__ constexpr int fast_kf(int R) { return R <= 3 ? 24 : (R <= 5 ? 20 : 16); }
__host__ __device__ constexpr int fast_k(int R, bool fused, int hs) {
    return fused ? (hs == 2 ? FK_FUSED2 : (R >= FK_WIDE_R ? SB_FK_FUSED_WIDE : FK_FUSED)) : (R >= FK_WIDE_R ? SB_FK_WIDE : FK_DEFAULT);
}
constexpr int FM = 4;           // disparities per thread
constexpr int FGROUP = 32 * FM; // disparities per warp ("group")
constexpr int FKEY_BITS = 7;    // log2(FGROUP): low bits of a key order candidates inside a group
constexpr int FRPS = 8;         // operand rows per pipeline stage
constexpr int FNST_MAX = 8;     // pipeline stages (fewer when the tile rows are wide, FastGeom::nst)
constexpr int FSMEM_BUDGET = 220 * 1024;   // dynamic shared memory the hot kernel may use
#ifndef SB_FWARPS
#define SB_FWARPS 8
#endif
constexpr int FWARPS = SB_FWARPS; // warps per CTA (K=24 pixels x 4 disparities per thread: ~254 registers).  4-warp CTAs (narrower
                                // tiles for small images) were measured: one warp per scheduler cannot hide the row code's
                                // latencies (511x640/96 fused pair: 91 us against 54 us with 8 warps)
// Fused pair launches: words of slack either side of a partner's partial-key map (see the row epilogue of fast_row): the
// merges of lanes whose partner pixel lies outside the image land at most one disparity range + a strip before the first
// row or behind the last one.
static inline size_t fused_part_pad_words(int G) { return size_t(G) * 128 + 512; }
#ifndef SB_FMAXJOBS
#define SB_FMAXJOBS 32
#endif
// directions (jobs) one launch sequence can carry: 16 pairs.  The parameter block (~5.6 KB) needs the large kernel parameters
// of CUDA 12.1+ (sm_70+, up to 32764 bytes); 16 jobs (SB_FMAXJOBS=16) stay below the classic 4 KB.  720p/64 x 16 pairs:
// 0.70 -> 0.67 ms per step with one launch sequence instead of two.
constexpr int FMAXJOBS = SB_FMAXJOBS;
constexpr int FMAXR = 7;        // largest window radius with 32-bit keys: 128*(2R+1)^2*255^2 < 2^31
constexpr uint32_t KEY_INVALID = 0xFFFFFFFFu;
constexpr int FFREE_MASK_R = 5;   // largest radius for which invalid candidates lose through the key alone

// Keys are unsigned:  key = BIAS + 128*(ER - 2C) + position,  BIAS = 128*Emax, Emax = (2R+1)^2*255^2,
// so valid keys lie in [0, 256*Emax + position].  A candidate whose centre is not a legal search
// position carries E2 = KEY_INVALID; its key KEY_INVALID - 256*C stays above every valid key as long
// as 512*Emax < 2^32 (R <= 5), i.e. border masking costs no instruction there.
__host__ __device__ static inline uint32_t key_emax(int R) { return uint32_t((2 * R + 1) * (2 * R + 1)) * 65025u; }
__host__ __device__ static inline uint32_t key_bias(int R) { return key_emax(R) << FKEY_BITS; }
__host__ __device__ static inline uint32_t key_invalid_threshold(int R) {
    return R <= FFREE_MASK_R ? KEY_INVALID - (key_emax(R) << (FKEY_BITS + 1)) : KEY_INVALID;
}

// ---------------------------------------------------------------------------------------------------
// Geometry shared by host and device
// ---------------------------------------------------------------------------------------------------
struct FastGeom {
    // problem (shared by every job of a launch)
    int rows, cols, R, D, cost;   // D = candidates per pixel (max_disp - min_disp + 1)
    int rb, re;            // output band
    int ar0, ar1;          // image rows present in the caller's buffers (full image: 0, rows); reads clamp into it
    int K;                 // pixels per thread (strip width): 24
    int nw;                // warps per CTA: 8
    int opf;               // 1: float operand rows (general float32 images), 0: packed 8-bit operands
    int hs;                // strips per warp: 1 (a warp = 24 px x 128 disparities) or 2 (2 x 24 px x 64 disparities, D <= 64)
    // derived
    int dg;                // disparities per strip and warp = 128 / hs
    int G;                 // number of dg-disparity groups
    int gc;                // groups per CTA (1 or 2)
    int spc;               // strips per CTA = nw * hs / gc
    int nstrips;           // ceil(cols / K)
    int tilesX;            // ceil(nstrips / spc)
    int gblocks;           // G / gc
    int base_y;            // step row of operand row 0 (multiple of FRPS, <= rb - (2R+1))
    int J;                 // operand rows (multiple of FRPS)
    int lp_pitch, rq_pitch, e2_pitch;   // words (maximum over the jobs)
    int lpw, rqw, e2w;     // tile widths in words (multiples of 4)
    int nst;               // pipeline stages that fit in shared memory (<= FNST_MAX)
    int wpart;             // partial-key map width (= tilesX*spc*K)
    int nrows;             // re - rb
    int njobs;             // directions in this launch
    int npairs;            // fused launches: image pairs (jobs 0..npairs-1 are the L->R directions the hot kernel
                           // walks, job i+npairs is the R->L partner of job i); 0 otherwise
    int elw;               // fused launches: tile width (words) of the partner's energy rows (= spc*K); 0 otherwise
    int border;            // fused launches: 1 = the partner's candidates centred in the right padding come from
                           // fused_border_kernel instead of R extra columns of strips (when those would cost a whole tile)
    int ctas;              // grid size
    int nrl;               // rows of a tile in the linear (tile, row) space the CTAs split: nrows, or nrows padded up to a
                           // multiple of L when there are fewer tiles than SMs (then no CTA straddles two tiles)
    long long total;       // tiles x nrl (all jobs)
    long long L;           // linear rows per CTA
    int sched;             // 0: CTA b owns the contiguous linear range [b*L, (b+1)*L);  1: row-band-major items (band, tile) of
                           // L rows, CTA b owns items b, b + ctas, ... - the CTAs of a wave walk the SAME rows of neighbouring
                           // tiles at the same time, so the target-side operand rows neighbouring tiles share (a tile is 80
                           // pixels wide, its search range 256) are fetched from HBM once and then hit in L2
    int ntiles, nbands;    // sched 1: tiles of the launch (all jobs), row bands per tile
};

// One direction of one image pair inside a launch.  All jobs of a launch share FastGeom; what depends
// on the sign of the search range (offsets, legal centre columns) and every pointer is per job.
struct FastJob {
    const uint8_t* A; size_t a_step;    // reference image (the one whose pixels get a disparity)
    const uint8_t* B; size_t b_step;    // target image (searched)
    int dmin, dmax;
    int dlo0;              // first disparity of group 0: dmin, or (fused pair launches, the direction the kernel walks)
                           // dmax - (G*dg - 1), i.e. groups aligned to the TOP of the range so that the partner's groups are
                           // this direction's groups reversed for any candidate count; candidates below dmin are masked
    int qoff, eoff;        // column offsets of the RQ / E2 arrays
    int cmin, cmax;        // legal centre columns (unpadded coordinates)
    void* disp; size_t disp_step; int elem;
    void* best; size_t best_step;
    int32_t* LP;       // [J][lp_pitch]   s16x2: (-l(y+R), +l(y-R-1));   opf: [J+2R+1][lp_pitch] float rows of the padded reference
                       //                 image, array row jj <-> image row base_y - R - 1 + jj
    uint32_t* RQ;      // [J/2][rq_pitch] u8x4 : (r(ye+R), r(ye-R-1), r(ye+1+R), r(ye-R));   opf: [J+2R+1][rq_pitch] float rows of the
                       //                 extended target image
    int32_t* E2;       // [J][e2_pitch]   SSD: BIAS + 128*ER + position, or KEY_INVALID;  NCC: ER
    int32_t* PART;     // [G][nrows][wpart] winning keys
    int32_t* V;        // [nrows][vpitch] vertical (2R+1)-sums of squares of the extended target image
    float* RS;         // NCC: 1/sqrt(ER) per position   [J][e2_pitch]
    float* SC;         // NCC: [strip][nrows] magic = 2^ceil(log2 sqrt(max EL of the strip row))
};

static inline int round_up(int v, int m) { return (v + m - 1) / m * m; }
static inline int floor_div(int a, int b) { int q = a / b; if ((a % b != 0) && ((a < 0) != (b < 0))) --q; return q; }

// ---------------------------------------------------------------------------------------------------
// Device helpers
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ int dp2a_lo(int a, unsigned b, int c) {
    int d; asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c)); return d;
}
__device__ __forceinline__ int dp2a_hi(int a, unsigned b, int c) {
    int d; asm("dp2a.hi.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c)); return d;
}
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}
// TMA bulk copy global -> shared, completion on an mbarrier (SASS: UBLKCP).
__device__ __forceinline__ void tma_load_1d(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

__device__ __forceinline__ int4 lds128(const int* p) { return *reinterpret_cast<const int4*>(p); }

// ---------------------------------------------------------------------------------------------------
// The hot kernel
// ---------------------------------------------------------------------------------------------------
struct FastKernelParams {
    FastGeom g;
    FastJob job[FMAXJOBS];
};

template <int R, int K>
struct RowShape {
    static constexpr int NC = K + 2 * R;              // columns whose sums a thread keeps
    static constexpr int NC4 = (NC + 3) / 4 * 4;
    static constexpr int NQ = NC + FM - 1;             // target positions a thread touches
    static constexpr int NQ4 = (NQ + 3) / 4 * 4;
    static constexpr int NE = K + FM - 1;              // centre positions
    static constexpr int NE4 = (NE + 3) / 4 * 4;
};

// One operand row for one warp.
//   MODE 0: warm-up (add the entering row only, no output)
//   MODE 1: regular row; SSD: invalid search positions lose through their E2 entry alone (R <= 5);
//           NCC: every candidate of the block is legal
//   MODE 2: MODE 1 + whole lanes beyond max_disp are excluded (one LOP3 per pixel)
//   MODE 3: explicit per-candidate selects (partially valid lanes, border positions)
// PAR selects the byte pair of the RQ words (even/odd step row).
// The column updates (IDP.2A, FMA-heavy pipe) are interleaved with the horizontal slide / WTA of the
// same row (IADD3, VIMNMX on the ALU pipe) so that a single warp keeps both half-rate pipes busy.
//
// NCC keys.  v = C * RS[pos] (f32, C an exact integer) orders the candidates of one pixel; the oracle's
// first-maximum rule (cv::minMaxLoc, DisparityNCorr.cpp:62-64) needs the full f32 precision of v AND the
// position in one 32-bit key, which an f32 bit pattern cannot hold.  So v is turned into a 23-bit
// fixed-point number first: r = v + magic with magic = the power of two just above sqrt(max EL) of the
// strip row (C*RS <= sqrt(EL) by Cauchy-Schwarz), i.e. r lies in the binade [magic, 2*magic) and its
// mantissa IS round(v * 2^23 / magic).  key = (bits(r) << 9) + (reversed position << 2 | 3): 23 value
// bits, 7 position bits, low bits 11 so that 0 can mean "no legal candidate".  Unsigned max.
// For (2R+1)^2*255^2 < 2^23 (R <= 5) the running sums carry the float bias 0x4B000000, i.e. they ARE
// the float 2^23 + C, and v = fma(2^23 + C, rs, -2^23*rs) is the correctly rounded product with no
// conversion instruction; larger windows convert with I2F and fold the magic add into the FFMA.
#ifndef SB_KEY_LEA_MASK
#define SB_KEY_LEA_MASK 0
#endif
#ifndef SB_KEY_LEA_FUSED
#define SB_KEY_LEA_FUSED 0
#endif
#ifndef SB_KEY2_LEA
#define SB_KEY2_LEA 0
#endif
// Fused kernels: a diagonal takes its four candidates of a lane in two three-input minima (VIMNMX3: acc, the key held over
// from the step before, this step's key) instead of four two-input ones.
#ifndef SB_DIAG_MIN3
#define SB_DIAG_MIN3 1
#endif
#ifndef SB_NCC_UNBIAS
#define SB_NCC_UNBIAS 1
#endif
#ifndef SB_NCC_CHAIN
#define SB_NCC_CHAIN 1
#endif
#ifndef SB_TAIL_BATCH
#define SB_TAIL_BATCH 1
#endif
constexpr int NCC_BIAS_MAX_R = 5;
constexpr int NCC_FLOAT_BIAS = 0x4B000000;        // bit pattern of 8388608.0f
constexpr int NCC_KEY_SHIFT = 9;                  // mantissa -> bits 9..31
constexpr uint32_t NCC_KEY_NONE = 0u;             // "no legal candidate" (loses every unsigned max)

//
// HS > 1 (narrow searches, D <= 128/HS): the warp is cut into HS sub-warps of 32/HS lanes, each with its
// own K-pixel strip; `sub` is the lane's sub-warp, `ll` its lane index inside it.  The per-pixel warp
// reduction then runs once per sub-warp over the full warp with the other lanes neutralised.
//
// FUSED: the R->L map of the same image pair comes out of the same cross terms (SURVEY.md §8 f2).  C(x, d) serves the L->R
// pixel x AND the R->L pixel x' = x + d, whose candidate -d it is (main.cpp:33,43: the second call swaps the images and mirrors
// the range).  A lane's four candidates at pixel step k lie on the diagonals t = k + 4*lane + m of the (x, x') plane
// (t = x' - x0 - dlo), so the warp keeps the running minimum (NCC: maximum) of 128 live diagonals in registers, 4 per lane: every
// step each lane merges its four keys  key2 = EL2[x] + 256*s  (EL2 = the partner direction's energy/position term for
// candidate x), hands the diagonal it will not touch again to the lane below (one SHFL) and lane 0 retires one finished diagonal
// into a shared-memory tail.  At the end of the row the tail and the 128 live diagonals are merged into the partner's
// partial-key map with RED.MIN / RED.MAX (several strips contribute to one x').  Any candidate count: the walked direction's
// groups are aligned to the TOP of its range (FastJob::dlo0) so that the partner's groups are these groups reversed, the
// candidates below dmin are masked in both maps (MODE 2 / 3).  R = 6, 7 and float operands take MODE 3 where a block holds
// illegal positions of either direction.
// OPF (float operands): the images are general float32 (noise / contrast variants, main.cpp:140-153,191-193), the
// operand rows are rows of the replicate-padded (extended) float images themselves - entering row and leaving row
// of the reference image (lp_row / lp_old) and of the target image (rq_row / rq_old) - and
//   SSD: col += q(l_new, r_new) - q(l_old, r_old) with q = the reference's per-element term (DisparitySSD.cpp:49-51)
//        (int)round(f32((l - r)^2)): FSUB, FMUL (separately rounded, never fused), FADD.RZ +0.5, FADD.RZ +2^23 - the
//        mantissa of the last sum IS floor(q + 0.5) = round-half-away(q) for q < 2^23 - 1, so the column sums are
//        exact int32 sums of the bit patterns (the 2^23 biases cancel in new - old): ONE IADD3 per unit.
//        key = 128 * SSD + position (no energy terms); illegal positions take the explicit selects of MODE 3.
//   NCC: col += l_new*r_new - l_old*r_old in float32 (two FFMA); key from v = C * RS[pos] shifted by 3*magic into
//        the binade [2*magic, 4*magic) because C may be negative for float images.
// The host only takes this path when the value range of the two images keeps every term inside those bounds.
__device__ __forceinline__ int ssd_q_bits(float a, float b) {
    const float d = __fsub_rn(a, b);
    const float q = __fmul_rn(d, d);
    return __float_as_int(__fadd_rz(__fadd_rz(q, 0.5f), 8388608.0f));
}
constexpr uint32_t FKEY_MUL_F32 = 1u << FKEY_BITS;     // OPF SSD keys: 128 * cost + position

template <int R, int K, int PAR, int MODE, int COST, int HS, bool FUSED = false, bool OPF = false>
__device__ __forceinline__ void fast_row(int (&col)[FM][RowShape<R, K>::NC], const int* __restrict__ lp_row,
                                         const int* __restrict__ rq_row, const int* __restrict__ e2_row,
                                         int32_t* __restrict__ out_row, int mmin, int mmax, uint32_t lane_or, int ll, int sub, int cbase,
                                         int cols, float magic, const int* __restrict__ el_row = nullptr,
                                         uint32_t* __restrict__ tail = nullptr, uint32_t* __restrict__ part2_row = nullptr,
                                         int x2base = 0, const int* __restrict__ lp_old = nullptr, const int* __restrict__ rq_old = nullptr) {
    using S = RowShape<R, K>;
    constexpr bool NCC = (COST == STEREO_COST_NCORR);
    constexpr bool BIASED = NCC && !OPF && (R <= NCC_BIAS_MAX_R);
    // (one-strip fused kernels lose with it: 8 bytes spilled, 4K/256 pairs 2.33 -> 2.40 ms; unfused 3.04 -> 2.87, two-strip fused 0.60 -> 0.59)
    constexpr bool NCC_CHAIN = NCC && SB_NCC_CHAIN && (!FUSED || HS == 2);
    constexpr uint32_t KEYMUL = OPF ? FKEY_MUL_F32 : uint32_t(2 << FKEY_BITS);
    int lpv[S::NC4];               // packed: s16x2 (new, old) of the reference image;  OPF: the entering row (float bits)
    int rqv[S::NQ4];               // packed: u8x4 of the target image;                 OPF: the entering row
    int lov[OPF ? S::NC4 : 1];     // OPF: the leaving rows
    int rov[OPF ? S::NQ4 : 1];
    // Packed operands are fetched four columns at a time, two quads ahead of their use (update below), not all at the start of
    // the row: with every operand word of the row live next to the column sums, ptxas split the column sums' live ranges and
    // copied them back into place every row (about 2 moves per pixel step of the fused 4K/256 kernel, 250 -> 233 registers).
    auto fetch_lp = [&](int i) {
        const int4 v = lds128(lp_row + 4 * i);
        lpv[4 * i] = v.x; lpv[4 * i + 1] = v.y; lpv[4 * i + 2] = v.z; lpv[4 * i + 3] = v.w;
    };
    auto fetch_rq = [&](int i) {
        const int4 v = lds128(rq_row + 4 * i);
        rqv[4 * i] = v.x; rqv[4 * i + 1] = v.y; rqv[4 * i + 2] = v.z; rqv[4 * i + 3] = v.w;
    };
    if (!OPF) {
#pragma unroll
        for (int i = 0; i < 2; ++i) { fetch_lp(i); fetch_rq(i); }
    }
    // OPF: operands are fetched four columns at a time right before their first use (twice the operand words of the
    // packed path would not fit next to the column sums)
    auto fetch4 = [&](int (&dst)[OPF ? S::NC4 : 1], const int* row, int i) {
        const int4 v = lds128(row + 4 * i);
        dst[OPF ? 4 * i : 0] = v.x; dst[OPF ? 4 * i + 1 : 0] = v.y; dst[OPF ? 4 * i + 2 : 0] = v.z; dst[OPF ? 4 * i + 3 : 0] = v.w;
    };
    auto fetch4q = [&](int (&dst)[OPF ? S::NQ4 : 1], const int* row, int i) {
        const int4 v = lds128(row + 4 * i);
        dst[OPF ? 4 * i : 0] = v.x; dst[OPF ? 4 * i + 1 : 0] = v.y; dst[OPF ? 4 * i + 2 : 0] = v.z; dst[OPF ? 4 * i + 3 : 0] = v.w;
    };
    auto update = [&](int c) {
        if (OPF) {
            if ((c & 3) == 0) {
                {
                    const int4 v = lds128(lp_row + c);
                    lpv[c] = v.x; lpv[c + 1] = v.y; lpv[c + 2] = v.z; lpv[c + 3] = v.w;
                }
                if (MODE != 0) fetch4(lov, lp_old, c / 4);
                if (c == 0) {
                    const int4 v = lds128(rq_row);
                    rqv[0] = v.x; rqv[1] = v.y; rqv[2] = v.z; rqv[3] = v.w;
                    if (MODE != 0) fetch4q(rov, rq_old, 0);
                }
                if (c + 4 < S::NQ4) {
                    const int4 v = lds128(rq_row + c + 4);
                    rqv[c + 4] = v.x; rqv[c + 5] = v.y; rqv[c + 6] = v.z; rqv[c + 7] = v.w;
                    if (MODE != 0) fetch4q(rov, rq_old, c / 4 + 1);
                }
            }
#pragma unroll
            for (int m = 0; m < FM; ++m) {
                if (!NCC) {
                    const int qn = ssd_q_bits(__int_as_float(lpv[c]), __int_as_float(rqv[c + m]));
                    if (MODE == 0) col[m][c] += qn - NCC_FLOAT_BIAS;      // warm-up: entering row only (remove its 2^23 bias)
                    else col[m][c] += qn - ssd_q_bits(__int_as_float(lov[OPF ? c : 0]), __int_as_float(rov[OPF ? c + m : 0]));
                } else {
                    float v = __fmaf_rn(__int_as_float(lpv[c]), __int_as_float(rqv[c + m]), __int_as_float(col[m][c]));
                    if (MODE != 0) v = __fmaf_rn(-__int_as_float(lov[OPF ? c : 0]), __int_as_float(rov[OPF ? c + m : 0]), v);
                    col[m][c] = __float_as_int(v);
                }
            }
            return;
        }
        if ((c & 3) == 0) {           // column c uses lpv[c] and rqv[c .. c + 3]
            if (c + 8 < S::NC4) fetch_lp(c / 4 + 2);
            if (c + 8 < S::NQ4) fetch_rq(c / 4 + 2);
        }
        const int a = (MODE == 0) ? (lpv[c] & 0xFFFF) : lpv[c];      // warm-up: entering row only
#pragma unroll
        for (int m = 0; m < FM; ++m)
            col[m][c] = PAR ? dp2a_hi(a, unsigned(rqv[c + m]), col[m][c]) : dp2a_lo(a, unsigned(rqv[c + m]), col[m][c]);
    };
    if (MODE == 0) {
#pragma unroll
        for (int c = 0; c < S::NC; ++c) update(c);
        return;
    }
    int e2v[S::NE4];
    // likewise the energy / position words, one quad ahead (step k reads e2v[k .. k + 3]); MODE 3 and the fused NCC
    // kernels derive per-position masks / scales from the whole row up front, and the float-operand kernels (which fetch
    // their operands per quad anyway) spill more with it (R = 7 NCC: 144 -> 160 bytes)
    constexpr bool E2LAZY = !OPF && MODE != 3 && !(FUSED && NCC);
    auto fetch_e2 = [&](int i) {
        const int4 v = lds128(e2_row + 4 * i);
        e2v[4 * i] = v.x; e2v[4 * i + 1] = v.y; e2v[4 * i + 2] = v.z; e2v[4 * i + 3] = v.w;
    };
#pragma unroll
    for (int i = 0; i < (E2LAZY ? 1 : S::NE4 / 4); ++i) fetch_e2(i);
    // MODE 3: the selects are turned into masks once per row - per position (K + 3 of them, each used by up to four
    // candidates) and per m - so that a candidate pays ONE three-input LOP3: key | inv[k + m] | mmask[m] (SSD: all-ones =
    // KEY_INVALID loses every min) or key & ok[k + m] & mmask[m] (NCC: 0 = NCC_KEY_NONE loses every max).
    uint32_t pmask[MODE == 3 ? S::NE : 1];
    uint32_t mmask[MODE == 3 ? FM : 1];
    if (MODE == 3) {
#pragma unroll
        for (int p = 0; p < S::NE; ++p) {
            if (!NCC) pmask[MODE == 3 ? p : 0] = uint32_t(e2v[p]) == KEY_INVALID ? KEY_INVALID : 0u;
            else pmask[MODE == 3 ? p : 0] = unsigned(cbase + p) < unsigned(cols) ? 0xFFFFFFFFu : 0u;
        }
#pragma unroll
        for (int m = 0; m < FM; ++m) {
            const bool out = m > mmax || m < mmin;
            mmask[MODE == 3 ? m : 0] = NCC ? (out ? 0u : 0xFFFFFFFFu) : (out ? KEY_INVALID : 0u);
        }
    }
    int s[FM];                   // horizontal window sums: int (packed, OPF SSD) or float bits (OPF NCC)
    int sbias = 0;
    // opaque to the compiler: a literal would be re-associated out of the running sums and re-added per use
    if (BIASED) asm("mov.b32 %0, 0x4B000000;" : "=r"(sbias));
#pragma unroll
    for (int m = 0; m < FM; ++m) s[m] = sbias;
    constexpr bool FSUM = OPF && NCC;           // float running sums
#pragma unroll
    for (int c = 0; c < 2 * R; ++c) {
        update(c);
#pragma unroll
        for (int m = 0; m < FM; ++m) {
            if (FSUM) s[m] = __float_as_int(__fadd_rn(__int_as_float(s[m]), __int_as_float(col[m][c])));
            else s[m] += col[m][c];
        }
    }
    uint32_t res[4];
    uint32_t acc[FM];            // FUSED: running minima of the diagonals k + 4*ll + m
    int elv[4];
    uint32_t einv[4] = {0u, 0u, 0u, 0u};
    uint32_t ret4[4] = {0u, 0u, 0u, 0u};
    if (FUSED) {
#pragma unroll
        for (int m = 0; m < FM; ++m) acc[m] = NCC ? NCC_KEY_NONE : KEY_INVALID;      // running minima (SSD) / maxima (NCC)
    }
    // SB_DIAG_MIN3: the keys of slots 3 and 1 wait one step - by then their diagonals sit in slots 2 and 0 and take them
    // together with that step's key
    constexpr bool DM3 = FUSED && SB_DIAG_MIN3 && FM == 4;
    uint32_t held3 = NCC ? NCC_KEY_NONE : KEY_INVALID, held1 = held3;
    constexpr int LSF = 32 / HS;                                          // lanes per strip
    const uint32_t top_or = (FUSED && ll == LSF - 1) ? KEY_INVALID : 0u;  // the top lane of a strip opens a fresh diagonal every step
    // FUSED NCC.  Both maps order candidates by C * rs with rs = 1/sqrt(energy of the OTHER image's window): the own pixel
    // x by rs_R[pos] (e2v), the partner pixel x' = pos by rs_L[x] (elv, the partner direction's RS row).  The fixed-point
    // scale of a key must be common to all candidates of ONE pixel and bound their scores: C * rs_R[pos] <= sqrt(EL(x)) =
    // 1 / rs_L[x] and C * rs_L[x] <= sqrt(ER(pos)) = 1 / rs_R[pos] (Cauchy-Schwarz), so the scale of either map is a power of
    // two read off the exponent of the OTHER map's rs - per PIXEL (the unfused kernels share one scale per strip row, which
    // costs mantissa bits where a dark window sits next to a bright one): 2^(127 - E) or 2^(128 - E) > 1/rs for rs = 2^(E-127) * 1.m.
    // rs = 0 (empty or illegal window) gives the scale inf, every key of that pixel then has value bits 0 and the position
    // bits alone decide - the first candidate, which is what an all-zero score row gives the oracle.
    // (the mantissa add carries into the exponent when rs is at least 2^-19 above a power of two: then 2^(127 - E) already
    // exceeds 1/rs by the slack the rounding of the sums needs, one more key bit than 2^(128 - E))
    auto scale_of = [](int rs_bits) -> float { return __int_as_float(0x7F800000 - ((rs_bits + 0x007FFFF0) & 0x7F800000)); };
    float own_scale[4];                                   // FUSED NCC: scale of the pixels k .. k+3
    float pos_scale[FUSED && NCC ? S::NE : 1];            // FUSED NCC: scale of the partner pixels (positions) of this lane
    const uint32_t lane_or2 = (uint32_t(FGROUP - 32 / HS * FM + FM * ll) << 2) | 3u;   // partner: reversed index of candidate (m = 0) in ITS group
    if (FUSED && NCC) {
#pragma unroll
        for (int p = 0; p < S::NE; ++p) pos_scale[FUSED && NCC ? p : 0] = scale_of(e2v[p]);
    }
#pragma unroll
    for (int k = 0; k < K; ++k) {                 // [pixel-loop-begin] (tests/test_capi.py checks that nothing spills in here)
        update(k + 2 * R);
        if (E2LAZY && (k & 3) == 0 && k + 4 < S::NE4) fetch_e2(k / 4 + 1);
        if (FUSED && (k & 3) == 0) {
            const int4 v = lds128(el_row + k);
            elv[0] = v.x; elv[1] = v.y; elv[2] = v.z; elv[3] = v.w;
            // a lane outside [dmin, dmax] contributes to neither map; for R <= 5 the partner's key of such a lane loses
            // through its energy term alone (KEY_INVALID - 256*C stays above every valid key), one OR per pixel
            if (MODE == 2 && R <= FFREE_MASK_R && !OPF && !NCC) {
#pragma unroll
                for (int i = 0; i < 4; ++i) elv[i] = int(uint32_t(elv[i]) | lane_or);
            }
            if (MODE == 3 && !NCC) {      // pixels the partner cannot centre a window on: one mask per pixel, shared by its four candidates
#pragma unroll
                for (int i = 0; i < 4; ++i) einv[i] = uint32_t(elv[i]) == KEY_INVALID ? KEY_INVALID : 0u;
            }
            if (NCC) {
#pragma unroll
                for (int i = 0; i < 4; ++i) own_scale[i] = scale_of(elv[i]);
            }
        }
        uint32_t key[FM];
        uint32_t key2[FM];       // (DM3: the partner keys of slots 1 and 3, held for the next step)
#pragma unroll
        for (int m = 0; m < FM; ++m) {
            if (FSUM) {
                float t = __fadd_rn(__int_as_float(s[m]), __int_as_float(col[m][k + 2 * R]));
                if (k > 0) t = __fsub_rn(t, __int_as_float(col[m][k - 1]));
                s[m] = __float_as_int(t);
            } else {
                s[m] = s[m] + col[m][k + 2 * R] - (k > 0 ? col[m][k - 1] : 0);
            }
            if (!NCC) {
                // packed: s = -C (the packed operand carries -l): key = BIAS + 128*(ER - 2C) + position; OPF: s = SSD,
                // key = 128*SSD + position.
                // literal multiplier: ptxas emits the immediate-form IMAD / LEA (2 register reads; the
                // register file delivers ~2 operands per cycle per SMSP, tools/microbench/rf.cu)
                uint32_t kv;
                // (shift-add variants of either key were measured on the fused 4K/256 kernel: 3.51 .. 3.69 ms against 3.57 ms,
                // i.e. inside the spread different register allocations of the same code produce - profiles/r2_hot_variants.md)
                if (!OPF && ((FUSED ? SB_KEY_LEA_FUSED : SB_KEY_LEA_MASK) & (1 << m))) {      // shift-add on the ALU pipe
                    asm("{.reg .b32 t; shl.b32 t, %1, 8; add.s32 %0, t, %2;}" : "=r"(kv) : "r"(s[m]), "r"(e2v[k + m]));
                } else {                                // IMAD (immediate) on the FMA-heavy pipe
                    kv = uint32_t(e2v[k + m]) + uint32_t(s[m]) * KEYMUL;
                }
                if (MODE == 3) kv = kv | pmask[MODE == 3 ? k + m : 0] | mmask[MODE == 3 ? m : 0];
                key[m] = kv;
                if (FUSED) {
                    // the partner direction's key of the same cross term: BIAS + 128*(EL(x) - 2C) + x; pixels x beyond its
                    // legal centres (x > cols-1+R) carry EL2 = KEY_INVALID and lose like illegal search positions do (R <= 5;
                    // wider windows and float operands take the explicit selects of MODE 3 in the blocks that hold such pixels)
                    uint32_t k2;
                    if (!OPF && (SB_KEY2_LEA & (1 << m))) asm("{.reg .b32 t; shl.b32 t, %1, 8; add.s32 %0, t, %2;}" : "=r"(k2) : "r"(s[m]), "r"(elv[k & 3]));
                    else k2 = uint32_t(elv[k & 3]) + uint32_t(s[m]) * KEYMUL;
                    if (MODE == 3) k2 = k2 | einv[k & 3] | mmask[MODE == 3 ? m : 0];
                    if (MODE == 2 && (R > FFREE_MASK_R || OPF)) k2 |= lane_or;
                    if (!DM3) acc[m] = min(acc[m], k2);
                    else if (m == 2) acc[2] = min(min(acc[2], held3), k2);
                    else if (m == 0) acc[0] = min(min(acc[0], held1), k2);
                    else key2[m] = k2;
                }
            } else {
                const float rs = __int_as_float(e2v[k + m]);
                const float mg = FUSED ? own_scale[k & 3] : magic;
                // BIASED: s is the float 2^23 + C, so C*rs + magic = fma(s, rs, magic - 2^23*rs); the addend is exact
                // (Sterbenz / common-ulp argument: 2^23*rs >= 2990 > magic/2 for R <= 5), i.e. ONE rounding (the per-pixel
                // scales of fused launches may be twice as large: the addend then rounds, by at most half a key unit)
                // OPF: `magic` arrives as 3 * 2^e (C may be negative): r lies in [2*2^e, 4*2^e)
                // fused pairs: both maps need C itself - one exact FADD (2^23 + C is a float, C < 2^23) shared by their two FFMAs
                // instead of one addend FFMA per map
                constexpr bool UNBIAS = BIASED && FUSED && SB_NCC_UNBIAS;
                const float cf = UNBIAS ? __fadd_rn(__int_as_float(s[m]), -8388608.0f)
                                        : (BIASED ? 0.f : (OPF ? __int_as_float(s[m]) : __int2float_rn(s[m])));
                const float r = (BIASED && !UNBIAS) ? __fmaf_rn(__int_as_float(s[m]), rs, __fmaf_rn(rs, -8388608.0f, mg)) : __fmaf_rn(cf, rs, mg);
                // lane_or carries ((127 - 4*lane) << 2) | 3: reversed position of the lane's first candidate
                // CHAIN (rows without explicit masks): the candidate's own two position bits join in the maximum below (add-then-max
                // is ONE instruction with the addend as an immediate; four distinct per-candidate constants would be four more
                // live registers, or an extra add each)
                uint32_t kv = (uint32_t(__float_as_int(r)) << NCC_KEY_SHIFT) + (NCC_CHAIN && MODE != 3 ? lane_or : lane_or - 4u * m);
                if (MODE == 3) kv = kv & pmask[MODE == 3 ? k + m : 0] & mmask[MODE == 3 ? m : 0];
                key[m] = kv;
                if (FUSED) {
                    // the partner's key of the same cross term: its candidate is THIS pixel (rs_L[x] = elv), its scale the one of
                    // position k + m, its candidate index inside its group runs against this lane's (d' = -d)
                    const float rs2 = __int_as_float(elv[k & 3]), mg2 = pos_scale[FUSED && NCC ? k + m : 0];
                    const float r2 = (BIASED && !UNBIAS) ? __fmaf_rn(__int_as_float(s[m]), rs2, __fmaf_rn(rs2, -8388608.0f, mg2)) : __fmaf_rn(cf, rs2, mg2);
                    uint32_t k2 = (uint32_t(__float_as_int(r2)) << NCC_KEY_SHIFT) + (lane_or2 + 4u * m);
                    if (MODE == 3) k2 = k2 & mmask[MODE == 3 ? m : 0];
                    if (MODE == 2) k2 = mmax < 0 ? NCC_KEY_NONE : k2;
                    if (!DM3) acc[m] = max(acc[m], k2);
                    else if (m == 2) acc[2] = max(max(acc[2], held3), k2);
                    else if (m == 0) acc[0] = max(max(acc[0], held1), k2);
                    else key2[m] = k2;
                }
            }
        }
        uint32_t best;
        if (!NCC) {
            best = min(min(key[0], key[1]), min(key[2], key[3]));
            if (MODE == 2) best |= lane_or;
        } else {
            if (NCC_CHAIN && MODE != 3) {
                best = key[0];
#pragma unroll
                for (int m = 1; m < FM; ++m) best = max(best, key[m] - 4u * m);
            } else {
                best = max(max(key[0], key[1]), max(key[2], key[3]));
            }
            if (MODE == 2) best = mmax < 0 ? NCC_KEY_NONE : best;
        }
        if (HS == 1) {
            res[k & 3] = NCC ? __reduce_max_sync(0xffffffffu, best) : __reduce_min_sync(0xffffffffu, best);
        } else {
            uint32_t mine = 0;
#pragma unroll
            for (int h = 0; h < HS; ++h) {
                const uint32_t v = (sub == h) ? best : (NCC ? NCC_KEY_NONE : KEY_INVALID);
                const uint32_t r = NCC ? __reduce_max_sync(0xffffffffu, v) : __reduce_min_sync(0xffffffffu, v);
                if (sub == h) mine = r;
            }
            res[k & 3] = mine;
        }
        if ((k & 3) == 3 && ll == 0)
            *reinterpret_cast<uint4*>(out_row + k - 3) = make_uint4(res[0], res[1], res[2], res[3]);
        if (FUSED) {
            // diagonal k + 4*ll is complete for this lane: it moves to the lane below (lane 0: into the tail);
            // the lane's other three diagonals move down one slot and the slot on top takes over lane ll+1's
            const uint32_t done = acc[0];
            uint32_t in;
            // (a fresh diagonal starts at "no candidate": all ones for the SSD minima, zero for the NCC maxima)
            // SSD: lane 0's retired diagonals go to the tail four at a time (one STS.128 per four pixels instead of four STS:
            // 3.58 -> 3.49 ms per four 4K/256 pairs; the NCC kernels have no registers to spare for it)
            constexpr bool TB = SB_TAIL_BATCH && !NCC;
            if (TB) ret4[k & 3] = done;
            uint32_t* const tl = tail + (HS == 1 ? 0 : 32 * sub);
            in = HS == 1 ? __shfl_down_sync(0xffffffffu, done, 1) : __shfl_down_sync(0xffffffffu, done, 1, LSF);
            if (TB) { if ((k & 3) == 3 && ll == 0) *reinterpret_cast<uint4*>(tl + k - 3) = make_uint4(ret4[0], ret4[1], ret4[2], ret4[3]); }
            else if (ll == 0) tl[k] = done;
            in = NCC ? (in & ~top_or) : (in | top_or);
            acc[0] = acc[1]; acc[1] = acc[2]; acc[2] = acc[3]; acc[3] = in;
            if (DM3) { held3 = key2[3]; held1 = key2[1]; }
        }
    }                                             // [pixel-loop-end]
    if (DM3) {        // the last step's held keys: their diagonals now sit in slots 2 and 0
        acc[2] = NCC ? max(acc[2], held3) : min(acc[2], held3);
        acc[0] = NCC ? max(acc[0], held1) : min(acc[0], held1);
    }
    if (FUSED) {
        // live diagonals: acc[m] <-> t = K + 4*ll + m <-> partner pixel x' = x2base + t; tail[t] <-> t < K
        __syncwarp();
        // Unconditional REDs: a lane whose partner pixel lies outside the image sends the neutral key instead of skipping the
        // merge (its address may fall into a neighbouring row or into the FUSED_PART_PAD words either side of the partner's
        // map, where a neutral key changes nothing).  As `if (in range) atomicMin(...)` every one of the five merges of a row
        // became its own divergence region (BSSY / BRA / R2UR x2 / REDG / BSYNC - ptxas does the same to a predicated `red`), and
        // the row epilogue took 20 % of the kernel's stall samples with 9 % of its instructions.
        auto merge = [&](uint32_t* row, int x, uint32_t v, bool ok) {
            const uint32_t vv = ok ? v : (NCC ? NCC_KEY_NONE : KEY_INVALID);
            if (NCC) atomicMax(row + x, vv); else atomicMin(row + x, vv);
        };
        if (HS == 1) {
            const uint32_t tv = (ll < K) ? tail[ll] : (NCC ? NCC_KEY_NONE : KEY_INVALID);
            const int xt = x2base + ll;
            merge(part2_row, xt, tv, unsigned(xt) < unsigned(cols));          // (tv is already neutral for ll >= K)
        } else {
            // every half-warp merges the tail of its own strip, one entry per lane (K <= lanes per strip)
            static_assert(!FUSED || HS == 1 || K <= 32 / HS, "two-strip warps: a strip's tail fits its half-warp");
            const uint32_t tv = (ll < K) ? tail[32 * sub + ll] : (NCC ? NCC_KEY_NONE : KEY_INVALID);
            const int xt = x2base + ll;
            merge(part2_row, xt, tv, unsigned(xt) < unsigned(cols));
        }
#pragma unroll
        for (int m = 0; m < FM; ++m) {
            const int xa = x2base + K + FM * ll + m;
            merge(part2_row, xa, acc[m], unsigned(xa) < unsigned(cols));
        }
        __syncwarp();             // the next row overwrites the tail
    }
}

// GEN (fused kernels only): false = every block of the launch is MODE 1 (whole disparity groups, R <= 5: the masks come
// free through the keys) - the kernel the 4K/256 and 1080p/128 configurations run, kept free of the other row flavours
// so that their code does not weigh on its register allocation; true = any candidate count, any radius.
// OPF: float operand rows (see fast_row): LP / RQ point at the extended float images, one row per image row; each
// stage stages the entering AND the leaving rows of both images.
template <int R, int K, int NW, int COST, int HS, bool FUSED = false, bool GEN = true, bool OPF = false>
__global__ void __launch_bounds__(NW * 32, 1) fast_cost_kernel(const __grid_constant__ FastKernelParams P) {
    static_assert(!FUSED || (K % 4 == 0 && K <= 32), "fused pair kernel: strips of 4k <= 32 pixels");
    static_assert(!FUSED || COST == STEREO_COST_SSD || !OPF, "fused NCC pairs: packed operands only");
    static_assert(!OPF || (HS == 1 && GEN && K % 4 == 0), "float operands: one strip per warp, general masks");
    constexpr bool NCC = (COST == STEREO_COST_NCORR);
    constexpr int LS = 32 / HS;                 // lanes per strip
    constexpr int DG = FM * LS;                 // disparities per strip and warp
    using S = RowShape<R, K>;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const FastGeom& g = P.g;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int sub = lane / LS, ll = lane % LS;
    const int nst = g.nst;
    constexpr int nw = NW;

    // stage layout (words): [lp (OPF: entering rows)] [OPF: lp leaving rows] [rq (OPF: entering)] [OPF: rq leaving] [e2] [FUSED: el]
    constexpr int NOP = OPF ? 2 : 1;
    const int lp_stage = FRPS * g.lpw, rq_stage = (OPF ? FRPS : FRPS / 2) * g.rqw, e2_stage = FRPS * g.e2w;
    const int el_stage = FUSED ? FRPS * g.elw : 0;
    const int rq_base = NOP * lp_stage, e2_base = NOP * (lp_stage + rq_stage), el_base = e2_base + e2_stage;
    const int stage_words = el_base + el_stage;
    int* smem = reinterpret_cast<int*>(smem_raw);
    unsigned long long* bars = reinterpret_cast<unsigned long long*>(smem_raw + size_t(nst) * stage_words * 4);
    const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + FNST_MAX);
    int* pcache = reinterpret_cast<int*>(bars + 2 * FNST_MAX) + warp * 8;                    // the warp's producer cache (below)
    uint32_t* tail = reinterpret_cast<uint32_t*>(bars + 2 * FNST_MAX) + NW * 8 + warp * (32 * HS);     // FUSED: 32 words per strip of the warp

    if (tid == 0) {
        for (int i = 0; i < nst; ++i) { mbar_init(full0 + 8 * i, nw); mbar_init(empty0 + 8 * i, nw); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    // ---- this CTA's share of the (job, tile, row) space ----------------------------------------------
    // Linear index = tile * nrl + row with nrl >= nrows (rows nrows..nrl-1 of a tile are padding: when the launch has fewer
    // tiles than SMs, nrl is a multiple of L and every CTA's share lies inside one tile).
    long long lin_begin = (long long)blockIdx.x * g.L;
    long long lin_end = lin_begin + g.L;
    if (lin_end > g.total) lin_end = g.total;
    if (g.sched == 1) { lin_begin = blockIdx.x; lin_end = (long long)g.ntiles * g.nbands; }     // item indices, stride gridDim.x
    if (lin_begin >= lin_end) return;
    const int w = 2 * R + 1;
    const int tpj = g.tilesX * g.gblocks;        // tiles per job
    const int npair = FUSED ? g.npairs : 0;      // the partner of job jb is job jb + npair
    // next non-empty segment [r0, r1) of one tile at or after `lin`; false when the share is exhausted
    auto next_segment = [&](long long& lin, int& tile, int& r0, int& r1) -> bool {
        if (g.sched == 1) {
            if (lin >= lin_end) return false;
            const int band = int(lin / g.ntiles);
            tile = int(lin - (long long)band * g.ntiles);
            r0 = band * int(g.L);
            r1 = min(r0 + int(g.L), g.nrows);
            lin += gridDim.x;
            return true;
        }
        while (lin < lin_end) {
            tile = int(lin / g.nrl);
            r0 = int(lin % g.nrl);
            const long long rem = lin_end - lin;
            const int e = (rem > g.nrl - r0) ? g.nrl : r0 + int(rem);
            lin += e - r0;
            r1 = e < g.nrows ? e : g.nrows;
            if (r0 < r1) return true;
        }
        return false;
    };

    // producer: EVERY warp iterates the same stage sequence, nst-2 stages ahead, warp-uniformly (all lanes
    // wait on the empty barrier), and its lane 0 issues the warp's share of the stage's row copies (row r of
    // a stage belongs to warp r mod nw).
    long long p_lin = lin_begin;   // start of the producer's next segment
    int p_sj = 0, p_sj_end = -1;   // stage range of the producer's segment
    int p_tile = 0;
    int p_slot = 0, p_round = 0;   // ring position of the next load
    // PCACHE (two-strip warps): the tile decomposition (two integer divisions) and the row-independent offsets are worked out
    // once per segment, by lane 0, into four words of shared memory, and a stage reads them back: 720p/64 launches 0.485 ->
    // 0.432 ms per 16 pairs.  The one-strip kernels keep redoing them per stage in all lanes (measured: 4K/256 3.23 ms
    // against 3.31 with the cache - the LDS -> indexed LDC -> address chain of lane 0 stalls the warp longer than the divisions).
    constexpr bool PCACHE = (HS == 2);
    auto tile_offsets = [&](int tile, int& jb, int& p0, int& q0, int& q20) {
        jb = tile / tpj;
        const int t2 = tile - jb * tpj;
        const FastJob& job = P.job[jb];
        const int xt = t2 % g.tilesX, gb = t2 / g.tilesX;
        p0 = xt * g.spc * K;
        q0 = p0 + job.dlo0 + g.dg * gb * g.gc + g.R + job.qoff;
        q20 = p0 + job.dlo0 + g.dg * gb * g.gc + job.eoff;
    };
    auto producer_issue = [&]() -> bool {     // returns false when nothing is left
        if (p_sj > p_sj_end) {
            int r0, r1;
            if (!next_segment(p_lin, p_tile, r0, r1)) return false;
            const int js = g.rb + r0 - w - g.base_y, je = g.rb + r1 - g.base_y;
            p_sj = js / FRPS; p_sj_end = (je - 1) / FRPS;
            if (PCACHE && lane == 0) {
                int jb, p0, q0, q20;
                tile_offsets(p_tile, jb, p0, q0, q20);
                *reinterpret_cast<int4*>(pcache) = make_int4(jb, p0, q0, q20);
            }
        }
        const int slot = p_slot;
        if (p_round > 0) mbar_wait(empty0 + 8 * slot, (p_round - 1) & 1);
        const int j0 = p_sj * FRPS;
        int jb = 0, p0 = 0, q0 = 0, q20 = 0;
        if (!PCACHE) tile_offsets(p_tile, jb, p0, q0, q20);
        if (lane == 0) {
            if (PCACHE) { const int4 pc = *reinterpret_cast<const int4*>(pcache); jb = pc.x; p0 = pc.y; q0 = pc.z; q20 = pc.w; }
            const FastJob& job = P.job[jb];
            const int32_t* e2src = NCC ? reinterpret_cast<const int32_t*>(job.RS) : job.E2;
            const uint32_t bar = full0 + 8 * slot;
            int* st = smem + size_t(slot) * stage_words;
            constexpr int NLP = (FRPS - 1) / NW + 1, NRQ = (FRPS / 2 - 1) / NW + 1;       // copies per warp, upper bounds
            uint32_t mine = 0;
#pragma unroll
            for (int i = 0; i < NLP; ++i)
                if (warp + i * nw < FRPS) mine += uint32_t(NOP * g.lpw + (OPF ? 2 * g.rqw : 0) + g.e2w + (FUSED ? g.elw : 0)) * 4u;
            if (!OPF) {
#pragma unroll
                for (int i = 0; i < NRQ; ++i) if (warp + i * nw < FRPS / 2) mine += uint32_t(g.rqw) * 4u;
            }
            if (mine) mbar_expect_tx(bar, mine); else mbar_arrive(bar);
#pragma unroll
            for (int i = 0; i < NLP; ++i) {
                const int r = warp + i * nw;
                if (r < FRPS) {
                    if (!OPF) {
                        tma_load_1d(smem_u32(st + r * g.lpw), job.LP + size_t(j0 + r) * g.lp_pitch + p0, uint32_t(g.lpw) * 4u, bar);
                    } else {
                        // image row of operand row j: leaving = array row j, entering = array row j + 2R + 1
                        tma_load_1d(smem_u32(st + r * g.lpw), job.LP + size_t(j0 + r + w) * g.lp_pitch + p0, uint32_t(g.lpw) * 4u, bar);
                        tma_load_1d(smem_u32(st + lp_stage + r * g.lpw), job.LP + size_t(j0 + r) * g.lp_pitch + p0, uint32_t(g.lpw) * 4u, bar);
                        tma_load_1d(smem_u32(st + rq_base + r * g.rqw), job.RQ + size_t(j0 + r + w) * g.rq_pitch + q0, uint32_t(g.rqw) * 4u, bar);
                        tma_load_1d(smem_u32(st + rq_base + rq_stage + r * g.rqw), job.RQ + size_t(j0 + r) * g.rq_pitch + q0, uint32_t(g.rqw) * 4u, bar);
                    }
                    tma_load_1d(smem_u32(st + e2_base + r * g.e2w), e2src + size_t(j0 + r) * g.e2_pitch + q20, uint32_t(g.e2w) * 4u, bar);
                    if (FUSED)      // the partner's energy rows: E2'[j][x] (NCC: RS'[j][x]), x = pixel column (its eoff is 0)
                        tma_load_1d(smem_u32(st + el_base + r * g.elw),
                                    (NCC ? reinterpret_cast<const int32_t*>(P.job[jb + npair].RS) : P.job[jb + npair].E2) + size_t(j0 + r) * g.e2_pitch + p0,
                                    uint32_t(g.elw) * 4u, bar);
                }
            }
            if (!OPF) {
#pragma unroll
                for (int i = 0; i < NRQ; ++i) {
                    const int r = warp + i * nw;
                    if (r < FRPS / 2)
                        tma_load_1d(smem_u32(st + rq_base + r * g.rqw), job.RQ + size_t(j0 / 2 + r) * g.rq_pitch + q0, uint32_t(g.rqw) * 4u, bar);
                }
            }
        }
        // reconverge here: without it lane 0 runs the following row on its own, up to the first warp
        // reduction, and every row instruction of that stretch issues twice
        __syncwarp();
        ++p_sj;
        if (++p_slot == nst) { p_slot = 0; ++p_round; }
        return true;
    };
    for (int i = 0; i < nst - 2; ++i) if (!producer_issue()) break;

    // ---- consumers -----------------------------------------------------------------------------------
    int c_slot = 0, c_round = 0;    // ring position of the next stage to consume
    long long lin = lin_begin;
    int col[FM][S::NC];
    int tile, r0, r1;
    while (next_segment(lin, tile, r0, r1)) {
        const int jb = tile / tpj, t2 = tile - jb * tpj;
        const FastJob& job = P.job[jb];
        const int xt = t2 % g.tilesX, gb = t2 / g.tilesX;
        const int wstrip = (warp / g.gc) * HS;                          // first strip of this warp inside the tile
        const int strip = xt * g.spc + wstrip + sub;
        const int grp = gb * g.gc + warp % g.gc;
        const int x0 = strip * K;
        const int x0w = (xt * g.spc + wstrip) * K;                       // first pixel of the warp (warp-uniform)
        // warp-uniform: the row code holds warp collectives.  FUSED: strips reach R columns into the right padding,
        // where the partner direction's last candidates are centred.
        const bool active = (x0w < g.cols + ((FUSED && !g.border) ? R : 0)) && (grp < g.G);
        const int y0 = g.rb + r0, y1 = g.rb + r1;
        const int js = y0 - w - g.base_y, je = y1 - g.base_y, jreg = y0 - g.base_y;
        // which flavour of candidate masking this warp's (HS x K pixels x DG disparities) block needs
        const int dlo = job.dlo0 + DG * grp;                              // first disparity of the group
        // (only the disparities of the group that lie inside [dmin, dmax] can name a position)
        bool pos_invalid = (x0w + max(dlo, job.dmin) < job.cmin) || (x0w + HS * K - 1 + min(dlo + DG - 1, job.dmax) > job.cmax);
        if (FUSED) pos_invalid = pos_invalid || (x0w + HS * K - 1 > P.job[jb + npair].cmax);   // pixels the partner cannot centre a window on
        const bool hi_invalid = dlo + DG - 1 > job.dmax, lo_invalid = dlo < job.dmin;
        const bool lane_invalid = hi_invalid || lo_invalid;
        const bool partial_lane = (hi_invalid && (((job.dmax - dlo + 1) % FM) != 0)) || (lo_invalid && (((job.dmin - dlo) % FM) != 0));
        // NCC: an illegal search position carries RS = 0, i.e. the score-0 key of its position; it can only win
        // when every legal candidate scores exactly 0 too, which the merge recognises (winner outside the image
        // -> first legal candidate, cv::minMaxLoc's first maximum).  So NCC never needs the explicit selects
        // for border positions, and SSD only for R > 5.
        // Float operands (OPF): no key headroom and scores may be negative, so illegal positions always take the selects.
        const int mode = (partial_lane || (pos_invalid && (OPF || (!NCC && R > FFREE_MASK_R)))) ? 3 : (lane_invalid ? 2 : 1);
        const int mmin = job.dmin - dlo - FM * ll;                        // mmin <= m <= mmax are inside [dmin, dmax]
        int mmax = job.dmax - dlo - FM * ll;
        if (mmin > FM - 1) mmax = -1;                                     // the whole lane lies below dmin: dead, like one above dmax
        // SSD: OR-mask that invalidates a whole lane; NCC: reversed position of the lane's first candidate
        const uint32_t lane_or = NCC ? (uint32_t(FGROUP - 1 - FM * ll) << 2 | 3u) : (mmax < 0 ? KEY_INVALID : 0u);
        const float* sc_row = (NCC && !FUSED) ? job.SC + size_t(strip) * g.nrows - (g.rb - g.base_y) : nullptr;   // indexed by operand row j
        const int cbase = x0 + dlo + FM * ll;                             // centre column of candidate (k=0, m=0)
        const int lp_off = (wstrip + sub) * K;
        const int rq_off = lp_off + DG * (warp % g.gc) + FM * ll;
        int32_t* part = job.PART + (size_t(grp) * g.nrows) * g.wpart + x0;
        // FUSED: the partner's candidates -d of this group are its group G-1-grp (the groups are aligned to the top of the range)
        uint32_t* part2 = FUSED ? reinterpret_cast<uint32_t*>(P.job[jb + npair].PART) + (size_t(g.G - 1 - grp) * g.nrows) * g.wpart : nullptr;
        const int x2base = x0 + dlo;                                      // partner pixel of diagonal 0
#pragma unroll
        for (int m = 0; m < FM; ++m)
#pragma unroll
            for (int c = 0; c < S::NC; ++c) col[m][c] = 0;

        for (int sj = js / FRPS; sj <= (je - 1) / FRPS; ++sj) {
            producer_issue();
            const int slot = c_slot;
            mbar_wait(full0 + 8 * slot, c_round & 1);
            if (active) {
                const int* st = smem + size_t(slot) * stage_words;
                const int jlo = max(js, sj * FRPS), jhi = min(je, sj * FRPS + FRPS);
                for (int j = jlo; j < jhi; ++j) {
                    const int r = j - sj * FRPS;
                    const int* lp_row = st + r * g.lpw + lp_off;
                    const int* rq_row = st + rq_base + (OPF ? r : (r >> 1)) * g.rqw + rq_off;
                    const int* e2_row = st + e2_base + r * g.e2w + rq_off;
                    int32_t* out_row = part + size_t(j - (g.rb - g.base_y)) * g.wpart;
                    const int par = j & 1;
                    const float magic = (NCC && !FUSED && j >= jreg) ? __ldg(sc_row + j) : 0.f;
#define SB_ROW(P_, M_) fast_row<R, K, P_, M_, COST, HS, false, OPF>(col, lp_row, rq_row, e2_row, out_row, mmin, mmax, lane_or, ll, sub, cbase, g.cols, magic, \
                                                          nullptr, nullptr, nullptr, 0, lp_row + lp_stage, rq_row + rq_stage)
#define SB_ROWF(P_, M_) fast_row<R, K, P_, M_, COST, HS, true, OPF>(col, lp_row, rq_row, e2_row, out_row, mmin, mmax, lane_or, ll, sub, cbase, g.cols, magic, \
                                                          st + el_base + r * g.elw + lp_off, tail, \
                                                          part2 + size_t(j - (g.rb - g.base_y)) * g.wpart, x2base, lp_row + lp_stage, rq_row + rq_stage)
                    if constexpr (OPF) {          // one row per operand row: no byte-pair parity
                        if (j < jreg) SB_ROW(0, 0);
                        else if constexpr (FUSED) { if (mode == 1) SB_ROWF(0, 1); else if (mode == 2) SB_ROWF(0, 2); else SB_ROWF(0, 3); }
                        else { if (mode == 1) SB_ROW(0, 1); else if (mode == 2) SB_ROW(0, 2); else SB_ROW(0, 3); }
                    }
                    else if (j < jreg)  { if (par) SB_ROW(1, 0); else SB_ROW(0, 0); }
                    else if constexpr (FUSED && !GEN) { if (par) SB_ROWF(1, 1); else SB_ROWF(0, 1); }   // the host vouches for mode 1
                    else if constexpr (FUSED) {
                        if (mode == 1)      { if (par) SB_ROWF(1, 1); else SB_ROWF(0, 1); }
                        else if (mode == 2) { if (par) SB_ROWF(1, 2); else SB_ROWF(0, 2); }
                        else                { if (par) SB_ROWF(1, 3); else SB_ROWF(0, 3); }
                    }
                    else if (mode == 1) { if (par) SB_ROW(1, 1); else SB_ROW(0, 1); }
                    else if (mode == 2) { if (par) SB_ROW(1, 2); else SB_ROW(0, 2); }
                    else                { if (par) SB_ROW(1, 3); else SB_ROW(0, 3); }
#undef SB_ROW
#undef SB_ROWF
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(empty0 + 8 * slot);
            if (++c_slot == nst) { c_slot = 0; ++c_round; }
        }
    }
}

typedef void (*fast_kernel_fn)(const FastKernelParams);
// The hot-kernel instantiations live in fast_inst.cu, compiled once per part (SB_PART = 0..15: cost x window
// radius subset x strips per warp) so that the translation units build in parallel; each part exports a
// lookup function.
constexpr int FAST_PARTS = 16;
#define SB_DECL_PART(n) fast_kernel_fn fast_pick_part##n(int R, int hs);
SB_DECL_PART(0) SB_DECL_PART(1) SB_DECL_PART(2) SB_DECL_PART(3) SB_DECL_PART(4) SB_DECL_PART(5) SB_DECL_PART(6) SB_DECL_PART(7)
SB_DECL_PART(8) SB_DECL_PART(9) SB_DECL_PART(10) SB_DECL_PART(11) SB_DECL_PART(12) SB_DECL_PART(13) SB_DECL_PART(14) SB_DECL_PART(15)
#undef SB_DECL_PART
// Fused pair kernels: SSD parts 16..25, NCC parts 38..47 (fast_inst.cu).
constexpr int FAST_FUSED_PARTS = 10;
#define SB_DECL_FPART(n) fast_kernel_fn fast_pick_fused_part##n(int R, int hs, int gen);
SB_DECL_FPART(16) SB_DECL_FPART(17) SB_DECL_FPART(18) SB_DECL_FPART(19) SB_DECL_FPART(20)
SB_DECL_FPART(21) SB_DECL_FPART(22) SB_DECL_FPART(23) SB_DECL_FPART(24) SB_DECL_FPART(25)
SB_DECL_FPART(38) SB_DECL_FPART(39) SB_DECL_FPART(40) SB_DECL_FPART(41) SB_DECL_FPART(42)
SB_DECL_FPART(43) SB_DECL_FPART(44) SB_DECL_FPART(45) SB_DECL_FPART(46) SB_DECL_FPART(47)
#undef SB_DECL_FPART
static inline fast_kernel_fn fast_pick_fused_ncc(int R, int hs) {
    typedef fast_kernel_fn (*part_fn)(int, int, int);
    static const part_fn parts[FAST_FUSED_PARTS] = {fast_pick_fused_part38, fast_pick_fused_part39, fast_pick_fused_part40, fast_pick_fused_part41,
                                                    fast_pick_fused_part42, fast_pick_fused_part43, fast_pick_fused_part44, fast_pick_fused_part45,
                                                    fast_pick_fused_part46, fast_pick_fused_part47};
    for (int i = 0; i < FAST_FUSED_PARTS; ++i)
        if (fast_kernel_fn fn = parts[i](R, hs, 1)) return fn;
    return nullptr;
}
// gen = 0: the launch's blocks are all MODE 1 (fast_fused_all_mode1); 1: any launch
static inline fast_kernel_fn fast_pick_fused(int R, int hs, int gen) {
    typedef fast_kernel_fn (*part_fn)(int, int, int);
    static const part_fn parts[FAST_FUSED_PARTS] = {fast_pick_fused_part16, fast_pick_fused_part17, fast_pick_fused_part18, fast_pick_fused_part19,
                                                    fast_pick_fused_part20, fast_pick_fused_part21, fast_pick_fused_part22, fast_pick_fused_part23,
                                                    fast_pick_fused_part24, fast_pick_fused_part25};
    for (int i = 0; i < FAST_FUSED_PARTS; ++i)
        if (fast_kernel_fn fn = parts[i](R, hs, gen)) return fn;
    return nullptr;
}
// Float-operand kernels: parts 26..37 = kind * 4 + radius subset; kind 0 = SSD, 1 = SSD fused pair, 2 = NCC.
constexpr int FAST_OPF_PARTS = 12;
enum { OPF_SSD = 0, OPF_SSD_FUSED = 1, OPF_NCC = 2 };
#define SB_DECL_OPART(n) fast_kernel_fn fast_pick_opf_part##n(int R, int kind);
SB_DECL_OPART(26) SB_DECL_OPART(27) SB_DECL_OPART(28) SB_DECL_OPART(29) SB_DECL_OPART(30) SB_DECL_OPART(31)
SB_DECL_OPART(32) SB_DECL_OPART(33) SB_DECL_OPART(34) SB_DECL_OPART(35) SB_DECL_OPART(36) SB_DECL_OPART(37)
#undef SB_DECL_OPART
static inline fast_kernel_fn fast_pick_opf(int R, int kind) {
    typedef fast_kernel_fn (*part_fn)(int, int);
    static const part_fn parts[FAST_OPF_PARTS] = {fast_pick_opf_part26, fast_pick_opf_part27, fast_pick_opf_part28, fast_pick_opf_part29,
                                                  fast_pick_opf_part30, fast_pick_opf_part31, fast_pick_opf_part32, fast_pick_opf_part33,
                                                  fast_pick_opf_part34, fast_pick_opf_part35, fast_pick_opf_part36, fast_pick_opf_part37};
    for (int i = 0; i < FAST_OPF_PARTS; ++i)
        if (fast_kernel_fn fn = parts[i](R, kind)) return fn;
    return nullptr;
}
static inline fast_kernel_fn fast_pick(int cost, int R, int hs) {
    typedef fast_kernel_fn (*part_fn)(int, int);
    static const part_fn parts[FAST_PARTS] = {fast_pick_part0, fast_pick_part1, fast_pick_part2, fast_pick_part3,
                                              fast_pick_part4, fast_pick_part5, fast_pick_part6, fast_pick_part7,
                                              fast_pick_part8, fast_pick_part9, fast_pick_part10, fast_pick_part11,
                                              fast_pick_part12, fast_pick_part13, fast_pick_part14, fast_pick_part15};
    for (int i = 0; i < FAST_PARTS; ++i)
        if (fast_kernel_fn fn = parts[i](R, hs | (cost << 8))) return fn;
    return nullptr;
}

} // namespace sb
