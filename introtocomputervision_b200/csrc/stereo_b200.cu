// stereo_b200 — C ABI implementation (context, validation, path selection, staging).
// Kernels: exact.cuh (general float path), fast.cuh (packed u8 path).  sm_100a only.
#include "common.cuh"
#include "exact.cuh"
#include "fast.cuh"
#include "compat.cuh"
#include "imgproc.cuh"
#include "lrcheck.cuh"
#include "speckle.cuh"
#include "sgm.cuh"
#include "prefilter.cuh"
#include "subpixel.cuh"
#include "host_pack.hpp"

#include <atomic>
#include <chrono>
#include <cstdarg>
#include <thread>
#include <new>
#include <initializer_list>
#include <utility>
#include <vector>

namespace sb {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int Arena::reserve(size_t bytes) {
    if (bytes <= cap) return STEREO_OK;
    release();
    size_t want = bytes + (bytes >> 3) + (1u << 20);
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&base), want);
    if (e != cudaSuccess) {
        base = nullptr; cap = 0;
        set_error("cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
        (void)cudaGetLastError();
        return STEREO_ERR_ALLOC;
    }
    cap = want;
    return STEREO_OK;
}

void Arena::release() {
    if (base) cudaFree(base);
    base = nullptr; cap = 0; used = 0;
}

static size_t align256(size_t v) { return (v + 255) & ~size_t(255); }
static int quiesce(stereo_ctx* ctx, cudaStream_t st);

// ---- validation ---------------------------------------------------------------------------------

static int validate(const Problem& p, size_t ref_min_step, size_t tgt_min_step) {
    if (!p.ref.ptr || !p.tgt.ptr || !p.disp.ptr) { set_error("null image/output pointer"); return STEREO_ERR_INVALID_ARG; }
    if (p.rows <= 0 || p.cols <= 0) { set_error("rows/cols must be positive (got %d x %d)", p.rows, p.cols); return STEREO_ERR_INVALID_ARG; }
    if (p.rows > 32768 || p.cols > 32768) { set_error("image larger than 32768 in a dimension"); return STEREO_ERR_UNSUPPORTED; }
    if (p.R < 0 || p.R > 64) { set_error("window_rad must be in [0, 64] (got %d)", p.R); return STEREO_ERR_INVALID_ARG; }
    if (p.cost != STEREO_COST_SSD && p.cost != STEREO_COST_NCORR) { set_error("unknown cost %d", p.cost); return STEREO_ERR_INVALID_ARG; }
    if (p.disp.elem != 1 && p.disp.elem != 2 && p.disp.elem != 4) { set_error("disp_elem_bytes must be 1, 2 or 4"); return STEREO_ERR_INVALID_ARG; }
    if (p.ref.step < ref_min_step || p.tgt.step < tgt_min_step) { set_error("image step smaller than a row"); return STEREO_ERR_INVALID_ARG; }
    if (p.disp.step < size_t(p.cols) * p.disp.elem) { set_error("disp_step smaller than a row"); return STEREO_ERR_INVALID_ARG; }
    if (p.best.ptr && p.best.step < size_t(p.cols) * 4) { set_error("best_step smaller than a row"); return STEREO_ERR_INVALID_ARG; }
    if (p.dmin > p.dmax) { set_error("min_disp (%d) > max_disp (%d)", p.dmin, p.dmax); return STEREO_ERR_INVALID_RANGE; }
    if (p.dmin < -32768 || p.dmax > 32768) { set_error("disparity range outside [-32768, 32768]"); return STEREO_ERR_INVALID_RANGE; }
    if (p.row_begin < 0 || p.row_end > p.rows || p.row_begin >= p.row_end) { set_error("bad row band [%d, %d)", p.row_begin, p.row_end); return STEREO_ERR_INVALID_ARG; }
    if (p.avail_begin < 0 || p.avail_end > p.rows || p.avail_begin > p.row_begin || p.avail_end < p.row_end) {
        set_error("available rows [%d, %d) do not cover the band [%d, %d)", p.avail_begin, p.avail_end, p.row_begin, p.row_end);
        return STEREO_ERR_INVALID_ARG;
    }
    if (p.cost == STEREO_COST_NCORR) {
        // Every pixel needs >= 1 candidate window; the reference would throw inside
        // cv::Mat::operator()(Rect) otherwise (DisparityNCorr.cpp:50-53).
        const int Wp = p.cols + 2 * p.R, w = 2 * p.R + 1;
        // ncand(x) is piecewise linear in x: checking both ends and the clamp knees suffices,
        // checking every column is cheap enough and obviously right.
        for (int x = p.R; x < Wp - p.R; ++x) {
            long s = long(x) + p.dmin - p.R; if (s < 0) s = 0;
            long e = long(x) + p.dmax + 1 + p.R; if (e > Wp) e = Wp;
            if (e - s - w + 1 <= 0) {
                set_error("NCC range [%d, %d] leaves column %d without a candidate", p.dmin, p.dmax, x - p.R);
                return STEREO_ERR_INVALID_RANGE;
            }
        }
    }
    return STEREO_OK;
}

// ---- problems -----------------------------------------------------------------------------------

// One direction: output rows [row_begin, row_end) of a rows x cols image pair whose buffers - addressed from the image's
// row 0 - hold rows [avail_begin, avail_end).
static Problem direction(int cost, PixType type, const void* ref, size_t ref_step, const void* tgt, size_t tgt_step, int rows,
                         int cols, int row_begin, int row_end, int avail_begin, int avail_end, int R, int dmin, int dmax,
                         void* disp, size_t disp_step, int elem, void* best, size_t best_step) {
    return Problem{cost, ImageView{ref, ref_step, type}, ImageView{tgt, tgt_step, type}, rows, cols, row_begin, row_end,
                   avail_begin, avail_end, R, dmin, dmax, OutView{disp, disp_step, elem}, OutView{best, best_step, 4}};
}

// Pair k of np: L->R over [-range, 0] at ps[k], then R->L with the images swapped over [0, +range] at ps[np + k]
// (main.cpp:21-48).  Left-referenced problems first is the order a fused launch takes pairs in (fused_layout).
static void pair_problems(Problem* ps, int np, int k, int cost, PixType type, const void* left, size_t left_step,
                          const void* right, size_t right_step, int rows, int cols, int row_begin, int row_end, int avail_begin,
                          int avail_end, int R, int range, void* disp_left, void* disp_right, size_t disp_step, int elem) {
    ps[k] = direction(cost, type, left, left_step, right, right_step, rows, cols, row_begin, row_end, avail_begin, avail_end, R,
                      -range, 0, disp_left, disp_step, elem, nullptr, 0);
    ps[np + k] = direction(cost, type, right, right_step, left, left_step, rows, cols, row_begin, row_end, avail_begin, avail_end,
                           R, 0, range, disp_right, disp_step, elem, nullptr, 0);
}

// ---- pair options: uniqueness ratio, left-right check (lrcheck.cuh), speckle filter (speckle.cuh), SGM (sgm.cuh) -------

// The uniqueness ratio, the texture threshold, the check and the filter mark removed pixels with -(range + 1), which must
// fit the maps' element type.  (An int8 map of more than 127 disparities already holds wrapped values.)
static int check_lr_sentinel(int elem, int range) {
    if (range <= (elem == 1 ? 127 : elem == 2 ? 32767 : 32768)) return STEREO_OK;
    set_error("uniqueness ratio / texture threshold / left-right check / speckle filter: the sentinel -(%d + 1) does not fit a "
              "%d-byte disparity element", range, elem);
    return STEREO_ERR_UNSUPPORTED;
}

// The uniqueness pass over the block matcher's SSD maps (run_uniqueness) holds C in int32 below SGM_ABSENT, the marker of
// absent candidates, so that no present cost reads as absent and C + m(q) of its path kernel cannot overflow:
// (2R + 1)^2 M < 2^30, M the largest per-element term as check_ssd_sgm_bound takes it.
static int check_uniq_bound(int R, double M) {
    if (double(2 * R + 1) * (2 * R + 1) * M < double(SGM_ABSENT)) return STEREO_OK;
    set_error("uniqueness ratio: the block matcher's window cost (2R + 1)^2 x %.0f (R = %d) does not stay below 2^30", M, R);
    return STEREO_ERR_UNSUPPORTED;
}

// Sub-pixel maps hold 16 d + offset, d in [-(range + 1), range] and the offset in [-7, 8], so 16 (range + 1) must fit:
// never a 1-byte map, a 2-byte map up to range 2047.  (The option marks no pixel itself: this is not check_lr_sentinel.)
static int check_subpixel_fit(int elem, int range) {
    if (elem == 4 || (elem == 2 && range <= 2047)) return STEREO_OK;
    set_error("sub-pixel disparity: 16 x (%d + 1) does not fit a %d-byte disparity element", range, elem);
    return STEREO_ERR_UNSUPPORTED;
}

// The options of PairOptions::needs_whole_maps, each with its refusal of a row band [%d, %d) by check_pair_options and of
// row-band sharding by band_sharding_refusal.  An option's entry is on while its field is positive.  check_pair_options
// names the first option on in this order, band_sharding_refusal the last.
struct WholeMapOption {
    int PairOptions::*field;
    const char* band;
    const char* sharding;
};
static const WholeMapOption WHOLE_MAP_OPTIONS[] = {
    {&PairOptions::pf_cap,
     "prefilter: rows [%d, %d) are not the whole map (its odd-height rule needs whole images: prefilter them with "
     "stereo_prefilter_*_device and call the band entry points with it off)",
     "prefilter on: row-band sharded pairs are not prefiltered (shard whole pairs, or prefilter the whole images)"},
    {&PairOptions::uniq,
     "uniqueness ratio: rows [%d, %d) are not the whole map (the uniqueness pass works on whole images)",
     "uniqueness ratio on: row-band sharded pairs are not checked (shard whole pairs)"},
    {&PairOptions::sgm_paths,
     "SGM: rows [%d, %d) are not the whole map (vertical and diagonal paths cross band seams)",
     "SGM on: row-band sharded pairs are not aggregated (shard whole pairs)"},
    {&PairOptions::spk_max_size,
     "speckle filter: rows [%d, %d) are not the whole map (filter the gathered map with stereo_filter_speckles_device)",
     "speckle filter on: row-band sharded pairs are not filtered (filter the gathered map with stereo_filter_speckles_device)"},
    {&PairOptions::subpix,
     "sub-pixel disparity: rows [%d, %d) are not the whole map (the sub-pixel pass works on whole images)",
     "sub-pixel disparity on: row-band sharded pairs are not refined (shard whole pairs)"},
};

// Why the row-band sharded pair calls (stereo_mgpu_disparity_pair_bands_*) refuse a context's options, or nullptr when
// they do not.  No band is filtered, aggregated, checked or prefiltered on its own, and no whole-pair call stands in for
// the bands: this holds for one device too, whose band is the whole image.
const char* band_sharding_refusal(const stereo_ctx* ctx) {
    if (!ctx->opt.needs_whole_maps()) return nullptr;
    const int n = int(sizeof(WHOLE_MAP_OPTIONS) / sizeof(WHOLE_MAP_OPTIONS[0]));
    for (int k = n - 1; k >= 0; --k)
        if (ctx->opt.*WHOLE_MAP_OPTIONS[k].field > 0) return WHOLE_MAP_OPTIONS[k].sharding;
    return nullptr;
}

// What a pair call must satisfy for the context's options, checked once per call before anything is staged or enqueued:
// the sentinel fits (PairOptions::writes_sentinel), SGM aggregates the SSD cost or, with an NCC scale set, the NCC cost,
// and the options of PairOptions::needs_whole_maps get whole maps.  Sub-pixel maps fit (check_subpixel_fit) and, with SGM
// off, need the SSD cost.  The uniqueness ratio on block-matcher maps needs the
// SSD cost, at most 512 candidates after clipping and, for 8-bit images, check_uniq_bound with M = 255^2 (float images:
// after their classification, check_uniq_classified; with the prefilter on every call matches 8-bit images).  run_sgm
// checks SGM's candidate count and int32 bound.
static int check_pair_options(const stereo_ctx* ctx, int cost, PixType type, int elem, int range, int R, int cols, int row_begin,
                              int row_end, int rows) {
    const PairOptions& o = ctx->opt;
    const bool sgm = o.sgm_paths > 0;
    if (o.pf_cap > 0) type = PixType::U8;
    if (o.writes_sentinel()) {
        const int rc = check_lr_sentinel(elem, range);
        if (rc != STEREO_OK) return rc;
    }
    if (o.subpix > 0) {
        const int rc = check_subpixel_fit(elem, range);
        if (rc != STEREO_OK) return rc;
        if (!sgm && cost != STEREO_COST_SSD) {
            set_error("sub-pixel disparity: NCC block-matcher maps rank float32 scores, which have no integer cost (switch SGM on with an NCC scale)");
            return STEREO_ERR_UNSUPPORTED;
        }
    }
    if (sgm && cost != STEREO_COST_SSD && o.sgm_ncc_scale == 0) {
        set_error("SGM aggregates the SSD cost only while no NCC scale is set (stereo_ctx_set_sgm_ncc_scale; or switch SGM off for NCC calls)");
        return STEREO_ERR_UNSUPPORTED;
    }
    if ((row_begin != 0 || row_end != rows) && o.needs_whole_maps())
        for (const WholeMapOption& w : WHOLE_MAP_OPTIONS)
            if (o.*w.field > 0) {
                set_error(w.band, row_begin, row_end);
                return STEREO_ERR_UNSUPPORTED;
            }
    if (o.uniq > 0 && !sgm) {
        if (cost != STEREO_COST_SSD) {
            set_error("uniqueness ratio: NCC block-matcher maps rank float32 scores, for which it has no rule (switch SGM on with an NCC scale)");
            return STEREO_ERR_UNSUPPORTED;
        }
        const int lim = cols - 1 + R, D = (range < lim ? range : lim) + 1;      // (sgm_shape's clipping of either direction)
        if (D > 32 * SGM_MAXK) {
            set_error("uniqueness ratio: %d candidates per pixel, at most %d are supported", D, 32 * SGM_MAXK);
            return STEREO_ERR_UNSUPPORTED;
        }
        if (type == PixType::U8) {
            const int rc = check_uniq_bound(R, 255.0 * 255.0);
            if (rc != STEREO_OK) return rc;
        }
    }
    return STEREO_OK;
}

// The check over `rows` rows of np pairs of maps, in place: maps[k] the left map of pair k, maps[np + k] its right map,
// each at its first row, all of one element type.
static int lr_check_pairs(stereo_ctx* ctx, const OutView* maps, int np, int rows, int cols, int max_diff, int sentinel,
                          cudaStream_t st) {
    LrParams P{};
    for (int k = 0; k < np; ++k) P.pair[k] = LrMaps{maps[k].ptr, maps[np + k].ptr, maps[k].step, maps[np + k].step};
    P.cols = cols;
    P.max_diff = max_diff;
    P.sentinel = sentinel;
    ctx->last_launches += 1;
    return lr_check_launch(P, rows, np, maps[0].elem, st);
}

// The filter over n whole rows x cols maps of one element type, in place.  Its scratch comes from the arena, which the
// caller sized for speckle_scratch_bytes(n, rows, cols) before it enqueued anything: the filter itself never grows it.
static int speckle_maps(stereo_ctx* ctx, const OutView* maps, int n, int rows, int cols, int new_val, int max_size, int max_diff,
                        cudaStream_t st) {
    SpeckleParams P{};
    for (int k = 0; k < n; ++k) P.map[k] = SpeckleMap{maps[k].ptr, maps[k].step, nullptr, nullptr};
    P.rows = rows; P.cols = cols; P.new_val = new_val; P.max_size = max_size; P.max_diff = max_diff;
    ctx->arena.reset();
    void* s = ctx->arena.take(speckle_scratch_bytes(n, rows, cols));
    if (!s) { set_error("scratch arena too small (internal)"); return STEREO_ERR_ALLOC; }
    speckle_bind_scratch(P, n, s);
    ctx->last_launches += SPK_LAUNCHES;
    return speckle_launch(P, n, maps[0].elem, st);
}

// The arena scratch finish_pairs needs for the n maps of a pair call.
static size_t finish_scratch_bytes(const stereo_ctx* ctx, int n, int rows, int cols) {
    return ctx->opt.spk_max_size > 0 ? speckle_scratch_bytes(n, rows, cols) : 0;
}

// The texture threshold on the n whole maps of ps, each against its own reference image, which prefilter_pairs made.
static int texture_maps(stereo_ctx* ctx, const Problem* ps, int n, int sentinel, cudaStream_t st) {
    static_assert(FMAXJOBS <= TX_MAXMAPS, "one texture launch covers the maps of one launch sequence");
    const Problem& p = ps[0];
    TxParams P{};
    for (int k = 0; k < n; ++k)
        P.map[k] = TxMap{static_cast<const uint8_t*>(ps[k].ref.ptr), ps[k].ref.step, ps[k].disp.ptr, ps[k].disp.step};
    P.rows = p.rows; P.cols = p.cols; P.R = p.R; P.cap = ctx->opt.pf_cap; P.threshold = ctx->opt.pf_texture; P.sentinel = sentinel;
    ctx->last_launches += 1;
    return texture_launch(P, n, p.disp.elem, st);
}

// The context's texture threshold, left-right check and speckle filter on the maps of the n/2 pairs of ps (laid out as
// pair_problems builds them), in that order (StereoBM's / StereoSGBM's): the threshold (whole maps only: the prefilter is
// refused for bands) and the check on the rows of ps, then, once `maps_complete` says every row of the maps is computed,
// the filter on the whole maps.
static int finish_pairs(stereo_ctx* ctx, const Problem* ps, int n, cudaStream_t st, bool maps_complete) {
    static_assert(FMAXJOBS / 2 <= LR_MAXPAIRS, "one check launch covers the pairs of one launch sequence");
    static_assert(FMAXJOBS <= SPK_MAXMAPS, "one filter launch covers the maps of one launch sequence");
    const Problem& p = ps[0];
    const int sentinel = -(ps[n / 2].dmax + 1);
    OutView maps[FMAXJOBS];
    for (int k = 0; k < n; ++k) maps[k] = ps[k].disp;
    int rc = STEREO_OK;
    if (ctx->opt.pf_cap > 0 && ctx->opt.pf_texture > 0) rc = texture_maps(ctx, ps, n, sentinel, st);
    if (rc == STEREO_OK && ctx->opt.lr_max_diff >= 0) rc = lr_check_pairs(ctx, maps, n / 2, p.row_end - p.row_begin, p.cols, ctx->opt.lr_max_diff, sentinel, st);
    if (rc != STEREO_OK || !maps_complete || ctx->opt.spk_max_size <= 0) return rc;
    for (int k = 0; k < n; ++k) maps[k].ptr = static_cast<char*>(maps[k].ptr) - size_t(ps[k].row_begin) * maps[k].step;
    return speckle_maps(ctx, maps, n, p.rows, p.cols, sentinel, ctx->opt.spk_max_size, ctx->opt.spk_max_diff, st);
}

// ---- exact path ---------------------------------------------------------------------------------

// Floats of one replicate-padded image of p with its guards (pad_images).
static size_t padded_elems(const Problem& p) {
    return size_t(p.rows + 2 * p.R) * (p.cols + 2 * p.R) + 2 * (size_t(p.R) + 64);
}

static size_t exact_scratch_bytes(const Problem& p) {
    const size_t band = size_t(p.row_end - p.row_begin) * p.cols;
    return 2 * align256(padded_elems(p) * sizeof(float)) + 2 * align256(band * 4) + 4096;
}

// Both images of p, padded by R with replicated borders, into two float images taken from the arena, each with R + 64
// guard floats on both sides; *Lp and *Rp point at their first pixels.  The target's guards are zeroed: they stand in for
// the reference's out-of-allocation reads.
static int pad_images(stereo_ctx* ctx, const Problem& p, cudaStream_t st, float** Lp, float** Rp) {
    const int Hp = p.rows + 2 * p.R, Wp = p.cols + 2 * p.R;
    const size_t guard = size_t(p.R) + 64;
    float* lbuf = static_cast<float*>(ctx->arena.take(padded_elems(p) * sizeof(float)));
    float* rbuf = static_cast<float*>(ctx->arena.take(padded_elems(p) * sizeof(float)));
    if (!lbuf || !rbuf) { set_error("scratch arena too small (internal)"); return STEREO_ERR_ALLOC; }
    SB_CUDA(cudaMemsetAsync(rbuf, 0, guard * sizeof(float), st));
    SB_CUDA(cudaMemsetAsync(rbuf + guard + size_t(Hp) * Wp, 0, guard * sizeof(float), st));
    *Lp = lbuf + guard;
    *Rp = rbuf + guard;
    dim3 pb(32, 8), pg(div_round_up(Wp, 32), div_round_up(Hp, 8));
    if (p.ref.type == PixType::F32)
        pad_replicate_kernel<float><<<pg, pb, 0, st>>>(static_cast<const float*>(p.ref.ptr), p.ref.step, p.rows, p.cols, p.R, *Lp, Hp, Wp, p.avail_begin, p.avail_end);
    else
        pad_replicate_kernel<uint8_t><<<pg, pb, 0, st>>>(static_cast<const uint8_t*>(p.ref.ptr), p.ref.step, p.rows, p.cols, p.R, *Lp, Hp, Wp, p.avail_begin, p.avail_end);
    if (p.tgt.type == PixType::F32)
        pad_replicate_kernel<float><<<pg, pb, 0, st>>>(static_cast<const float*>(p.tgt.ptr), p.tgt.step, p.rows, p.cols, p.R, *Rp, Hp, Wp, p.avail_begin, p.avail_end);
    else
        pad_replicate_kernel<uint8_t><<<pg, pb, 0, st>>>(static_cast<const uint8_t*>(p.tgt.ptr), p.tgt.step, p.rows, p.cols, p.R, *Rp, Hp, Wp, p.avail_begin, p.avail_end);
    ctx->last_launches += 2;
    return STEREO_OK;
}

static int run_exact(stereo_ctx* ctx, const Problem& p, cudaStream_t st) {
    float *Lp, *Rp;
    const int rc = pad_images(ctx, p, st, &Lp, &Rp);
    if (rc != STEREO_OK) return rc;
    const int band_rows = p.row_end - p.row_begin;
    int32_t* d_disp = static_cast<int32_t*>(ctx->arena.take(size_t(band_rows) * p.cols * 4));
    uint32_t* d_best = static_cast<uint32_t*>(ctx->arena.take(size_t(band_rows) * p.cols * 4));
    if (!d_disp || !d_best) { set_error("scratch arena too small (internal)"); return STEREO_ERR_ALLOC; }
    dim3 kb(128), kg(div_round_up(p.cols, 128), band_rows);
    if (p.cost == STEREO_COST_SSD)
        ssd_exact_kernel<<<kg, kb, 0, st>>>(Lp, Rp, p.rows, p.cols, p.R, p.dmin, p.dmax, p.row_begin, d_disp,
                                            reinterpret_cast<int32_t*>(d_best), 0, p.cols);
    else
        ncorr_exact_kernel<<<kg, kb, 0, st>>>(Lp, Rp, p.rows, p.cols, p.R, p.dmin, p.dmax, p.row_begin, d_disp,
                                              reinterpret_cast<float*>(d_best));
    store_output_kernel<<<kg, kb, 0, st>>>(d_disp, d_best, band_rows, p.cols, p.disp.ptr, p.disp.step, p.disp.elem,
                                           p.best.ptr, p.best.step);
    ctx->last_launches += 2;
    SB_CUDA(cudaGetLastError());
    return STEREO_OK;
}

// ---- path selection -------------------------------------------------------------------------------

// Float images: which kernel family applies (decided from the device-side classification, see classify_convert_kernel).
enum { CLS_U8 = 0, CLS_F32_FAST = 1, CLS_EXACT = 2 };

static Problem as_u8(Problem p) { p.ref.type = PixType::U8; p.tgt.type = PixType::U8; return p; }

// The two u8 copies classify_flags takes from the arena.
static size_t u8_copies_bytes(const Problem& p) { return 2 * align256(size_t(p.rows) * align256(p.cols)); }

// Scratch for a float problem whose kernel family is only known after the classification: the larger of the three
// families' needs plus the u8 copies of both images.  `dirs` = directions that share one launch sequence.
static size_t f32_scratch_bytes(stereo_ctx* ctx, const Problem& p, int dirs) {
    size_t need = exact_scratch_bytes(p);
    const size_t f = size_t(dirs) * fast_scratch_bytes(ctx, p), u = size_t(dirs) * fast_scratch_bytes(ctx, as_u8(p));
    if (f > need) need = f;
    if (u > need) need = u;
    return need + u8_copies_bytes(p) + 4096;
}

// Resets the arena and converts both float images of p into u8 copies at its start (u8[0] of ref, u8[1] of tgt) while
// classifying them, then reads the verdict back into ctx->h_flag (one 16-byte copy and a stream synchronize: the kernel
// family is a host decision).
static int classify_flags(stereo_ctx* ctx, const Problem& p, cudaStream_t st, ImageView u8[2]) {
    ctx->arena.reset();
    const size_t pitch = align256(p.cols);
    uint8_t* a8 = static_cast<uint8_t*>(ctx->arena.take(size_t(p.rows) * pitch));
    uint8_t* b8 = static_cast<uint8_t*>(ctx->arena.take(size_t(p.rows) * pitch));
    if (!a8 || !b8) { set_error("scratch arena too small (internal)"); return STEREO_ERR_ALLOC; }
    u8[0] = ImageView{a8, pitch, PixType::U8};
    u8[1] = ImageView{b8, pitch, PixType::U8};
    SB_CUDA(cudaMemsetAsync(ctx->d_flag, 0, 4 * sizeof(int), st));
    dim3 cb(32, 8), cg(div_round_up(p.cols, 32), div_round_up(p.rows, 8), 2);
    classify_convert_kernel<<<cg, cb, 0, st>>>(static_cast<const float*>(p.ref.ptr), p.ref.step, a8, static_cast<const float*>(p.tgt.ptr), p.tgt.step, b8,
                                               p.rows, p.cols, pitch, ctx->d_flag);
    ctx->last_launches += 1;
    SB_CUDA(cudaMemcpyAsync(ctx->h_flag, ctx->d_flag, 4 * sizeof(int), cudaMemcpyDeviceToHost, st));
    SB_CUDA(cudaEventRecord(ctx->ev_gap0, st));
    SB_CUDA(cudaStreamSynchronize(st));
    SB_CUDA(cudaEventRecord(ctx->ev_gap1, st));          // (the kernels chosen below follow this mark)
    ctx->gap_recorded = true;
    return STEREO_OK;
}

// The tracked extremes [tlo, thi] of the blocks that hold a non-8-bit pixel, and the value range [lo, hi] of both images:
// [0, 255] for the blocks without a non-8-bit pixel, the tracked extremes for the others.
static void classified_range(const stereo_ctx* ctx, double* tlo, double* thi, double* lo, double* hi) {
    const unsigned* hf = reinterpret_cast<const unsigned*>(ctx->h_flag);
    *tlo = hf[1] ? -double(f32_from_ordered(hf[1])) : 0.0;
    *thi = hf[2] ? double(f32_from_ordered(hf[2])) : 0.0;
    *lo = *tlo < 0.0 ? *tlo : 0.0;
    *hi = *thi > 255.0 ? *thi : 255.0;
}

// Classifies the float images of one pair (classify_flags) and says which kernel family serves it.
static int classify_images(stereo_ctx* ctx, const Problem& p, cudaStream_t st, ImageView u8[2], int* cls) {
    const int rc = classify_flags(ctx, p, st, u8);
    if (rc != STEREO_OK) return rc;
    const unsigned* hf = reinterpret_cast<const unsigned*>(ctx->h_flag);
    if (hf[0] == 0 && ctx->force_path != STEREO_PATH_FAST_F32) { *cls = CLS_U8; return STEREO_OK; }
    *cls = CLS_EXACT;
    if (hf[0] & 2u) return STEREO_OK;                                  // a pixel that is not finite
    if (ctx->force_path == STEREO_PATH_FAST_U8) return STEREO_OK;      // (reported as "not applicable" by the caller)
    double tlo, thi, lo, hi;
    classified_range(ctx, &tlo, &thi, &lo, &hi);
    const double range = (hi - lo) * (1.0 + 1e-6), wnd = double(2 * p.R + 1) * (2 * p.R + 1);
    bool ok;
    if (p.cost == STEREO_COST_SSD) {
        // per element: round((l - r)^2) + 0.5 < 2^23 (mantissa trick of ssd_q_bits); per window: 128 * SSD + position < 2^32 - 1
        ok = range * range + 1.0 < 8388607.0 && wnd * (range * range + 1.0) < 33554432.0 - 8193.0;
    } else {
        // Overflow: float32 sums of products stay far from it below 1e6.  Resolution: the key ranks C * rs in a power-of-two
        // binade with about 16 value bits, i.e. to ~2^-16 of the score bound (DESIGN.md §4.5).  When every pixel has one sign
        // (a DC offset), two windows of values in [tlo, thi] meet at an angle whose cosine is at least 1 - band with
        // band = (thi - tlo)^2 / (tlo^2 + thi^2), so every score crowds into [1 - band, 1].  band >= 2^-4 keeps >= 2^12 key
        // steps across it; the oracle's first maximum then survives on textured images (measured on 8-bit textures moved
        // up by 1000: band ~0.013, 99.69-99.97 % agreement; by 300: band ~0.09, 100 %).  The tracked extremes are those of the
        // non-8-bit blocks alone, the narrowest range the image can have, so the bound errs towards the exact kernels.
        const double band = (tlo > 0.0 || thi < 0.0) ? (thi - tlo) * (thi - tlo) / (tlo * tlo + thi * thi) : 1.0;
        ok = -lo < 1.0e6 && hi < 1.0e6 && band >= 1.0 / 16;
    }
    if (ok) *cls = CLS_F32_FAST;
    return STEREO_OK;
}

// M of check_ssd_sgm_bound for float images from their classification (classify_flags): 255^2 when 8-bit-valued, otherwise
// ceil((hi - lo)^2) of their value range, widened by 1e-6 for the float rounding of l - r and its square.
static double classified_ssd_max_elem(const stereo_ctx* ctx) {
    if (*reinterpret_cast<const unsigned*>(ctx->h_flag) == 0) return 255.0 * 255.0;
    double tlo, thi, lo, hi;
    classified_range(ctx, &tlo, &thi, &lo, &hi);
    const double range = (hi - lo) * (1.0 + 1e-6);
    return ceil(range * range);
}

// check_uniq_bound for float images from the classification the call made; a pixel that is not finite has no bound.
static int check_uniq_classified(const stereo_ctx* ctx, int R) {
    if (*reinterpret_cast<const unsigned*>(ctx->h_flag) & 2u) {
        set_error("uniqueness ratio: an image holds a pixel that is not finite");
        return STEREO_ERR_UNSUPPORTED;
    }
    return check_uniq_bound(R, classified_ssd_max_elem(ctx));
}

// Grows the scratch arena to `need` bytes; nothing enqueued by earlier calls may still use it then.
static int reserve_arena(stereo_ctx* ctx, cudaStream_t st, size_t need) {
    if (need <= ctx->arena.cap) return STEREO_OK;
    const int rc = quiesce(ctx, st);
    return rc != STEREO_OK ? rc : ctx->arena.reserve(need);
}

// Enqueues one direction on the exact kernels.
static int run_exact_direction(stereo_ctx* ctx, const Problem& p, cudaStream_t st) {
    if (ctx->force_path == STEREO_PATH_FAST_U8 || ctx->force_path == STEREO_PATH_FAST_F32) {
        set_error("fast path forced but not applicable (pixel values or window/range outside what the running-sum kernels cover)");
        return STEREO_ERR_UNSUPPORTED;
    }
    const int rc = reserve_arena(ctx, st, exact_scratch_bytes(p));
    if (rc != STEREO_OK) return rc;
    ctx->arena.reset();
    ctx->last_path = STEREO_PATH_EXACT_F32;
    return run_exact(ctx, p, st);
}

// True when ps = n/2 left-referenced problems followed by their right-referenced partners, each pair fusable.
static bool fused_layout(const stereo_ctx* ctx, const Problem* ps, int n) {
    if (!ctx->fuse_pairs || n < 2 || (n & 1) || n > FMAXJOBS) return false;
    const int np = n / 2;
    for (int k = 0; k < np; ++k)
        if (!fast_pair_fusable(ps[k], ps[np + k]) || !fast_batchable(ps[0], ps[k])) return false;
    return true;
}

// The float images of ONE image pair - ps[0], and its mirror ps[1] when n == 2 - classified once, then every direction
// from one launch sequence (one cost volume where the pair is fusable) on u8 copies or the float operands, or from the
// exact kernels.
static int run_f32_pair(stereo_ctx* ctx, Problem* ps, int n, cudaStream_t st) {
    const Problem& p = ps[0];
    int rc = reserve_arena(ctx, st, f32_scratch_bytes(ctx, p, n));
    if (rc != STEREO_OK) return rc;
    ImageView u8[2];
    int cls = CLS_EXACT;
    rc = classify_images(ctx, p, st, u8, &cls);
    if (rc == STEREO_OK && n == 2 && ctx->opt.uniq > 0) rc = check_uniq_classified(ctx, p.R);      // (before any map is written)
    if (rc != STEREO_OK) return rc;
    if (cls == CLS_EXACT) {
        for (int d = 0; d < n && rc == STEREO_OK; ++d) rc = run_exact_direction(ctx, ps[d], st);
        return rc;
    }
    if (cls == CLS_U8) {
        // ps[0]: ref = left, tgt = right; ps[1] the other way round
        ps[0].ref = u8[0]; ps[0].tgt = u8[1];
        if (n == 2) { ps[1].ref = ps[0].tgt; ps[1].tgt = ps[0].ref; }
    }
    ctx->last_path = cls == CLS_U8 ? STEREO_PATH_FAST_U8 : STEREO_PATH_FAST_F32;
    return run_fast_batch(ctx, ps, n, st, fused_layout(ctx, ps, n) ? n / 2 : 0);
}

// One launch sequence over batchable problems, fused when they are whole pairs.
static int run_fast_auto(stereo_ctx* ctx, const Problem* ps, int n, cudaStream_t st) {
    return run_fast_batch(ctx, ps, n, st, fused_layout(ctx, ps, n) ? n / 2 : 0);
}

// Enqueues `n` u8 problems that all take the packed path, several directions per launch sequence where they are
// batchable (same shape, band, window, cost and candidate count), one fused launch sequence when they are whole pairs.
// `budget` bounds the scratch one unfused launch sequence may hold.
static int run_fast_jobs(stereo_ctx* ctx, const Problem* ps, int n, cudaStream_t st) {
    const size_t budget = size_t(3) << 30;
    const bool fused = fused_layout(ctx, ps, n);         // (n <= FMAXJOBS: one launch sequence)
    for (int i = 0, m = 0; i < n; i += m) {
        const size_t per_job = fast_scratch_bytes(ctx, ps[i]);
        m = fused ? n : 1;
        while (i + m < n && m < FMAXJOBS && fast_batchable(ps[i], ps[i + m]) && size_t(m + 1) * per_job <= budget) ++m;
        int rc = reserve_arena(ctx, st, size_t(m) * per_job);
        if (rc != STEREO_OK) return rc;
        ctx->arena.reset();
        ctx->last_path = STEREO_PATH_FAST_U8;
        rc = run_fast_batch(ctx, ps + i, m, st, fused ? n / 2 : 0);
        if (rc != STEREO_OK) return rc;
    }
    return STEREO_OK;
}

// Enqueues every direction of a call: one problem, or n/2 left-referenced problems followed by their right-referenced
// partners (pair k = ps[k], ps[n/2 + k]).  The one place that picks the kernel family.
static int run_families(stereo_ctx* ctx, Problem* ps, int n, cudaStream_t st, bool fast, bool u8) {
    if (fast && u8) return run_fast_jobs(ctx, ps, n, st);
    if (fast && n <= 2) return run_f32_pair(ctx, ps, n, st);      // (float images come one pair per call)
    const int np = n / 2;
    if (np == 0) return run_exact_direction(ctx, ps[0], st);
    for (int k = 0; k < np; ++k) {
        int rc = run_exact_direction(ctx, ps[k], st);
        if (rc == STEREO_OK) rc = run_exact_direction(ctx, ps[np + k], st);
        if (rc != STEREO_OK) return rc;
    }
    return STEREO_OK;
}

// ---- semi-global matching (sgm.cuh) ----------------------------------------------------------------------------------

// Candidates of one direction: [dmin, dmax] clipped to the ones some pixel has present (|d| <= cols - 1 + R for SSD,
// |d| <= cols - 1 for NCC), padded to 32 K for the path kernels.
struct SgmShape { int dlo, D, K; size_t Dp; };
static SgmShape sgm_shape(const Problem& p) {
    const int lim = p.cost == STEREO_COST_NCORR ? p.cols - 1 : p.cols - 1 + p.R;
    const int dlo = p.dmin > -lim ? p.dmin : -lim, dhi = p.dmax < lim ? p.dmax : lim;
    const int D = dhi - dlo + 1, K = (D + 31) / 32;
    return SgmShape{dlo, D, K, size_t(32) * K};
}

// One direction's scratch: both padded images, the cost volume and the aggregate, for NCC the two window-norm maps (plus,
// for float images, the u8 copies the classification writes).  Directions of a call run one after the other on the same
// scratch.
static size_t sgm_scratch_bytes(const Problem& p) {
    const size_t cells = size_t(p.rows) * p.cols * sgm_shape(p).Dp;
    size_t need = 2 * align256(padded_elems(p) * sizeof(float)) + 2 * align256(cells * 4) + 4096;
    if (p.cost == STEREO_COST_NCORR) need += 2 * align256(size_t(p.rows) * p.cols * sizeof(double));
    return p.ref.type == PixType::F32 ? need + u8_copies_bytes(p) : need;
}

// Every L_r is at most C_max + P2: S stays in int32 when paths (C_max + P2) <= 2^31 - 1.  C_max is (2R + 1)^2 M for SSD,
// M the largest per-element term, and 2q for NCC.
static int check_sgm_bound(const stereo_ctx* ctx, double c_max, const char* what) {
    if (double(ctx->opt.sgm_paths) * (c_max + ctx->opt.sgm_p2) <= 2147483647.0) return STEREO_OK;
    set_error("SGM: %d paths x (C_max %.0f [%s] + P2 %d) exceeds 2^31 - 1", ctx->opt.sgm_paths, c_max, what, ctx->opt.sgm_p2);
    return STEREO_ERR_UNSUPPORTED;
}
static int check_ssd_sgm_bound(const stereo_ctx* ctx, int R, double M) {
    return check_sgm_bound(ctx, double(2 * R + 1) * (2 * R + 1) * M, "(2R + 1)^2 x the largest element");
}

// C of one direction (sgm_cost_kernel; SSD, or NCC of 8-bit-valued images) from its padded images.
static void launch_sgm_cost(stereo_ctx* ctx, const Problem& p, const SgmShape& g, const float* Lp, const float* Rp, const SgmNcc& ncc,
                            int32_t* C, cudaStream_t st) {
    // rows per cost block: as many as still leave about four blocks per SM (each block recomputes 2R + 1 rows first)
    const long long tiles = (long long)div_round_up(p.cols, SGM_XT) * (g.Dp / 32);
    int rpb = 64;
    while (rpb > 8 && tiles * div_round_up(p.rows, rpb) < 4LL * ctx->sm_count) rpb /= 2;
    const dim3 cg(div_round_up(p.cols, SGM_XT), div_round_up(p.rows, rpb), unsigned(g.Dp / 32));
    const size_t smem = size_t(SGM_XT + 2 * p.R) * 32 * sizeof(int32_t);
    if (p.cost == STEREO_COST_NCORR) sgm_cost_kernel<true><<<cg, SGM_COST_THREADS, smem, st>>>(Lp, Rp, p.rows, p.cols, p.R, g.dlo, g.D, int(g.Dp), rpb, ncc, C);
    else sgm_cost_kernel<false><<<cg, SGM_COST_THREADS, smem, st>>>(Lp, Rp, p.rows, p.cols, p.R, g.dlo, g.D, int(g.Dp), rpb, ncc, C);
    ctx->last_launches += 1;
}

// One sgm_path_kernel launch of direction (dy, dx) over C of shape g.
static int launch_sgm_path(stereo_ctx* ctx, const Problem& p, const SgmShape& g, const int32_t* C, int32_t* S, int dy, int dx, int P1,
                           int P2, bool first, const SgmOut& out, cudaStream_t st) {
    const unsigned blocks = div_round_up(sgm_lines(p.rows, p.cols, dy, dx), SGM_PATH_WARPS);
#define SB_SGM_PATH(K) case K: sgm_path_kernel<K><<<blocks, SGM_PATH_WARPS * 32, 0, st>>>(C, S, p.rows, p.cols, dy, dx, P1, P2, first, out); break
    switch (g.K) {
        SB_SGM_PATH(1); SB_SGM_PATH(2); SB_SGM_PATH(3); SB_SGM_PATH(4); SB_SGM_PATH(5); SB_SGM_PATH(6); SB_SGM_PATH(7); SB_SGM_PATH(8);
        SB_SGM_PATH(9); SB_SGM_PATH(10); SB_SGM_PATH(11); SB_SGM_PATH(12); SB_SGM_PATH(13); SB_SGM_PATH(14); SB_SGM_PATH(15); SB_SGM_PATH(16);
        default: set_error("SGM: no path kernel for %d candidates per lane (internal)", g.K); return STEREO_ERR_UNSUPPORTED;
    }
#undef SB_SGM_PATH
    ctx->last_launches += 1;
    return STEREO_OK;
}

// One direction by SGM into p.disp, on scratch the caller reserved.  ref / tgt: the caller's images (u8 or float).
// `per_cell`: NCC on float images that are not 8-bit-valued, whose numerators are summed cell by cell (sgm_ncc_cell_kernel).
// `sentinel`: the value of pixels the uniqueness ratio rejects.
// `subpix`: rows x cols bytes for the sub-pixel offsets of the map (nullptr: off).
static int run_sgm_direction(stereo_ctx* ctx, const Problem& p, cudaStream_t st, bool per_cell, int sentinel, int8_t* subpix) {
    static constexpr int DIRS[8][2] = {{0, 1}, {0, -1}, {1, 0}, {-1, 0}, {1, 1}, {1, -1}, {-1, 1}, {-1, -1}};
    const SgmShape g = sgm_shape(p);
    const size_t cells = size_t(p.rows) * p.cols * g.Dp;
    float *Lp, *Rp;
    const int rc = pad_images(ctx, p, st, &Lp, &Rp);
    if (rc != STEREO_OK) return rc;
    int32_t* C = static_cast<int32_t*>(ctx->arena.take(cells * 4));
    int32_t* S = static_cast<int32_t*>(ctx->arena.take(cells * 4));
    if (!C || !S) { set_error("scratch arena too small (internal)"); return STEREO_ERR_ALLOC; }
    SgmNcc ncc{nullptr, nullptr, ctx->opt.sgm_ncc_scale};
    const bool is_ncc = p.cost == STEREO_COST_NCORR;
    if (is_ncc) {
        double* nref = static_cast<double*>(ctx->arena.take(size_t(p.rows) * p.cols * sizeof(double)));
        double* ntgt = static_cast<double*>(ctx->arena.take(size_t(p.rows) * p.cols * sizeof(double)));
        if (!nref || !ntgt) { set_error("scratch arena too small (internal)"); return STEREO_ERR_ALLOC; }
        ncc.nref = nref;
        ncc.ntgt = ntgt;
        sgm_ncc_norm_kernel<<<dim3(div_round_up(p.cols, 128), p.rows, 2), 128, 0, st>>>(Lp, Rp, p.cols, p.R, nref, ntgt);
        ctx->last_launches += 1;
    }
    if (per_cell) {
        const dim3 cg(div_round_up(p.cols, SGM_CELL_XT), p.rows, unsigned(g.Dp / 32));
        const size_t smem = size_t(2 * (SGM_CELL_XT + 2 * p.R) + 31) * sizeof(float);
        sgm_ncc_cell_kernel<<<cg, SGM_COST_THREADS, smem, st>>>(Lp, Rp, p.cols, p.R, g.dlo, g.D, int(g.Dp), ncc, C);
        ctx->last_launches += 1;
    } else {
        launch_sgm_cost(ctx, p, g, Lp, Rp, ncc, C, st);
    }
    for (int k = 0; k < ctx->opt.sgm_paths; ++k) {
        const bool last = k == ctx->opt.sgm_paths - 1;
        const SgmOut out{last ? p.disp.ptr : nullptr, p.disp.step, p.disp.elem, g.dlo, ctx->opt.uniq, sentinel, 0, last ? subpix : nullptr};
        const int rc2 = launch_sgm_path(ctx, p, g, C, S, DIRS[k][0], DIRS[k][1], ctx->opt.sgm_p1, ctx->opt.sgm_p2, k == 0, out, st);
        if (rc2 != STEREO_OK) return rc2;
    }
    SB_CUDA(cudaGetLastError());
    return STEREO_OK;
}

// The uniqueness pass's scratch for one direction: both padded images and C (plus, for float images, the u8 copies a
// classification writes).  Directions run one after the other on the same scratch.
static size_t uniq_scratch_bytes(const Problem& p) {
    const size_t need = 2 * align256(padded_elems(p) * sizeof(float)) + align256(size_t(p.rows) * p.cols * sgm_shape(p).Dp * 4) + 4096;
    return p.ref.type == PixType::F32 ? need + u8_copies_bytes(p) : need;
}

// The uniqueness ratio on the block matcher's SSD maps of the n directions of ps (pair_problems' layout, the caller's
// images), after the block matcher wrote them: per direction, on scratch the caller reserved, the padded images, C
// (sgm_cost_kernel<false>, the block matcher's window costs exactly) and one vertical path kernel with P1 = P2 = 0, so
// that L_r = C, which stores no S and writes only the sentinel (SgmOut::only_invalid).
static int run_uniqueness(stereo_ctx* ctx, const Problem* ps, int n, cudaStream_t st) {
    const int sentinel = -(ps[n / 2].dmax + 1);
    for (int i = 0; i < n; ++i) {
        const Problem& p = ps[i];
        const SgmShape g = sgm_shape(p);
        ctx->arena.reset();
        float *Lp, *Rp;
        int rc = pad_images(ctx, p, st, &Lp, &Rp);
        if (rc != STEREO_OK) return rc;
        int32_t* C = static_cast<int32_t*>(ctx->arena.take(size_t(p.rows) * p.cols * g.Dp * 4));
        if (!C) { set_error("scratch arena too small (internal)"); return STEREO_ERR_ALLOC; }
        launch_sgm_cost(ctx, p, g, Lp, Rp, SgmNcc{nullptr, nullptr, 0}, C, st);
        const SgmOut out{p.disp.ptr, p.disp.step, p.disp.elem, g.dlo, ctx->opt.uniq, sentinel, 1, nullptr};
        rc = launch_sgm_path(ctx, p, g, C, nullptr, 1, 0, 0, 0, true, out, st);
        if (rc != STEREO_OK) return rc;
    }
    SB_CUDA(cudaGetLastError());
    return STEREO_OK;
}

// Every direction of a pair call by SGM: n/2 left-referenced problems and their partners, one at a time on one scratch.
// SSD: 8-bit images are checked against the int32 bound with M = 255^2 before anything is enqueued; float images (one
// pair per call) are classified first, refused when a pixel is not finite, and checked with M = ceil((hi - lo)^2) of
// their value range (widened by 1e-6 for the float rounding of l - r and its square).  NCC: the bound (C_max = 2q) is
// checked before anything is enqueued; float images are classified, refused when a pixel is not finite, and take the
// per-cell cost kernel unless they are 8-bit-valued.
static int run_sgm(stereo_ctx* ctx, Problem* ps, int n, cudaStream_t st, bool u8) {
    const bool ncc = ps[0].cost == STEREO_COST_NCORR;
    size_t need = 0;
    for (int i = 0; i < n; ++i) {
        if (sgm_shape(ps[i]).K > SGM_MAXK) {
            set_error("SGM: %d candidates per pixel, at most %d are supported", sgm_shape(ps[i]).D, 32 * SGM_MAXK);
            return STEREO_ERR_UNSUPPORTED;
        }
        const size_t b = sgm_scratch_bytes(ps[i]);
        if (b > need) need = b;
    }
    int rc = ncc ? check_sgm_bound(ctx, 2.0 * ctx->opt.sgm_ncc_scale, "2q")
           : u8 ? check_ssd_sgm_bound(ctx, ps[0].R, 255.0 * 255.0) : STEREO_OK;
    if (rc == STEREO_OK) rc = reserve_arena(ctx, st, need);
    if (rc != STEREO_OK) return rc;
    bool per_cell = false;
    if (!u8) {
        const Problem& p = ps[0];
        ImageView copies[2];
        rc = classify_flags(ctx, p, st, copies);
        if (rc != STEREO_OK) return rc;
        const unsigned flags = *reinterpret_cast<const unsigned*>(ctx->h_flag);
        if (flags & 2u) { set_error("SGM: an image holds a pixel that is not finite"); return STEREO_ERR_UNSUPPORTED; }
        per_cell = ncc && flags != 0;
        if (!ncc) {
            rc = check_ssd_sgm_bound(ctx, p.R, classified_ssd_max_elem(ctx));
            if (rc != STEREO_OK) return rc;
        }
    }
    ctx->last_path = STEREO_PATH_SGM;
    for (int i = 0; i < n && rc == STEREO_OK; ++i) {
        ctx->arena.reset();
        int8_t* off = ctx->opt.subpix > 0 ? reinterpret_cast<int8_t*>(ctx->sp.base) + size_t(i) * ps[i].rows * ps[i].cols : nullptr;
        rc = run_sgm_direction(ctx, ps[i], st, per_cell, -(ps[n / 2].dmax + 1), off);
    }
    return rc;
}

// ---- prefilter (prefilter.cuh) ----------------------------------------------------------------------------------------
// Both images of every pair of ps (pair_problems' layout, whole images) prefiltered once, in one launch, into ctx->pf:
// u8 images of align256(cols) pitch that stay live while the arena is reset.  Every problem is then repointed at them
// (L->R: ref pf(left), tgt pf(right); R->L swapped), so everything after matches 8-bit images.  The buffer grows (after
// quiesce) only for a larger shape: after one call of a shape nothing is allocated.
static int prefilter_pairs(stereo_ctx* ctx, Problem* ps, int n, cudaStream_t st) {
    static_assert(FMAXJOBS <= PF_MAXIMGS, "one prefilter launch covers the images of one launch sequence");
    const int np = n / 2;
    const Problem& p = ps[0];
    const size_t pitch = align256(p.cols), img = size_t(p.rows) * pitch;
    if (size_t(n) * align256(img) > ctx->pf.cap) {
        int rc = quiesce(ctx, st);
        if (rc == STEREO_OK) rc = ctx->pf.reserve(size_t(n) * align256(img));
        if (rc != STEREO_OK) return rc;
    }
    ctx->pf.reset();
    const bool f32 = p.ref.type == PixType::F32;
    PfParams P{};
    for (int k = 0; k < np; ++k) {
        uint8_t* l8 = static_cast<uint8_t*>(ctx->pf.take(img));
        uint8_t* r8 = static_cast<uint8_t*>(ctx->pf.take(img));
        if (!l8 || !r8) { set_error("prefilter buffer too small (internal)"); return STEREO_ERR_ALLOC; }
        P.img[2 * k] = PfImage{ps[k].ref.ptr, l8, ps[k].ref.step, pitch};
        P.img[2 * k + 1] = PfImage{ps[k].tgt.ptr, r8, ps[k].tgt.step, pitch};
        ps[k].ref = ImageView{l8, pitch, PixType::U8};
        ps[k].tgt = ImageView{r8, pitch, PixType::U8};
        ps[np + k].ref = ps[k].tgt;
        ps[np + k].tgt = ps[k].ref;
    }
    P.rows = p.rows; P.cols = p.cols; P.cap = ctx->opt.pf_cap;
    ctx->last_launches += 1;
    return prefilter_launch(P, n, f32, st);
}

// ---- sub-pixel disparity (subpixel.cuh) -------------------------------------------------------------------------------

// The SGM maps' offsets of the n directions of a launch sequence in ctx->sp, n x rows x cols bytes that stay live while the
// arena is reset.  The buffer grows (after quiesce) only for a larger shape: after one call of a shape nothing is allocated.
static int reserve_subpix_offsets(stereo_ctx* ctx, cudaStream_t st, size_t bytes) {
    if (bytes <= ctx->sp.cap) return STEREO_OK;
    const int rc = quiesce(ctx, st);
    return rc != STEREO_OK ? rc : ctx->sp.reserve(bytes);
}

// The block-matcher pass's scratch: each image of the n/2 pairs padded once (both directions of a pair read the same two).
static size_t subpix_scratch_bytes(const Problem& p, int n) {
    return size_t(n) * align256(padded_elems(p) * sizeof(float)) + 4096;
}

// The last step of a pair call: every map of the n directions of ps (pair_problems' layout, whole maps, the caller's or the
// prefiltered images) rewritten in place in 1/16 pixels.  SGM maps apply the offsets their last path stored in ctx->sp;
// block-matcher SSD maps pad the images once into the arena, which the caller sized for subpix_scratch_bytes, and
// recompute V(d - 1), V(d), V(d + 1) of each final d.
static int subpixel_maps(stereo_ctx* ctx, const Problem* ps, int n, cudaStream_t st, bool sgm) {
    static_assert(FMAXJOBS <= SP_MAXMAPS, "one sub-pixel launch covers the maps of one launch sequence");
    const Problem& p = ps[0];
    const int np = n / 2;
    SpParams P{};
    P.rows = p.rows; P.cols = p.cols; P.R = p.R; P.sentinel = -(ps[np].dmax + 1);
    for (int k = 0; k < n; ++k) P.map[k] = SpMap{ps[k].disp.ptr, ps[k].disp.step, nullptr, nullptr, nullptr, ps[k].dmin, ps[k].dmax};
    if (sgm) {
        for (int k = 0; k < n; ++k) P.map[k].off = reinterpret_cast<const int8_t*>(ctx->sp.base) + size_t(k) * p.rows * p.cols;
        ctx->last_launches += 1;
        return subpix_apply_launch(P, n, p.disp.elem, st);
    }
    ctx->arena.reset();
    const size_t guard = size_t(p.R) + 64;
    SpPadParams Q{};
    Q.rows = p.rows; Q.cols = p.cols; Q.R = p.R;
    for (int k = 0; k < np; ++k) {
        float* l = static_cast<float*>(ctx->arena.take(padded_elems(p) * sizeof(float)));
        float* r = static_cast<float*>(ctx->arena.take(padded_elems(p) * sizeof(float)));
        if (!l || !r) { set_error("scratch arena too small (internal)"); return STEREO_ERR_ALLOC; }
        Q.img[2 * k] = SpImage{ps[k].ref.ptr, ps[k].ref.step, l + guard};
        Q.img[2 * k + 1] = SpImage{ps[k].tgt.ptr, ps[k].tgt.step, r + guard};
        P.map[k].Lp = P.map[np + k].Rp = l + guard;
        P.map[k].Rp = P.map[np + k].Lp = r + guard;
    }
    ctx->last_launches += 2;
    return subpix_bm_launch(Q, n, P, n, p.disp.elem, p.ref.type == PixType::U8, st);
}

// Validates every direction, runs them - pairs with the context's SGM on by SGM, everything else on the kernel family
// run_families picks - then, for pairs of block-matcher maps, applies the context's uniqueness ratio (run_uniqueness;
// SGM maps apply it in their last path) and finishes pairs with the texture threshold, the left-right check and the
// speckle filter (finish_pairs), and last refines them to 1/16 pixel (subpixel_maps).  Pairs with the prefilter on match
// the prefiltered images (prefilter_pairs) from the start.
static int run_directions(stereo_ctx* ctx, Problem* ps, int n, cudaStream_t st) {
    bool fast = ctx->force_path != STEREO_PATH_EXACT_F32, u8 = true;
    for (int i = 0; i < n; ++i) {
        const Problem& p = ps[i];
        const size_t row = size_t(p.cols) * (p.ref.type == PixType::F32 ? 4 : 1);
        const int rc = validate(p, row, row);
        if (rc != STEREO_OK) return rc;
        if (p.ref.type != p.tgt.type) { set_error("mixed pixel types (internal)"); return STEREO_ERR_INVALID_ARG; }
        fast = fast && fast_supported(p);
        u8 = u8 && p.ref.type == PixType::U8;
    }
    const bool pair = n >= 2;      // (every pair of a call has the same shape, band, range and element type)
    const bool uniq_pass = pair && ctx->opt.uniq > 0 && ctx->opt.sgm_paths == 0;
    const bool subpix = pair && ctx->opt.subpix > 0, sgm = pair && ctx->opt.sgm_paths > 0;
    if (pair) {
        const Problem& p = ps[0];
        int rc = check_pair_options(ctx, p.cost, p.ref.type, p.disp.elem, ps[n / 2].dmax, p.R, p.cols, p.row_begin, p.row_end, p.rows);
        if (rc == STEREO_OK && ctx->opt.pf_cap > 0) {
            rc = prefilter_pairs(ctx, ps, n, st);
            u8 = true;
        }
        size_t need = finish_scratch_bytes(ctx, n, p.rows, p.cols);
        if (uniq_pass && uniq_scratch_bytes(p) > need) need = uniq_scratch_bytes(p);      // (both directions have one shape)
        if (subpix && !sgm && subpix_scratch_bytes(p, n) > need) need = subpix_scratch_bytes(p, n);
        if (rc == STEREO_OK) rc = reserve_arena(ctx, st, need);
        if (rc == STEREO_OK && subpix && sgm) rc = reserve_subpix_offsets(ctx, st, size_t(n) * p.rows * p.cols);
        if (rc == STEREO_OK && uniq_pass && !u8 && !(fast && n <= 2)) {
            // float images the exact kernels take without a classification: classify them for the bound
            ImageView copies[2];
            rc = classify_flags(ctx, p, st, copies);
            if (rc == STEREO_OK) rc = check_uniq_classified(ctx, p.R);
        }
        if (rc != STEREO_OK) return rc;
    }
    Problem callers[FMAXJOBS];      // (run_f32_pair points ps at u8 copies in the arena, which the later passes reuse)
    for (int i = 0; (uniq_pass || subpix) && i < n; ++i) callers[i] = ps[i];
    int rc = sgm ? run_sgm(ctx, ps, n, st, u8) : run_families(ctx, ps, n, st, fast, u8);
    if (rc == STEREO_OK && uniq_pass) rc = run_uniqueness(ctx, callers, n, st);
    if (rc == STEREO_OK && pair) rc = finish_pairs(ctx, ps, n, st, true);
    return rc == STEREO_OK && subpix ? subpixel_maps(ctx, callers, n, st, sgm) : rc;
}

// Every call of a context shares one scratch arena (and the classification flag), so calls are ordered: a call
// enqueued on another stream than its predecessor first waits for the predecessor's end-of-call event.
static void begin_call(stereo_ctx* ctx, cudaStream_t st) {
    if (ctx->have_prev_call && ctx->prev_stream != st) cudaStreamWaitEvent(st, ctx->ev1, 0);
    ctx->prev_stream = st;
    ctx->last_launches = 0;
    ctx->last_ms = -1.f;
    ctx->last_path = STEREO_PATH_NONE;
    ctx->hot_used = 0;
    ctx->hot_total = 0;
    ctx->hot_jobs = 0;
    ctx->fused_pairs_done = 0;
    ctx->gap_recorded = false;
    cudaEventRecord(ctx->ev0, st);
}
static void end_call(stereo_ctx* ctx, cudaStream_t st) {
    cudaEventRecord(ctx->ev1, st);
    ctx->timing_pending = true;
    ctx->have_prev_call = true;
}

// Before the scratch arena is reallocated: nothing enqueued by earlier calls may still use it.
static int quiesce(stereo_ctx* ctx, cudaStream_t st) {
    SB_CUDA(cudaStreamSynchronize(st));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    if (ctx->have_prev_call && ctx->prev_stream != st && ctx->prev_stream != ctx->stream) SB_CUDA(cudaEventSynchronize(ctx->ev1));
    return STEREO_OK;
}

static int check_ctx(stereo_ctx* ctx) {
    if (!ctx) { set_error("null context"); return STEREO_ERR_INVALID_ARG; }
    cudaError_t e = cudaSetDevice(ctx->device);
    if (e != cudaSuccess) { set_error("cudaSetDevice(%d): %s", ctx->device, cudaGetErrorString(e)); return STEREO_ERR_CUDA; }
    return STEREO_OK;
}

static int ensure_pinned(stereo_ctx* ctx, size_t bytes) {
    if (bytes <= ctx->pinned_cap) return STEREO_OK;
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    ctx->pinned = nullptr; ctx->pinned_cap = 0;
    cudaError_t e = cudaHostAlloc(&ctx->pinned, bytes, cudaHostAllocDefault);
    if (e != cudaSuccess) { set_error("cudaHostAlloc(%zu): %s", bytes, cudaGetErrorString(e)); (void)cudaGetLastError(); return STEREO_ERR_ALLOC; }
    ctx->pinned_cap = bytes;
    return STEREO_OK;
}

// ---- pipelined host entry points --------------------------------------------------------------------
// The reference wrapper uploads, computes and downloads strictly one after the other on pageable
// memory (DisparitySSD.cu:171-206).  Here a host call is cut into (pair, row band) work items that flow
// through three streams — H2D of band b+1, compute of band b (both directions) and D2H of band b-1 run
// concurrently — so a call costs about max(upload, compute, download) instead of their sum.  Bands are
// the same R(+1)-row-halo bands the multi-GPU sharding uses (SURVEY.md §8e): bit-identical results.
// f32 images are converted to u8 band by band while the "is it really 8-bit" flag accumulates; it is
// read once at the end, and a non-8-bit image makes the caller redo the call on the exact path.

struct HostDir {          // one direction of a host pair job
    bool swap;            // false: ref = left, tgt = right; true: ref = right, tgt = left
    int dmin, dmax;
    void* const* out;     // per pair: host output pointer
};
struct HostPairIn { const void* left; size_t left_step; const void* right; size_t right_step; };

enum { PIPE_NOT_APPLICABLE = 1, PIPE_NOT_8BIT = 2 };

// STEREO_PIPE_TRACE=1: the pipeline's events keep timestamps and every pipelined call prints, per work item and band, when
// its upload, compute and download finished (ms after the call's first enqueue) - a diagnostic for the e2e numbers.
static bool pipe_trace() {
    static const bool on = getenv("STEREO_PIPE_TRACE") != nullptr;
    return on;
}

static int ensure_pipe(stereo_ctx* ctx, int events) {
    if (!ctx->s_in) SB_CUDA(cudaStreamCreateWithFlags(&ctx->s_in, cudaStreamNonBlocking));
    if (!ctx->s_out) SB_CUDA(cudaStreamCreateWithFlags(&ctx->s_out, cudaStreamNonBlocking));
    if (events > ctx->pipe_ev_cap) {
        const int cap = events + 64;
        cudaEvent_t* ev = new (std::nothrow) cudaEvent_t[cap]();
        if (!ev) { set_error("out of host memory"); return STEREO_ERR_ALLOC; }
        for (int i = 0; i < ctx->pipe_ev_cap; ++i) ev[i] = ctx->pipe_ev[i];
        for (int i = ctx->pipe_ev_cap; i < cap; ++i) {
            cudaError_t e = cudaEventCreateWithFlags(&ev[i], pipe_trace() ? cudaEventDefault : cudaEventDisableTiming);
            if (e != cudaSuccess) {
                for (int k = ctx->pipe_ev_cap; k < i; ++k) cudaEventDestroy(ev[k]);
                delete[] ev;
                set_error("cudaEventCreate: %s", cudaGetErrorString(e));
                return STEREO_ERR_CUDA;
            }
        }
        delete[] ctx->pipe_ev;
        ctx->pipe_ev = ev;
        ctx->pipe_ev_cap = cap;
    }
    return STEREO_OK;
}

static int pipe_bands(const stereo_ctx* ctx, int n_pairs, int rows) {
    if (ctx->pipe_bands > 0) return ctx->pipe_bands < rows ? ctx->pipe_bands : rows;
    if (rows < 512) return 1;                           // too small to be worth cutting
    if (n_pairs >= 4) return rows >= 1024 ? 2 : 1;      // enough pairs in flight; two bands shorten the fill and the drain (tools/e2e_sweep.py)
    int nb = (rows + 255) / 512;                        // ~512-row bands: the (2R+1)-row warm-up stays < 3 %
    return nb < 1 ? 1 : (nb > 8 ? 8 : nb);
}

// Pairs per work item of the pipeline.  Small images (BASELINE config 5: 1280x720, 64 disparities) ride several
// pairs per item so that one launch sequence carries several pairs, as the device batch entry point does (which takes
// up to FMAXJOBS / 2; items stay at PIPE_CPMAX so that uploads, kernels and downloads of different items overlap); large
// images stay one pair (or one band of a pair) per item.
constexpr int PIPE_CPMAX = 4;
static_assert(2 * PIPE_CPMAX <= FMAXJOBS, "a pipeline item is one launch sequence");
static int pipe_chunk_pairs(int n_pairs, int nb, int rows, int cols) {
    if (nb > 1) return 1;
    const long long px = (long long)rows * cols;
    long long cp = ((4ll << 20) + px - 1) / px;           // ~4 Mpix of reference image per item
    if (cp > PIPE_CPMAX) cp = PIPE_CPMAX;
    if (cp > n_pairs / 3) cp = n_pairs / 3;               // keep at least three items in flight
    return cp < 1 ? 1 : int(cp);
}


// Large images (4K): the first work item of a call starts with a short band and the last one ends with a short band, so
// that the part of a call nothing overlaps - the first upload and the last download - is an eighth of an image, and the
// items in between go as whole images (every launch sequence costs ~65 us of ramp-up, warm-up rows and tail whatever
// its size: tools/e2e_sweep.py, STEREO_PIPE_TRACE).
static bool pipe_ramped(const stereo_ctx* ctx, int rows, int cols) {
    return ctx->pipe_bands == 0 && rows >= 1024 && (long long)rows * cols >= (4ll << 20);
}

// Row-band boundaries of work item w of a pipelined call: ascending, from 0 to rows.
static void pipe_item_bounds(const stereo_ctx* ctx, int n_pairs, int n_items, int w, int rows, int cols, std::vector<int>& b) {
    b.clear();
    b.push_back(0);
    if (pipe_ramped(ctx, rows, cols)) {
        const int e = rows / 8;
        if (w == 0) { b.push_back(e); b.push_back(3 * e); }
        if (w == n_items - 1) { if (rows - 3 * e > b.back()) b.push_back(rows - 3 * e); b.push_back(rows - e); }
        b.push_back(rows);
        return;
    }
    const int nb = pipe_bands(ctx, n_pairs, rows);
    const int band_rows = (rows + nb - 1) / nb;
    for (int r = band_rows; r < rows; r += band_rows) b.push_back(r);
    b.push_back(rows);
}

static int pairs_host_pipelined_body(stereo_ctx* ctx, int cost, PixType type, int n_pairs, const HostPairIn* in,
                                     const HostDir* dirs, int n_dirs, int rows, int cols, int R, size_t disp_step, int elem);

// Failures inside the pipeline leave asynchronous copies from / to the CALLER's host buffers queued on the three
// streams: drain them before the error reaches the caller, who may free or reuse those buffers.
static int pairs_host_pipelined(stereo_ctx* ctx, int cost, PixType type, int n_pairs, const HostPairIn* in,
                                const HostDir* dirs, int n_dirs, int rows, int cols, int R, size_t disp_step, int elem) {
    const int rc = pairs_host_pipelined_body(ctx, cost, type, n_pairs, in, dirs, n_dirs, rows, cols, R, disp_step, elem);
    if (rc < STEREO_OK) {
        if (ctx->s_in) cudaStreamSynchronize(ctx->s_in);
        if (ctx->stream) cudaStreamSynchronize(ctx->stream);
        if (ctx->s_out) cudaStreamSynchronize(ctx->s_out);
        (void)cudaGetLastError();
    }
    return rc;
}

// Host-side packing of CV_32FC1 images (host_pack.cpp): on when the context has enough host threads to convert faster
// than the link would carry the floats (stereo_ctx_set_host_threads; automatic: min(16, cores / LOCAL_WORLD_SIZE) threads,
// packing from HOST_PACK_MIN_THREADS up).
constexpr int HOST_PACK_MIN_THREADS = 8;
static bool host_pack_enabled(stereo_ctx* ctx) {
    if (ctx->host_threads == 0) ctx->host_threads = default_host_threads();
    if (ctx->host_threads < 0) return false;                  // switched off
    if (ctx->host_threads < HOST_PACK_MIN_THREADS && !ctx->host_pack_forced) return false;
    if (!ctx->pool || ctx->pool->threads() != ctx->host_threads) {
        delete ctx->pool;
        ctx->pool = new (std::nothrow) HostPool(ctx->host_threads);
    }
    return ctx->pool != nullptr;
}

// A few pixels of a host float image: false as soon as one is not an integer in 0..255.  Noisy / contrast-scaled images
// (main.cpp:140-153,191-193) fail on the first samples, so they skip the optimistic 8-bit pipeline instead of running
// it, finding the flag set and being computed a second time by the float kernels.
static bool host_sample_is_8bit(const void* img, size_t step, int rows, int cols) {
    const int ny = rows < 8 ? rows : 8, nx = cols < 16 ? cols : 16;
    for (int iy = 0; iy < ny; ++iy) {
        const float* row = reinterpret_cast<const float*>(static_cast<const char*>(img) + size_t((long long)iy * (rows - 1) / (ny > 1 ? ny - 1 : 1)) * step);
        for (int ix = 0; ix < nx; ++ix) {
            const float v = row[(long long)ix * (cols - 1) / (nx > 1 ? nx - 1 : 1)];
            if (!(v >= 0.f && v <= 255.f && v == float(int(v)))) return false;
        }
    }
    return true;
}

static int pairs_host_pipelined_body(stereo_ctx* ctx, int cost, PixType type, int n_pairs, const HostPairIn* in,
                                     const HostDir* dirs, int n_dirs, int rows, int cols, int R, size_t disp_step, int elem) {
    if (ctx->force_path == STEREO_PATH_EXACT_F32 || ctx->force_path == STEREO_PATH_FAST_F32) return PIPE_NOT_APPLICABLE;
    if (n_dirs == 2 && ctx->opt.computed_whole()) return PIPE_NOT_APPLICABLE;      // (run_directions computes them whole)
    const auto t_call = std::chrono::steady_clock::now();       // (trace only)
    double t_pack = 0.0, t_ring = 0.0;
    auto since = [](std::chrono::steady_clock::time_point t0) { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); };
    if (type == PixType::F32)
        for (int i = 0; i < n_pairs; ++i)
            if (!host_sample_is_8bit(in[i].left, in[i].left_step, rows, cols) || !host_sample_is_8bit(in[i].right, in[i].right_step, rows, cols))
                return PIPE_NOT_8BIT;
    // CV_32FC1 host images with enough host threads: converted to u8 on the HOST (checking that every pixel is 8-bit), so the
    // link carries 1 byte per pixel; otherwise the float rows are uploaded and converted / classified on the device.
    // (Sending a share of the rows as floats next to the host conversion was measured and dropped: the copy engine's reads
    // and the converting threads compete for the same host memory bandwidth - 4K x 4 pairs: 4.88 ms with none, 5.01 ms with a
    // quarter, 5.57 ms with half of the rows as floats.)
    const bool pack = type == PixType::F32 && host_pack_enabled(ctx);
    const bool any_f32 = type == PixType::F32 && !pack, any_pack = pack;
    const size_t f_pitch = align256(size_t(cols) * 4), u8_pitch = align256(cols), d_pitch = align256(size_t(cols) * elem);
    // validate each direction on a full-image problem (pointers only need to be non-null here)
    Problem full = direction(cost, PixType::U8, in, u8_pitch, in, u8_pitch, rows, cols, 0, rows, 0, rows, R, 0, 0, ctx, d_pitch,
                             elem, nullptr, 0);
    const int nb_uniform = pipe_bands(ctx, n_pairs, rows);
    const int cp = pipe_chunk_pairs(n_pairs, nb_uniform, rows, cols);
    const int n_items = (n_pairs + cp - 1) / cp;
    // row bands of every work item (pipe_item_bounds): item w owns bounds[boff[w]] .. bounds[boff[w + 1] - 1]
    std::vector<int> bounds, boff(n_items + 1, 0), tmpb;
    for (int w = 0; w < n_items; ++w) {
        pipe_item_bounds(ctx, n_pairs, n_items, w, rows, cols, tmpb);
        bounds.insert(bounds.end(), tmpb.begin(), tmpb.end());
        boff[w + 1] = int(bounds.size());
    }
    auto nbw = [&](int w) { return boff[w + 1] - boff[w] - 1; };                           // bands of item w
    std::vector<int> uoff(n_items + 1, 0);                                                 // units (item, band) before item w
    for (int w = 0; w < n_items; ++w) uoff[w + 1] = uoff[w] + nbw(w);
    const int n_units = uoff[n_items];
    size_t scratch = 0;
    int max_up = 0;                                       // most rows one unit uploads
    for (int d = 0; d < n_dirs; ++d) {
        full.dmin = dirs[d].dmin; full.dmax = dirs[d].dmax;
        int rc = validate(full, u8_pitch, u8_pitch);
        if (rc != STEREO_OK) return rc;
        if (!fast_supported(full)) return PIPE_NOT_APPLICABLE;
        // every band: the operand-row count depends on where the band starts relative to the FRPS-row stages
        for (int w = 0; w < n_items; ++w) {
            int up = 0;
            for (int b = 0; b < nbw(w); ++b) {
                Problem band = full; band.row_begin = bounds[boff[w] + b]; band.row_end = bounds[boff[w] + b + 1];
                const size_t need = size_t(n_dirs) * cp * fast_scratch_bytes(ctx, band);
                scratch = need > scratch ? need : scratch;
                const int up_hi = (b == nbw(w) - 1) ? rows : ((band.row_end + R + 16 < rows) ? band.row_end + R + 16 : rows);
                max_up = up_hi - up > max_up ? up_hi - up : max_up;
                up = up_hi;
            }
        }
    }
    // pairs with the speckle filter: an item's maps are filtered whole after its last band, then downloaded
    const bool spk = n_dirs == 2 && ctx->opt.spk_max_size > 0;
    const size_t finish = n_dirs == 2 ? finish_scratch_bytes(ctx, 2 * cp, rows, cols) : 0;
    if (finish > scratch) scratch = finish;
    constexpr int NSTG = 4;                               // pinned staging ring of the host-packed uploads
    int rc = ensure_pipe(ctx, 3 * n_units + 4 + NSTG);
    if (rc != STEREO_OK) return rc;
    cudaStream_t s_in = ctx->s_in, s_cmp = ctx->stream, s_out = ctx->s_out;
    // uploads go chunk by chunk (~a quarter of a large image): the first copy of a unit leaves while the host threads are
    // still converting the rest of it
    const int chunk_rows = cp > 1 || rows < 1024 ? max_up : ((rows + 3) / 4 < 128 ? 128 : (rows + 3) / 4);
    const int stg_rows = chunk_rows < max_up ? chunk_rows : max_up;
    const size_t stg_pitch = (size_t(cols) + 63) & ~size_t(63);
    const size_t stg_slot = 2 * size_t(cp) * stg_rows * stg_pitch;
    if (any_pack) { rc = ensure_pinned(ctx, NSTG * stg_slot); if (rc != STEREO_OK) return rc; }

    const int S = n_items < 3 ? n_items : 3;            // device slots (ring), one work item each
    const size_t pair_bytes = 2 * align256(u8_pitch * rows) + (any_f32 ? 2 * align256(f_pitch * rows) : 0) + size_t(n_dirs) * align256(d_pitch * rows);
    const size_t slot_bytes = size_t(cp) * pair_bytes;
    if (size_t(S) * slot_bytes + 1024 > ctx->io.cap || scratch > ctx->arena.cap) {
        SB_CUDA(cudaStreamSynchronize(s_in)); SB_CUDA(cudaStreamSynchronize(s_cmp)); SB_CUDA(cudaStreamSynchronize(s_out));
        if (size_t(S) * slot_bytes + 1024 > ctx->io.cap) { rc = ctx->io.reserve(size_t(S) * slot_bytes + 1024); if (rc != STEREO_OK) return rc; }
        if (scratch > ctx->arena.cap) { rc = ctx->arena.reserve(scratch); if (rc != STEREO_OK) return rc; }
    }
    ctx->io.reset();
    struct Slot { char* lf; char* rf; uint8_t* l8; uint8_t* r8; char* out[2]; };      // lf / rf: float rows awaiting conversion
    constexpr int CPMAX = PIPE_CPMAX;
    Slot slot[3][CPMAX] = {};
    for (int k = 0; k < S; ++k)
        for (int c = 0; c < cp; ++c) {
            Slot& sl = slot[k][c];
            sl.l8 = static_cast<uint8_t*>(ctx->io.take(u8_pitch * rows));
            sl.r8 = static_cast<uint8_t*>(ctx->io.take(u8_pitch * rows));
            if (any_f32) {
                sl.lf = static_cast<char*>(ctx->io.take(f_pitch * rows));
                sl.rf = static_cast<char*>(ctx->io.take(f_pitch * rows));
            }
            for (int d = 0; d < n_dirs; ++d) sl.out[d] = static_cast<char*>(ctx->io.take(d_pitch * rows));
            if (!sl.l8 || !sl.r8 || (any_f32 && (!sl.lf || !sl.rf)) || !sl.out[n_dirs - 1]) { set_error("io arena too small (internal)"); return STEREO_ERR_ALLOC; }
        }
    auto ev = [&](int item, int band, int kind) { return ctx->pipe_ev[3 * (uoff[item] + band) + kind + 1]; };   // kind: 0 in, 1 cmp, 2 out

    begin_call(ctx, s_cmp);
    // copy streams start after whatever the context's stream was doing with these buffers
    SB_CUDA(cudaEventRecord(ctx->pipe_ev[0], s_cmp));
    SB_CUDA(cudaStreamWaitEvent(s_in, ctx->pipe_ev[0], 0));
    SB_CUDA(cudaStreamWaitEvent(s_out, ctx->pipe_ev[0], 0));
    if (any_f32) SB_CUDA(cudaMemsetAsync(ctx->d_flag, 0, 4 * sizeof(int), s_cmp));
    ctx->last_path = STEREO_PATH_FAST_U8;
    auto stg_ev = [&](int k) { return ctx->pipe_ev[3 * n_units + 1 + k]; };
    struct FloatRows { int r0, n; };                      // float row ranges of the unit being uploaded (converted on the device)
    std::vector<FloatRows> frows;
    // host conversion runs one upload chunk ahead of the enqueueing thread: the chunks in the order the loops below meet them
    struct PackChunk { int w, r0, n; };
    std::vector<PackChunk> pchunks;
    if (any_pack)
        for (int w = 0; w < n_items; ++w) {
            int up = 0;
            for (int b = 0; b < nbw(w); ++b) {
                const int re = bounds[boff[w] + b + 1];
                const int up_hi = (b == nbw(w) - 1) ? rows : ((re + R + 16 < rows) ? re + R + 16 : rows);
                for (int r0 = up; r0 < up_hi; r0 += chunk_rows) pchunks.push_back(PackChunk{w, r0, up_hi - r0 < chunk_rows ? up_hi - r0 : chunk_rows});
                if (up_hi > up) up = up_hi;
            }
        }
    // STEREO_PACK_AHEAD=0 (diagnostic): convert each chunk only when the loop reaches it, as before the look-ahead
    static const bool pack_ahead = [] { const char* e = getenv("STEREO_PACK_AHEAD"); return !(e && atoi(e) == 0); }();
    PackAsync pa;
    struct PoolDrain { HostPool* p; ~PoolDrain() { if (p) p->end(); } } pool_drain{any_pack ? ctx->pool : nullptr};   // no conversion outlives `pa`
    int pk = 0, pk_begun = 0;
    auto pack_begin = [&](int idx) -> int {
        const PackChunk& ch = pchunks[idx];
        const int k = idx % NSTG;
        const auto t_r = std::chrono::steady_clock::now();
        if (idx >= NSTG) SB_CUDA(cudaEventSynchronize(stg_ev(k)));      // the upload that last read this staging slot
        t_ring += since(t_r);
        uint8_t* stg = static_cast<uint8_t*>(ctx->pinned) + size_t(k) * stg_slot;
        const int i0 = ch.w * cp, np = (n_pairs - i0 < cp) ? n_pairs - i0 : cp;
        PackJob jobs[2 * PIPE_CPMAX];
        for (int c = 0; c < np; ++c) {
            const HostPairIn& hp = in[i0 + c];
            jobs[2 * c] = PackJob{reinterpret_cast<const float*>(static_cast<const char*>(hp.left) + size_t(ch.r0) * hp.left_step), hp.left_step,
                                  stg + size_t(2 * c) * stg_rows * stg_pitch, stg_pitch, ch.n, cols};
            jobs[2 * c + 1] = PackJob{reinterpret_cast<const float*>(static_cast<const char*>(hp.right) + size_t(ch.r0) * hp.right_step), hp.right_step,
                                      stg + size_t(2 * c + 1) * stg_rows * stg_pitch, stg_pitch, ch.n, cols};
        }
        pa.begin(*ctx->pool, jobs, 2 * np);
        pk_begun = idx + 1;
        return STEREO_OK;
    };

    for (int w = 0; w < n_items; ++w) {
        const Slot* sl = slot[w % S];
        const int i0 = w * cp, np = (n_pairs - i0 < cp) ? n_pairs - i0 : cp;     // pairs i0 .. i0+np-1 ride this item
        int uploaded = 0;
        for (int b = 0; b < nbw(w); ++b) {
            const int rb = bounds[boff[w] + b], re = bounds[boff[w] + b + 1];
            // ---- upload the rows this band adds: window halo R, the +1 row of the SSD flat-index wrap, and the
            //      operand rows the FRPS-row pipeline stages round up to
            const int up_hi = (b == nbw(w) - 1) ? rows : ((re + R + 16 < rows) ? re + R + 16 : rows);
            if (b == 0 && w >= S) SB_CUDA(cudaStreamWaitEvent(s_in, ev(w - S, nbw(w - S) - 1, 1), 0));   // slot inputs free again
            frows.clear();
            for (int r0 = uploaded; r0 < up_hi; r0 += chunk_rows) {
                const int n = up_hi - r0 < chunk_rows ? up_hi - r0 : chunk_rows;
                if (type == PixType::U8) {
                    for (int c = 0; c < np; ++c) {
                        const HostPairIn& hp = in[i0 + c];
                        SB_CUDA(cudaMemcpy2DAsync(sl[c].l8 + size_t(r0) * u8_pitch, u8_pitch, static_cast<const char*>(hp.left) + size_t(r0) * hp.left_step,
                                                  hp.left_step, cols, n, cudaMemcpyHostToDevice, s_in));
                        SB_CUDA(cudaMemcpy2DAsync(sl[c].r8 + size_t(r0) * u8_pitch, u8_pitch, static_cast<const char*>(hp.right) + size_t(r0) * hp.right_step,
                                                  hp.right_step, cols, n, cudaMemcpyHostToDevice, s_in));
                    }
                    continue;
                }
                // float rows as they are (converted by classify_convert_kernel in front of the unit's kernels), or through the
                // pinned staging ring as 8-bit pixels
                const int nf = any_pack ? 0 : n;
                if (nf > 0) {
                    for (int c = 0; c < np; ++c) {
                        const HostPairIn& hp = in[i0 + c];
                        SB_CUDA(cudaMemcpy2DAsync(sl[c].lf + size_t(r0) * f_pitch, f_pitch, static_cast<const char*>(hp.left) + size_t(r0) * hp.left_step,
                                                  hp.left_step, size_t(cols) * 4, nf, cudaMemcpyHostToDevice, s_in));
                        SB_CUDA(cudaMemcpy2DAsync(sl[c].rf + size_t(r0) * f_pitch, f_pitch, static_cast<const char*>(hp.right) + size_t(r0) * hp.right_step,
                                                  hp.right_step, size_t(cols) * 4, nf, cudaMemcpyHostToDevice, s_in));
                    }
                    frows.push_back(FloatRows{r0, nf});
                }
                const int p0 = r0 + nf, npk = n - nf;
                if (npk > 0) {
                    // this chunk's conversion was started while the previous chunk's copies and launches were being enqueued
                    // (the very first one starts here); the next chunk's starts before this one's copies are enqueued
                    const int idx = pk++, k = idx % NSTG;
                    if (idx >= int(pchunks.size()) || pchunks[idx].w != w || pchunks[idx].r0 != p0 || pchunks[idx].n != npk) {
                        set_error("upload chunk list out of step (internal)"); return STEREO_ERR_INVALID_ARG;
                    }
                    if (pk_begun <= idx) { rc = pack_begin(idx); if (rc != STEREO_OK) return rc; }
                    const auto t_p = std::chrono::steady_clock::now();
                    const bool all8 = pa.end(*ctx->pool);
                    t_pack += since(t_p);
                    if (!all8) {
                        // a pixel that is not 8-bit: give the call to the float kernels (nothing of it has reached the caller's
                        // maps that will not be overwritten)
                        SB_CUDA(cudaStreamSynchronize(s_in)); SB_CUDA(cudaStreamSynchronize(s_cmp)); SB_CUDA(cudaStreamSynchronize(s_out));
                        return PIPE_NOT_8BIT;
                    }
                    if (pack_ahead && idx + 1 < int(pchunks.size())) { rc = pack_begin(idx + 1); if (rc != STEREO_OK) return rc; }
                    const uint8_t* stg = static_cast<const uint8_t*>(ctx->pinned) + size_t(k) * stg_slot;
                    for (int c = 0; c < np; ++c) {
                        SB_CUDA(cudaMemcpy2DAsync(sl[c].l8 + size_t(p0) * u8_pitch, u8_pitch, stg + size_t(2 * c) * stg_rows * stg_pitch, stg_pitch, cols, npk,
                                                  cudaMemcpyHostToDevice, s_in));
                        SB_CUDA(cudaMemcpy2DAsync(sl[c].r8 + size_t(p0) * u8_pitch, u8_pitch, stg + size_t(2 * c + 1) * stg_rows * stg_pitch, stg_pitch, cols, npk,
                                                  cudaMemcpyHostToDevice, s_in));
                    }
                    SB_CUDA(cudaEventRecord(stg_ev(k), s_in));
                }
            }
            if (up_hi > uploaded) uploaded = up_hi;
            SB_CUDA(cudaEventRecord(ev(w, b, 0), s_in));
            // ---- compute
            SB_CUDA(cudaStreamWaitEvent(s_cmp, ev(w, b, 0), 0));
            if (b == 0 && w >= S) SB_CUDA(cudaStreamWaitEvent(s_cmp, ev(w - S, nbw(w - S) - 1, 2), 0));  // slot outputs downloaded
            for (const FloatRows& fr : frows) {
                dim3 cb(32, 8), cg(div_round_up(cols, 32), div_round_up(fr.n, 8), 2);
                for (int c = 0; c < np; ++c) {
                    classify_convert_kernel<<<cg, cb, 0, s_cmp>>>(reinterpret_cast<const float*>(sl[c].lf + size_t(fr.r0) * f_pitch), f_pitch,
                                                                 sl[c].l8 + size_t(fr.r0) * u8_pitch,
                                                                 reinterpret_cast<const float*>(sl[c].rf + size_t(fr.r0) * f_pitch), f_pitch,
                                                                 sl[c].r8 + size_t(fr.r0) * u8_pitch, fr.n, cols, u8_pitch, ctx->d_flag);
                    ctx->last_launches += 1;
                }
            }
            {
                // direction-major: jobs with the same range sign are neighbours (they share offsets and pitches)
                Problem pd[FMAXJOBS];
                for (int d = 0; d < n_dirs; ++d)
                    for (int c = 0; c < np; ++c) {
                        Problem& p = pd[d * np + c];
                        p = full;
                        p.row_begin = rb; p.row_end = re;
                        p.dmin = dirs[d].dmin; p.dmax = dirs[d].dmax;
                        p.ref = ImageView{dirs[d].swap ? sl[c].r8 : sl[c].l8, u8_pitch, PixType::U8};
                        p.tgt = ImageView{dirs[d].swap ? sl[c].l8 : sl[c].r8, u8_pitch, PixType::U8};
                        p.disp = OutView{sl[c].out[d] + size_t(rb) * d_pitch, d_pitch, elem};
                    }
                const int nj = n_dirs * np;
                bool together = true;
                for (int k = 1; k < nj; ++k) together = together && fast_batchable(pd[0], pd[k]);
                if (together) {
                    ctx->arena.reset();
                    rc = run_fast_auto(ctx, pd, nj, s_cmp);
                } else {
                    for (int k = 0; k < nj && rc == STEREO_OK; ++k) { ctx->arena.reset(); rc = run_fast(ctx, pd[k], s_cmp); }
                }
                // two directions: pd holds the np left-referenced problems, then their partners
                if (rc == STEREO_OK && n_dirs == 2) rc = finish_pairs(ctx, pd, nj, s_cmp, b == nbw(w) - 1);
                if (rc != STEREO_OK) return rc;
            }
            SB_CUDA(cudaEventRecord(ev(w, b, 1), s_cmp));
            // ---- download: this band's rows, or with the speckle filter every row of the item after its last band
            SB_CUDA(cudaStreamWaitEvent(s_out, ev(w, b, 1), 0));
            const int d0 = !spk ? rb : (b == nbw(w) - 1 ? 0 : re);
            for (int c = 0; c < np && re > d0; ++c)
                for (int d = 0; d < n_dirs; ++d)
                    SB_CUDA(cudaMemcpy2DAsync(static_cast<char*>(dirs[d].out[i0 + c]) + size_t(d0) * disp_step, disp_step, sl[c].out[d] + size_t(d0) * d_pitch, d_pitch,
                                              size_t(cols) * elem, re - d0, cudaMemcpyDeviceToHost, s_out));
            SB_CUDA(cudaEventRecord(ev(w, b, 2), s_out));
        }
    }
    if (any_f32) SB_CUDA(cudaMemcpyAsync(ctx->h_flag, ctx->d_flag, sizeof(int), cudaMemcpyDeviceToHost, s_cmp));
    end_call(ctx, s_cmp);
    const double t_enq = since(t_call);
    SB_CUDA(cudaStreamSynchronize(s_cmp));
    SB_CUDA(cudaStreamSynchronize(s_out));
    SB_CUDA(cudaStreamSynchronize(s_in));
    if (pipe_trace()) {
        fprintf(stderr, "[pipe] host: everything enqueued after %.3f ms (converting %.3f, waiting for a staging slot %.3f), streams idle after %.3f ms\n",
                t_enq, t_pack, t_ring, since(t_call));
        fprintf(stderr, "[pipe] %d pairs %dx%d, %d items, %d units, %s\n", n_pairs, rows, cols, n_items, n_units,
                any_pack ? "host pack" : (type == PixType::F32 ? "float upload" : "u8"));
        for (int w = 0; w < n_items; ++w)
            for (int b = 0; b < nbw(w); ++b) {
                float t[3] = {-1.f, -1.f, -1.f};
                for (int k = 0; k < 3; ++k) cudaEventElapsedTime(&t[k], ctx->pipe_ev[0], ev(w, b, k));
                fprintf(stderr, "[pipe]   item %d rows %d..%d: in %.3f  compute %.3f  out %.3f ms\n", w, bounds[boff[w] + b], bounds[boff[w] + b + 1], t[0], t[1], t[2]);
            }
        (void)cudaGetLastError();
    }
    if (any_f32 && *ctx->h_flag != 0) return PIPE_NOT_8BIT;
    return STEREO_OK;
}

// What every host entry point checks before it touches a buffer: the context, non-null pointers, an image of at most
// 32768 pixels a side (validate() reports larger ones to device callers as UNSUPPORTED), a disparity element of 1, 2 or
// 4 bytes and every {step, row bytes} step at least its row.  A pair's negative `range` is rejected with `range_rc` (single
// directions pass range 0).
static int check_host_args(stereo_ctx* ctx, std::initializer_list<const void*> ptrs, int rows, int cols, int elem,
                           std::initializer_list<std::pair<size_t, size_t>> steps, int range = 0,
                           int range_rc = STEREO_ERR_INVALID_RANGE) {
    const int rc = check_ctx(ctx);
    if (rc != STEREO_OK) return rc;
    for (const void* p : ptrs)
        if (!p) { set_error("null pointer"); return STEREO_ERR_INVALID_ARG; }
    if (rows <= 0 || cols <= 0 || rows > 32768 || cols > 32768) { set_error("bad image size %d x %d", rows, cols); return STEREO_ERR_INVALID_ARG; }
    if (elem != 1 && elem != 2 && elem != 4) { set_error("disp_elem_bytes must be 1, 2 or 4"); return STEREO_ERR_INVALID_ARG; }
    for (const auto& s : steps)
        if (s.first < s.second) { set_error("a step is smaller than its row"); return STEREO_ERR_INVALID_ARG; }
    if (range < 0) { set_error("disparity_range must be >= 0"); return range_rc; }
    return STEREO_OK;
}

// Sequential host call: upload (2D async copies), compute, download, synchronize - the shape of cuda::disparitySSD
// (DisparitySSD.cu:171-206) without per-call allocation.
struct HostRows { const void* ptr; size_t step, row_bytes; };     // host input rows
struct HostMap { void* ptr; size_t step, row_bytes; };            // host output rows; ptr == nullptr: not wanted
struct DevRows { char* ptr; size_t pitch; };

// Uploads in_rows rows of both inputs, runs compute(device inputs, device outputs) on ctx->stream and downloads out_rows
// rows of every wanted output.  `compute` brackets its kernels with begin_call / end_call, so the copies stay out of
// last_kernel_ms.  The stream is synchronized on every return, errors included: nothing may still touch the caller's buffers.
template <class Compute>
static int staged_host_call(stereo_ctx* ctx, const HostRows (&in)[2], int in_rows, const HostMap (&out)[2], int out_rows,
                            Compute compute) {
    cudaStream_t st = ctx->stream;
    DevRows din[2], dout[2] = {};
    size_t need = 1024;
    for (const HostRows& h : in) need += align256(h.row_bytes) * in_rows;
    for (const HostMap& h : out) need += h.ptr ? align256(h.row_bytes) * out_rows : 0;
    if (need > ctx->io.cap) {
        SB_CUDA(cudaStreamSynchronize(st));
        const int rc = ctx->io.reserve(need);
        if (rc != STEREO_OK) return rc;
    }
    ctx->io.reset();
    bool ok = true;
    for (int i = 0; i < 2; ++i) {
        din[i].pitch = align256(in[i].row_bytes);
        din[i].ptr = static_cast<char*>(ctx->io.take(din[i].pitch * in_rows));
        ok = ok && din[i].ptr;
        if (!out[i].ptr) continue;
        dout[i].pitch = align256(out[i].row_bytes);
        dout[i].ptr = static_cast<char*>(ctx->io.take(dout[i].pitch * out_rows));
        ok = ok && dout[i].ptr;
    }
    if (!ok) { set_error("io arena too small (internal)"); return STEREO_ERR_ALLOC; }
    cudaError_t e = cudaSuccess;
    for (int i = 0; i < 2 && e == cudaSuccess; ++i)
        e = cudaMemcpy2DAsync(din[i].ptr, din[i].pitch, in[i].ptr, in[i].step, in[i].row_bytes, in_rows, cudaMemcpyHostToDevice, st);
    int rc = e == cudaSuccess ? compute(din, dout) : STEREO_ERR_CUDA;
    for (int i = 0; i < 2 && rc == STEREO_OK && e == cudaSuccess; ++i)
        if (out[i].ptr)
            e = cudaMemcpy2DAsync(out[i].ptr, out[i].step, dout[i].ptr, dout[i].pitch, out[i].row_bytes, out_rows, cudaMemcpyDeviceToHost, st);
    if (e != cudaSuccess) { set_error("host copy failed: %s", cudaGetErrorString(e)); rc = STEREO_ERR_CUDA; }
    e = cudaStreamSynchronize(st);
    if (rc == STEREO_OK && e != cudaSuccess) { set_error("host call failed: %s", cudaGetErrorString(e)); rc = STEREO_ERR_CUDA; }
    return rc;
}

// One call of a device entry point: every direction on `stream` (nullptr: the context's stream).
static int device_call(stereo_ctx* ctx, Problem* ps, int n, void* stream) {
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    begin_call(ctx, st);
    const int rc = run_directions(ctx, ps, n, st);
    end_call(ctx, st);
    return rc;
}

static int device_single(stereo_ctx* ctx, Problem p, void* stream) {
    const int rc = check_ctx(ctx);
    return rc != STEREO_OK ? rc : device_call(ctx, &p, 1, stream);
}

static int host_single(stereo_ctx* ctx, int cost, PixType type, const void* ref, size_t ref_step, const void* tgt,
                       size_t tgt_step, int rows, int cols, int R, int dmin, int dmax, void* disp_out,
                       size_t disp_step, int elem, void* best_out, size_t best_step) {
    const size_t row = size_t(cols) * (type == PixType::F32 ? 4 : 1), disp_row = size_t(cols) * elem, best_row = size_t(cols) * 4;
    int rc = check_host_args(ctx, {ref, tgt, disp_out}, rows, cols, elem,
                             {{ref_step, row}, {tgt_step, row}, {disp_step, disp_row}, {best_step, best_out ? best_row : 0}});
    if (rc != STEREO_OK) return rc;
    if (!best_out) {      // pipelined band-by-band; falls through to the sequential path when the packed kernels do not apply
        const HostPairIn in{ref, ref_step, tgt, tgt_step};
        void* outs[1] = {disp_out};
        const HostDir dir{false, dmin, dmax, outs};
        rc = pairs_host_pipelined(ctx, cost, type, 1, &in, &dir, 1, rows, cols, R, disp_step, elem);
        if (rc <= STEREO_OK) return rc;
    }
    const HostRows in[2] = {{ref, ref_step, row}, {tgt, tgt_step, row}};
    const HostMap out[2] = {{disp_out, disp_step, disp_row}, {best_out, best_step, best_row}};
    return staged_host_call(ctx, in, rows, out, rows, [&](const DevRows* d, const DevRows* o) {
        Problem p = direction(cost, type, d[0].ptr, d[0].pitch, d[1].ptr, d[1].pitch, rows, cols, 0, rows, 0, rows, R, dmin, dmax,
                              o[0].ptr, o[0].pitch, elem, o[1].ptr, o[1].pitch);
        return device_call(ctx, &p, 1, ctx->stream);
    });
}

} // namespace sb

using namespace sb;

// =================================================================================================
// C ABI
// =================================================================================================

extern "C" {

int stereo_abi_version(void) { return STEREO_B200_ABI_VERSION; }

const char* stereo_last_error(void) { return g_err; }

const char* stereo_status_string(int status) {
    switch (status) {
    case STEREO_OK: return "ok";
    case STEREO_ERR_INVALID_ARG: return "invalid argument";
    case STEREO_ERR_INVALID_RANGE: return "invalid disparity range";
    case STEREO_ERR_NO_DEVICE: return "no sm_100 CUDA device";
    case STEREO_ERR_CUDA: return "CUDA error";
    case STEREO_ERR_ALLOC: return "allocation failed";
    case STEREO_ERR_UNSUPPORTED: return "unsupported parameters";
    default: return "unknown status";
    }
}

int stereo_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { (void)cudaGetLastError(); return 0; }
    int ok = 0;
    for (int i = 0; i < n; ++i) {
        int major = 0;
        if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, i) == cudaSuccess && major == 10) ++ok;
    }
    return ok;
}

int stereo_ctx_create(int device, stereo_ctx** ctx_out) {
    if (!ctx_out) { set_error("ctx_out is null"); return STEREO_ERR_INVALID_ARG; }
    *ctx_out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
        (void)cudaGetLastError();
        set_error("no CUDA device available (this library has no CPU fallback)");
        return STEREO_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= n) { set_error("device %d out of range [0, %d)", device, n); return STEREO_ERR_INVALID_ARG; }
    int major = 0, sms = 0;
    SB_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
    SB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    if (major != 10) { set_error("device %d is sm_%d0; this library is built for sm_100a only", device, major); return STEREO_ERR_NO_DEVICE; }
    SB_CUDA(cudaSetDevice(device));
    stereo_ctx* c = new (std::nothrow) stereo_ctx();
    if (!c) { set_error("out of host memory"); return STEREO_ERR_ALLOC; }
    c->device = device;
    c->sm_count = sms;
    cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev1);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev_gap0);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev_gap1);
    for (int i = 0; i < stereo_ctx::HOT_EVENTS && e == cudaSuccess; ++i) {
        e = cudaEventCreate(&c->hot0[i]);
        if (e == cudaSuccess) e = cudaEventCreate(&c->hot1[i]);
    }
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&c->d_flag), 256);
    if (e == cudaSuccess) e = cudaHostAlloc(reinterpret_cast<void**>(&c->h_flag), 256, cudaHostAllocDefault);
    if (e != cudaSuccess) {
        set_error("context setup failed: %s", cudaGetErrorString(e));
        stereo_ctx_destroy(c);
        return STEREO_ERR_CUDA;
    }
    int rc = fast_ctx_init(c);
    if (rc == STEREO_OK) rc = lr_check_init();
    if (rc == STEREO_OK) rc = texture_init();
    if (rc != STEREO_OK) { stereo_ctx_destroy(c); return rc; }
    *ctx_out = c;
    return STEREO_OK;
}

void stereo_ctx_destroy(stereo_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) { cudaStreamSynchronize(ctx->stream); }
    ctx->arena.release();
    ctx->io.release();
    ctx->pf.release();
    ctx->sp.release();
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    delete ctx->pool;
    if (ctx->d_flag) cudaFree(ctx->d_flag);
    if (ctx->h_flag) cudaFreeHost(ctx->h_flag);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    if (ctx->ev_gap0) cudaEventDestroy(ctx->ev_gap0);
    if (ctx->ev_gap1) cudaEventDestroy(ctx->ev_gap1);
    for (int i = 0; i < stereo_ctx::HOT_EVENTS; ++i) {
        if (ctx->hot0[i]) cudaEventDestroy(ctx->hot0[i]);
        if (ctx->hot1[i]) cudaEventDestroy(ctx->hot1[i]);
    }
    for (int i = 0; i < ctx->pipe_ev_cap; ++i) cudaEventDestroy(ctx->pipe_ev[i]);
    delete[] ctx->pipe_ev;
    for (int i = 0; i < stereo_ctx::PEER_STREAMS; ++i) if (ctx->s_peer[i]) { cudaStreamSynchronize(ctx->s_peer[i]); cudaStreamDestroy(ctx->s_peer[i]); }
    if (ctx->peer_ready) cudaEventDestroy(ctx->peer_ready);
    for (int t = 0; t < stereo_ctx::PEER_TICKETS; ++t)
        for (int i = 0; i < stereo_ctx::PEER_STREAMS; ++i) if (ctx->peer_done[t][i]) cudaEventDestroy(ctx->peer_done[t][i]);
    if (ctx->s_in) cudaStreamDestroy(ctx->s_in);
    if (ctx->s_out) cudaStreamDestroy(ctx->s_out);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

int stereo_ctx_last_path(const stereo_ctx* ctx) { return ctx ? ctx->last_path : 0; }

float stereo_ctx_last_kernel_ms(const stereo_ctx* ctx) {
    if (!ctx) return -1.f;
    stereo_ctx* c = const_cast<stereo_ctx*>(ctx);
    if (c->timing_pending) {
        float ms = -1.f;
        if (cudaEventSynchronize(c->ev1) == cudaSuccess && cudaEventElapsedTime(&ms, c->ev0, c->ev1) == cudaSuccess) {
            float gap = 0.f;      // float device calls: the host round trip of the classification verdict is not kernel time
            if (c->gap_recorded && cudaEventElapsedTime(&gap, c->ev_gap0, c->ev_gap1) == cudaSuccess && gap > 0.f && gap < ms) ms -= gap;
            c->last_ms = ms;
        }
        else (void)cudaGetLastError();
        c->timing_pending = false;
    }
    return c->last_ms;
}

int stereo_ctx_last_launches(const stereo_ctx* ctx) { return ctx ? ctx->last_launches : 0; }

float stereo_ctx_last_hot_kernel_ms(const stereo_ctx* ctx, int* launches_measured) {
    if (launches_measured) *launches_measured = 0;
    if (!ctx || ctx->hot_used == 0) return -1.f;
    float total = 0.f;
    for (int i = 0; i < ctx->hot_used; ++i) {
        float ms = 0.f;
        if (cudaEventSynchronize(ctx->hot1[i]) != cudaSuccess || cudaEventElapsedTime(&ms, ctx->hot0[i], ctx->hot1[i]) != cudaSuccess) {
            (void)cudaGetLastError();
            return -1.f;
        }
        total += ms;
    }
    if (launches_measured) *launches_measured = ctx->hot_used;
    return total;
}

int stereo_ctx_last_hot_jobs(const stereo_ctx* ctx) { return ctx ? ctx->hot_jobs : 0; }

int stereo_ctx_force_path(stereo_ctx* ctx, int path) {
    if (!ctx || path < 0 || path > STEREO_PATH_FAST_F32) { set_error("bad force_path argument"); return STEREO_ERR_INVALID_ARG; }
    ctx->force_path = path;
    return STEREO_OK;
}

int stereo_ctx_set_pipe_bands(stereo_ctx* ctx, int bands) {
    if (!ctx || bands < 0 || bands > 4096) { set_error("bad pipe_bands argument"); return STEREO_ERR_INVALID_ARG; }
    ctx->pipe_bands = bands;
    return STEREO_OK;
}

// Pure host arithmetic (no device): how a host batch call is cut into pipeline items.
int stereo_host_pipeline_plan(int n_pairs, int rows, int cols, int bands_override, int* bands_per_pair, int* pairs_per_item) {
    if (n_pairs <= 0 || rows <= 0 || cols <= 0 || bands_override < 0 || !bands_per_pair || !pairs_per_item) {
        set_error("bad arguments"); return STEREO_ERR_INVALID_ARG;
    }
    stereo_ctx tmp;
    tmp.pipe_bands = bands_override;
    const int nb = pipe_bands(&tmp, n_pairs, rows);
    const int cp = pipe_chunk_pairs(n_pairs, nb, rows, cols);
    const int n_items = (n_pairs + cp - 1) / cp;
    std::vector<int> b;
    int most = 0;
    for (int w = 0; w < n_items; w = (w == 0 && n_items > 2) ? n_items - 1 : w + 1) {      // first and last item hold the most bands
        pipe_item_bounds(&tmp, n_pairs, n_items, w, rows, cols, b);
        most = int(b.size()) - 1 > most ? int(b.size()) - 1 : most;
    }
    *bands_per_pair = most;
    *pairs_per_item = cp;
    return STEREO_OK;
}

int stereo_host_pipeline_item_bands(int n_pairs, int rows, int cols, int bands_override, int item, int* bounds, int cap) {
    if (n_pairs <= 0 || rows <= 0 || cols <= 0 || bands_override < 0 || item < 0 || !bounds || cap < 2) {
        set_error("bad arguments"); return STEREO_ERR_INVALID_ARG;
    }
    stereo_ctx tmp;
    tmp.pipe_bands = bands_override;
    const int cp = pipe_chunk_pairs(n_pairs, pipe_bands(&tmp, n_pairs, rows), rows, cols);
    const int n_items = (n_pairs + cp - 1) / cp;
    if (item >= n_items) { set_error("item %d of %d", item, n_items); return STEREO_ERR_INVALID_ARG; }
    std::vector<int> b;
    pipe_item_bounds(&tmp, n_pairs, n_items, item, rows, cols, b);
    if (int(b.size()) > cap) { set_error("%d boundaries, room for %d", int(b.size()), cap); return STEREO_ERR_INVALID_ARG; }
    for (size_t i = 0; i < b.size(); ++i) bounds[i] = b[i];
    return int(b.size());
}

// Pure host arithmetic (no device): the geometry of the hot-kernel launch a batch of `n_pairs` pair problems would get.
int stereo_launch_plan(int cost, int float_operands, int n_pairs, int rows, int cols, int window_rad, int disparity_range, int fuse,
                       int sm_count, stereo_launch_plan_t* plan) {
    if (!plan || n_pairs < 1 || 2 * n_pairs > FMAXJOBS || rows <= 0 || cols <= 0 || window_rad < 0 || window_rad > FMAXR || disparity_range < 0 ||
        sm_count < 1 || (cost != STEREO_COST_SSD && cost != STEREO_COST_NCORR)) {
        set_error("bad launch plan arguments"); return STEREO_ERR_INVALID_ARG;
    }
    stereo_ctx tmp;
    tmp.sm_count = sm_count;
    Problem ps[FMAXJOBS];
    static const char dummy_l = 0, dummy_r = 0;
    for (int k = 0; k < n_pairs; ++k)
        pair_problems(ps, n_pairs, k, cost, float_operands ? PixType::F32 : PixType::U8, &dummy_l + k, size_t(cols), &dummy_r + k,
                      size_t(cols), rows, cols, 0, rows, 0, rows, window_rad, disparity_range, nullptr, nullptr, 0, 1);
    if (!fast_supported(ps[0])) { set_error("outside what the running-sum kernels cover"); return STEREO_ERR_UNSUPPORTED; }
    tmp.fuse_pairs = fuse ? 1 : 0;
    const bool fused = fused_layout(&tmp, ps, 2 * n_pairs);
    FastKernelParams kp{};
    fast_geometry(&tmp, ps, 2 * n_pairs, kp.g, kp.job, fused ? n_pairs : 0);
    const FastGeom& g = kp.g;
    plan->fused = fused ? 1 : 0;
    plan->strip_px = g.K; plan->strips_per_warp = g.hs; plan->groups = g.G; plan->tile_px = g.spc * g.K; plan->tiles = g.ntiles;
    plan->ctas = g.ctas; plan->schedule = g.sched == 1 ? 2 : (g.nrl != g.nrows ? 1 : 0); plan->rows_per_item = int(g.L);
    plan->bands = g.sched == 1 ? g.nbands : 0; plan->stages = g.nst; plan->smem_bytes = int(fast_smem_bytes(g)); plan->border_kernel = g.border;
    return STEREO_OK;
}

int stereo_ctx_last_fused_pairs(const stereo_ctx* ctx) { return ctx ? ctx->fused_pairs_done : 0; }

// Pure host code (no device): the conversion the pipelined CV_32FC1 entry points run on their host threads.
int stereo_host_pack_f32_u8(const float* src, size_t src_step, uint8_t* dst, size_t dst_step, int rows, int cols, int threads, int* all_8bit) {
    if (!src || !dst || !all_8bit || rows <= 0 || cols <= 0 || src_step < size_t(cols) * 4 || dst_step < size_t(cols) || threads < 1 || threads > 256) {
        set_error("bad pack arguments"); return STEREO_ERR_INVALID_ARG;
    }
    HostPool pool(threads);
    *all_8bit = pack_f32_u8(pool, src, src_step, dst, dst_step, rows, cols) ? 1 : 0;
    return STEREO_OK;
}

int stereo_host_pool_selftest(int threads, int rounds) {
    if (threads < 1 || threads > 256 || rounds < 1) { set_error("bad selftest arguments"); return STEREO_ERR_INVALID_ARG; }
    HostPool pool(threads);
    std::vector<std::atomic<int>> hits(257);
    for (int r = 0; r < rounds; ++r) {
        const int n_tasks = 1 + (r * 37) % 257;
        for (int i = 0; i < n_tasks; ++i) hits[i].store(0, std::memory_order_relaxed);
        // odd rounds: the asynchronous form the host pipeline uses - the caller does something else between begin() and end()
        if (r & 1) {
            pool.begin(n_tasks, [&](int t) { hits[t].fetch_add(1, std::memory_order_relaxed); });
            volatile int spin = 0;
            for (int i = 0; i < (r % 7) * 300; ++i) spin = spin + i;
            pool.end();
        } else {
            pool.run(n_tasks, [&](int t) { hits[t].fetch_add(1, std::memory_order_relaxed); });
        }
        for (int i = 0; i < n_tasks; ++i)
            if (hits[i].load() != 1) { set_error("round %d: task %d of %d ran %d times", r, i, n_tasks, hits[i].load()); return STEREO_ERR_UNSUPPORTED; }
        if (r % 64 == 63) std::this_thread::sleep_for(std::chrono::microseconds(600));     // let the workers fall asleep now and then
    }
    return STEREO_OK;
}

int stereo_ctx_set_host_threads(stereo_ctx* ctx, int threads) {
    if (!ctx || threads < -1 || threads > 256) { set_error("bad host_threads argument"); return STEREO_ERR_INVALID_ARG; }
    ctx->host_threads = threads;
    ctx->host_pack_forced = threads > 0;
    return STEREO_OK;
}

int stereo_ctx_host_threads(const stereo_ctx* ctx) {
    if (!ctx) return 0;
    return ctx->host_threads == 0 ? default_host_threads() : ctx->host_threads;
}

int stereo_ctx_set_fuse_pairs(stereo_ctx* ctx, int on) {
    if (!ctx) { set_error("null context"); return STEREO_ERR_INVALID_ARG; }
    ctx->fuse_pairs = on ? 1 : 0;
    return STEREO_OK;
}

int stereo_ctx_set_lr_check(stereo_ctx* ctx, int max_diff) {
    if (!ctx) { set_error("null context"); return STEREO_ERR_INVALID_ARG; }
    ctx->opt.lr_max_diff = max_diff < 0 ? -1 : max_diff;
    return STEREO_OK;
}

int stereo_ctx_lr_check(const stereo_ctx* ctx) { return ctx ? ctx->opt.lr_max_diff : -1; }

int stereo_lr_check_device(stereo_ctx* ctx, void* disp_left, void* disp_right, size_t disp_step, int disp_elem_bytes, int rows,
                           int cols, int disparity_range, int max_diff, void* cuda_stream) {
    int rc = check_ctx(ctx);
    if (rc != STEREO_OK) return rc;
    if (!disp_left || !disp_right) { set_error("null map pointer"); return STEREO_ERR_INVALID_ARG; }
    if (rows <= 0 || cols <= 0) { set_error("rows/cols must be positive (got %d x %d)", rows, cols); return STEREO_ERR_INVALID_ARG; }
    if (rows > 32768 || cols > LR_MAXCOLS) { set_error("map larger than 32768 in a dimension"); return STEREO_ERR_UNSUPPORTED; }
    if (disp_elem_bytes != 1 && disp_elem_bytes != 2 && disp_elem_bytes != 4) { set_error("disp_elem_bytes must be 1, 2 or 4"); return STEREO_ERR_INVALID_ARG; }
    if (disp_step < size_t(cols) * disp_elem_bytes) { set_error("disp_step smaller than a row"); return STEREO_ERR_INVALID_ARG; }
    if (disparity_range < 0 || disparity_range > 32768) { set_error("disparity_range must be in [0, 32768]"); return STEREO_ERR_INVALID_RANGE; }
    if (max_diff < 0) { set_error("max_diff must be >= 0"); return STEREO_ERR_INVALID_ARG; }
    rc = check_lr_sentinel(disp_elem_bytes, disparity_range);
    if (rc != STEREO_OK) return rc;
    cudaStream_t st = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->stream;
    begin_call(ctx, st);
    const OutView maps[2] = {{disp_left, disp_step, disp_elem_bytes}, {disp_right, disp_step, disp_elem_bytes}};
    rc = lr_check_pairs(ctx, maps, 1, rows, cols, max_diff, -(disparity_range + 1), st);
    end_call(ctx, st);
    return rc;
}

int stereo_ctx_set_speckle_filter(stereo_ctx* ctx, int max_size, int max_diff) {
    if (!ctx) { set_error("null context"); return STEREO_ERR_INVALID_ARG; }
    if (max_size > 0 && max_diff < 0) { set_error("max_diff must be >= 0"); return STEREO_ERR_INVALID_ARG; }
    ctx->opt.spk_max_size = max_size > 0 ? max_size : 0;
    ctx->opt.spk_max_diff = max_size > 0 ? max_diff : 0;
    return STEREO_OK;
}

int stereo_ctx_speckle_filter(const stereo_ctx* ctx, int* max_size, int* max_diff) {
    if (!ctx || !max_size || !max_diff) { set_error("null argument"); return STEREO_ERR_INVALID_ARG; }
    *max_size = ctx->opt.spk_max_size;
    *max_diff = ctx->opt.spk_max_diff;
    return STEREO_OK;
}

int stereo_ctx_set_sgm(stereo_ctx* ctx, int paths, int p1, int p2) {
    if (!ctx) { set_error("null context"); return STEREO_ERR_INVALID_ARG; }
    if (paths != 0 && paths != 4 && paths != 8) { set_error("SGM paths must be 0, 4 or 8 (got %d)", paths); return STEREO_ERR_INVALID_ARG; }
    if (p1 < 0 || p1 > p2) { set_error("SGM penalties need 0 <= P1 <= P2 (got %d, %d)", p1, p2); return STEREO_ERR_INVALID_ARG; }
    ctx->opt.sgm_paths = paths;
    ctx->opt.sgm_p1 = paths ? p1 : 0;
    ctx->opt.sgm_p2 = paths ? p2 : 0;
    return STEREO_OK;
}

int stereo_ctx_sgm(const stereo_ctx* ctx, int* paths, int* p1, int* p2) {
    if (!ctx || !paths || !p1 || !p2) { set_error("null argument"); return STEREO_ERR_INVALID_ARG; }
    *paths = ctx->opt.sgm_paths;
    *p1 = ctx->opt.sgm_p1;
    *p2 = ctx->opt.sgm_p2;
    return STEREO_OK;
}

int stereo_ctx_set_sgm_ncc_scale(stereo_ctx* ctx, int q) {
    if (!ctx) { set_error("null context"); return STEREO_ERR_INVALID_ARG; }
    if (q < 0 || q > (1 << 24)) { set_error("SGM NCC scale must be in [0, 2^24] (got %d)", q); return STEREO_ERR_INVALID_ARG; }
    ctx->opt.sgm_ncc_scale = q;
    return STEREO_OK;
}

int stereo_ctx_sgm_ncc_scale(const stereo_ctx* ctx) {
    if (!ctx) { set_error("null context"); return STEREO_ERR_INVALID_ARG; }
    return ctx->opt.sgm_ncc_scale;
}

int stereo_ctx_set_uniqueness(stereo_ctx* ctx, int uniqueness_ratio) {
    if (!ctx) { set_error("null context"); return STEREO_ERR_INVALID_ARG; }
    if (uniqueness_ratio < 0 || uniqueness_ratio > 99) {
        set_error("uniqueness ratio must be in [0, 99] (got %d)", uniqueness_ratio);
        return STEREO_ERR_INVALID_ARG;
    }
    ctx->opt.uniq = uniqueness_ratio;
    return STEREO_OK;
}

int stereo_ctx_uniqueness(const stereo_ctx* ctx) {
    if (!ctx) { set_error("null context"); return STEREO_ERR_INVALID_ARG; }
    return ctx->opt.uniq;
}

int stereo_ctx_set_subpixel(stereo_ctx* ctx, int on) {
    if (!ctx) { set_error("null context"); return STEREO_ERR_INVALID_ARG; }
    if (on != 0 && on != 1) { set_error("sub-pixel disparity: on must be 0 or 1 (got %d)", on); return STEREO_ERR_INVALID_ARG; }
    ctx->opt.subpix = on;
    return STEREO_OK;
}

int stereo_ctx_subpixel(const stereo_ctx* ctx) {
    if (!ctx) { set_error("null context"); return STEREO_ERR_INVALID_ARG; }
    return ctx->opt.subpix;
}

int stereo_ctx_set_prefilter(stereo_ctx* ctx, int cap, int texture_threshold) {
    if (!ctx) { set_error("null context"); return STEREO_ERR_INVALID_ARG; }
    if (cap < 0 || cap > 63 || texture_threshold < 0 || (cap == 0 && texture_threshold != 0)) {
        set_error("prefilter: cap must be in [1, 63] (0: off) and the texture threshold >= 0 (0 while off) (got %d, %d)", cap,
                  texture_threshold);
        return STEREO_ERR_INVALID_ARG;
    }
    ctx->opt.pf_cap = cap;
    ctx->opt.pf_texture = texture_threshold;
    return STEREO_OK;
}

int stereo_ctx_prefilter(const stereo_ctx* ctx, int* cap, int* texture_threshold) {
    if (!ctx || !cap || !texture_threshold) { set_error("null argument"); return STEREO_ERR_INVALID_ARG; }
    *cap = ctx->opt.pf_cap;
    *texture_threshold = ctx->opt.pf_texture;
    return STEREO_OK;
}

// pf(src) into dst, one image, on the caller's stream.
static int prefilter_device(stereo_ctx* ctx, const void* src, size_t src_step, size_t px, int rows, int cols, int cap, uint8_t* dst,
                            size_t dst_step, void* cuda_stream) {
    int rc = check_ctx(ctx);
    if (rc != STEREO_OK) return rc;
    if (!src || !dst) { set_error("null pointer"); return STEREO_ERR_INVALID_ARG; }
    if (rows <= 0 || cols <= 0) { set_error("rows/cols must be positive (got %d x %d)", rows, cols); return STEREO_ERR_INVALID_ARG; }
    if (rows > 32768 || cols > 32768) { set_error("image larger than 32768 in a dimension"); return STEREO_ERR_UNSUPPORTED; }
    if (src_step < size_t(cols) * px || dst_step < size_t(cols)) { set_error("a step is smaller than its row"); return STEREO_ERR_INVALID_ARG; }
    if (cap < 1 || cap > 63) { set_error("prefilter cap must be in [1, 63] (got %d)", cap); return STEREO_ERR_INVALID_ARG; }
    const uintptr_t s0 = reinterpret_cast<uintptr_t>(src), s1 = s0 + size_t(rows - 1) * src_step + size_t(cols) * px;
    const uintptr_t d0 = reinterpret_cast<uintptr_t>(dst), d1 = d0 + size_t(rows - 1) * dst_step + size_t(cols);
    if (s0 < d1 && d0 < s1) { set_error("prefilter: dst overlaps src"); return STEREO_ERR_INVALID_ARG; }
    cudaStream_t st = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->stream;
    begin_call(ctx, st);
    PfParams P{};
    P.img[0] = PfImage{src, dst, src_step, dst_step};
    P.rows = rows; P.cols = cols; P.cap = cap;
    ctx->last_launches += 1;
    rc = prefilter_launch(P, 1, px == 4, st);
    end_call(ctx, st);
    return rc;
}

int stereo_prefilter_u8_device(stereo_ctx* ctx, const uint8_t* src, size_t src_step, int rows, int cols, int cap, uint8_t* dst,
                               size_t dst_step, void* cuda_stream) {
    return prefilter_device(ctx, src, src_step, 1, rows, cols, cap, dst, dst_step, cuda_stream);
}

int stereo_prefilter_f32_device(stereo_ctx* ctx, const float* src, size_t src_step, int rows, int cols, int cap, uint8_t* dst,
                                size_t dst_step, void* cuda_stream) {
    return prefilter_device(ctx, src, src_step, 4, rows, cols, cap, dst, dst_step, cuda_stream);
}

int stereo_filter_speckles_device(stereo_ctx* ctx, void* disp, size_t disp_step, int disp_elem_bytes, int rows, int cols, int new_val,
                                  int max_size, int max_diff, void* cuda_stream) {
    int rc = check_ctx(ctx);
    if (rc != STEREO_OK) return rc;
    if (!disp) { set_error("null map pointer"); return STEREO_ERR_INVALID_ARG; }
    if (rows <= 0 || cols <= 0) { set_error("rows/cols must be positive (got %d x %d)", rows, cols); return STEREO_ERR_INVALID_ARG; }
    if (rows > SPK_MAXDIM || cols > SPK_MAXDIM) { set_error("map larger than 32768 in a dimension"); return STEREO_ERR_UNSUPPORTED; }
    if (disp_elem_bytes != 1 && disp_elem_bytes != 2 && disp_elem_bytes != 4) { set_error("disp_elem_bytes must be 1, 2 or 4"); return STEREO_ERR_INVALID_ARG; }
    if (disp_step < size_t(cols) * disp_elem_bytes) { set_error("disp_step smaller than a row"); return STEREO_ERR_INVALID_ARG; }
    if (max_size < 0 || max_diff < 0) { set_error("max_size and max_diff must be >= 0"); return STEREO_ERR_INVALID_ARG; }
    const int lim = disp_elem_bytes == 1 ? 127 : disp_elem_bytes == 2 ? 32767 : INT32_MAX;
    if (new_val > lim || new_val < -lim - 1) { set_error("new_val %d does not fit a %d-byte element", new_val, disp_elem_bytes); return STEREO_ERR_INVALID_ARG; }
    cudaStream_t st = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->stream;
    if (max_size > 0) rc = reserve_arena(ctx, st, speckle_scratch_bytes(1, rows, cols));
    if (rc != STEREO_OK) return rc;
    begin_call(ctx, st);
    const OutView map{disp, disp_step, disp_elem_bytes};
    if (max_size > 0) rc = speckle_maps(ctx, &map, 1, rows, cols, new_val, max_size, max_diff, st);
    end_call(ctx, st);
    return rc;
}

// ---- peer gather: results pushed into other ranks' buffers by the copy engines ---------------------
static int ensure_peer(stereo_ctx* ctx) {
    if (ctx->peer_ready) return STEREO_OK;
    for (int i = 0; i < stereo_ctx::PEER_STREAMS; ++i) SB_CUDA(cudaStreamCreateWithFlags(&ctx->s_peer[i], cudaStreamNonBlocking));
    for (int t = 0; t < stereo_ctx::PEER_TICKETS; ++t)
        for (int i = 0; i < stereo_ctx::PEER_STREAMS; ++i) SB_CUDA(cudaEventCreateWithFlags(&ctx->peer_done[t][i], cudaEventDisableTiming));
    SB_CUDA(cudaEventCreateWithFlags(&ctx->peer_ready, cudaEventDisableTiming));
    return STEREO_OK;
}

int stereo_peer_buffer_create(stereo_ctx* ctx, size_t bytes, void** dev_ptr, unsigned char* handle_out) {
    int rc = check_ctx(ctx);
    if (rc != STEREO_OK) return rc;
    if (!dev_ptr || !handle_out || bytes == 0) { set_error("bad peer buffer arguments"); return STEREO_ERR_INVALID_ARG; }
    static_assert(sizeof(cudaIpcMemHandle_t) == STEREO_IPC_HANDLE_BYTES, "IPC handle size");
    void* p = nullptr;
    if (cudaMalloc(&p, bytes) != cudaSuccess) { (void)cudaGetLastError(); set_error("peer buffer of %zu bytes: out of device memory", bytes); return STEREO_ERR_ALLOC; }
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) { cudaFree(p); set_error("cudaIpcGetMemHandle failed: %s", cudaGetErrorString(e)); return STEREO_ERR_CUDA; }
    memcpy(handle_out, &h, sizeof(h));
    *dev_ptr = p;
    return STEREO_OK;
}

int stereo_peer_buffer_open(stereo_ctx* ctx, const unsigned char* handle, void** peer_ptr) {
    int rc = check_ctx(ctx);
    if (rc != STEREO_OK) return rc;
    if (!handle || !peer_ptr) { set_error("bad peer buffer arguments"); return STEREO_ERR_INVALID_ARG; }
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    SB_CUDA(cudaIpcOpenMemHandle(peer_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return STEREO_OK;
}

int stereo_peer_buffer_close(stereo_ctx* ctx, void* peer_ptr) {
    int rc = check_ctx(ctx);
    if (rc != STEREO_OK) return rc;
    if (peer_ptr) SB_CUDA(cudaIpcCloseMemHandle(peer_ptr));
    return STEREO_OK;
}

int stereo_peer_buffer_destroy(stereo_ctx* ctx, void* dev_ptr) {
    int rc = check_ctx(ctx);
    if (rc != STEREO_OK) return rc;
    if (dev_ptr) SB_CUDA(cudaFree(dev_ptr));
    return STEREO_OK;
}

int stereo_peer_push(stereo_ctx* ctx, void* const* dst_ptrs, int n_dst, size_t dst_offset, const void* src, size_t bytes,
                     void* after_stream) {
    int rc = check_ctx(ctx);
    if (rc != STEREO_OK) return rc;
    if (!dst_ptrs || n_dst < 0 || (!src && bytes)) { set_error("bad peer push arguments"); return STEREO_ERR_INVALID_ARG; }
    rc = ensure_peer(ctx);
    if (rc != STEREO_OK) return rc;
    cudaStream_t producer = after_stream ? static_cast<cudaStream_t>(after_stream) : ctx->stream;
    SB_CUDA(cudaEventRecord(ctx->peer_ready, producer));
    for (int i = 0; i < stereo_ctx::PEER_STREAMS; ++i) SB_CUDA(cudaStreamWaitEvent(ctx->s_peer[i], ctx->peer_ready, 0));
    for (int i = 0; i < n_dst; ++i) {
        if (!dst_ptrs[i]) continue;
        cudaStream_t s = ctx->s_peer[ctx->peer_next_stream];
        ctx->peer_next_stream = (ctx->peer_next_stream + 1) % stereo_ctx::PEER_STREAMS;
        SB_CUDA(cudaMemcpyAsync(static_cast<char*>(dst_ptrs[i]) + dst_offset, src, bytes, cudaMemcpyDeviceToDevice, s));
    }
    return STEREO_OK;
}

int stereo_peer_mark(stereo_ctx* ctx, int* ticket_out) {
    int rc = check_ctx(ctx);
    if (rc != STEREO_OK) return rc;
    if (!ticket_out) { set_error("ticket_out is null"); return STEREO_ERR_INVALID_ARG; }
    rc = ensure_peer(ctx);
    if (rc != STEREO_OK) return rc;
    const int t = ctx->peer_next_ticket;
    ctx->peer_next_ticket = (t + 1) % stereo_ctx::PEER_TICKETS;
    for (int i = 0; i < stereo_ctx::PEER_STREAMS; ++i) SB_CUDA(cudaEventRecord(ctx->peer_done[t][i], ctx->s_peer[i]));
    *ticket_out = t;
    return STEREO_OK;
}

int stereo_peer_wait(stereo_ctx* ctx, int ticket, void* cuda_stream) {
    int rc = check_ctx(ctx);
    if (rc != STEREO_OK) return rc;
    if (ticket < 0 || ticket >= stereo_ctx::PEER_TICKETS || !ctx->peer_ready) { set_error("bad peer ticket"); return STEREO_ERR_INVALID_ARG; }
    cudaStream_t s = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->stream;
    for (int i = 0; i < stereo_ctx::PEER_STREAMS; ++i) SB_CUDA(cudaStreamWaitEvent(s, ctx->peer_done[ticket][i], 0));
    return STEREO_OK;
}

int stereo_ctx_synchronize(stereo_ctx* ctx, void* cuda_stream) {
    int rc = check_ctx(ctx);
    if (rc != STEREO_OK) return rc;
    SB_CUDA(cudaStreamSynchronize(cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->stream));
    return STEREO_OK;
}

int stereo_disparity_f32_host(stereo_ctx* ctx, int cost, const float* ref, size_t ref_step, const float* tgt,
                              size_t tgt_step, int rows, int cols, int window_rad, int min_disp, int max_disp,
                              void* disp_out, size_t disp_step, int disp_elem_bytes, void* best_out, size_t best_step) {
    return host_single(ctx, cost, PixType::F32, ref, ref_step, tgt, tgt_step, rows, cols, window_rad, min_disp,
                       max_disp, disp_out, disp_step, disp_elem_bytes, best_out, best_step);
}

int stereo_disparity_u8_host(stereo_ctx* ctx, int cost, const uint8_t* ref, size_t ref_step, const uint8_t* tgt,
                             size_t tgt_step, int rows, int cols, int window_rad, int min_disp, int max_disp,
                             void* disp_out, size_t disp_step, int disp_elem_bytes, void* best_out, size_t best_step) {
    return host_single(ctx, cost, PixType::U8, ref, ref_step, tgt, tgt_step, rows, cols, window_rad, min_disp,
                       max_disp, disp_out, disp_step, disp_elem_bytes, best_out, best_step);
}

// ---- device images and preprocessing (imgproc.cuh) ---------------------------------------------------------------------------
int stereo_dev_alloc(stereo_ctx* ctx, size_t bytes, void** ptr) {
    int rc = check_ctx(ctx);
    if (rc != STEREO_OK) return rc;
    if (!ptr || bytes == 0) { set_error("bad allocation arguments"); return STEREO_ERR_INVALID_ARG; }
    if (cudaMalloc(ptr, bytes) != cudaSuccess) { (void)cudaGetLastError(); *ptr = nullptr; set_error("device allocation of %zu bytes failed", bytes); return STEREO_ERR_ALLOC; }
    return STEREO_OK;
}

int stereo_dev_free(stereo_ctx* ctx, void* ptr) {
    int rc = check_ctx(ctx);
    if (rc != STEREO_OK) return rc;
    if (ptr) { SB_CUDA(cudaStreamSynchronize(ctx->stream)); SB_CUDA(cudaFree(ptr)); }
    return STEREO_OK;
}

int stereo_dev_upload(stereo_ctx* ctx, void* dst, size_t dst_step, const void* src, size_t src_step, size_t row_bytes, int rows) {
    int rc = check_ctx(ctx);
    if (rc != STEREO_OK) return rc;
    if (!dst || !src || rows <= 0 || row_bytes == 0 || dst_step < row_bytes || src_step < row_bytes) { set_error("bad upload arguments"); return STEREO_ERR_INVALID_ARG; }
    SB_CUDA(cudaMemcpy2DAsync(dst, dst_step, src, src_step, row_bytes, rows, cudaMemcpyHostToDevice, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));          // the host buffer is the caller's again
    return STEREO_OK;
}

int stereo_dev_download(stereo_ctx* ctx, void* dst, size_t dst_step, const void* src, size_t src_step, size_t row_bytes, int rows) {
    int rc = check_ctx(ctx);
    if (rc != STEREO_OK) return rc;
    if (!dst || !src || rows <= 0 || row_bytes == 0 || dst_step < row_bytes || src_step < row_bytes) { set_error("bad download arguments"); return STEREO_ERR_INVALID_ARG; }
    SB_CUDA(cudaMemcpy2DAsync(dst, dst_step, src, src_step, row_bytes, rows, cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return STEREO_OK;
}

int stereo_image_gray_f32_device(stereo_ctx* ctx, const uint8_t* img, size_t step, int rows, int cols, int channels, int shift,
                                 float* out, size_t out_step, void* cuda_stream) {
    int rc = check_ctx(ctx);
    if (rc != STEREO_OK) return rc;
    if (!img || !out || rows <= 0 || cols <= 0 || (channels != 1 && channels != 3 && channels != 4) || (shift != 14 && shift != 15) ||
        step < size_t(cols) * channels || out_step < size_t(cols) * 4) { set_error("bad gray conversion arguments"); return STEREO_ERR_INVALID_ARG; }
    cudaStream_t st = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->stream;
    gray_f32_kernel<<<dim3(div_round_up(cols, 256), rows), 256, 0, st>>>(img, step, rows, cols, channels, shift, out, out_step);
    SB_CUDA(cudaGetLastError());
    return STEREO_OK;
}

int stereo_image_scale_add_f32_device(stereo_ctx* ctx, const float* a, size_t a_step, const float* add, size_t add_step, float scale,
                                      int rows, int cols, float* out, size_t out_step, void* cuda_stream) {
    int rc = check_ctx(ctx);
    if (rc != STEREO_OK) return rc;
    if (!a || !out || rows <= 0 || cols <= 0 || a_step < size_t(cols) * 4 || out_step < size_t(cols) * 4 || (add && add_step < size_t(cols) * 4)) {
        set_error("bad scale/add arguments"); return STEREO_ERR_INVALID_ARG;
    }
    cudaStream_t st = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->stream;
    scale_add_f32_kernel<<<dim3(div_round_up(cols, 256), rows), 256, 0, st>>>(a, a_step, add, add_step, scale, rows, cols, out, out_step);
    SB_CUDA(cudaGetLastError());
    return STEREO_OK;
}

// ---- reference-GPU-semantics mode (compat.cuh) ------------------------------------------------------------------------------
int stereo_disparity_refgpu_f32_device(stereo_ctx* ctx, int cost, const float* ref, size_t ref_step, const float* tgt, size_t tgt_step,
                                       int rows, int cols, int window_rad, int min_disp, int max_disp, int8_t* disp_out,
                                       size_t disp_step, float* best_out, size_t best_step, void* cuda_stream) {
    int rc = check_ctx(ctx);
    if (rc != STEREO_OK) return rc;
    if (!ref || !tgt || !disp_out) { set_error("null pointer"); return STEREO_ERR_INVALID_ARG; }
    if (rows <= 0 || cols <= 0 || rows > 32768 || cols > 32768) { set_error("bad image size %d x %d", rows, cols); return STEREO_ERR_INVALID_ARG; }
    if (cost != STEREO_COST_SSD && cost != STEREO_COST_NCORR) { set_error("unknown cost %d", cost); return STEREO_ERR_INVALID_ARG; }
    if (ref_step < size_t(cols) * 4 || tgt_step < size_t(cols) * 4 || disp_step < size_t(cols) || (best_out && best_step < size_t(cols) * 4)) {
        set_error("a step is smaller than its row"); return STEREO_ERR_INVALID_ARG;
    }
    if (window_rad < 0 || window_rad > 64) { set_error("window_rad must be in [0, 64]"); return STEREO_ERR_INVALID_ARG; }
    if (min_disp > max_disp) { set_error("min_disp (%d) > max_disp (%d)", min_disp, max_disp); return STEREO_ERR_INVALID_RANGE; }
    // the reference's loop variable is a `char` (DisparitySSD.cu:41,56): ranges beyond int8 never terminate there
    if (min_disp < -128 || max_disp > 126) { set_error("the reference's GPU kernels index disparities with a char: range must lie in [-128, 126]"); return STEREO_ERR_INVALID_RANGE; }
    cudaStream_t st = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->stream;
    begin_call(ctx, st);
    const dim3 grid(div_round_up(cols, CG_TILE), div_round_up(rows, CG_ROWS));
    const int threads = CG_TILE + 2 * window_rad;
    const size_t smem = size_t(3) * threads * sizeof(float);
    if (cost == STEREO_COST_SSD)
        refgpu_kernel<STEREO_COST_SSD><<<grid, threads, smem, st>>>(ref, ref_step, tgt, tgt_step, rows, cols, window_rad, min_disp, max_disp, disp_out, disp_step, best_out, best_step);
    else
        refgpu_kernel<STEREO_COST_NCORR><<<grid, threads, smem, st>>>(ref, ref_step, tgt, tgt_step, rows, cols, window_rad, min_disp, max_disp, disp_out, disp_step, best_out, best_step);
    ctx->last_launches += 1;
    ctx->last_path = STEREO_PATH_REFGPU;
    end_call(ctx, st);
    SB_CUDA(cudaGetLastError());
    return STEREO_OK;
}

int stereo_disparity_refgpu_f32_host(stereo_ctx* ctx, int cost, const float* ref, size_t ref_step, const float* tgt, size_t tgt_step,
                                     int rows, int cols, int window_rad, int min_disp, int max_disp, int8_t* disp_out,
                                     size_t disp_step, float* best_out, size_t best_step) {
    const size_t row = size_t(cols) * 4;
    const int rc = check_host_args(ctx, {ref, tgt, disp_out}, rows, cols, 1, {{ref_step, row}, {tgt_step, row}});
    if (rc != STEREO_OK) return rc;
    const HostRows in[2] = {{ref, ref_step, row}, {tgt, tgt_step, row}};
    const HostMap out[2] = {{disp_out, disp_step, size_t(cols)}, {best_out, best_step, row}};
    return staged_host_call(ctx, in, rows, out, rows, [&](const DevRows* d, const DevRows* o) {
        return stereo_disparity_refgpu_f32_device(ctx, cost, reinterpret_cast<const float*>(d[0].ptr), d[0].pitch,
                                                  reinterpret_cast<const float*>(d[1].ptr), d[1].pitch, rows, cols, window_rad, min_disp,
                                                  max_disp, reinterpret_cast<int8_t*>(o[0].ptr), o[0].pitch,
                                                  reinterpret_cast<float*>(o[1].ptr), o[1].pitch, ctx->stream);
    });
}

int stereo_disparity_f32_device(stereo_ctx* ctx, int cost, const float* ref, size_t ref_step, const float* tgt,
                                size_t tgt_step, int rows, int cols, int window_rad, int min_disp, int max_disp,
                                void* disp_out, size_t disp_step, int disp_elem_bytes, void* best_out,
                                size_t best_step, void* cuda_stream) {
    return device_single(ctx, direction(cost, PixType::F32, ref, ref_step, tgt, tgt_step, rows, cols, 0, rows, 0, rows, window_rad,
                                        min_disp, max_disp, disp_out, disp_step, disp_elem_bytes, best_out, best_step), cuda_stream);
}

int stereo_disparity_u8_device(stereo_ctx* ctx, int cost, const uint8_t* ref, size_t ref_step, const uint8_t* tgt,
                               size_t tgt_step, int rows, int cols, int window_rad, int min_disp, int max_disp,
                               void* disp_out, size_t disp_step, int disp_elem_bytes, void* best_out,
                               size_t best_step, void* cuda_stream) {
    return device_single(ctx, direction(cost, PixType::U8, ref, ref_step, tgt, tgt_step, rows, cols, 0, rows, 0, rows, window_rad,
                                        min_disp, max_disp, disp_out, disp_step, disp_elem_bytes, best_out, best_step), cuda_stream);
}

int stereo_disparity_band_u8_device(stereo_ctx* ctx, int cost, const uint8_t* ref, size_t ref_step,
                                    const uint8_t* tgt, size_t tgt_step, int rows, int cols, int row_begin,
                                    int row_end, int window_rad, int min_disp, int max_disp, void* disp_out,
                                    size_t disp_step, int disp_elem_bytes, void* cuda_stream) {
    return device_single(ctx, direction(cost, PixType::U8, ref, ref_step, tgt, tgt_step, rows, cols, row_begin, row_end, 0, rows,
                                        window_rad, min_disp, max_disp, disp_out, disp_step, disp_elem_bytes, nullptr, 0), cuda_stream);
}

int stereo_disparity_band_halo_u8_device(stereo_ctx* ctx, int cost, const uint8_t* ref_halo, size_t ref_step,
                                         const uint8_t* tgt_halo, size_t tgt_step, int rows, int cols, int row_begin,
                                         int row_end, int halo_begin, int halo_end, int window_rad, int min_disp,
                                         int max_disp, void* disp_out, size_t disp_step, int disp_elem_bytes,
                                         void* cuda_stream) {
    if (!ref_halo || !tgt_halo) { set_error("null image pointer"); return STEREO_ERR_INVALID_ARG; }
    if (halo_begin < 0 || halo_end > rows || halo_begin >= halo_end) { set_error("bad halo rows [%d, %d)", halo_begin, halo_end); return STEREO_ERR_INVALID_ARG; }
    // Full-image origins that are never dereferenced outside [halo_begin, halo_end): every row index is clamped
    // into the available range, which changes nothing when the halo covers what the band needs.
    const uint8_t* ref0 = ref_halo - size_t(halo_begin) * ref_step;
    const uint8_t* tgt0 = tgt_halo - size_t(halo_begin) * tgt_step;
    return device_single(ctx, direction(cost, PixType::U8, ref0, ref_step, tgt0, tgt_step, rows, cols, row_begin, row_end, halo_begin,
                                        halo_end, window_rad, min_disp, max_disp, disp_out, disp_step, disp_elem_bytes, nullptr, 0),
                         cuda_stream);
}

int stereo_band_halo_rows(int rows, int row_begin, int row_end, int window_rad, int* halo_begin, int* halo_end) {
    if (!halo_begin || !halo_end || rows <= 0 || row_begin < 0 || row_end > rows || row_begin >= row_end || window_rad < 0) {
        set_error("bad arguments"); return STEREO_ERR_INVALID_ARG;
    }
    // R rows of window above and below, +1 for the neighbouring padded row the reference's SSD reads
    // through its flat index (SURVEY.md A.1 item 3); clamped to the image (replicate padding).
    int b = row_begin - window_rad - 1, e = row_end + window_rad + 1;
    *halo_begin = b < 0 ? 0 : b;
    *halo_end = e > rows ? rows : e;
    return STEREO_OK;
}

// ---- pairs: L->R over [-range, 0], then R->L with images swapped over [0, +range] (main.cpp:21-48) ----

// Both maps of a pair of device images, or of a row band of them (avail_begin / avail_end as in direction()).
static int pair_device(stereo_ctx* ctx, int cost, PixType type, const void* left, size_t left_step, const void* right,
                       size_t right_step, int rows, int cols, int row_begin, int row_end, int avail_begin, int avail_end, int R,
                       int range, void* disp_left, void* disp_right, size_t disp_step, int elem, void* stream) {
    if (range < 0) { set_error("disparity_range must be >= 0"); return STEREO_ERR_INVALID_RANGE; }
    Problem p[2];
    pair_problems(p, 1, 0, cost, type, left, left_step, right, right_step, rows, cols, row_begin, row_end, avail_begin, avail_end, R,
                  range, disp_left, disp_right, disp_step, elem);
    return device_call(ctx, p, 2, stream);
}

static int pair_host(stereo_ctx* ctx, int cost, PixType type, const void* left, size_t left_step, const void* right,
                     size_t right_step, int rows, int cols, int R, int range, void* disp_left, void* disp_right,
                     size_t disp_step, int elem) {
    const size_t row = size_t(cols) * (type == PixType::F32 ? 4 : 1), disp_row = size_t(cols) * elem;
    int rc = check_host_args(ctx, {left, right, disp_left, disp_right}, rows, cols, elem,
                             {{left_step, row}, {right_step, row}, {disp_step, disp_row}}, range);
    if (rc == STEREO_OK) rc = check_pair_options(ctx, cost, type, elem, range, R, cols, 0, rows, rows);      // (as run_directions would, but before staging)
    if (rc != STEREO_OK) return rc;
    {
        const HostPairIn in{left, left_step, right, right_step};
        void* outs_l[1] = {disp_left};
        void* outs_r[1] = {disp_right};
        const HostDir dirs[2] = {{false, -range, 0, outs_l}, {true, 0, range, outs_r}};
        rc = pairs_host_pipelined(ctx, cost, type, 1, &in, dirs, 2, rows, cols, R, disp_step, elem);
        if (rc <= STEREO_OK) return rc;
    }
    const HostRows in[2] = {{left, left_step, row}, {right, right_step, row}};
    const HostMap out[2] = {{disp_left, disp_step, disp_row}, {disp_right, disp_step, disp_row}};
    return staged_host_call(ctx, in, rows, out, rows, [&](const DevRows* d, const DevRows* o) {
        return pair_device(ctx, cost, type, d[0].ptr, d[0].pitch, d[1].ptr, d[1].pitch, rows, cols, 0, rows, 0, rows, R, range,
                           o[0].ptr, o[1].ptr, o[0].pitch, elem, ctx->stream);
    });
}

int stereo_disparity_pair_f32_host(stereo_ctx* ctx, int cost, const float* left, size_t left_step, const float* right,
                                   size_t right_step, int rows, int cols, int window_rad, int disparity_range,
                                   void* disp_left, void* disp_right, size_t disp_step, int disp_elem_bytes) {
    return pair_host(ctx, cost, PixType::F32, left, left_step, right, right_step, rows, cols, window_rad,
                     disparity_range, disp_left, disp_right, disp_step, disp_elem_bytes);
}

int stereo_disparity_pair_u8_host(stereo_ctx* ctx, int cost, const uint8_t* left, size_t left_step,
                                  const uint8_t* right, size_t right_step, int rows, int cols, int window_rad,
                                  int disparity_range, void* disp_left, void* disp_right, size_t disp_step,
                                  int disp_elem_bytes) {
    return pair_host(ctx, cost, PixType::U8, left, left_step, right, right_step, rows, cols, window_rad,
                     disparity_range, disp_left, disp_right, disp_step, disp_elem_bytes);
}

int stereo_disparity_pair_u8_device(stereo_ctx* ctx, int cost, const uint8_t* left, size_t left_step,
                                    const uint8_t* right, size_t right_step, int rows, int cols, int window_rad,
                                    int disparity_range, void* disp_left, void* disp_right, size_t disp_step,
                                    int disp_elem_bytes, void* cuda_stream) {
    const int rc = check_ctx(ctx);
    if (rc != STEREO_OK) return rc;
    return pair_device(ctx, cost, PixType::U8, left, left_step, right, right_step, rows, cols, 0, rows, 0, rows, window_rad,
                       disparity_range, disp_left, disp_right, disp_step, disp_elem_bytes, cuda_stream);
}

int stereo_disparity_pair_f32_device(stereo_ctx* ctx, int cost, const float* left, size_t left_step, const float* right,
                                     size_t right_step, int rows, int cols, int window_rad, int disparity_range,
                                     void* disp_left, void* disp_right, size_t disp_step, int disp_elem_bytes,
                                     void* cuda_stream) {
    const int rc = check_ctx(ctx);
    if (rc != STEREO_OK) return rc;
    return pair_device(ctx, cost, PixType::F32, left, left_step, right, right_step, rows, cols, 0, rows, 0, rows, window_rad,
                       disparity_range, disp_left, disp_right, disp_step, disp_elem_bytes, cuda_stream);
}

// Both maps of a row band from one launch sequence (one rank's share of a row-band sharded PAIR, BASELINE config 4).
int stereo_disparity_pair_band_halo_u8_device(stereo_ctx* ctx, int cost, const uint8_t* left_halo, size_t left_step,
                                              const uint8_t* right_halo, size_t right_step, int rows, int cols,
                                              int row_begin, int row_end, int halo_begin, int halo_end, int window_rad,
                                              int disparity_range, void* disp_left, void* disp_right, size_t disp_step,
                                              int disp_elem_bytes, void* cuda_stream) {
    const int rc = check_ctx(ctx);
    if (rc != STEREO_OK) return rc;
    if (!left_halo || !right_halo || !disp_left || !disp_right) { set_error("null pointer"); return STEREO_ERR_INVALID_ARG; }
    if (halo_begin < 0 || halo_end > rows || halo_begin >= halo_end) { set_error("bad halo rows [%d, %d)", halo_begin, halo_end); return STEREO_ERR_INVALID_ARG; }
    const uint8_t* l0 = left_halo - size_t(halo_begin) * left_step;       // full-image origins, see above
    const uint8_t* r0 = right_halo - size_t(halo_begin) * right_step;
    return pair_device(ctx, cost, PixType::U8, l0, left_step, r0, right_step, rows, cols, row_begin, row_end, halo_begin, halo_end,
                       window_rad, disparity_range, disp_left, disp_right, disp_step, disp_elem_bytes, cuda_stream);
}

// ---- one row band of a pair from HOST images (a device's share of a row-band sharded pair) ------------------------------
// Uploads only the slab of rows the band needs (window halo + the row of the SSD flat-index wrap), computes both maps of
// the band in one launch sequence and downloads them into the caller's band rows.  CV_32FC1 images are converted to u8 on
// the host while the slab is staged; an image that is not 8-bit-valued makes the call return STEREO_ERR_UNSUPPORTED (the
// band entry points are 8-bit only; callers then take a whole-image call).
static int pair_band_host(stereo_ctx* ctx, int cost, PixType type, const void* left, size_t left_step, const void* right,
                          size_t right_step, int rows, int cols, int row_begin, int row_end, int R, int range,
                          void* disp_left, void* disp_right, size_t disp_step, int elem) {
    const size_t row = size_t(cols) * (type == PixType::F32 ? 4 : 1), disp_row = size_t(cols) * elem;
    int rc = check_host_args(ctx, {left, right, disp_left, disp_right}, rows, cols, elem,
                             {{left_step, row}, {right_step, row}, {disp_step, disp_row}}, range, STEREO_ERR_INVALID_ARG);
    if (rc != STEREO_OK) return rc;
    int h0 = 0, h1 = 0;
    rc = stereo_band_halo_rows(rows, row_begin, row_end, R, &h0, &h1);      // (rejects a bad band or window radius)
    if (rc != STEREO_OK) return rc;
    rc = check_pair_options(ctx, cost, type, elem, range, R, cols, row_begin, row_end, rows);      // (as run_directions would, but before staging)
    if (rc != STEREO_OK) return rc;
    const int nh = h1 - h0;
    HostRows in[2] = {{static_cast<const char*>(left) + size_t(h0) * left_step, left_step, size_t(cols)},
                      {static_cast<const char*>(right) + size_t(h0) * right_step, right_step, size_t(cols)}};
    if (type == PixType::F32) {
        const size_t stg_pitch = (size_t(cols) + 63) & ~size_t(63);
        SB_CUDA(cudaStreamSynchronize(ctx->stream));            // (the staging may still feed an earlier upload)
        rc = ensure_pinned(ctx, 2 * stg_pitch * nh);
        if (rc != STEREO_OK) return rc;
        if (ctx->host_threads == 0) ctx->host_threads = default_host_threads();
        const int nt = ctx->host_threads > 0 ? ctx->host_threads : 1;
        if (!ctx->pool || ctx->pool->threads() != nt) { delete ctx->pool; ctx->pool = new (std::nothrow) HostPool(nt); }
        if (!ctx->pool) { set_error("out of host memory"); return STEREO_ERR_ALLOC; }
        uint8_t* sl = static_cast<uint8_t*>(ctx->pinned);
        uint8_t* sr = sl + stg_pitch * nh;
        const bool ok = pack_f32_u8(*ctx->pool, static_cast<const float*>(in[0].ptr), left_step, sl, stg_pitch, nh, cols) &&
                        pack_f32_u8(*ctx->pool, static_cast<const float*>(in[1].ptr), right_step, sr, stg_pitch, nh, cols);
        if (!ok) { set_error("row-band entry points take 8-bit-valued images only"); return STEREO_ERR_UNSUPPORTED; }
        in[0] = HostRows{sl, stg_pitch, size_t(cols)};
        in[1] = HostRows{sr, stg_pitch, size_t(cols)};
    }
    const HostMap out[2] = {{disp_left, disp_step, disp_row}, {disp_right, disp_step, disp_row}};
    return staged_host_call(ctx, in, nh, out, row_end - row_begin, [&](const DevRows* d, const DevRows* o) {
        return stereo_disparity_pair_band_halo_u8_device(ctx, cost, reinterpret_cast<const uint8_t*>(d[0].ptr), d[0].pitch,
                                                         reinterpret_cast<const uint8_t*>(d[1].ptr), d[1].pitch, rows, cols, row_begin,
                                                         row_end, h0, h1, R, range, o[0].ptr, o[1].ptr, o[0].pitch, elem, ctx->stream);
    });
}

int stereo_disparity_pair_band_u8_host(stereo_ctx* ctx, int cost, const uint8_t* left, size_t left_step, const uint8_t* right,
                                       size_t right_step, int rows, int cols, int row_begin, int row_end, int window_rad,
                                       int disparity_range, void* disp_left, void* disp_right, size_t disp_step, int disp_elem_bytes) {
    return pair_band_host(ctx, cost, PixType::U8, left, left_step, right, right_step, rows, cols, row_begin, row_end, window_rad,
                          disparity_range, disp_left, disp_right, disp_step, disp_elem_bytes);
}

int stereo_disparity_pair_band_f32_host(stereo_ctx* ctx, int cost, const float* left, size_t left_step, const float* right,
                                        size_t right_step, int rows, int cols, int row_begin, int row_end, int window_rad,
                                        int disparity_range, void* disp_left, void* disp_right, size_t disp_step, int disp_elem_bytes) {
    return pair_band_host(ctx, cost, PixType::F32, left, left_step, right, right_step, rows, cols, row_begin, row_end, window_rad,
                          disparity_range, disp_left, disp_right, disp_step, disp_elem_bytes);
}

int stereo_disparity_pair_batch_u8_device(stereo_ctx* ctx, int cost, int n_pairs, const uint8_t* left,
                                          const uint8_t* right, size_t img_step, size_t pair_stride, int rows,
                                          int cols, int window_rad, int disparity_range, void* disp_left,
                                          void* disp_right, size_t disp_step, size_t disp_pair_stride,
                                          int disp_elem_bytes, void* cuda_stream) {
    int rc = check_ctx(ctx);
    if (rc != STEREO_OK) return rc;
    if (n_pairs <= 0) { set_error("n_pairs must be positive"); return STEREO_ERR_INVALID_ARG; }
    if (!left || !right || !disp_left || !disp_right) { set_error("null pointer"); return STEREO_ERR_INVALID_ARG; }
    cudaStream_t st = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->stream;
    if (disparity_range < 0) { set_error("disparity_range must be >= 0"); return STEREO_ERR_INVALID_RANGE; }
    begin_call(ctx, st);
    // jobs of FMAXJOBS/2 pairs at a time: up to FMAXJOBS directions share one launch sequence
    constexpr int CHUNK = FMAXJOBS / 2;
    Problem ps[FMAXJOBS];
    for (int i0 = 0; i0 < n_pairs && rc == STEREO_OK; i0 += CHUNK) {
        const int np = (n_pairs - i0 < CHUNK) ? n_pairs - i0 : CHUNK;
        for (int k = 0; k < np; ++k) {
            const int i = i0 + k;
            pair_problems(ps, np, k, cost, PixType::U8, left + size_t(i) * pair_stride, img_step, right + size_t(i) * pair_stride,
                          img_step, rows, cols, 0, rows, 0, rows, window_rad, disparity_range,
                          static_cast<char*>(disp_left) + size_t(i) * disp_pair_stride,
                          static_cast<char*>(disp_right) + size_t(i) * disp_pair_stride, disp_step, disp_elem_bytes);
        }
        rc = run_directions(ctx, ps, 2 * np, st);
    }
    end_call(ctx, st);
    return rc;
}

// Host batches, both pixel types.  Strides are in bytes.
static int pair_batch_host(stereo_ctx* ctx, int cost, PixType type, int n_pairs, const void* left_v, const void* right_v,
                           size_t img_step, size_t pair_stride, int rows, int cols, int window_rad, int disparity_range,
                           void* disp_left, void* disp_right, size_t disp_step, size_t disp_pair_stride, int disp_elem_bytes) {
    const char* left = static_cast<const char*>(left_v);
    const char* right = static_cast<const char*>(right_v);
    const size_t px = type == PixType::F32 ? 4 : 1;
    if (n_pairs <= 0) { set_error("n_pairs must be positive"); return STEREO_ERR_INVALID_ARG; }
    int rc = check_host_args(ctx, {left, right, disp_left, disp_right}, rows, cols, disp_elem_bytes,
                             {{img_step, size_t(cols) * px}, {disp_step, size_t(cols) * disp_elem_bytes}}, disparity_range);
    if (rc == STEREO_OK) rc = check_pair_options(ctx, cost, type, disp_elem_bytes, disparity_range, window_rad, cols, 0, rows, rows);
    if (rc != STEREO_OK) return rc;
    {   // pipelined: item i+1 uploads while item i computes and item i-1 downloads (3 device slots)
        std::vector<HostPairIn> in(n_pairs);
        std::vector<void*> outs_l(n_pairs), outs_r(n_pairs);
        for (int i = 0; i < n_pairs; ++i) {
            in[i] = HostPairIn{left + size_t(i) * pair_stride, img_step, right + size_t(i) * pair_stride, img_step};
            outs_l[i] = static_cast<char*>(disp_left) + size_t(i) * disp_pair_stride;
            outs_r[i] = static_cast<char*>(disp_right) + size_t(i) * disp_pair_stride;
        }
        const HostDir dirs[2] = {{false, -disparity_range, 0, outs_l.data()}, {true, 0, disparity_range, outs_r.data()}};
        rc = pairs_host_pipelined(ctx, cost, type, n_pairs, in.data(), dirs, 2, rows, cols, window_rad, disp_step, disp_elem_bytes);
        if (rc <= STEREO_OK) return rc;
    }
    // Sequential fallback (parameters the packed kernels do not cover, or float images that are not 8-bit):
    // pair by pair through the single-pair host path (which picks the exact kernels where needed).
    int launches = 0;
    for (int i = 0; i < n_pairs; ++i) {
        rc = pair_host(ctx, cost, type, left + size_t(i) * pair_stride, img_step, right + size_t(i) * pair_stride, img_step, rows, cols,
                       window_rad, disparity_range, static_cast<char*>(disp_left) + size_t(i) * disp_pair_stride,
                       static_cast<char*>(disp_right) + size_t(i) * disp_pair_stride, disp_step, disp_elem_bytes);
        if (rc != STEREO_OK) return rc;
        launches += ctx->last_launches;
    }
    ctx->last_launches = launches;
    return STEREO_OK;
}

int stereo_disparity_pair_batch_u8_host(stereo_ctx* ctx, int cost, int n_pairs, const uint8_t* left,
                                        const uint8_t* right, size_t img_step, size_t pair_stride, int rows, int cols,
                                        int window_rad, int disparity_range, void* disp_left, void* disp_right,
                                        size_t disp_step, size_t disp_pair_stride, int disp_elem_bytes) {
    return pair_batch_host(ctx, cost, PixType::U8, n_pairs, left, right, img_step, pair_stride, rows, cols, window_rad,
                           disparity_range, disp_left, disp_right, disp_step, disp_pair_stride, disp_elem_bytes);
}

int stereo_disparity_pair_batch_f32_host(stereo_ctx* ctx, int cost, int n_pairs, const float* left,
                                         const float* right, size_t img_step, size_t pair_stride, int rows, int cols,
                                         int window_rad, int disparity_range, void* disp_left, void* disp_right,
                                         size_t disp_step, size_t disp_pair_stride, int disp_elem_bytes) {
    return pair_batch_host(ctx, cost, PixType::F32, n_pairs, left, right, img_step, pair_stride, rows, cols, window_rad,
                           disparity_range, disp_left, disp_right, disp_step, disp_pair_stride, disp_elem_bytes);
}

} // extern "C"
