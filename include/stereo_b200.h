/*
 * stereo_b200.h — C ABI of the B200-native (sm_100a) dense stereo block matcher.
 *
 * This is the drop-in boundary for ONE path of tanmaniac/IntroToComputerVision: the Problem Set 2
 * window-based stereo matcher.  Every entry point cites the reference interface it replaces; paths
 * are relative to the reference repository root.
 *
 *   cuda::disparitySSD     ProblemSets/ps2_cpp/include/DisparitySSD.h:18-23
 *                          (wrapper being replaced: ProblemSets/ps2_cpp/lib/DisparitySSD.cu:143-207)
 *   cuda::disparityNCorr   ProblemSets/ps2_cpp/include/DisparityNCorr.h:19-24
 *                          (wrapper being replaced: ProblemSets/ps2_cpp/lib/DisparityNCorr.cu:177-251)
 *   disparitySSDPair / disparityNCorrPair   ProblemSets/ps2_cpp/src/main.cpp:21-48, 51-78
 *
 * RESULTS follow the reference's CPU semantics (serial::disparitySSD, lib/DisparitySSD.cpp:9-62 and
 * serial::disparityNCorr, lib/DisparityNCorr.cpp:12-71) — the reference's GPU kernels compute a
 * different window and thresholds (SURVEY.md §A.3) and are not the parity target.
 *
 * Conventions
 *   - "ref" is the reference image (first argument of the reference functions), "tgt" the image
 *     that is searched.  L->R maps pass (left, right, -range, 0); R->L maps pass (right, left, 0,
 *     +range) — main.cpp:33,43.
 *   - Images are single channel, row-major; `*_step` arguments are row strides in BYTES
 *     (cv::Mat::step).  f32 images carry raw 0..255 intensities (no /255 — main.cpp:87-88) and may
 *     be non-integer/negative (main.cpp:140-153); u8 entry points are the same computation for
 *     images that are exactly 8-bit.
 *   - Disparity output element size is 1 (int8, the reference's CV_8SC1 with its `char` narrowing,
 *     DisparitySSD.cpp:59), 2 (int16) or 4 (int32); 2/4 hold the un-narrowed value, which is what
 *     >127-disparity searches need.
 *   - Every function returns STEREO_OK (0) or a negative stereo_status; nothing in this library
 *     calls exit() (the reference does: common/include/common/CudaCommon.cuh:11-22).
 *     stereo_last_error() returns a per-thread description of the last failure.
 *   - There is no CPU fallback: without a CUDA device every compute entry point fails with
 *     STEREO_ERR_NO_DEVICE.
 *   - A context owns all device buffers, streams and scratch; it is created once and reused (the
 *     reference re-allocates per call, DisparitySSD.cu:171-178).  A context is not thread-safe;
 *     use one per host thread.  Different contexts are independent (the reference's file-scope
 *     texture references, DisparitySSD.cu:19-20, made it non-reentrant).
 *   - Calls on one context execute in call order even when they are enqueued on different CUDA
 *     streams: all of them share the context's scratch arena, so a call enqueued on another stream
 *     than its predecessor first waits (on the device) for the predecessor's last kernel.  Use one
 *     context per stream for concurrent execution.
 */
#ifndef STEREO_B200_H_
#define STEREO_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define STEREO_B200_ABI_VERSION 1

typedef enum stereo_status {
    STEREO_OK = 0,
    STEREO_ERR_INVALID_ARG = -1,   /* null pointer, non-positive size, bad element size, step too small */
    STEREO_ERR_INVALID_RANGE = -2, /* min_disp > max_disp, or an NCC range that leaves a pixel without candidates */
    STEREO_ERR_NO_DEVICE = -3,     /* no CUDA device / wrong architecture (needs sm_100) */
    STEREO_ERR_CUDA = -4,          /* a CUDA runtime/driver call failed; see stereo_last_error() */
    STEREO_ERR_ALLOC = -5,         /* device or pinned-host allocation failed */
    STEREO_ERR_UNSUPPORTED = -6    /* parameter combination outside what the kernels cover */
} stereo_status;

typedef enum stereo_cost {
    STEREO_COST_SSD = 0,   /* sum of squared differences, argmin, first minimum wins   (DisparitySSD.cpp:45-57) */
    STEREO_COST_NCORR = 1  /* TM_CCORR_NORMED, argmax, first maximum wins              (DisparityNCorr.cpp:60-67) */
} stereo_cost;

/* Which kernel family served the last call (for tests and reports). */
typedef enum stereo_path {
    STEREO_PATH_NONE = 0,
    STEREO_PATH_EXACT_F32 = 1,  /* any float input, window and range: per-element reference arithmetic, no running sums */
    STEREO_PATH_FAST_U8 = 2,    /* integer-valued 0..255 inputs: packed dot-product running sums */
    STEREO_PATH_REFGPU = 4,     /* stereo_disparity_refgpu_*: the function the reference's GPU kernels compute (SURVEY.md A.3) */
    STEREO_PATH_SGM = 5,        /* pair calls with stereo_ctx_set_sgm on: semi-global matching (sgm.cuh) */
    STEREO_PATH_FAST_F32 = 3    /* general float inputs of bounded range (noise / contrast variants, main.cpp:140-153,191-193):
                                   per-element round((l-r)^2) as exact int32 running sums (SSD), float32 running sums (NCC).
                                   Bounds: SSD keys 128*SSD + position < 2^32 and (l-r)^2 < 2^23; NCC |v| < 1e6 and, when
                                   every value has one sign, (hi-lo)^2 / (lo^2 + hi^2) >= 2^-4 - a larger DC offset crowds
                                   every score towards 1 below the keys' ~2^-16 resolution (DESIGN.md §4.5) */
} stereo_path;

typedef struct stereo_ctx stereo_ctx;

/* ---- library / context ------------------------------------------------------------------- */

int stereo_abi_version(void);
const char* stereo_last_error(void);
const char* stereo_status_string(int status);

/* Number of visible CUDA devices of compute capability 10.x (0 if none / no driver). */
int stereo_device_count(void);

/* Creates a context on `device` (ordinal).  Replaces the per-call GpuMat/Stream setup of
 * DisparitySSD.cu:163-182 and common::warmup() (common/src/CudaWarmup.cu:14-19). */
int stereo_ctx_create(int device, stereo_ctx** ctx_out);
void stereo_ctx_destroy(stereo_ctx* ctx);

/* Kernel family used by the most recent compute call on this context (stereo_path). */
int stereo_ctx_last_path(const stereo_ctx* ctx);
/* Device time of the most recent compute call's kernels in milliseconds (cudaEvent pair; the
 * reference logs the same quantity, DisparitySSD.cu:192-203).  <0 if unavailable.  For the pipelined
 * HOST entry points the pair brackets the compute stream, which waits for every band's upload: the
 * figure then includes upload time the kernels were blocked on (stereo_ctx_last_hot_kernel_ms is
 * kernels only).  CV_32FC1 DEVICE calls: the time the device idles while the host reads the classification
 * verdict is left out (classification kernels + the kernels of the chosen family). */
float stereo_ctx_last_kernel_ms(const stereo_ctx* ctx);
/* Device time (ms) of the most recent call's HOT kernels only (the packed cost/WTA kernels; one launch
 * covers up to 32 directions of equally shaped problems), summed over the launches that were measured
 * (at most 16 per call); *launches_measured (nullable) receives how many that was.  <0 if the call used
 * no hot kernel.  This is the number the roofline report divides by. */
float stereo_ctx_last_hot_kernel_ms(const stereo_ctx* ctx, int* launches_measured);
/* Directions (disparity maps) the measured hot launches of the most recent call computed. */
int stereo_ctx_last_hot_jobs(const stereo_ctx* ctx);
/* Number of kernel launches issued by the most recent compute call. */
int stereo_ctx_last_launches(const stereo_ctx* ctx);
/* Force a kernel family (debug/testing): 0 = automatic, else a stereo_path value. */
int stereo_ctx_force_path(stereo_ctx* ctx, int path);
/* Host entry points overlap upload, compute and download by cutting each image pair into row bands
 * (with the window halo) that flow through three streams.  bands = 0 (default) picks the band count
 * from the image size and the number of pairs; bands >= 1 forces it (1 = whole images).  Results do not
 * depend on it.  The reference uploads, computes and downloads one after the other
 * (DisparitySSD.cu:171-206). */
int stereo_ctx_set_pipe_bands(stereo_ctx* ctx, int bands);

/* How the pipelined host entry points cut a call of `n_pairs` rows x cols pairs into work items: row bands per pair
 * (bands_override = stereo_ctx_set_pipe_bands' value, 0 = automatic) and pairs per item (small images ride several
 * pairs per launch sequence).  Pure host arithmetic, no device needed. */
int stereo_host_pipeline_plan(int n_pairs, int rows, int cols, int bands_override, int* bands_per_pair, int* pairs_per_item);
/* The row bands of work item `item` of such a call: writes the ascending boundaries (first 0, last rows) to bounds[0 .. n-1]
 * and returns n (negative: error; cap = room in bounds).  With automatic bands, 4K-sized images are cut unevenly: the
 * first item of a call begins and the last item ends with a band of an eighth of the image - the first upload and the last
 * download are the only copies no kernel overlaps - and the items in between go as whole images. */
int stereo_host_pipeline_item_bands(int n_pairs, int rows, int cols, int bands_override, int item, int* bounds, int cap);

/* CV_32FC1 HOST entry points: images whose pixels are all integers in 0..255 (everything convertTo(CV_32FC1) produces,
 * main.cpp:87-88) are converted to u8 by `threads` host threads into pinned staging and uploaded as 1 byte per pixel; the
 * reference uploads the float Mats (DisparitySSD.cu:171-174).  threads = 0 (default): min(16, hardware threads /
 * LOCAL_WORLD_SIZE), and host conversion only from 8 threads up (below that the floats are uploaded and converted on the
 * device); threads = -1: never convert on the host; threads >= 1: that many, always.  Results do not depend on it. */
int stereo_ctx_set_host_threads(stereo_ctx* ctx, int threads);
int stereo_ctx_host_threads(const stereo_ctx* ctx);
/* The conversion itself, on `threads` host threads (pure host code, no device needed): rows x cols float32 -> u8;
 * *all_8bit = 1 when every pixel is an integer in 0..255 (otherwise the u8 image is meaningless). */
int stereo_host_pack_f32_u8(const float* src, size_t src_step, uint8_t* dst, size_t dst_step, int rows, int cols, int threads,
                            int* all_8bit);
/* Self-test of the worker pool behind the conversion (pure host code): `rounds` dispatches of 1..257 tasks on ONE pool of
 * `threads` threads (blocking and begin / end form alternating), with pauses long enough for the polling workers to fall asleep; STEREO_OK when every task of every
 * dispatch ran exactly once (STEREO_ERR_UNSUPPORTED with the offending task in stereo_last_error() otherwise). */
int stereo_host_pool_selftest(int threads, int rounds);

/* How the hot kernel of a batch of `n_pairs` (<= 16) equally shaped pair problems would be launched on a device with
 * `sm_count` SMs (pure host arithmetic, no device needed; tests pin the scheduling decisions with it).
 * schedule: 0 = linear split of the (tile, row) space, 1 = equal row segments per tile (fewer tiles than SMs),
 * 2 = row-band-major items strided over the CTAs (many tiles: neighbouring tiles walk the same rows together). */
typedef struct stereo_launch_plan_t {
    int fused;            /* both maps from one cost volume */
    int strip_px;         /* pixels per thread (K) */
    int strips_per_warp;  /* 1, or 2 for searches of at most 64 candidates */
    int groups;           /* 128- (64-) disparity groups */
    int tile_px;          /* pixels per CTA tile */
    int tiles;            /* tiles of the launch */
    int ctas;             /* grid size */
    int schedule;
    int rows_per_item;    /* rows per CTA share (schedule 0, 1) or per band (2) */
    int bands;            /* schedule 2: row bands per tile */
    int stages;           /* TMA pipeline stages */
    int smem_bytes;
    int border_kernel;    /* fused SSD: candidates centred in the right padding come from fused_border_kernel */
} stereo_launch_plan_t;
int stereo_launch_plan(int cost, int float_operands, int n_pairs, int rows, int cols, int window_rad, int disparity_range, int fuse,
                       int sm_count, stereo_launch_plan_t* plan);

/* Pair calls (stereo_disparity_pair_*): compute BOTH maps of a pair from one cost volume where the kernels allow it -
 * SSD with any disparity_range and window_rad <= 7 on 8-bit-valued or float images, NCC on 8-bit-valued images - the
 * reference's disparitySSDPair / disparityNCorrPair always want both (main.cpp:21-78) and the window cost of (x, d) in
 * one direction IS the window cost of (x + d, -d) in the other.  SSD results are identical either way (bit-exact), NCC
 * results agree like any two evaluations of the same scores (per-pixel instead of per-strip key scales); on (the default)
 * is faster.  0 switches back to one cost volume per direction. */
int stereo_ctx_set_fuse_pairs(stereo_ctx* ctx, int on);
/* Image pairs of the last call whose two maps came out of one cost volume. */
int stereo_ctx_last_fused_pairs(const stereo_ctx* ctx);

/* Left-right consistency check of pair calls (OpenCV's disp12MaxDiff occlusion / mismatch filter), on the device right
 * after both maps are computed.  max_diff < 0 (the default) switches it off: results are then exactly those without it.
 * max_diff >= 0 switches it on for every pair entry point of this context - pair host and device, f32 and u8, the batches,
 * the host row band and the device band halo; single-direction and stereo_disparity_refgpu_* calls ignore it.  For every
 * output row y of every pair of a call, with both maps read as they were before any pixel was invalidated:
 *   left pixel x, value dL, is consistent when xr = x + dL lies in [0, cols) and |dL + dR(y, xr)| <= max_diff;
 *   right pixel x, value dR, is consistent when xl = x + dR lies in [0, cols) and |dR + dL(y, xl)| <= max_diff.
 * An inconsistent pixel gets -(disparity_range + 1) in either map (below every valid disparity of both, OpenCV's
 * minDisparity - 1); every other pixel keeps its value.  SSD candidates centred in the replicate padding have their
 * partner outside the image and so are inconsistent.  The sentinel must fit the map: disp_elem_bytes 1 needs
 * disparity_range <= 127, 2 needs <= 32767; a pair call with the check on that breaks this returns STEREO_ERR_UNSUPPORTED
 * before it enqueues or uploads anything and leaves the outputs untouched.  The check needs no scratch: device calls with
 * it stay capturable in CUDA graphs. */
int stereo_ctx_set_lr_check(stereo_ctx* ctx, int max_diff);
/* The context's current max_diff (-1: off). */
int stereo_ctx_lr_check(const stereo_ctx* ctx);
/* The same check in place on two device maps the caller holds: rows x cols elements of disp_elem_bytes each, row stride
 * disp_step bytes, disp_left over [-disparity_range, 0] and disp_right over [0, +disparity_range] (values outside those
 * ranges are checked by the same rule).  Asynchronous on `cuda_stream` (NULL = the context's stream), like every device
 * entry point.  max_diff must be >= 0; arguments are checked like those of the pair device entry points, and a sentinel
 * that does not fit the element type returns STEREO_ERR_UNSUPPORTED. */
int stereo_lr_check_device(stereo_ctx* ctx, void* disp_left, void* disp_right, size_t disp_step, int disp_elem_bytes,
                           int rows, int cols, int disparity_range, int max_diff, void* cuda_stream);

/* Speckle filter of pair calls (OpenCV's cv::filterSpeckles, StereoSGBM's speckleWindowSize / speckleRange), on the device
 * after both maps are computed and, with it on too, after the left-right check.  max_size <= 0 (the default) switches it
 * off: results are then exactly those without it.  max_size > 0 switches it on for the pair entry points of this context
 * that compute whole maps - pair host and device, f32 and u8, the batches - and needs max_diff >= 0
 * (STEREO_ERR_INVALID_ARG otherwise).  In each map, two 4-neighbours are connected when neither holds the sentinel and
 * their values differ by at most max_diff (disparity units); every pixel of a connected component of at most max_size
 * pixels gets the sentinel -(disparity_range + 1), every other pixel keeps its value.  Pixels the left-right check
 * invalidated therefore split regions.  The sentinel rule is the left-right check's (disp_elem_bytes 1 needs
 * disparity_range <= 127, 2 needs <= 32767; otherwise STEREO_ERR_UNSUPPORTED before anything is enqueued or uploaded).
 * A speckle region can cross a band seam, so the row-band entry points (stereo_disparity_pair_band_halo_u8_device,
 * stereo_disparity_pair_band_{u8,f32}_host) accept only the whole image as their band, and stereo_mgpu_disparity_pair_bands_*
 * refuse: those calls return STEREO_ERR_UNSUPPORTED and enqueue, upload and write nothing.  Callers of band-sharded pairs
 * filter the gathered maps with stereo_filter_speckles_device.  Single-direction and stereo_disparity_refgpu_* calls
 * ignore the setting.  The filter takes about 8 bytes of scratch per pixel and map from the context's arena; after one
 * call of a shape, device calls of that shape allocate nothing and stay capturable in CUDA graphs. */
int stereo_ctx_set_speckle_filter(stereo_ctx* ctx, int max_size, int max_diff);
/* The context's current setting (max_size 0: off). */
int stereo_ctx_speckle_filter(const stereo_ctx* ctx, int* max_size, int* max_diff);
/* cv::filterSpeckles(map, new_val, max_size, max_diff) in place on one device map the caller holds: rows x cols elements
 * of disp_elem_bytes each (signed), row stride disp_step bytes; the bytes past a row's cols elements are never touched.
 * Asynchronous on `cuda_stream` (NULL = the context's stream), like every device entry point.  A null map, a non-positive
 * size, an element size other than 1, 2 or 4, a short step, a negative max_size or max_diff or a new_val the element type
 * cannot hold return STEREO_ERR_INVALID_ARG; rows or cols over 32768 STEREO_ERR_UNSUPPORTED; max_size 0 is a valid no-op. */
int stereo_filter_speckles_device(stereo_ctx* ctx, void* disp, size_t disp_step, int disp_elem_bytes, int rows, int cols,
                                  int new_val, int max_size, int max_diff, void* cuda_stream);

/* Semi-global matching of pair calls: path aggregation of the matching cost along scanlines, in place of the
 * winner-take-all of the block matcher.  paths 0 (the default) switches it off: results are then exactly those without
 * it.  paths 4 or 8 switch it on for the pair entry points of this context that compute whole maps - pair host and
 * device, f32 and u8, the batches; any other paths, p1 < 0 or p1 > p2 return STEREO_ERR_INVALID_ARG and keep the old
 * setting.  Each direction of a pair is aggregated on its own (L->R over [-range, 0] referenced on the left image, R->L
 * over [0, +range] referenced on the right).  SSD: for reference image ref, radius R and padded column xp = x + R of a
 * Wp = cols + 2R wide padded image, candidate d is present at (y, x) when xp + d lies in [0, Wp - 1] (the candidates the
 * SSD single-direction call evaluates; d = 0 always is).  C(p, d) is that call's window sum for the candidate (replicate
 * padding, the flat-index row-wrap reads, per element round(float((l - r)^2)), integer accumulation).  NCC pair calls are
 * served only while an NCC scale q is set (stereo_ctx_set_sgm_ncc_scale), with C defined there.  For each path
 * direction r - (0,+-1), (+-1,0), and with 8 paths also (+-1,+-1) - and q = p - r:
 *     L_r(p, d) = C(p, d)                                                               where q is outside the image,
 *     L_r(p, d) = C(p, d) + min(L_r(q, d), L_r(q, d-1) + p1, L_r(q, d+1) + p1, m(q) + p2) - m(q)   otherwise,
 * with m(q) the minimum of L_r(q, .) over the candidates present at q; terms of candidates absent at q are left out.
 * S(p, d) is the sum of L_r(p, d) over the paths, and the disparity the first minimum of S over the present candidates in
 * ascending d, stored in the map's element type as every other call does (1-byte maps narrow like the reference's char).
 * For SSD, p1 = p2 = 0 gives L_r = C and so the SSD maps themselves (wherever every present window cost is below 99999999).
 * The left-right check, then the speckle filter, run on the SGM maps when they are on too (SGM -> check -> filter).
 * Refused with STEREO_ERR_UNSUPPORTED before anything is enqueued or written (float images: after their classification):
 * NCC pair calls while the NCC scale is 0; SSD with paths * ((2R + 1)^2 M + p2) > 2^31 - 1, with M = 255^2 for 8-bit-valued
 * images and ceil((hi - lo)^2) (widened by 1e-6 for float rounding) over the value range of other float images; float
 * images with a pixel that is not finite; more than 512 candidates after clipping [-range, range] to |d| <= cols - 1 + R
 * (SSD) or |d| <= cols - 1 (NCC).  Paths cross band seams, so
 * the row-band entry points (stereo_disparity_pair_band_halo_u8_device, stereo_disparity_pair_band_{u8,f32}_host) accept
 * only the whole image as their band and stereo_mgpu_disparity_pair_bands_* refuse.  Single-direction and
 * stereo_disparity_refgpu_* calls ignore the setting.  Calls served by SGM report STEREO_PATH_SGM, 0 fused pairs and no
 * hot-kernel time.  Scratch, from the context's arena, is 8 bytes per pixel and padded candidate (32 K >= the clipped
 * candidate count) for one direction at a time, plus the padded images; after one call of a shape, device calls of that
 * shape allocate nothing and stay capturable in CUDA graphs. */
int stereo_ctx_set_sgm(stereo_ctx* ctx, int paths, int p1, int p2);
/* The context's current setting (paths 0: off, with p1 = p2 = 0). */
int stereo_ctx_sgm(const stereo_ctx* ctx, int* paths, int* p1, int* p2);

/* Integer scale q of the NCC matching cost for SGM.  0 (the default): SGM refuses NCC pair calls, as before.
 * 1 <= q <= 2^24: NCC pair calls are served by SGM while stereo_ctx_set_sgm is on.  Other values: STEREO_ERR_INVALID_ARG,
 * old setting kept.  The scale and stereo_ctx_set_sgm are independent: switching SGM off keeps q, q alone changes nothing,
 * and SSD calls ignore it.
 * NCC cost.  Candidate d is present at (y, x) when 0 <= x + d <= cols - 1: the reference's own NCC candidates in both
 * directions (L->R over [-range, 0] right-aligned, DisparityNCorr.cpp:67; R->L over [0, range] from startX = x), so
 * [-range, range] is clipped to |d| <= cols - 1.  s(p, d) is the candidate's float32 TM_CCORR_NORMED score in the
 * reference's arithmetic (the double numerator summed in (wy, k) order and rounded to float32, double window energies in
 * the same order, the 10 FLT_EPSILON zero-energy rule and the 1.125 t rule; stereo_disparity_* with the exact kernels
 * return it as best_out), and
 *     C(p, d) = q - floor(fl32(q * s(p, d)))        in [0, 2q]
 * (the product is exact for a power-of-two q and correctly rounded otherwise).  L_r, S and the first minimum of S are as
 * above; the left-right check and the speckle filter follow.  Float images are classified once and refused when a pixel is
 * not finite.  paths * (2q + p2) > 2^31 - 1 returns STEREO_ERR_UNSUPPORTED before anything is enqueued, whatever the
 * image.  With p1 = p2 = 0 the map is the first d that maximises floor(fl32(q * s)): the block matcher's NCC map except
 * where a candidate before the block matcher's winner falls in the same quantum of q * s (not an exact identity, as it is
 * for SSD).  Scratch adds 16 bytes per pixel (the two images' window norms) to the SSD figure. */
int stereo_ctx_set_sgm_ncc_scale(stereo_ctx* ctx, int q);
/* The context's current q (0: off); STEREO_ERR_INVALID_ARG for a null context. */
int stereo_ctx_sgm_ncc_scale(const stereo_ctx* ctx);

/* Uniqueness ratio of pair calls (StereoSGBM's uniquenessRatio u), on the device before the left-right check and the
 * speckle filter (StereoSGBM's order: uniqueness -> check -> filter; the check and the filter see the pixels it rejected).
 * u = 0 (the default) switches it off: the rule below can then never fire and results are exactly those without it.
 * 1 <= u <= 99 switches it on for the pair entry points of this context that compute whole maps - pair host and device,
 * f32 and u8, the batches; any other u returns STEREO_ERR_INVALID_ARG and keeps the old setting.  For each map of each pair,
 * over the candidates d present at the pixel (SSD: xp + d in [0, Wp - 1]; NCC: x + d in [0, cols - 1]; as defined for SGM
 * above), V(d) is the value the map minimises - S(p, d) for SGM maps, the SSD window sum C(p, d) for block-matcher maps -
 * and j* its first minimum in ascending d (the map's own winner), V* = V(j*).  The pixel gets the sentinel
 * -(disparity_range + 1) when some present d with |d - j*| > 1 has
 *     V(d) (100 - u) < V* 100        (in 64-bit; StereoSGBM's integer form),
 * and, for block-matcher maps, when every present window cost is >= 99999999 (the map holds the reference's default 0
 * there: no candidate was accepted).  Every other pixel keeps its value.  StereoBM's form (sad[d] <= minsad (1 + u / 100))
 * is not offered: one rule serves both matchers.  OpenCV applies the ratio to its left map only; here it applies to both
 * maps of a pair, each against its own V, because each direction is matched on its own.
 * Refused with STEREO_ERR_UNSUPPORTED before anything is enqueued, uploaded or written (float images: after their
 * classification): a sentinel that does not fit the map (the left-right check's rule); NCC pair calls with SGM off (the NCC
 * block matcher ranks float32 scores, for which OpenCV has no ratio rule; NCC SGM maps are served); row bands other than the
 * whole image and stereo_mgpu_disparity_pair_bands_*; and, with SGM off, more than 512 candidates after clipping (as SGM)
 * or a window cost that can reach 2^30: (2R + 1)^2 M >= 2^30 with M as for SGM (255^2 for 8-bit images, ceil((hi - lo)^2)
 * of other float images, none for a pixel that is not finite).  Single-direction and stereo_disparity_refgpu_* calls
 * ignore the setting.
 * Block-matcher maps come from the same kernels as without it (same last path, same fused pairs); a second pass then
 * recomputes each direction's exact cost volume (SGM's cost kernel, 4 bytes per pixel and padded candidate, one direction
 * at a time, plus the padded images) and reads it once.  SGM maps apply the ratio in their last path at no extra scratch.
 * After one call of a shape, device calls of that shape allocate nothing and stay capturable in CUDA graphs. */
int stereo_ctx_set_uniqueness(stereo_ctx* ctx, int uniqueness_ratio);
/* The context's current u (0: off); STEREO_ERR_INVALID_ARG for a null context. */
int stereo_ctx_uniqueness(const stereo_ctx* ctx);

/* Sub-pixel disparity of pair calls: StereoSGBM's 1/16-pixel fixed point (DISP_SHIFT = 4), the parabola through the cost of
 * the winner and the costs of its two neighbours.
 * on = 0 (the default) switches it off, and results are then exactly those without it.  on = 1 switches it on for the pair
 * entry points of this context that compute whole maps - pair host and device, f32 and u8, the batches; any other value
 * returns STEREO_ERR_INVALID_ARG and keeps the old setting.
 * For each map of each pair, V is the value the map minimises over the present candidates, as for the uniqueness ratio:
 * S(p, d) for SGM maps (SSD cost, or NCC cost with scale q), the single-direction SSD window sum C(p, d) for block-matcher
 * maps.  Present is as defined for SGM above (SSD: xp + d in [0, Wp - 1]; NCC: x + d in [0, cols - 1]), each inside the
 * direction's candidate range.  With d the map's integer value at the pixel after every other step (uniqueness ratio,
 * texture threshold, left-right check, speckle filter), the pixel is written as
 *     16 sentinel                                                  where d is the sentinel -(disparity_range + 1),
 *     16 d + ((V(d-1) - V(d+1)) 16 + den) / (2 den),
 *            den = max(V(d-1) + V(d+1) - 2 V(d), 1)               where d - 1 and d + 1 are both present,
 *     16 d                                                         otherwise (a range edge or an absent neighbour),
 * in 64-bit, with C division (truncation toward zero): StereoSGBM's formula ("do subpixel quadratic interpolation",
 * stereosgbm.cpp) over ascending signed d, so L->R maps stay negative.  V(d) is the first minimum, so the offset lies in
 * [-7, 8] and (out + 7) >> 4 is the integer map without the option at every pixel, the sentinel included.  A block-matcher
 * pixel that accepted no candidate holds 0, a range edge in both directions, and stays 0.  Two differences from OpenCV:
 * the left-right check, the speckle filter and the texture threshold run on the integer maps, before the refinement
 * (OpenCV's validateDisparity and filterSpeckles see the 16S values); and both maps of a pair are refined, each against its
 * own V (OpenCV refines its left map only), as for the uniqueness ratio.
 *   Order: prefilter -> block matcher or SGM -> uniqueness ratio -> texture threshold -> left-right check -> speckle filter
 *   -> sub-pixel.
 * Refused with STEREO_ERR_UNSUPPORTED before anything is enqueued, uploaded or written: 1-byte maps; 2-byte maps with
 * disparity_range > 2047 (16 (disparity_range + 1) must fit); NCC pair calls with SGM off (the NCC block matcher ranks
 * float32 scores, which have no integer V; NCC SGM maps are served); row bands other than the whole image
 * (stereo_disparity_pair_band_halo_u8_device, stereo_disparity_pair_band_{u8,f32}_host) and
 * stereo_mgpu_disparity_pair_bands_*.  Single-direction and stereo_disparity_refgpu_* calls ignore the setting.  Host pair
 * calls take the staged whole-image path.
 * SGM maps: the last path kernel stores each pixel's offset in a grow-only buffer of the context (1 byte per pixel and map of
 * a launch sequence), applied by one launch at the end.  Block-matcher maps come from the same kernels as without it (same
 * last path, same fused pairs); a pass at the end pads each image once (4 bytes per padded pixel, from the context's arena)
 * and recomputes V(d - 1), V(d), V(d + 1) of each pixel.  After one call of a shape, device calls of that shape allocate
 * nothing and stay capturable in CUDA graphs. */
int stereo_ctx_set_subpixel(stereo_ctx* ctx, int on);
/* The context's current setting (0: off, 1: on); STEREO_ERR_INVALID_ARG for a null context. */
int stereo_ctx_subpixel(const stereo_ctx* ctx);

/* StereoBM's X-Sobel prefilter (preFilterCap, PREFILTER_XSOBEL) and texture threshold (textureThreshold) of pair calls.
 * cap = 0 (the default) switches both off; texture_threshold must then be 0, and results are exactly those without them.
 * 1 <= cap <= 63 (StereoBM's range) switches the prefilter on for the pair entry points of this context that compute whole
 * maps - pair host and device, f32 and u8, the batches; texture_threshold >= 0 adds the threshold (0 never fires).  Anything
 * else returns STEREO_ERR_INVALID_ARG and keeps the old setting.
 *   P = pf(I, cap), per image (OpenCV's prefilterXSobel), 8-bit: columns 0 and cols - 1 get cap; when rows is odd, the whole
 *   last row gets cap (OpenCV filters rows in pairs; rows == 1 too); every other pixel takes rows a = y - 1 and b = y + 1
 *   reflected 101-style (-1 -> 1, rows -> rows - 2) and
 *       v = (I[a][x+1] - I[a][x-1]) + 2 (I[y][x+1] - I[y][x-1]) + (I[b][x+1] - I[b][x-1]),   P = min(max(v, -cap), cap) + cap
 *   exactly for u8 images.  f32 images (OpenCV takes 8U only): d = fl32(I[.][x+1] - I[.][x-1]) per row,
 *   v = fl32(fl32(d_a + 2 d_y) + d_b), P = cap + clamp(rint(v), -cap, cap) rounding half to even, P = cap where v is NaN;
 *   for 8-bit-valued float images this equals the u8 result.
 *   Matching: pf(left) and pf(right) are computed once per pair; the L->R map matches ref pf(left) in tgt pf(right), R->L the
 *   other way round, with every definition above (SSD, NCC, SGM with the NCC scale, the uniqueness ratio) applied to the
 *   prefiltered images as to given ones.  Float pair calls then run as u8 calls (no classification, no host round trip).
 *   Texture: with T = texture_threshold, a pixel of a map gets the sentinel -(disparity_range + 1) when the sum of |P(q) - cap|
 *   over the (2R + 1)^2 window centred on it (coordinates clamped to the image, the matcher's replicate padding) is < T, P the
 *   map's own reference image prefiltered.  OpenCV thresholds its left map only; here both maps, each against its own
 *   reference, as for the uniqueness ratio.
 *   Order: prefilter -> block matcher or SGM -> uniqueness ratio -> texture threshold -> left-right check -> speckle filter.
 * Refused with STEREO_ERR_UNSUPPORTED before anything is enqueued, uploaded or written: row bands other than the whole image
 * (stereo_disparity_pair_band_halo_u8_device, stereo_disparity_pair_band_{u8,f32}_host) and
 * stereo_mgpu_disparity_pair_bands_* (the odd-height rule needs whole images: prefilter them with stereo_prefilter_*_device
 * below and call the band entry points with it off), and a texture threshold whose sentinel does not fit the map (the
 * left-right check's rule).  Single-direction and stereo_disparity_refgpu_* calls ignore the setting.  Host pair calls take
 * the staged whole-image path (CV_32FC1 host images are uploaded as floats).  The prefiltered images live in a grow-only
 * buffer of the context (2 x rows x align256(cols) bytes per pair of a launch sequence): after one call of a shape, device
 * calls of that shape allocate nothing and stay capturable in CUDA graphs. */
int stereo_ctx_set_prefilter(stereo_ctx* ctx, int cap, int texture_threshold);
/* The context's current cap (0: off) and texture threshold; STEREO_ERR_INVALID_ARG for a null argument. */
int stereo_ctx_prefilter(const stereo_ctx* ctx, int* cap, int* texture_threshold);

/* pf(src, cap) as defined above, one rows x cols image of DEVICE memory into the 8-bit DEVICE image dst, asynchronously on
 * cuda_stream (nullptr: the context's stream).  For callers that shard a pair by row bands: prefilter the whole images, then
 * call the band entry points with the option off.  Bytes past cols in each dst row are never written.  STEREO_ERR_INVALID_ARG:
 * a null pointer, a non-positive size, a step smaller than its row, a cap outside 1 .. 63, or a dst that overlaps src. */
int stereo_prefilter_u8_device(stereo_ctx* ctx, const uint8_t* src, size_t src_step, int rows, int cols, int cap,
                               uint8_t* dst, size_t dst_step, void* cuda_stream);
int stereo_prefilter_f32_device(stereo_ctx* ctx, const float* src, size_t src_step, int rows, int cols, int cap,
                                uint8_t* dst, size_t dst_step, void* cuda_stream);

/* ---- single direction, HOST buffers (the drop-in form) ------------------------------------ */
/*
 * One disparity map for reference image `ref` searched in `tgt` over [min_disp, max_disp].
 * Replaces cuda::disparitySSD / cuda::disparityNCorr (host cv::Mat in, host cv::Mat out;
 * upload, kernels and download happen inside, synchronously — DisparitySSD.cu:171-206).
 *   disp_out        rows x cols elements of disp_elem_bytes (1, 2 or 4), row stride disp_step bytes
 *   best_out        optional (NULL to skip) rows x cols winning values, row stride best_step bytes:
 *                   SSD  -> int32 cost  (99999999 where no candidate exists, DisparitySSD.cpp:37)
 *                   NCC  -> float32 score (the result[] value minMaxLoc selected, DisparityNCorr.cpp:60-64)
 */
int stereo_disparity_f32_host(stereo_ctx* ctx, int cost,
                              const float* ref, size_t ref_step, const float* tgt, size_t tgt_step,
                              int rows, int cols, int window_rad, int min_disp, int max_disp,
                              void* disp_out, size_t disp_step, int disp_elem_bytes,
                              void* best_out, size_t best_step);

int stereo_disparity_u8_host(stereo_ctx* ctx, int cost,
                             const uint8_t* ref, size_t ref_step, const uint8_t* tgt, size_t tgt_step,
                             int rows, int cols, int window_rad, int min_disp, int max_disp,
                             void* disp_out, size_t disp_step, int disp_elem_bytes,
                             void* best_out, size_t best_step);

/* ---- single direction, DEVICE buffers, asynchronous on `cuda_stream` ----------------------- */
/* Same computation with every pointer a device pointer on the context's device.  `cuda_stream` is a
 * cudaStream_t passed as void* (NULL = the context's own stream; pass cudaStreamLegacy, (void*)1, for the
 * CUDA legacy default stream).  Returns after enqueueing. */
int stereo_disparity_f32_device(stereo_ctx* ctx, int cost,
                                const float* ref, size_t ref_step, const float* tgt, size_t tgt_step,
                                int rows, int cols, int window_rad, int min_disp, int max_disp,
                                void* disp_out, size_t disp_step, int disp_elem_bytes,
                                void* best_out, size_t best_step, void* cuda_stream);

int stereo_disparity_u8_device(stereo_ctx* ctx, int cost,
                               const uint8_t* ref, size_t ref_step, const uint8_t* tgt, size_t tgt_step,
                               int rows, int cols, int window_rad, int min_disp, int max_disp,
                               void* disp_out, size_t disp_step, int disp_elem_bytes,
                               void* best_out, size_t best_step, void* cuda_stream);

/* ---- both directions (the reference's *Pair helpers, main.cpp:21-78) ------------------------ */
/* left-referenced map over [-disparity_range, 0] into disp_left, right-referenced map over
 * [0, +disparity_range] (images swapped) into disp_right.  Host buffers, synchronous. */
int stereo_disparity_pair_f32_host(stereo_ctx* ctx, int cost,
                                   const float* left, size_t left_step, const float* right, size_t right_step,
                                   int rows, int cols, int window_rad, int disparity_range,
                                   void* disp_left, void* disp_right, size_t disp_step, int disp_elem_bytes);

int stereo_disparity_pair_u8_host(stereo_ctx* ctx, int cost,
                                  const uint8_t* left, size_t left_step, const uint8_t* right, size_t right_step,
                                  int rows, int cols, int window_rad, int disparity_range,
                                  void* disp_left, void* disp_right, size_t disp_step, int disp_elem_bytes);

/* Device buffers, asynchronous on `cuda_stream`. */
int stereo_disparity_pair_u8_device(stereo_ctx* ctx, int cost,
                                    const uint8_t* left, size_t left_step, const uint8_t* right, size_t right_step,
                                    int rows, int cols, int window_rad, int disparity_range,
                                    void* disp_left, void* disp_right, size_t disp_step, int disp_elem_bytes,
                                    void* cuda_stream);

/* The same for CV_32FC1 device images (what the reference's wrapper holds after its uploads, DisparitySSD.cu:171-174).
 * The kernel family depends on the pixel values (8-bit-valued, bounded float range, anything else), which the
 * host learns from a device-side classification: this call synchronises `cuda_stream` once before it enqueues
 * the matching kernels; the kernels themselves run asynchronously. */
int stereo_disparity_pair_f32_device(stereo_ctx* ctx, int cost,
                                     const float* left, size_t left_step, const float* right, size_t right_step,
                                     int rows, int cols, int window_rad, int disparity_range,
                                     void* disp_left, void* disp_right, size_t disp_step, int disp_elem_bytes,
                                     void* cuda_stream);

/* ---- batches of equally-shaped pairs (BASELINE config 5) ------------------------------------ */
/* `n_pairs` image pairs stored back to back: pair i's left image starts at left + i*pair_stride
 * bytes (same for right); outputs start at disp_* + i*disp_pair_stride bytes.  Device buffers,
 * asynchronous on `cuda_stream`. */
int stereo_disparity_pair_batch_u8_device(stereo_ctx* ctx, int cost, int n_pairs,
                                          const uint8_t* left, const uint8_t* right, size_t img_step,
                                          size_t pair_stride, int rows, int cols, int window_rad,
                                          int disparity_range, void* disp_left, void* disp_right,
                                          size_t disp_step, size_t disp_pair_stride, int disp_elem_bytes,
                                          void* cuda_stream);

/* Host buffers, synchronous: uploads, computes and downloads with copies overlapped across pairs. */
int stereo_disparity_pair_batch_u8_host(stereo_ctx* ctx, int cost, int n_pairs,
                                        const uint8_t* left, const uint8_t* right, size_t img_step,
                                        size_t pair_stride, int rows, int cols, int window_rad,
                                        int disparity_range, void* disp_left, void* disp_right,
                                        size_t disp_step, size_t disp_pair_stride, int disp_elem_bytes);

/* The same for CV_32FC1 host images (the type the reference's entry points take, DisparitySSD.cu:150): a batch
 * of the reference's disparitySSDPair / disparityNCorrPair calls (main.cpp:21-78) in one call.  img_step and
 * pair_stride are in BYTES.  8-bit-valued images ride the packed kernels with uploads, conversion, compute and
 * downloads overlapped across pairs; anything else is computed pair by pair on the exact path. */
int stereo_disparity_pair_batch_f32_host(stereo_ctx* ctx, int cost, int n_pairs,
                                         const float* left, const float* right, size_t img_step,
                                         size_t pair_stride, int rows, int cols, int window_rad,
                                         int disparity_range, void* disp_left, void* disp_right,
                                         size_t disp_step, size_t disp_pair_stride, int disp_elem_bytes);

/* ---- row-band form for sharding one large image across GPUs (BASELINE config 4) -------------- */
/* Computes output rows [row_begin, row_end) of the full rows x cols problem.  `ref`/`tgt` point at
 * FULL images (device); only rows within the band's halo are read.  disp_out points at the band's
 * first output row.  Results equal the corresponding rows of the full-image call, including the
 * reference's row-wrap reads at band seams (SURVEY.md §A.1, §8e). */
int stereo_disparity_band_u8_device(stereo_ctx* ctx, int cost,
                                    const uint8_t* ref, size_t ref_step, const uint8_t* tgt, size_t tgt_step,
                                    int rows, int cols, int row_begin, int row_end,
                                    int window_rad, int min_disp, int max_disp,
                                    void* disp_out, size_t disp_step, int disp_elem_bytes, void* cuda_stream);

/* Same, for callers that hold only a slab of the images (one rank of a row-band sharded job): `ref_halo`/
 * `tgt_halo` point at image row `halo_begin`; rows [halo_begin, halo_end) are present.  The slab must
 * contain the rows stereo_band_halo_rows() reports for the band — window_rad rows above and below plus
 * one more for the reference's row-wrap reads, clamped to the image — then the result equals the
 * corresponding rows of the full-image call bit for bit. */
int stereo_disparity_band_halo_u8_device(stereo_ctx* ctx, int cost,
                                         const uint8_t* ref_halo, size_t ref_step, const uint8_t* tgt_halo, size_t tgt_step,
                                         int rows, int cols, int row_begin, int row_end, int halo_begin, int halo_end,
                                         int window_rad, int min_disp, int max_disp,
                                         void* disp_out, size_t disp_step, int disp_elem_bytes, void* cuda_stream);

/* Both maps of the band in one call (a rank's share of a row-band sharded pair): left-referenced map over
 * [-disparity_range, 0] into disp_left, right-referenced map over [0, +disparity_range] into disp_right, each
 * pointing at the band's first output row; from one cost volume where stereo_ctx_set_fuse_pairs allows it. */
int stereo_disparity_pair_band_halo_u8_device(stereo_ctx* ctx, int cost,
                                              const uint8_t* left_halo, size_t left_step, const uint8_t* right_halo, size_t right_step,
                                              int rows, int cols, int row_begin, int row_end, int halo_begin, int halo_end,
                                              int window_rad, int disparity_range,
                                              void* disp_left, void* disp_right, size_t disp_step, int disp_elem_bytes,
                                              void* cuda_stream);

/* Input rows [*halo_begin, *halo_end) a band [row_begin, row_end) of a rows-high image needs (pure host
 * arithmetic, no device). */
int stereo_band_halo_rows(int rows, int row_begin, int row_end, int window_rad, int* halo_begin, int* halo_end);

/* ---- peer gather: the exchange step of the sharded configs, on the copy engines -----------------------
 * The reference has no multi-GPU path (SURVEY.md §0.9); BASELINE configs 4 and 5 gather the per-rank maps.
 * The hot kernel is persistent (one CTA per SM, full register file), so a collective that needs SMs cannot
 * overlap it.  These calls let each rank push its finished maps straight into every other rank's gather
 * buffer with device-to-device copies over NVLink (copy engines, no SM), stream-ordered after the kernels
 * that produced them, while the SMs already work on the next launch sequence.
 *   create  : device buffer other processes of this box can map + the 64-byte handle to send them
 *   open    : map a peer's buffer from its handle (a different process; never the creating one)
 *   push    : once `after_stream` reaches this point, copy src -> dst_ptrs[i] + dst_offset for every i
 *             (NULL entries are skipped; pointers may be local or opened peers)
 *   mark    : returns a ticket that completes when every push enqueued so far has finished
 *   wait    : makes `cuda_stream` wait for a ticket (at most 64 tickets are live) */
#define STEREO_IPC_HANDLE_BYTES 64
int stereo_peer_buffer_create(stereo_ctx* ctx, size_t bytes, void** dev_ptr, unsigned char* handle_out);
int stereo_peer_buffer_open(stereo_ctx* ctx, const unsigned char* handle, void** peer_ptr);
int stereo_peer_buffer_close(stereo_ctx* ctx, void* peer_ptr);
int stereo_peer_buffer_destroy(stereo_ctx* ctx, void* dev_ptr);
int stereo_peer_push(stereo_ctx* ctx, void* const* dst_ptrs, int n_dst, size_t dst_offset, const void* src, size_t bytes,
                     void* after_stream);
int stereo_peer_mark(stereo_ctx* ctx, int* ticket_out);
int stereo_peer_wait(stereo_ctx* ctx, int ticket, void* cuda_stream);

/* ---- device images and preprocessing (SURVEY.md §8 f3) ----------------------------------------------------- */
/*
 * What the ps2 executable does to an image between imread and the disparity call, on the device, so that an image pair
 * is uploaded ONCE (as 8-bit pixels) and serves both directions and every problem that uses it; the reference uploads
 * both float Mats again for every direction (DisparitySSD.cu:171-174).
 *   stereo_dev_alloc/free/upload/download : plain device buffers for callers without the CUDA runtime (synchronous copies)
 *   gray   : channels == 1: Mat::convertTo(CV_32FC1) unscaled (main.cpp:87-88); 3 or 4: cvtColor(COLOR_RGB2GRAY) on the
 *            interleaved data as loaded (BGR from imread, main.cpp:114-117) with OpenCV's fixed-point coefficients
 *            (shift 14 = OpenCV 3.4.1, 15 = later), then convertTo
 *   scale_add : out = a * scale (+ add, nullable): `left * 1.1f` (main.cpp:191-193) and `first + noise` (main.cpp:146-152),
 *            separately rounded float32 operations.  The noise field itself is cv::randn's sequential stream: host.
 */
int stereo_dev_alloc(stereo_ctx* ctx, size_t bytes, void** ptr);
int stereo_dev_free(stereo_ctx* ctx, void* ptr);
int stereo_dev_upload(stereo_ctx* ctx, void* dst, size_t dst_step, const void* src, size_t src_step, size_t row_bytes, int rows);
int stereo_dev_download(stereo_ctx* ctx, void* dst, size_t dst_step, const void* src, size_t src_step, size_t row_bytes, int rows);
int stereo_image_gray_f32_device(stereo_ctx* ctx, const uint8_t* img, size_t step, int rows, int cols, int channels, int shift,
                                 float* out, size_t out_step, void* cuda_stream);
int stereo_image_scale_add_f32_device(stereo_ctx* ctx, const float* a, size_t a_step, const float* add, size_t add_step, float scale,
                                      int rows, int cols, float* out, size_t out_step, void* cuda_stream);

/* ---- reference-GPU-semantics mode (SURVEY.md A.3, §8 f4) ------------------------------------------------- */
/*
 * Everything above reproduces the reference's CPU functions (the parity target).  Its GTX-1080 kernels compute a
 * different function: a (2R+1) x 2R window, clamp-to-edge addressing, every d in [min_disp, max_disp], float32 rolling
 * column sums restarted every 40 rows, SSD accepted only below 5e6 and NCC only above 0, -1 where nothing won
 * (lib/DisparitySSD.cu:16,27-141,177; lib/DisparityNCorr.cu:16,28-175,211).  These two entry points compute THAT function,
 * every float operation in the kernels' order, so maps the reference's GPU build produced can be reproduced.
 * disp_out: int8 (the kernels store `char`); best_out (nullable): the kernels' running best SSD / score map.
 * The range must fit the kernels' `char` loop variable.  Checked bit for bit against oracle_disparity_refgpu. */
int stereo_disparity_refgpu_f32_host(stereo_ctx* ctx, int cost,
                                     const float* ref, size_t ref_step, const float* tgt, size_t tgt_step,
                                     int rows, int cols, int window_rad, int min_disp, int max_disp,
                                     int8_t* disp_out, size_t disp_step, float* best_out, size_t best_step);
int stereo_disparity_refgpu_f32_device(stereo_ctx* ctx, int cost,
                                       const float* ref, size_t ref_step, const float* tgt, size_t tgt_step,
                                       int rows, int cols, int window_rad, int min_disp, int max_disp,
                                       int8_t* disp_out, size_t disp_step, float* best_out, size_t best_step,
                                       void* cuda_stream);

/* ---- one row band of a pair, HOST images (a device's share of a row-band sharded pair) -------------- */
/* left / right: FULL-image host origins (cv::Mat data pointers); only the slab of rows the band [row_begin, row_end) needs -
 * window halo plus the row of the SSD flat-index wrap, stereo_band_halo_rows - is uploaded.  disp_left / disp_right point
 * at the band's first output row.  Synchronous.  The f32 form converts the slab to u8 on the host; images that are not
 * 8-bit-valued return STEREO_ERR_UNSUPPORTED (callers take a whole-image call then). */
int stereo_disparity_pair_band_u8_host(stereo_ctx* ctx, int cost,
                                       const uint8_t* left, size_t left_step, const uint8_t* right, size_t right_step,
                                       int rows, int cols, int row_begin, int row_end, int window_rad, int disparity_range,
                                       void* disp_left, void* disp_right, size_t disp_step, int disp_elem_bytes);
int stereo_disparity_pair_band_f32_host(stereo_ctx* ctx, int cost,
                                        const float* left, size_t left_step, const float* right, size_t right_step,
                                        int rows, int cols, int row_begin, int row_end, int window_rad, int disparity_range,
                                        void* disp_left, void* disp_right, size_t disp_step, int disp_elem_bytes);

/* ---- several GPUs in ONE process (SURVEY.md §8b "context create/destroy taking a device list", §8e) ---------- */
/*
 * The reference is single-GPU (lib/DisparitySSD.cu:143-207).  A stereo_mgpu owns one stereo_ctx per listed device
 * (devices = NULL: every visible sm_100 device) and one host thread per device during a call.  The path has no exchange
 * inside the computation: batches are sharded by pair (contiguous blocks), one pair by row bands with halo; every device
 * uploads only its share and downloads its maps straight into the caller's host arrays - results are bit-identical to the
 * single-GPU calls.  A device ordinal may be listed more than once (several contexts on one GPU).
 */
typedef struct stereo_mgpu stereo_mgpu;
int stereo_mgpu_create(const int* devices, int n_devices, stereo_mgpu** out);
void stereo_mgpu_destroy(stereo_mgpu* mg);
int stereo_mgpu_device_count(const stereo_mgpu* mg);
/* The context of the index-th listed device (for stereo_ctx_set_* knobs); owned by the stereo_mgpu. */
stereo_ctx* stereo_mgpu_ctx(stereo_mgpu* mg, int index);
/* stereo_ctx_set_lr_check on every device's context.  The check works row by row, so row bands and pair shards give the
 * single-GPU result. */
int stereo_mgpu_set_lr_check(stereo_mgpu* mg, int max_diff);
/* stereo_ctx_set_speckle_filter on every device's context.  Pair batches shard whole pairs and so give the single-GPU
 * result; row-band sharded pairs return STEREO_ERR_UNSUPPORTED while the filter is on. */
int stereo_mgpu_set_speckle_filter(stereo_mgpu* mg, int max_size, int max_diff);
/* stereo_ctx_set_sgm on every device's context.  Pair batches shard whole pairs and so give the single-GPU result;
 * row-band sharded pairs return STEREO_ERR_UNSUPPORTED while SGM is on. */
int stereo_mgpu_set_sgm(stereo_mgpu* mg, int paths, int p1, int p2);
/* stereo_ctx_set_sgm_ncc_scale on every device's context. */
int stereo_mgpu_set_sgm_ncc_scale(stereo_mgpu* mg, int q);
/* stereo_ctx_set_uniqueness on every device's context.  Pair batches shard whole pairs and so give the single-GPU result;
 * row-band sharded pairs return STEREO_ERR_UNSUPPORTED while it is on. */
int stereo_mgpu_set_uniqueness(stereo_mgpu* mg, int uniqueness_ratio);
/* stereo_ctx_set_prefilter on every device's context.  Pair batches shard whole pairs and so give the single-GPU result;
 * row-band sharded pairs return STEREO_ERR_UNSUPPORTED while it is on. */
int stereo_mgpu_set_prefilter(stereo_mgpu* mg, int cap, int texture_threshold);
/* stereo_ctx_set_subpixel on every device's context.  Pair batches shard whole pairs and so give the single-GPU result;
 * row-band sharded pairs return STEREO_ERR_UNSUPPORTED while it is on. */
int stereo_mgpu_set_subpixel(stereo_mgpu* mg, int on);
/* Batches (BASELINE config 5): same arguments as stereo_disparity_pair_batch_{u8,f32}_host. */
int stereo_mgpu_disparity_pair_batch_u8_host(stereo_mgpu* mg, int cost, int n_pairs,
                                             const uint8_t* left, const uint8_t* right, size_t img_step, size_t pair_stride,
                                             int rows, int cols, int window_rad, int disparity_range,
                                             void* disp_left, void* disp_right, size_t disp_step, size_t disp_pair_stride,
                                             int disp_elem_bytes);
int stereo_mgpu_disparity_pair_batch_f32_host(stereo_mgpu* mg, int cost, int n_pairs,
                                              const float* left, const float* right, size_t img_step, size_t pair_stride,
                                              int rows, int cols, int window_rad, int disparity_range,
                                              void* disp_left, void* disp_right, size_t disp_step, size_t disp_pair_stride,
                                              int disp_elem_bytes);
/* One pair in row bands (BASELINE config 4): same arguments as stereo_disparity_pair_{u8,f32}_host.  Float images that are
 * not 8-bit-valued are computed whole on the first device. */
int stereo_mgpu_disparity_pair_bands_u8_host(stereo_mgpu* mg, int cost,
                                             const uint8_t* left, size_t left_step, const uint8_t* right, size_t right_step,
                                             int rows, int cols, int window_rad, int disparity_range,
                                             void* disp_left, void* disp_right, size_t disp_step, int disp_elem_bytes);
int stereo_mgpu_disparity_pair_bands_f32_host(stereo_mgpu* mg, int cost,
                                              const float* left, size_t left_step, const float* right, size_t right_step,
                                              int rows, int cols, int window_rad, int disparity_range,
                                              void* disp_left, void* disp_right, size_t disp_step, int disp_elem_bytes);

/* Blocks until everything enqueued on `cuda_stream` (NULL = the context's stream) has finished and
 * returns any asynchronous error. */
int stereo_ctx_synchronize(stereo_ctx* ctx, void* cuda_stream);

#ifdef __cplusplus
} /* extern "C" */
#endif

#endif /* STEREO_B200_H_ */
