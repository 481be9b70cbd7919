// Shared declarations for the stereo_b200 library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstddef>
#include <cstdio>
#include <cstring>
#include <string>

#include "../../include/stereo_b200.h"

namespace sb {

class HostPool;

// ---- error plumbing: status codes out, never exit() (contrast: common/CudaCommon.cuh:11-22) ----
void set_error(const char* fmt, ...);
#define SB_CUDA(expr)                                                                         \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess) {                                                              \
            sb::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return STEREO_ERR_CUDA;                                                           \
        }                                                                                     \
    } while (0)

// The reference's launch-geometry helper (common/include/common/Utils.h:12-15): ceil-div, min 1.
static inline unsigned div_round_up(long long num, long long den) {
    long long v = (num + den - 1) / den;
    return (unsigned)(v < 1 ? 1 : v);
}

__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

enum class PixType : int { U8 = 0, F32 = 1 };

struct ImageView {       // device image
    const void* ptr;
    size_t step;         // bytes
    PixType type;
};

struct OutView {         // device output
    void* ptr;
    size_t step;         // bytes
    int elem;            // 1,2,4 (disparity) — best maps are always 4 bytes
};

// One direction of one image pair.
struct Problem {
    int cost;            // stereo_cost
    ImageView ref, tgt;
    int rows, cols;      // full image
    int row_begin, row_end;   // output band (full image: 0, rows)
    int avail_begin, avail_end;   // image rows the buffers actually hold (pointers are full-image origins)
    int R, dmin, dmax;
    OutView disp;        // first row of the band
    OutView best;        // optional (ptr == nullptr)
};

// Grow-only device scratch arena owned by a context; sub-allocations are 256-byte aligned and
// valid until the next reset().
struct Arena {
    char* base = nullptr;
    size_t cap = 0, used = 0;
    int reserve(size_t bytes);          // (re)allocate to at least `bytes`; invalidates contents
    void reset() { used = 0; }
    void* take(size_t bytes) {
        size_t off = (used + 255) & ~size_t(255);
        if (off + bytes > cap) return nullptr;
        used = off + bytes;
        return base + off;
    }
    void release();
};

// The pair options of a context: what pair calls do beyond the block matcher.  Single-direction calls ignore them.
struct PairOptions {
    int lr_max_diff = -1;     // left-right consistency check with this disp12MaxDiff (< 0: off)
    int spk_max_size = 0;     // speckle filter of components up to this many pixels (0: off) ...
    int spk_max_diff = 0;     // ... whose neighbours differ by at most this much
    int sgm_paths = 0;        // semi-global matching over 4 or 8 paths (0: off) ...
    int sgm_p1 = 0, sgm_p2 = 0;   // ... with these penalties
    int sgm_ncc_scale = 0;    // ... and, for NCC pair calls, this integer scale of the NCC cost (0: NCC refused)
    int uniq = 0;             // StereoSGBM's uniquenessRatio, 1 .. 99 (0: off)
    int pf_cap = 0;           // StereoBM's X-Sobel prefilter with this preFilterCap, 1 .. 63 (0: off) ...
    int pf_texture = 0;       // ... and this textureThreshold (0: off)
    int subpix = 0;           // StereoSGBM's sub-pixel disparity, 1/16-pixel fixed point, after every other step (0: off)

    // Removed pixels are marked with -(range + 1), which must fit the maps' element type.
    bool writes_sentinel() const { return lr_max_diff >= 0 || spk_max_size > 0 || uniq > 0 || pf_texture > 0; }
    // Row bands are refused: speckle regions and SGM paths cross band seams, the uniqueness pass, the sub-pixel pass and
    // the prefilter's odd-height rule work on whole images.
    bool needs_whole_maps() const { return pf_cap > 0 || uniq > 0 || sgm_paths > 0 || spk_max_size > 0 || subpix > 0; }
    // The maps are computed from whole images in one go, so the host pipeline's row bands do not apply.  (The speckle
    // filter is not here: the pipeline filters an item's maps after its last band.)
    bool computed_whole() const { return sgm_paths > 0 || uniq > 0 || pf_cap > 0 || subpix > 0; }
};

} // namespace sb

struct stereo_ctx {
    int device = -1;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t s_in = nullptr, s_out = nullptr;   // copy streams of the pipelined host entry points
    cudaEvent_t* pipe_ev = nullptr;                 // pool of timing-free events for the pipeline
    int pipe_ev_cap = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaEvent_t ev_gap0 = nullptr, ev_gap1 = nullptr;   // float device calls: the device idles between these two while the host reads
    bool gap_recorded = false;                          // the classification verdict; last_kernel_ms leaves that gap out
    bool timing_pending = false;
    bool have_prev_call = false;                    // ev1 marks the end of the previous call ...
    cudaStream_t prev_stream = nullptr;             // ... which was enqueued on this stream
    sb::Arena arena;          // per-call scratch (padded images, packed rows, partial keys)
    sb::Arena io;             // device staging of host-API inputs/outputs
    void* pinned = nullptr;   // pinned host staging
    size_t pinned_cap = 0;
    sb::HostPool* pool = nullptr;   // host threads that convert CV_32FC1 host images to u8 (host_pack.cpp)
    int host_threads = 0;           // 0 = automatic, -1 = host packing off, n = use n threads (and pack whatever n is)
    bool host_pack_forced = false;
    int* d_flag = nullptr;    // device classification flag
    int* h_flag = nullptr;    // pinned mirror
    int last_path = 0;
    int last_launches = 0;
    float last_ms = -1.f;
    int force_path = 0;
    int pipe_bands = 0;       // 0 = automatic
    int fuse_pairs = 1;       // both maps of a pair from one cost volume where the problem allows it
    sb::PairOptions opt;      // what pair calls do beyond the block matcher (stereo_ctx_set_lr_check .. _set_prefilter)
    sb::Arena pf;             // the prefiltered images of a pair call, live while the arena is reset (grow-only)
    sb::Arena sp;             // the SGM maps' sub-pixel offsets of a pair call, live while the arena is reset (grow-only)
    // device time of the hot kernels only (fast_*_kernel), per direction, for the roofline report
    static constexpr int HOT_EVENTS = 16;
    cudaEvent_t hot0[HOT_EVENTS] = {}, hot1[HOT_EVENTS] = {};
    int hot_used = 0;          // event pairs recorded by the last call
    int hot_total = 0;         // hot-kernel launches of the last call (may exceed HOT_EVENTS)
    int hot_jobs = 0;          // directions (jobs) covered by the measured hot launches
    int fused_pairs_done = 0;  // image pairs of the last call whose two maps came out of one cost volume
    // peer gather (stereo_peer_*): copy-engine pushes of finished maps into other ranks' buffers over NVLink
    static constexpr int PEER_STREAMS = 2, PEER_TICKETS = 64;
    cudaStream_t s_peer[PEER_STREAMS] = {};
    cudaEvent_t peer_ready = nullptr;                            // "producer stream reached this point"
    cudaEvent_t peer_done[PEER_TICKETS][PEER_STREAMS] = {};      // ring of completion marks
    int peer_next_stream = 0, peer_next_ticket = 0;
};
