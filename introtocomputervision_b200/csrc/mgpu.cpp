// stereo_mgpu_*: one process, several B200s.  The path shards with no exchange inside the computation (SURVEY.md §8e):
// by stereo pair for batches, by row band with halo for one pair.  Each device has its own stereo_ctx and is driven by its
// own host thread through the single-GPU HOST entry points, so every device uploads only its share, computes it and
// downloads straight into the caller's arrays - the gather's consumer is the host, over each GPU's own link.  (The
// device-to-device gather of one-process-per-GPU jobs is stereo_peer_*.)  Plain C++ on top of the C ABI.
#include "../../include/stereo_b200.h"

#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

namespace sb {
void set_error(const char* fmt, ...);
const char* band_sharding_refusal(const stereo_ctx* ctx);
}

struct stereo_mgpu {
    std::vector<stereo_ctx*> ctx;
    std::vector<int> device;
};

namespace {

// contiguous block [begin, end) of `n` items owned by part k of `parts` (sizes differ by at most one)
void block_shard(int n, int parts, int k, int* begin, int* end) {
    const int base = n / parts, extra = n % parts;
    *begin = k * base + (k < extra ? k : extra);
    *end = *begin + base + (k < extra ? 1 : 0);
}

// Runs fn(k) on one host thread per device; returns the first failing status and republishes its message on this thread.
template <class F>
int for_each_device(stereo_mgpu* mg, F fn) {
    const int n = int(mg->ctx.size());
    std::vector<int> rc(n, STEREO_OK);
    std::vector<std::string> msg(n);
    std::vector<std::thread> th;
    auto body = [&](int k) {
        rc[k] = fn(k);
        if (rc[k] != STEREO_OK) msg[k] = stereo_last_error();      // (the message is per thread)
    };
    for (int k = 1; k < n; ++k) th.emplace_back(body, k);
    body(0);
    for (auto& t : th) t.join();
    for (int k = 0; k < n; ++k)
        if (rc[k] != STEREO_OK) { sb::set_error("device %d: %s", mg->device[k], msg[k].c_str()); return rc[k]; }
    return STEREO_OK;
}

// One pair-option setter on the context of every device; stops at the first refusal.
template <class... A>
int set_all(stereo_mgpu* mg, int (*set)(stereo_ctx*, A...), A... args) {
    if (!mg || mg->ctx.empty()) { sb::set_error("null multi-GPU context"); return STEREO_ERR_INVALID_ARG; }
    for (stereo_ctx* c : mg->ctx) {
        const int rc = set(c, args...);
        if (rc != STEREO_OK) return rc;
    }
    return STEREO_OK;
}

template <class T>
int pair_batch(stereo_mgpu* mg, int cost, int n_pairs, const T* left, const T* right, size_t img_step, size_t pair_stride, int rows,
               int cols, int window_rad, int disparity_range, void* disp_left, void* disp_right, size_t disp_step,
               size_t disp_pair_stride, int elem, bool f32) {
    if (!mg || mg->ctx.empty()) { sb::set_error("null multi-GPU context"); return STEREO_ERR_INVALID_ARG; }
    if (n_pairs <= 0 || !left || !right || !disp_left || !disp_right) { sb::set_error("bad batch arguments"); return STEREO_ERR_INVALID_ARG; }
    const int parts = int(mg->ctx.size());
    return for_each_device(mg, [&](int k) -> int {
        int b, e;
        block_shard(n_pairs, parts, k, &b, &e);
        if (b >= e) return STEREO_OK;
        const char* l = reinterpret_cast<const char*>(left) + size_t(b) * pair_stride;
        const char* r = reinterpret_cast<const char*>(right) + size_t(b) * pair_stride;
        char* dl = static_cast<char*>(disp_left) + size_t(b) * disp_pair_stride;
        char* dr = static_cast<char*>(disp_right) + size_t(b) * disp_pair_stride;
        if (f32)
            return stereo_disparity_pair_batch_f32_host(mg->ctx[k], cost, e - b, reinterpret_cast<const float*>(l), reinterpret_cast<const float*>(r),
                                                        img_step, pair_stride, rows, cols, window_rad, disparity_range, dl, dr, disp_step, disp_pair_stride, elem);
        return stereo_disparity_pair_batch_u8_host(mg->ctx[k], cost, e - b, reinterpret_cast<const uint8_t*>(l), reinterpret_cast<const uint8_t*>(r),
                                                   img_step, pair_stride, rows, cols, window_rad, disparity_range, dl, dr, disp_step, disp_pair_stride, elem);
    });
}

template <class T>
int pair_bands(stereo_mgpu* mg, int cost, const T* left, size_t left_step, const T* right, size_t right_step, int rows, int cols,
               int window_rad, int disparity_range, void* disp_left, void* disp_right, size_t disp_step, int elem, bool f32) {
    if (!mg || mg->ctx.empty()) { sb::set_error("null multi-GPU context"); return STEREO_ERR_INVALID_ARG; }
    if (rows <= 0) { sb::set_error("rows must be positive"); return STEREO_ERR_INVALID_ARG; }
    for (stereo_ctx* c : mg->ctx)
        if (const char* why = sb::band_sharding_refusal(c)) { sb::set_error("%s", why); return STEREO_ERR_UNSUPPORTED; }
    int parts = int(mg->ctx.size());
    const int band = (rows + parts - 1) / parts;            // equal bands of ceil(rows / parts) rows, the last one(s) shorter or empty
    int rc = for_each_device(mg, [&](int k) -> int {
        const int r0 = k * band < rows ? k * band : rows, r1 = r0 + band < rows ? r0 + band : rows;
        if (r0 >= r1) return STEREO_OK;
        char* dl = static_cast<char*>(disp_left) + size_t(r0) * disp_step;
        char* dr = static_cast<char*>(disp_right) + size_t(r0) * disp_step;
        if (f32)
            return stereo_disparity_pair_band_f32_host(mg->ctx[k], cost, reinterpret_cast<const float*>(left), left_step, reinterpret_cast<const float*>(right),
                                                       right_step, rows, cols, r0, r1, window_rad, disparity_range, dl, dr, disp_step, elem);
        return stereo_disparity_pair_band_u8_host(mg->ctx[k], cost, reinterpret_cast<const uint8_t*>(left), left_step, reinterpret_cast<const uint8_t*>(right),
                                                  right_step, rows, cols, r0, r1, window_rad, disparity_range, dl, dr, disp_step, elem);
    });
    if (rc == STEREO_ERR_UNSUPPORTED && f32)
        // float images that are not 8-bit-valued (noise / contrast variants): the band kernels are 8-bit only - the whole
        // pair on the first device (float running-sum kernels)
        rc = stereo_disparity_pair_f32_host(mg->ctx[0], cost, reinterpret_cast<const float*>(left), left_step, reinterpret_cast<const float*>(right),
                                            right_step, rows, cols, window_rad, disparity_range, disp_left, disp_right, disp_step, elem);
    return rc;
}

} // namespace

extern "C" {

int stereo_mgpu_create(const int* devices, int n_devices, stereo_mgpu** out) {
    if (!out) { sb::set_error("out is null"); return STEREO_ERR_INVALID_ARG; }
    *out = nullptr;
    std::vector<int> dev;
    if (devices && n_devices > 0) dev.assign(devices, devices + n_devices);
    else {
        const int n = stereo_device_count();
        for (int i = 0; i < n; ++i) dev.push_back(i);
    }
    if (dev.empty()) { sb::set_error("no sm_100 CUDA device available (this library has no CPU fallback)"); return STEREO_ERR_NO_DEVICE; }
    if (dev.size() > 64) { sb::set_error("more than 64 devices"); return STEREO_ERR_INVALID_ARG; }
    stereo_mgpu* mg = new (std::nothrow) stereo_mgpu();
    if (!mg) { sb::set_error("out of host memory"); return STEREO_ERR_ALLOC; }
    for (int d : dev) {
        stereo_ctx* c = nullptr;
        const int rc = stereo_ctx_create(d, &c);
        if (rc != STEREO_OK) { stereo_mgpu_destroy(mg); return rc; }
        mg->ctx.push_back(c);
        mg->device.push_back(d);
    }
    // the devices' host threads share the cores: each context packs CV_32FC1 images with its share of them, or (fewer
    // than the packing threshold of 8 each) uploads the floats and converts on the device
    const int share = stereo_ctx_host_threads(mg->ctx[0]) / int(mg->ctx.size());
    for (stereo_ctx* c : mg->ctx) stereo_ctx_set_host_threads(c, share >= 8 ? share : -1);
    *out = mg;
    return STEREO_OK;
}

void stereo_mgpu_destroy(stereo_mgpu* mg) {
    if (!mg) return;
    for (stereo_ctx* c : mg->ctx) stereo_ctx_destroy(c);
    delete mg;
}

int stereo_mgpu_device_count(const stereo_mgpu* mg) { return mg ? int(mg->ctx.size()) : 0; }

stereo_ctx* stereo_mgpu_ctx(stereo_mgpu* mg, int index) {
    if (!mg || index < 0 || index >= int(mg->ctx.size())) return nullptr;
    return mg->ctx[index];
}

int stereo_mgpu_set_lr_check(stereo_mgpu* mg, int max_diff) { return set_all(mg, stereo_ctx_set_lr_check, max_diff); }

int stereo_mgpu_set_speckle_filter(stereo_mgpu* mg, int max_size, int max_diff) {
    return set_all(mg, stereo_ctx_set_speckle_filter, max_size, max_diff);
}

int stereo_mgpu_set_sgm(stereo_mgpu* mg, int paths, int p1, int p2) { return set_all(mg, stereo_ctx_set_sgm, paths, p1, p2); }

int stereo_mgpu_set_sgm_ncc_scale(stereo_mgpu* mg, int q) { return set_all(mg, stereo_ctx_set_sgm_ncc_scale, q); }

int stereo_mgpu_set_uniqueness(stereo_mgpu* mg, int uniqueness_ratio) { return set_all(mg, stereo_ctx_set_uniqueness, uniqueness_ratio); }

int stereo_mgpu_set_subpixel(stereo_mgpu* mg, int on) { return set_all(mg, stereo_ctx_set_subpixel, on); }

int stereo_mgpu_set_prefilter(stereo_mgpu* mg, int cap, int texture_threshold) {
    return set_all(mg, stereo_ctx_set_prefilter, cap, texture_threshold);
}

int stereo_mgpu_disparity_pair_batch_u8_host(stereo_mgpu* mg, int cost, int n_pairs, const uint8_t* left, const uint8_t* right,
                                             size_t img_step, size_t pair_stride, int rows, int cols, int window_rad,
                                             int disparity_range, void* disp_left, void* disp_right, size_t disp_step,
                                             size_t disp_pair_stride, int disp_elem_bytes) {
    return pair_batch(mg, cost, n_pairs, left, right, img_step, pair_stride, rows, cols, window_rad, disparity_range, disp_left, disp_right,
                      disp_step, disp_pair_stride, disp_elem_bytes, false);
}

int stereo_mgpu_disparity_pair_batch_f32_host(stereo_mgpu* mg, int cost, int n_pairs, const float* left, const float* right,
                                              size_t img_step, size_t pair_stride, int rows, int cols, int window_rad,
                                              int disparity_range, void* disp_left, void* disp_right, size_t disp_step,
                                              size_t disp_pair_stride, int disp_elem_bytes) {
    return pair_batch(mg, cost, n_pairs, left, right, img_step, pair_stride, rows, cols, window_rad, disparity_range, disp_left, disp_right,
                      disp_step, disp_pair_stride, disp_elem_bytes, true);
}

int stereo_mgpu_disparity_pair_bands_u8_host(stereo_mgpu* mg, int cost, const uint8_t* left, size_t left_step, const uint8_t* right,
                                             size_t right_step, int rows, int cols, int window_rad, int disparity_range,
                                             void* disp_left, void* disp_right, size_t disp_step, int disp_elem_bytes) {
    return pair_bands(mg, cost, left, left_step, right, right_step, rows, cols, window_rad, disparity_range, disp_left, disp_right,
                      disp_step, disp_elem_bytes, false);
}

int stereo_mgpu_disparity_pair_bands_f32_host(stereo_mgpu* mg, int cost, const float* left, size_t left_step, const float* right,
                                              size_t right_step, int rows, int cols, int window_rad, int disparity_range,
                                              void* disp_left, void* disp_right, size_t disp_step, int disp_elem_bytes) {
    return pair_bands(mg, cost, left, left_step, right, right_step, rows, cols, window_rad, disparity_range, disp_left, disp_right,
                      disp_step, disp_elem_bytes, true);
}

} // extern "C"
