// Host-side plumbing of the library: context, grow-only device buffers, per-image geometry.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <deque>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>
#include "../../include/b200jpeg.h"
#include "bj_dev.h"

#define BJ_STR2(x) #x
#define BJ_STR(x) BJ_STR2(x)

namespace bj {

// Grow-only device allocation: batches reuse HBM instead of paying cudaMalloc per call.
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return BJ_OK;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        if (cudaMalloc(&p, want) != cudaSuccess) { cudaGetLastError(); p = nullptr; return BJ_ERR_NOMEM; }
        cap = want;
        return BJ_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

// Host worker pool: the per-image host work of a batch (header parse, packing file bytes into pinned staging) is
// independent per image, like everything else on this path; the calling thread takes part.  Replaces the
// reference's single producer thread (src/decoder_host.cpp:101-211).
class HostPool {
    std::vector<std::thread> workers_;
    std::mutex m_;
    std::condition_variable cv_, done_cv_;
    const std::function<void(int, int)> *job_ = nullptr;
    std::atomic<int> next_{0};
    int n_ = 0, chunk_ = 1, epoch_ = 0, active_ = 0;
    bool stop_ = false;

    void drain() {
        for (;;) {
            const int b = next_.fetch_add(chunk_);
            if (b >= n_) break;
            (*job_)(b, b + chunk_ < n_ ? b + chunk_ : n_);
        }
    }
    void run() {
        int seen = 0;
        for (;;) {
            {
                std::unique_lock<std::mutex> l(m_);
                cv_.wait(l, [&] { return stop_ || epoch_ != seen; });
                if (stop_) return;
                seen = epoch_;
            }
            drain();
            {
                std::lock_guard<std::mutex> l(m_);
                if (--active_ == 0) done_cv_.notify_one();
            }
        }
    }

public:
    int threads() const { return (int)workers_.size() + 1; }
    void resize(int nthreads) {                       // total threads including the caller
        shutdown();
        stop_ = false;
        for (int i = 1; i < nthreads; i++) workers_.emplace_back([this] { run(); });
    }
    void shutdown() {
        { std::lock_guard<std::mutex> l(m_); stop_ = true; }
        cv_.notify_all();
        for (auto &t : workers_) t.join();
        workers_.clear();
    }
    ~HostPool() { shutdown(); }
    // fn(begin, end) over [0, n) in chunks; returns when all of it is done
    void parallel_for(int n, int chunk, const std::function<void(int, int)> &fn) {
        if (n <= 0) return;
        if (workers_.empty() || n <= chunk) { fn(0, n); return; }
        {
            std::lock_guard<std::mutex> l(m_);
            job_ = &fn; n_ = n; chunk_ = chunk > 0 ? chunk : 1; next_.store(0);
            active_ = (int)workers_.size();
            epoch_++;
        }
        cv_.notify_all();
        drain();
        std::unique_lock<std::mutex> l(m_);
        done_cv_.wait(l, [&] { return active_ == 0; });
    }
};

// Page-locked host ranges this library knows about (bj_host_alloc, bj_host_register): files that lie inside one of
// them are uploaded straight from the caller's memory, without a staging copy.
class PinnedRanges {
    std::mutex m_;
    std::vector<std::pair<uintptr_t, uintptr_t>> r_;
public:
    void add(const void *p, size_t bytes) { std::lock_guard<std::mutex> l(m_); r_.emplace_back((uintptr_t)p, (uintptr_t)p + bytes); }
    void remove(const void *p) {
        std::lock_guard<std::mutex> l(m_);
        for (size_t i = 0; i < r_.size(); i++) if (r_[i].first == (uintptr_t)p) { r_[i] = r_.back(); r_.pop_back(); return; }
    }
    bool contains(uintptr_t lo, uintptr_t hi) {
        std::lock_guard<std::mutex> l(m_);
        for (auto &r : r_) if (lo >= r.first && hi <= r.second) return true;
        return false;
    }
};
inline PinnedRanges &pinned_ranges() { static PinnedRanges r; return r; }

constexpr int kSlots = 3;             // sub-batches in flight inside bj_decode_batch
constexpr size_t kDefaultMaxImagePixels = (size_t)1 << 28;   // option "max_image_pixels"

enum { POOL_COMPAT_MD = 0, POOL_COMPAT_MCUS, POOL_COEF, POOL_OUT, POOL_IMGS, POOL_TILES, POOL_COUNT };

// counters of one bj_decode_batch / job (bj_get_stat: "decode_batch_<name>", "total_<name>")
enum { ST_SUB = 0, ST_LAUNCH, ST_H2D, ST_D2H, ST_HOST_MS, ST_WAIT_MS, ST_D2H_COPIES, ST_MS_UNSTUFF, ST_MS_SYNC, ST_MS_WRITE, ST_MS_IDCT, ST_DIRECT, ST_MS_RESIZE, ST_MS_PROG, ST_COUNT };

}  // namespace bj

struct bj_job;
struct bj_batch;

namespace bj {
// The thread behind bj_submit / bj_wait: runs the submitted batches one after the other (b200jpeg.cu).
struct AsyncWorker {
    std::mutex m;
    std::condition_variable cv, done_cv;
    std::deque<bj_job *> q;              // front = the job that is running
    bool stop = false;
    std::thread th;
    void run();
    bool pending() { std::lock_guard<std::mutex> l(m); return !q.empty(); }
};
struct Device;
}  // namespace bj

// A context: the options and counters, and the GPUs it drives (one for bj_create, several for bj_create_multi).
struct bj_ctx {
    int subseq_bits = 0;                 // sub-sequence length of the synchronisation pass; 0 = automatic (per image)
    int slices = 0;                      // slices (write pass) per sub-sequence: 1, 2, 4, 8; 0 = default (1)
    int sync_threads = 0;                // CTA width of the synchronisation pass: 128, 256; 0 = automatic (per batch)
    size_t sub_batch_bytes = 0;          // 0 = default
    int sub_batch_ramp = 1;              // the first two sub-batches of a call are smaller (the copy-out starts earlier)
    int packed_outputs = 0;              // see batch_download_async
    int packed_inputs = 0;               // see batch_assign: 0 = upload straight from the caller's memory when it is known to be page-locked
                                         // (bj_host_alloc / bj_host_register), 1 = the caller says it is, -1 = always stage
    int ref_m = 100;                     // BJ_OUT_REF_MCUS: MAX_MCU_PER_DPU of the host that reads the buffer (Makefile:2 of the reference)
    int debug_poison = 0;                // fill coefficient / DC / output buffers with 0xA5 before every decode (tests: every byte must be written)
    size_t max_image_pixels = bj::kDefaultMaxImagePixels;   // larger images are refused (BJ_ERR_UNSUPPORTED), like the reference's "Too high resolution"
    size_t sub_batch_out_bytes = (size_t)1 << 30; // decoded bytes per sub-batch of bj_decode_batch
    int sync_rounds = 0;                 // 0 = default (3 launches of the fix-up kernel before the first check)
    int progressive = 0;                 // 1: the data-loader entries decode progressive (SOF2) files too (kernels_prog.cuh)
    std::vector<bj::Device *> devs;      // never empty; staged and stage-level entries run on devs[0]
    bj::AsyncWorker *async = nullptr;    // bj_submit / bj_wait
    double stats[bj::ST_COUNT] = {};     // counters of the last bj_decode_batch / job, folded over the devices
    double totals[bj::ST_COUNT] = {};    // ... summed over every call since bj_create
    std::mutex error_m;                  // the devices' host threads report errors side by side
    std::string last_error;
    void set_error(const char *what) { std::lock_guard<std::mutex> l(error_m); last_error = what; }
};

namespace bj {

// One GPU of a context: what its host thread works with.
struct Device {
    bj_ctx *ctx = nullptr;
    int ordinal = 0;
    int sm_count = 0;
    bj_batch *slots[kSlots] = {};        // sub-batches of bj_decode_batch in flight (one stream each)
    cudaStream_t streams[kSlots] = {};
    cudaEvent_t ev_exec[2] = {nullptr, nullptr};      // bj_exec_mcus: around the kernel ("DPU execution" profile line)
    DevBuf pool[POOL_COUNT];
    HostPool host_pool;
    float last_exec_ms = 0.f;
    int check(cudaError_t e) {
        if (e == cudaSuccess) return BJ_OK;
        ctx->set_error(cudaGetErrorString(e));
        cudaGetLastError();
        return BJ_ERR_CUDA;
    }
};

struct Geometry {
    uint32_t nmx, nmy, nmcu, bpm, ndu;   // MCUs per row/column, total, data units per MCU, total data units
    uint32_t tile_mcus;                  // MCUs per K2/K3 tile
};

inline Geometry geometry_of(const bj_image_desc &d) {
    Geometry g;
    g.nmx = (d.mcu_w + d.hs - 1) / d.hs;
    g.nmy = (d.mcu_h + d.vs - 1) / d.vs;
    g.nmcu = g.nmx * g.nmy;
    g.bpm = 0;
    for (int j = 0; j < d.ncomp; j++) g.bpm += (uint32_t)d.comp_h[j] * d.comp_v[j];
    g.ndu = g.nmcu * g.bpm;
    g.tile_mcus = kTileThreads / g.bpm;
    return g;
}

// Reduced-size output: log2 of a scale denominator 1, 2, 4 or 8; -1 for any other value.
inline int scale_log2_of(uint32_t scale) { return scale == 1 ? 0 : scale == 2 ? 1 : scale == 4 ? 2 : scale == 8 ? 3 : -1; }

// The rectangle a region of interest selects in the image scaled by 1 / scale (ceil(width / scale) x ceil(height / scale),
// include/b200jpeg.h): false if the scale is not 1, 2, 4 or 8 or the ROI does not fit the scaled image.  roi == nullptr or
// {0,0,0,0}: the whole scaled image.  The sums are taken in 64 bits: x + w must not wrap into range.
inline bool roi_rect(const bj_image_desc &d, const bj_roi *roi, uint32_t scale, bj_roi *r) {
    const int sl = scale_log2_of(scale);
    if (sl < 0) return false;
    const uint32_t W = (d.width + scale - 1) >> sl, H = (d.height + scale - 1) >> sl;
    if (!roi || (roi->x == 0 && roi->y == 0 && roi->w == 0 && roi->h == 0)) { *r = bj_roi{0, 0, W, H}; return true; }
    if (roi->w == 0 || roi->h == 0 || (uint64_t)roi->x + roi->w > W || (uint64_t)roi->y + roi->h > H) return false;
    *r = *roi;
    return true;
}

// The crop window of an image: its pixels in the scaled image, and the MCUs that hold their full-size footprint
// [s cx, min(s (cx + cw), width)) x [s cy, min(s (cy + ch), height)) (the only ones the K2/K3 tile list covers).
inline void set_crop(const bj_roi &r, int scale_log2, ImgDev *im) {
    im->cx = r.x; im->cy = r.y; im->cw = r.w; im->ch = r.h;
    im->scale_log2 = (uint8_t)scale_log2;
    const uint32_t mw = im->hs * 8u, mh = im->vs * 8u;
    const uint32_t x_lo = r.x << scale_log2, x_hi = (uint32_t)std::min<uint64_t>((uint64_t)(r.x + r.w) << scale_log2, im->width);
    const uint32_t y_lo = r.y << scale_log2, y_hi = (uint32_t)std::min<uint64_t>((uint64_t)(r.y + r.h) << scale_log2, im->height);
    im->mx_lo = (uint16_t)(x_lo / mw); im->mx_hi = (uint16_t)((x_hi + mw - 1) / mw);
    im->my_lo = (uint16_t)(y_lo / mh); im->my_hi = (uint16_t)((y_hi + mh - 1) / mh);
}

// The output layout of a w x h image in the RGB8 or BMP format whose first byte is at out_base: the fields of the
// image record the copy-out reads (tile_copy_out).  Shared by the IDCT + colour stage's records and the resize records.
inline void set_layout(int format, uint32_t w, uint32_t h, uint64_t out_base, ImgDev *im) {
    im->row_bytes = w * 3;
    if (format == BJ_OUT_BMP) {
        im->row_pad = w % 4;
        im->out_pitch = w * 3 + im->row_pad;
        im->out_row0 = out_base + 26 + (uint64_t)(h - 1) * im->out_pitch;
        im->row_dir = -1;
        im->bgr = 1;
    } else {
        im->row_pad = 0;
        im->out_pitch = w * 3;
        im->out_row0 = out_base;
        im->row_dir = 1;
        im->bgr = 0;
    }
}

// out_base: byte offset of this image's output inside the batch output buffer.  roi, scale: a request roi_rect accepted
// (nullptr, 1: the whole image; BJ_OUT_REF_MCUS always takes the whole image at full size).
inline void fill_imgdev(const bj_image_desc &d, const Geometry &g, int format, uint32_t du_base, uint64_t out_base, ImgDev *im,
                        const bj_roi *roi = nullptr, uint32_t scale = 1) {
    memset(im, 0, sizeof(*im));
    im->width = d.width; im->height = d.height;
    im->nmx = g.nmx; im->nmy = g.nmy;
    im->du_base = du_base;
    im->hs = d.hs; im->vs = d.vs; im->ncomp = d.ncomp; im->bpm = (uint8_t)g.bpm;
    im->valid = 1;
    if (format == BJ_OUT_REF_MCUS) { roi = nullptr; scale = 1; }
    bj_roi r{};
    roi_rect(d, roi, scale, &r);
    set_crop(r, scale_log2_of(scale), im);
    if (format == BJ_OUT_REF_MCUS) {
        im->row_bytes = r.w * 3;
        im->row_pad = 0; im->out_pitch = 0; im->row_dir = 1; im->bgr = 0;
        im->out_row0 = out_base;                       // byte offset of the image's first chunk
    } else
        set_layout(format, r.w, r.h, out_base, im);
}

// Fixed-size output: 0 when `size` asks for none (nullptr or {0,0}), 1 when it asks for a w x h output, -1 when it is
// refused: only one of w, h is 0, or either is above 65535 (the BMP header holds 16-bit sizes).
inline int resize_kind(const bj_size *size) {
    if (!size || (size->w == 0 && size->h == 0)) return 0;
    return (size->w == 0 || size->h == 0 || size->w > 65535u || size->h > 65535u) ? -1 : 1;
}

// The resize record of an image whose IDCT-stage record `src` (an RGB8 output of its scaled crop at src_off) is resized
// to `size` (resize_kind 1) in `format` at out_base.
inline void fill_resize(const bj_size &size, int format, uint64_t out_base, const ImgDev &src, ResizeDev *rz) {
    memset(rz, 0, sizeof(*rz));
    ImgDev &o = rz->out;
    o.width = size.w; o.height = size.h; o.valid = 1;
    o.cw = size.w; o.ch = size.h;                      // (cx = cy = 0, mx_lo = my_lo = 0: the tile at (0, 0) writes a BMP header)
    set_layout(format, size.w, size.h, out_base, &o);
    rz->src_off = src.out_row0;
    rz->sw = src.cw; rz->sh = src.ch;
    rz->tiles_x = (size.w + kResizeTileW - 1) / kResizeTileW;
}
inline uint32_t resize_tile_count(const bj_size &size) {
    return ((size.w + kResizeTileW - 1) / kResizeTileW) * ((size.h + kResizeTileH - 1) / kResizeTileH);
}

// The image's quantiser set as the K2 kernel stages it.
inline void fill_qtab(const bj_image_desc &d, QTab *q) {
    memset(q, 0, sizeof(*q));
    // The reference forwards quantisation tables to the DPUs only up to the first unset table id
    // (src/decoder_host.cpp:173-178): a table behind a gap reads as zeros.
    bool reachable[4];
    bool ok = true;
    for (int t = 0; t < 4; t++) { ok = ok && d.qt_set[t]; reachable[t] = ok; }
    for (int j = 0; j < 3; j++)
        for (int k = 0; k < 64; k++)
            q->q16[j][k] = (j < d.ncomp && reachable[d.qt_id[j] & 3]) ? ((uint32_t)d.qt_zz[d.qt_id[j] & 3][k] << 16) : 0u;
}
// Same quantiser set?  (what fill_qtab reads of the two descriptors)
inline bool same_qtab(const bj_image_desc &a, const bj_image_desc &b) {
    return a.ncomp == b.ncomp && !memcmp(a.qt_id, b.qt_id, 3) && !memcmp(a.qt_set, b.qt_set, 4) && !memcmp(a.qt_zz, b.qt_zz, sizeof(a.qt_zz));
}

// Descriptors that do not come from parse_header (bj_stage_idct_color, bj_decode_batch_desc) are checked before they
// reach a kernel: the tile and shared-memory sizes assume what the reference's parser enforces
// (src/jpeg_scanner.cpp:187-285: 1..3 components, luma sampling 1 or 2, chroma 1x1, table ids below 4).
inline bool desc_is_sane(const bj_image_desc &d) {
    if (d.width == 0 || d.height == 0 || d.width > 65535u || d.height > 65535u) return false;
    if (d.ncomp < 1 || d.ncomp > 3) return false;
    if ((d.hs != 1 && d.hs != 2) || (d.vs != 1 && d.vs != 2)) return false;
    if (d.comp_h[0] != d.hs || d.comp_v[0] != d.vs) return false;
    for (int j = 1; j < d.ncomp; j++) if (d.comp_h[j] != 1 || d.comp_v[j] != 1) return false;
    for (int j = 0; j < d.ncomp; j++) if (d.qt_id[j] > 3 || d.dc_id[j] > 3 || d.ac_id[j] > 3) return false;
    if (d.mcu_w != (d.width + 7) / 8 || d.mcu_h != (d.height + 7) / 8) return false;
    return true;
}

// BJ_OUT_REF_MCUS: DPU chunks of an image (src/decoder_host.cpp:125-128) and the bytes of its `mcus` buffers.
inline uint32_t ref_mcus_chunks(const bj_image_desc &d, int M) {
    const uint32_t pw = (d.mcu_w_real + 1) / 2 * 2, ph = (d.mcu_h_real + 1) / 2 * 2;
    return (pw * ph + (uint32_t)M - 1) / (uint32_t)M;
}
// Bytes of a w x h image in the RGB8 or BMP format (0 for any other)
inline size_t layout_bytes(int format, size_t w, size_t h) {
    if (format == BJ_OUT_RGB8) return w * h * 3;
    if (format == BJ_OUT_BMP) return 26 + h * (w * 3 + w % 4);
    return 0;
}
// roi, scale: as for fill_imgdev (BJ_OUT_REF_MCUS ignores them); size: a target size (resize_kind 1) or nullptr
inline size_t output_bytes(const bj_image_desc &d, int format, int M, const bj_roi *roi = nullptr, uint32_t scale = 1,
                           const bj_size *size = nullptr) {
    if (format == BJ_OUT_REF_MCUS) return (size_t)ref_mcus_chunks(d, M) * 64 * (size_t)M * 3 * sizeof(int16_t);
    if (size) return layout_bytes(format, size->w, size->h);
    bj_roi r{};
    roi_rect(d, roi, scale, &r);
    return layout_bytes(format, r.w, r.h);
}

inline void append_tiles(const Geometry &g, uint32_t img, uint32_t du_base, std::vector<TileDev> *tiles) {
    for (uint32_t my = 0; my < g.nmy; my++)
        for (uint32_t mx = 0; mx < g.nmx; mx += g.tile_mcus) {
            TileDev t;
            t.img = img; t.my = (uint16_t)my; t.mx0 = (uint16_t)mx;
            t.nm = (uint16_t)std::min<uint32_t>(g.tile_mcus, g.nmx - mx);
            t.ndu = (uint16_t)(t.nm * g.bpm);
            t.du0 = du_base + (my * g.nmx + mx) * g.bpm;
            tiles->push_back(t);
        }
}

}  // namespace bj
