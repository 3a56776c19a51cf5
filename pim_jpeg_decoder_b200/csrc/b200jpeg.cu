// libb200jpeg.so - C ABI (include/b200jpeg.h) and host orchestration of the sm_100a kernels.
// No CPU decode path exists in this library: every compute entry needs a CUDA device.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <stddef.h>
#include <string.h>

#include <algorithm>
#include <time.h>
#include <string>
#include <thread>
#include <vector>

#include "../../include/b200jpeg.h"
#include "bj_dev.h"
#include "bj_host.h"
#include "kernels_idct.cuh"
#include "parse.h"
#include "batch.h"

using namespace bj;

// ------------------------------------------------------------------------------------------------ context

extern "C" const char *bj_status_string(int s) {
    switch (s) {
        case BJ_OK: return "ok";
        case BJ_ERR_ARG: return "bad argument";
        case BJ_ERR_CUDA: return "CUDA error";
        case BJ_ERR_NOMEM: return "out of memory";
        case BJ_ERR_INVALID_JPEG: return "invalid JPEG (the reference's read_JPEG rejects it)";
        case BJ_ERR_UNSUPPORTED: return "unsupported JPEG (not a single-scan baseline file)";
        case BJ_ERR_CORRUPT_SCAN: return "corrupt entropy-coded data";
    }
    return "unknown status";
}

extern "C" const char *bj_build_info(void) { return "b200jpeg sm_100a (CUDA " BJ_STR(CUDART_VERSION) "), built " __DATE__; }

extern "C" void bj_destroy(bj_ctx *c);

// CUDA devices this process sees; none: says so (there is no CPU fallback) and returns 0.
static int visible_devices() {
    int count = 0;
    const cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        fprintf(stderr, "b200jpeg: no CUDA device (%s) - this library has no CPU fallback\n", cudaGetErrorString(e));
        return 0;
    }
    return count;
}

static int open_device(Device *dev) {
    int rc = dev->check(cudaSetDevice(dev->ordinal));
    cudaDeviceProp prop;
    if (rc == BJ_OK) rc = dev->check(cudaGetDeviceProperties(&prop, dev->ordinal));
    if (rc == BJ_OK) dev->sm_count = prop.multiProcessorCount;
    if (rc == BJ_OK) rc = dev->check(cudaFuncSetAttribute(k_idct_color<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemIdctColor));
    if (rc == BJ_OK) rc = dev->check(cudaFuncSetAttribute(k_idct_color<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemIdctColor));
    if (rc == BJ_OK) rc = batch_kernels_init(dev);
    for (int i = 0; i < kSlots && rc == BJ_OK; i++) rc = dev->check(cudaStreamCreateWithFlags(&dev->streams[i], cudaStreamNonBlocking));
    for (int i = 0; i < 2 && rc == BJ_OK; i++) rc = dev->check(cudaEventCreate(&dev->ev_exec[i]));
    return rc;
}

// A context on the devices `ordinals[0..n)` (of `count`), one host thread each.
static int create_ctx(bj_ctx **out, const int *ordinals, int n, int count) {
    for (int i = 0; i < n; i++) if (ordinals[i] < 0 || ordinals[i] >= count) return BJ_ERR_ARG;
    bj_ctx *c = new (std::nothrow) bj_ctx();
    if (!c) return BJ_ERR_NOMEM;
    for (int i = 0; i < n; i++) {
        Device *dev = new (std::nothrow) Device{c, ordinals[i]};
        if (!dev) { bj_destroy(c); return BJ_ERR_NOMEM; }
        c->devs.push_back(dev);
    }
    // one CUDA context per device, created side by side (a context takes some hundred milliseconds)
    std::vector<int> rcs(n, BJ_OK);
    std::vector<std::thread> th;
    for (int i = 1; i < n; i++) th.emplace_back([&, i] { rcs[i] = open_device(c->devs[i]); });
    rcs[0] = open_device(c->devs[0]);
    for (auto &t : th) t.join();
    for (int i = 0; i < n; i++) if (rcs[i] != BJ_OK) { bj_destroy(c); return rcs[i]; }    // (releases whatever was created)
    // worker threads for the per-image host work (header parse; staging copies for pageable inputs): a few per device
    // are enough - the host reads some hundred bytes per file - and more only take memory bandwidth from the copy
    // engines.  All devices' threads together stay within what this process may run on (cgroup / affinity).
    const int avail = std::max(1, (int)std::thread::hardware_concurrency());
    for (Device *dev : c->devs) dev->host_pool.resize(std::max(1, std::min(4, avail / (2 * n))));
    *out = c;
    return BJ_OK;
}

extern "C" int bj_create(bj_ctx **out, int device) {
    if (!out) return BJ_ERR_ARG;
    *out = nullptr;
    const int count = visible_devices();
    return count ? create_ctx(out, &device, 1, count) : BJ_ERR_CUDA;
}

// All the GPUs of one process: replaces `DpuSet::allocate(DPU_ALLOCATE_ALL)` (src/decoder_host.cpp:32-33) - the
// reference's single process spreads its work over every DPU of the machine; here one context drives `ndev` GPUs,
// one host thread each.  devices == NULL: the first ndev devices; ndev <= 0: all of them.
extern "C" int bj_create_multi(bj_ctx **out, const int *devices, int ndev) {
    if (!out) return BJ_ERR_ARG;
    *out = nullptr;
    const int count = visible_devices();
    if (!count) return BJ_ERR_CUDA;
    if (ndev <= 0) { ndev = count; devices = nullptr; }
    if (ndev > count && !devices) return BJ_ERR_ARG;
    // no list given and fewer devices wanted than there are: every (count / ndev)-th one - neighbouring ordinals
    // often share a PCIe uplink, and the copy-out is what bounds this path (profiles/r2_bench_*gpu_spread.json)
    const int stride = (!devices && count >= 2 * ndev) ? count / ndev : 1;
    std::vector<int> ordinals(ndev);
    for (int i = 0; i < ndev; i++) ordinals[i] = devices ? devices[i] : i * stride;
    return create_ctx(out, ordinals.data(), ndev, count);
}

extern "C" int bj_device_count(const bj_ctx *c) { return c ? (int)c->devs.size() : 0; }

extern "C" void bj_destroy(bj_ctx *c) {
    if (!c) return;
    if (c->async) {
        { std::lock_guard<std::mutex> l(c->async->m); c->async->stop = true; }
        c->async->cv.notify_all();
        if (c->async->th.joinable()) c->async->th.join();                      // (finishes the queued jobs first)
        delete c->async;
        c->async = nullptr;
    }
    for (Device *dev : c->devs) {
        cudaSetDevice(dev->ordinal);
        cudaDeviceSynchronize();
        for (auto &p : dev->pool) p.release();
        for (auto &b : dev->slots) if (b) { b->release(); delete b; b = nullptr; }
        for (int i = 0; i < kSlots; i++) if (dev->streams[i]) cudaStreamDestroy(dev->streams[i]);
        for (auto &ev : dev->ev_exec) if (ev) cudaEventDestroy(ev);
        delete dev;
    }
    delete c;
}

extern "C" const char *bj_last_error(const bj_ctx *c) { return c ? c->last_error.c_str() : "null context"; }
extern "C" int bj_device_sm_count(const bj_ctx *c) { return c ? c->devs[0]->sm_count : 0; }

extern "C" void *bj_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    pinned_ranges().add(p, bytes ? bytes : 1);
    return p;
}
extern "C" void bj_host_free(void *p) { if (p) { pinned_ranges().remove(p); cudaFreeHost(p); } }

extern "C" int bj_host_register(void *p, size_t bytes) {
    if (!p || !bytes) return BJ_ERR_ARG;
    const cudaError_t e = cudaHostRegister(p, bytes, cudaHostRegisterDefault);
    if (e != cudaSuccess && e != cudaErrorHostMemoryAlreadyRegistered) { cudaGetLastError(); return BJ_ERR_CUDA; }
    if (e != cudaSuccess) cudaGetLastError();
    pinned_ranges().add(p, bytes);
    return BJ_OK;
}
extern "C" int bj_host_unregister(void *p) {
    if (!p) return BJ_ERR_ARG;
    pinned_ranges().remove(p);
    if (cudaHostUnregister(p) != cudaSuccess) { cudaGetLastError(); return BJ_ERR_CUDA; }
    return BJ_OK;
}

extern "C" int bj_set_option(bj_ctx *c, const char *name, long value) {
    if (!c || !name) return BJ_ERR_ARG;
    if (!strcmp(name, "subseq_bits")) { if (value != 0 && (value < 128 || value % 32 || value > (1 << 18))) return BJ_ERR_ARG; c->subseq_bits = (int)value; return BJ_OK; }
    if (!strcmp(name, "sub_batch_ramp")) { c->sub_batch_ramp = value != 0; return BJ_OK; }
    // the synchronisation pass with early stop of re-decodes is the only one; the option stays for bench.py --sync-phased
    if (!strcmp(name, "sync_phased")) return value == 1 ? BJ_OK : BJ_ERR_ARG;
    if (!strcmp(name, "slices")) { if (value != 0 && value != 1 && value != 2 && value != 4 && value != 8) return BJ_ERR_ARG; c->slices = (int)value; return BJ_OK; }
    if (!strcmp(name, "sub_batch_bytes")) { if (value < (1 << 16)) return BJ_ERR_ARG; c->sub_batch_bytes = (size_t)value; return BJ_OK; }
    if (!strcmp(name, "packed_outputs")) { c->packed_outputs = value != 0; return BJ_OK; }
    if (!strcmp(name, "packed_inputs")) { if (value < -1 || value > 1) return BJ_ERR_ARG; c->packed_inputs = (int)value; return BJ_OK; }
    if (!strcmp(name, "ref_max_mcu_per_dpu")) { if (value < 4 || value % 4 || value > (1 << 20)) return BJ_ERR_ARG; c->ref_m = (int)value; return BJ_OK; }
    if (!strcmp(name, "debug_poison")) { c->debug_poison = value != 0; return BJ_OK; }
    if (!strcmp(name, "max_image_pixels")) { if (value < 1) return BJ_ERR_ARG; c->max_image_pixels = (size_t)value; return BJ_OK; }
    if (!strcmp(name, "sub_batch_out_bytes")) { if (value < (1 << 16)) return BJ_ERR_ARG; c->sub_batch_out_bytes = (size_t)value; return BJ_OK; }
    if (!strcmp(name, "host_threads")) { if (value < 1 || value > 256) return BJ_ERR_ARG; for (Device *dev : c->devs) dev->host_pool.resize((int)value); return BJ_OK; }
    // the synchronisation pass starts every sub-sequence from its own first bit; the option stays for bench.py --sync-preroll
    if (!strcmp(name, "sync_preroll_bits")) return value == 0 ? BJ_OK : BJ_ERR_ARG;
    if (!strcmp(name, "sync_rounds")) { if (value < 0 || value > kMaxRounds) return BJ_ERR_ARG; c->sync_rounds = (int)value; return BJ_OK; }
    return BJ_ERR_ARG;
}

extern "C" int bj_get_stat(const bj_ctx *c, const char *name, double *value) {
    if (!c || !name || !value) return BJ_ERR_ARG;
    if (!strcmp(name, "exec_ms")) { *value = 0; for (const Device *dev : c->devs) *value = std::max(*value, (double)dev->last_exec_ms); return BJ_OK; }  // of the last bj_exec_mcus
    // "decode_batch_<name>": of the last bj_decode_batch / job, "total_<name>": summed over every call since bj_create.
    // host_ms: parse + layout + pack, wait_ms: host blocked on the GPU; ms_*: kernel time per stage, summed over the
    // sub-batches (CUDA events) - the reference's per-stage "Profiles" lines (src/decoder_host.cpp:379-394)
    static const char *const names[ST_COUNT] = {"sub_batches", "launches", "h2d_bytes", "d2h_bytes", "host_ms", "wait_ms", "d2h_copies",
                                                "ms_unstuff", "ms_sync", "ms_write", "ms_idct", "direct_uploads"};
    const struct { const char *prefix; const double *counters; } sets[] = {{"decode_batch_", c->stats}, {"total_", c->totals}};
    for (const auto &set : sets) {
        const size_t len = strlen(set.prefix);
        if (strncmp(name, set.prefix, len)) continue;
        for (int i = 0; i < ST_COUNT; i++) if (!strcmp(name + len, names[i])) { *value = set.counters[i]; return BJ_OK; }
        return BJ_ERR_ARG;
    }
    if (!strcmp(name, "devices")) { *value = (double)c->devs.size(); return BJ_OK; }
    if (!strcmp(name, "host_threads")) { *value = c->devs[0]->host_pool.threads(); return BJ_OK; }
    return BJ_ERR_ARG;
}

// ------------------------------------------------------------------------------------------------ compat entry

static int launch_exec_mcus(Device *dev, const uint32_t *d_md, int16_t *d_mcus, int nchunk, int M, cudaStream_t s) {
    if (nchunk == 0) return BJ_OK;
    const int blk_per_chunk = M / 4;
    const long long nblk = (long long)nchunk * blk_per_chunk;
    const int grid = (int)((nblk + 15) / 16);
    k_exec_mcus<<<grid, kTileThreads, 0, s>>>(d_md, d_mcus, nchunk, blk_per_chunk, 64 * M * 3);
    return dev->check(cudaGetLastError());
}

extern "C" int bj_exec_mcus_device(bj_ctx *c, const uint32_t *d_md, int16_t *d_mcus, int nchunk, int M, void *stream) {
    if (!c || !d_md || !d_mcus || nchunk < 0 || M < 4 || M % 4 || c->devs.size() != 1) return BJ_ERR_ARG;   // (pointers of one GPU)
    return launch_exec_mcus(c->devs[0], d_md, d_mcus, nchunk, M, (cudaStream_t)stream);
}

static int exec_mcus_one(Device *dev, const uint32_t *metadata, int16_t *mcus, int nchunk, int M) {
    if (dev->check(cudaSetDevice(dev->ordinal)) != BJ_OK) return BJ_ERR_CUDA;
    const size_t md_bytes = (size_t)nchunk * 276 * 4, mc_bytes = (size_t)nchunk * 64 * M * 3 * 2;
    DevBuf &dmd = dev->pool[POOL_COMPAT_MD], &dmc = dev->pool[POOL_COMPAT_MCUS];
    if (dmd.reserve(md_bytes) != BJ_OK || dmc.reserve(mc_bytes) != BJ_OK) return BJ_ERR_NOMEM;
    cudaStream_t s = dev->streams[0];
    // the three pim.copy calls + pim.exec of src/decoder_host.cpp:276-308
    int rc = dev->check(cudaMemcpyAsync(dmd.p, metadata, md_bytes, cudaMemcpyHostToDevice, s));
    if (rc == BJ_OK) rc = dev->check(cudaMemcpyAsync(dmc.p, mcus, mc_bytes, cudaMemcpyHostToDevice, s));
    cudaEventRecord(dev->ev_exec[0], s);
    if (rc == BJ_OK) rc = launch_exec_mcus(dev, (const uint32_t *)dmd.p, (int16_t *)dmc.p, nchunk, M, s);
    cudaEventRecord(dev->ev_exec[1], s);
    if (rc == BJ_OK) rc = dev->check(cudaMemcpyAsync(mcus, dmc.p, mc_bytes, cudaMemcpyDeviceToHost, s));
    if (rc == BJ_OK) rc = dev->check(cudaStreamSynchronize(s));
    if (rc == BJ_OK) cudaEventElapsedTime(&dev->last_exec_ms, dev->ev_exec[0], dev->ev_exec[1]);
    return rc;
}

extern "C" int bj_exec_mcus(bj_ctx *c, const uint32_t *metadata, int16_t *mcus, int nchunk) {
    if (!c || !metadata || !mcus || nchunk < 0) return BJ_ERR_ARG;
    if (nchunk == 0) return BJ_OK;
    int M = 0;                                   // MAX_MCU_PER_DPU as the host compiled it (metadata[19], decoder_host.cpp:172)
    for (int i = 0; i < nchunk && M == 0; i++) M = (int)metadata[(size_t)i * 276 + 19];
    if (M == 0) return BJ_OK;                    // only idle DPUs: the program touches nothing
    if (M < 4 || M % 4) return BJ_ERR_ARG;       // the DPU program works on whole blocks of 4 positions (src/decoder_dpu.c:130)
    for (int i = 0; i < nchunk; i++) { const uint32_t m = metadata[(size_t)i * 276 + 19]; if (m != 0 && m != (uint32_t)M) return BJ_ERR_ARG; }
    // the DPUs are dealt to the GPUs in equal contiguous shares, one host thread per GPU (the first: the caller's)
    const int nd = (int)c->devs.size();
    std::vector<int> rcs(nd, BJ_OK);
    std::vector<std::thread> th;
    auto share = [&](int d) {
        const int lo = (int)((long long)nchunk * d / nd), hi = (int)((long long)nchunk * (d + 1) / nd);
        if (hi > lo) rcs[d] = exec_mcus_one(c->devs[d], metadata + (size_t)lo * 276, mcus + (size_t)lo * 64 * M * 3, hi - lo, M);
    };
    for (int d = 1; d < nd; d++) th.emplace_back(share, d);
    share(0);
    for (auto &t : th) t.join();
    for (int rc : rcs) if (rc != BJ_OK) return rc;
    return BJ_OK;
}

// ------------------------------------------------------------------------------------------------ descriptors

extern "C" int bj_parse_header(const uint8_t *file, size_t len, bj_image_desc *desc) {
    if (!file || !desc) return BJ_ERR_ARG;
    return parse_header(file, len, desc);
}

extern "C" int bj_peek_header(const uint8_t *file, size_t len, bj_image_desc *desc) {
    if (!file || !desc) return BJ_ERR_ARG;
    return parse_header(file, len, desc, /*walk_scan=*/false);
}

extern "C" size_t bj_output_size(const bj_image_desc *d, int format) { return d ? output_bytes(*d, format, 100) : 0; }

extern "C" size_t bj_ref_mcus_size(const bj_image_desc *d, int max_mcu_per_dpu, int *nchunks) {
    if (!d || max_mcu_per_dpu < 4 || max_mcu_per_dpu % 4) return 0;
    if (nchunks) *nchunks = (int)ref_mcus_chunks(*d, max_mcu_per_dpu);
    return output_bytes(*d, BJ_OUT_REF_MCUS, max_mcu_per_dpu);
}

// ------------------------------------------------------------------------------------------------ stage entry

extern "C" int bj_stage_idct_color(bj_ctx *c, const bj_image_desc *desc, const int16_t *coef_zz, int format, uint8_t *out) {
    if (!c || !desc || !coef_zz || !out) return BJ_ERR_ARG;
    if (format != BJ_OUT_RGB8 && format != BJ_OUT_BMP) return BJ_ERR_ARG;
    if (!desc_is_sane(*desc)) return BJ_ERR_ARG;                 // a caller-made descriptor: checked before it sizes anything
    Device *dev = c->devs[0];
    if (dev->check(cudaSetDevice(dev->ordinal)) != BJ_OK) return BJ_ERR_CUDA;
    struct StageRec { ImgDev im; QTab q; } rec;                  // one upload: the image record and its quantiser set
    std::vector<TileDev> tiles;
    Geometry g = geometry_of(*desc);
    fill_imgdev(*desc, g, format, /*du_base=*/0, /*out_base=*/0, &rec.im);
    fill_qtab(*desc, &rec.q);
    append_tiles(g, 0, 0, &tiles);
    const size_t coef_bytes = (size_t)g.ndu * 128, out_bytes = bj_output_size(desc, format);
    DevBuf &dco = dev->pool[POOL_COEF], &dout = dev->pool[POOL_OUT], &dim = dev->pool[POOL_IMGS], &dti = dev->pool[POOL_TILES];
    if (dco.reserve(coef_bytes) || dout.reserve(out_bytes + 64) || dim.reserve(sizeof(rec)) || dti.reserve(tiles.size() * sizeof(TileDev))) return BJ_ERR_NOMEM;
    cudaStream_t s = dev->streams[0];
    int rc = dev->check(cudaMemcpyAsync(dco.p, coef_zz, coef_bytes, cudaMemcpyHostToDevice, s));
    if (rc == BJ_OK) rc = dev->check(cudaMemcpyAsync(dim.p, &rec, sizeof(rec), cudaMemcpyHostToDevice, s));
    if (rc == BJ_OK) rc = dev->check(cudaMemcpyAsync(dti.p, tiles.data(), tiles.size() * sizeof(TileDev), cudaMemcpyHostToDevice, s));
    if (rc == BJ_OK) {
        const uint8_t *base = (const uint8_t *)dim.p;
        k_idct_color<false><<<(unsigned)tiles.size(), kTileThreads, kSmemIdctColor, s>>>((const int16_t *)dco.p, nullptr, (const ImgDev *)base, (const QTab *)(base + offsetof(StageRec, q)),
                                                                                 (const TileDev *)dti.p, (uint8_t *)dout.p);
        rc = dev->check(cudaGetLastError());
    }
    if (rc == BJ_OK) rc = dev->check(cudaMemcpyAsync(out, dout.p, out_bytes, cudaMemcpyDeviceToHost, s));
    if (rc == BJ_OK) rc = dev->check(cudaStreamSynchronize(s));
    return rc;
}

// ------------------------------------------------------------------------------------------------ full path, staged

extern "C" int bj_batch_create(bj_ctx *c, const uint8_t *const *files, const size_t *lens, int n, int format, bj_batch **out) {
    if (!c || !out || n < 0 || (n > 0 && (!files || !lens))) return BJ_ERR_ARG;
    *out = nullptr;
    bj_batch *b = new (std::nothrow) bj_batch();
    if (!b) return BJ_ERR_NOMEM;
    const int rc = batch_assign(b, c->devs[0], files, lens, n, format);     // a staged batch lives on one device
    if (rc != BJ_OK) { b->release(); delete b; return rc; }
    *out = b;
    return BJ_OK;
}

extern "C" void bj_batch_destroy(bj_batch *b) {
    if (!b) return;
    cudaSetDevice(b->dev->ordinal);
    if (b->last_stream) cudaStreamSynchronize(b->last_stream);
    b->release();
    delete b;
}

static cudaStream_t stream_or_default(bj_batch *b, void *stream) { return stream ? (cudaStream_t)stream : b->dev->streams[0]; }

extern "C" int bj_batch_upload(bj_batch *b, void *stream) { return b ? batch_upload(b, stream_or_default(b, stream)) : BJ_ERR_ARG; }
extern "C" int bj_batch_decode(bj_batch *b, void *stream) { return b ? batch_decode(b, stream_or_default(b, stream)) : BJ_ERR_ARG; }
extern "C" int bj_batch_sync(bj_batch *b) { return b ? batch_sync(b) : BJ_ERR_ARG; }
extern "C" int bj_batch_download(bj_batch *b, uint8_t *const *outs, void *stream) {
    if (!b || (b->n > 0 && !outs)) return BJ_ERR_ARG;
    return batch_download(b, outs, stream_or_default(b, stream));
}

extern "C" int bj_batch_status(const bj_batch *b, int *status) {
    if (!b || !status) return BJ_ERR_ARG;
    for (int i = 0; i < b->n; i++) status[i] = batch_image_status(b, i);
    return BJ_OK;
}

extern "C" int bj_batch_get_info(const bj_batch *b, bj_batch_info *info) {
    if (!b || !info) return BJ_ERR_ARG;
    memset(info, 0, sizeof(*info));
    info->pixels = b->pixels; info->scan_bytes = b->scan_bytes_max; info->data_units = b->coef_units; info->out_bytes = b->out_bytes;
    if (b->synced) {                                             // the scans' true lengths are found on the device
        info->scan_bytes = 0;
        for (int i = 0; i < b->n; i++) info->scan_bytes += const_cast<bj_batch *>(b)->h_state()[i].raw_len;
    }
    info->h2d_bytes = b->files_bytes + b->meta_bytes; info->d2h_bytes = b->d2h_bytes;
    uint32_t nsub = 0;
    if (b->synced) for (int i = 0; i < b->n; i++) nsub += const_cast<bj_batch *>(b)->h_state()[i].nsub;
    info->subsequences = nsub; info->sync_rounds = b->sync_rounds; info->launches = b->launches;
    info->ms_entropy = b->ms_entropy; info->ms_idct = b->ms_idct;
    info->ms_unstuff = b->ms_unstuff; info->ms_sync = b->ms_sync; info->ms_write = b->ms_write;
    info->clean_bytes = 0;
    if (b->synced) for (int i = 0; i < b->n; i++) info->clean_bytes += const_cast<bj_batch *>(b)->h_state()[i].clean_len;
    return BJ_OK;
}

extern "C" int bj_batch_output_offset(const bj_batch *b, int i, size_t *offset, size_t *bytes) {
    if (!b || i < 0 || i >= b->n) return BJ_ERR_ARG;
    if (offset) *offset = b->out_off[i];
    if (bytes) *bytes = b->out_size[i];
    return b->parse_status[i];
}

extern "C" int bj_batch_device_output(const bj_batch *b, int i, void **dptr, size_t *bytes) {
    if (!b || i < 0 || i >= b->n || b->parse_status[i] != BJ_OK) return BJ_ERR_ARG;
    if (dptr) *dptr = (uint8_t *)b->d_out.p + b->out_off[i];
    if (bytes) *bytes = b->out_size[i];
    return BJ_OK;
}

extern "C" int bj_batch_device_coefficients(const bj_batch *b, int i, void **dptr, size_t *bytes, void **dc_dptr) {
    if (!b || i < 0 || i >= b->n || b->parse_status[i] != BJ_OK) return BJ_ERR_ARG;
    if (dptr) *dptr = (int16_t *)b->d_coef.p + (size_t)b->du_base[i] * 64;
    if (bytes) *bytes = (size_t)b->ndu[i] * 128;
    if (dc_dptr) *dc_dptr = (int16_t *)b->d_dc.p + b->du_base[i];
    return BJ_OK;
}

// Stage-level entry for known-answer tests: K0 + K1 only; coefficients (zig-zag, DC un-differenced) back to the host.
extern "C" int bj_stage_entropy(bj_ctx *c, const uint8_t *file, size_t len, int16_t *coef_zz, size_t capacity_bytes, int *status) {
    if (!c || !file || !coef_zz) return BJ_ERR_ARG;
    bj_batch *b = nullptr;
    const uint8_t *files[1] = {file};
    const size_t lens[1] = {len};
    int rc = bj_batch_create(c, files, lens, 1, BJ_OUT_RGB8, &b);
    if (rc != BJ_OK) return rc;
    if (b->parse_status[0] != BJ_OK) { rc = b->parse_status[0]; bj_batch_destroy(b); return rc; }
    if ((size_t)b->ndu[0] * 128 > capacity_bytes) { bj_batch_destroy(b); return BJ_ERR_ARG; }
    Device *dev = b->dev;
    cudaStream_t s = dev->streams[0];
    rc = batch_upload(b, s);
    if (rc == BJ_OK) rc = batch_decode(b, s);
    if (rc == BJ_OK) rc = batch_sync(b);
    std::vector<int16_t> dcs(b->ndu[0]);
    if (rc == BJ_OK) rc = dev->check(cudaMemcpyAsync(coef_zz, b->d_coef.p, (size_t)b->ndu[0] * 128, cudaMemcpyDeviceToHost, s));
    if (rc == BJ_OK && b->ndu[0]) rc = dev->check(cudaMemcpyAsync(dcs.data(), b->d_dc.p, (size_t)b->ndu[0] * 2, cudaMemcpyDeviceToHost, s));
    if (rc == BJ_OK) rc = dev->check(cudaStreamSynchronize(s));
    if (rc == BJ_OK) for (uint32_t u = 0; u < b->ndu[0]; u++) coef_zz[(size_t)u * 64] = dcs[u];   // the device keeps DC in its own plane
    if (rc == BJ_OK && status) *status = batch_image_status(b, 0);
    bj_batch_destroy(b);
    return rc;
}

// ------------------------------------------------------------------------------------------------ full path, one call
// Sub-batches rotate over kSlots batch objects, each with its own stream: while sub-batch k copies out (PCIe D2H is
// the bound of this call: 3 bytes per pixel), sub-batch k+1 decodes and the host reads the headers of sub-batch k+2.
// The image list is cut into sub-batches by a RangeSource; the devices of a context (several with bj_create_multi) pull
// from ONE source, so the list is dealt dynamically - by sub-batch, in list order, no collective - like the reference
// deals its images over all DPUs of the machine (src/decoder_host.cpp:32-33,125-149).
static double wall_ms() {
    struct timespec t;
    clock_gettime(CLOCK_MONOTONIC, &t);
    return t.tv_sec * 1e3 + t.tv_nsec * 1e-6;
}

namespace {
struct RangeSource {
    std::mutex m;
    const size_t *lens;
    int n, next = 0;
    size_t budget;
    bool ramp;
    // k = how many ranges the asking device has had: its first two are small, so that its copy-out starts early
    bool take(int k, int *i0, int *i1) {
        std::lock_guard<std::mutex> l(m);
        if (next >= n) return false;
        const size_t cap = !ramp ? budget : (k == 0 ? budget / 8 : (k == 1 ? budget / 3 : budget));
        int j = next;
        size_t bytes = 0;
        while (j < n && (j == next || bytes + lens[j] <= cap)) bytes += lens[j++];
        *i0 = next; *i1 = j; next = j;
        return true;
    }
};
}  // namespace

struct CallInput {                       // what a call decodes: files, or (bj_decode_batch_desc) descriptors + scans
    const uint8_t *const *files; const size_t *lens;
    const bj_image_desc *descs; const int *kinds;
};

// One device's share of a call: pull ranges from `src` until it runs dry.  st[ST_COUNT]: this device's counters.
static int decode_worker(Device *dev, RangeSource *src, const CallInput &in, int format, uint8_t *const *outs, int *status, double *st) {
    const uint8_t *const *files = in.files;
    const size_t *lens = in.lens;
    const bj_ctx *c = dev->ctx;
    if (dev->check(cudaSetDevice(dev->ordinal)) != BJ_OK) return BJ_ERR_CUDA;
    for (auto &b : dev->slots) if (!b) { b = new (std::nothrow) bj_batch(); if (!b) return BJ_ERR_NOMEM; }
    int first[kSlots] = {}, count[kSlots] = {};
    bool busy[kSlots] = {};
    int rc = BJ_OK;
    // B200JPEG_TRACE=1: one line per sub-batch on stderr - when its kernels ran and its copy-out ended (ms since the
    // first sub-batch was enqueued) - to see whether the copy-out engine is kept busy.  (No event is recorded in front
    // of the upload: on a stream whose last operation was a copy-out it waits for the copy-out engine.)
    static const bool trace = getenv("B200JPEG_TRACE") != nullptr;
    cudaEvent_t ev_base = nullptr;
    double host_t[kSlots][2] = {};
    const double wall0 = wall_ms();
    auto finish = [&](int slot) -> int {
        bj_batch *b = dev->slots[slot];
        const double t0 = wall_ms();
        // sleep until the sub-batch's copy-out is done instead of polling for it (cudaStreamSynchronize spins by
        // default, and a polling host thread takes bandwidth from the copy-out it is waiting for)
        if (b->ev_done) cudaEventSynchronize(b->ev_done);
        int r = batch_sync(b);
        if (trace && r == BJ_OK && ev_base) {
            float k0 = 0, k1 = 0, out = 0;
            cudaEventSynchronize(b->ev[5]);
            cudaEventElapsedTime(&k0, ev_base, b->ev[0]);
            cudaEventElapsedTime(&k1, ev_base, b->ev[4]); cudaEventElapsedTime(&out, ev_base, b->ev[5]);
            fprintf(stderr, "b200jpeg trace: dev %d sub-batch of %4d images (%6.1f MB out, %s)  host prepare %6.2f..%6.2f  kernels %6.2f..%6.2f  copied out %6.2f\n",
                    dev->ordinal, b->n, b->d2h_bytes / 1e6, b->direct_src ? "direct upload" : "staged upload", host_t[slot][0], host_t[slot][1], k0, k1, out);
        }
        if (r == BJ_OK && b->redone)                                   // extra fix-up rounds ran: the early copy-out is stale
            r = batch_download(b, outs + first[slot], dev->streams[slot]);
        st[ST_WAIT_MS] += wall_ms() - t0;
        if (status) for (int i = 0; i < count[slot]; i++) status[first[slot] + i] = r == BJ_OK ? batch_image_status(b, i) : r;
        st[ST_LAUNCH] += b->launches; st[ST_H2D] += (double)(b->files_bytes + b->meta_bytes); st[ST_D2H] += (double)b->d2h_bytes; st[ST_D2H_COPIES] += b->d2h_copies;
        if (r == BJ_OK) { st[ST_MS_UNSTUFF] += b->ms_unstuff; st[ST_MS_SYNC] += b->ms_sync; st[ST_MS_WRITE] += b->ms_write; st[ST_MS_IDCT] += b->ms_idct; }
        busy[slot] = false;
        return r;
    };
    int k = 0, r0 = 0, r1 = 0, nranges = 0;
    while (rc == BJ_OK && src->take(nranges, &r0, &r1)) {
        nranges++;
        int i0 = r0;
        while (rc == BJ_OK && i0 < r1) {
            const int slot = k % kSlots;
            if (busy[slot]) rc = finish(slot);
            if (rc != BJ_OK) break;
            bj_batch *b = dev->slots[slot];
            cudaStream_t s = dev->streams[slot];
            const double t0 = wall_ms();
            rc = batch_assign(b, dev, files + i0, lens + i0, r1 - i0, format, c->sub_batch_out_bytes, in.descs ? in.descs + i0 : nullptr, in.kinds ? in.kinds + i0 : nullptr);
            const int m = rc == BJ_OK ? b->n : 0;
            st[ST_HOST_MS] += wall_ms() - t0;
            host_t[slot][0] = t0 - wall0; host_t[slot][1] = wall_ms() - wall0;
            if (rc == BJ_OK && trace && !ev_base) { cudaEventCreate(&ev_base); cudaEventRecord(ev_base, s); }
            if (rc == BJ_OK) rc = batch_upload(b, s);
            if (rc == BJ_OK) rc = batch_decode(b, s);
            if (rc == BJ_OK) {                                            // enqueue the copy-out behind the kernels, no host wait
                b->synced = true;                                         // (checked for real in finish())
                rc = batch_download_async(b, outs + i0, s);
                b->synced = false;
                if (trace) cudaEventRecord(b->ev[5], s);
                if (!b->ev_done) cudaEventCreateWithFlags(&b->ev_done, cudaEventBlockingSync | cudaEventDisableTiming);
                if (b->ev_done) cudaEventRecord(b->ev_done, s);
            }
            if (rc != BJ_OK) {                                            // nothing (complete) was enqueued for this range: report it, do not wait for it
                cudaStreamSynchronize(s);
                if (status) for (int i = i0; i < r1; i++) status[i] = rc;
                break;
            }
            first[slot] = i0; count[slot] = m; busy[slot] = true;
            st[ST_SUB] += 1; st[ST_DIRECT] += b->direct_src ? 1 : 0;
            i0 += m; k++;
        }
    }
    // drain in submission order
    for (int j = 0; j < kSlots; j++) { const int slot = (k + j) % kSlots; if (busy[slot]) { const int r = finish(slot); if (rc == BJ_OK) rc = r; } }
    // after a failure nobody may be left wondering: the images this device will not get to carry the error, too
    if (rc != BJ_OK && status) while (src->take(nranges, &r0, &r1)) for (int i = r0; i < r1; i++) status[i] = rc;
    if (ev_base) cudaEventDestroy(ev_base);
    return rc;
}

static int decode_batch_now(bj_ctx *c, const CallInput &in, int n, int format, uint8_t *const *outs, int *status) {
    RangeSource src;
    src.lens = in.lens; src.n = n;
    src.budget = c->sub_batch_bytes ? c->sub_batch_bytes : ((size_t)24 << 20);    // compressed bytes per sub-batch
    src.ramp = c->sub_batch_ramp != 0;
    // one host thread per device (the first: the caller's), all pulling sub-batches from the same source
    if (status) for (int i = 0; i < n; i++) status[i] = BJ_ERR_CUDA;                // (overwritten by whoever decodes the image)
    const size_t nd = c->devs.size();
    std::vector<int> rcs(nd, BJ_OK);
    std::vector<double> st(nd * ST_COUNT, 0.0);
    std::vector<std::thread> th;
    for (size_t d = 1; d < nd; d++)
        th.emplace_back([&, d] { rcs[d] = decode_worker(c->devs[d], &src, in, format, outs, status, &st[d * ST_COUNT]); });
    rcs[0] = decode_worker(c->devs[0], &src, in, format, outs, status, &st[0]);
    for (auto &t : th) t.join();
    // the devices work side by side: counts add up, a time is the longest device's
    for (int i = 0; i < ST_COUNT; i++) {
        const bool is_time = i == ST_HOST_MS || i == ST_WAIT_MS || (i >= ST_MS_UNSTUFF && i <= ST_MS_IDCT);
        double v = st[i];
        for (size_t d = 1; d < nd; d++) v = is_time ? std::max(v, st[d * ST_COUNT + i]) : v + st[d * ST_COUNT + i];
        c->stats[i] = v; c->totals[i] += v;
    }
    for (int rc : rcs) if (rc != BJ_OK) return rc;
    return BJ_OK;
}

extern "C" int bj_decode_batch(bj_ctx *c, const uint8_t *const *files, const size_t *lens, int n, int format,
                               uint8_t *const *outs, int *status) {
    if (!c || n < 0 || (n > 0 && (!files || !lens || !outs))) return BJ_ERR_ARG;
    if (format != BJ_OUT_RGB8 && format != BJ_OUT_BMP && format != BJ_OUT_REF_MCUS) return BJ_ERR_ARG;
    if (c->async && c->async->pending()) return BJ_ERR_ARG;                          // jobs of bj_submit are still running on this context
    return decode_batch_now(c, CallInput{files, lens, nullptr, nullptr}, n, format, outs, status);
}

// The same for a caller that already holds the parsed header (the reference's `Header`, src/headers/jpeg.h:146-179) and
// the scan bytes: replaces decode_Huffman_data + the DPU round trip (src/decoder_host.cpp:181, :268-312) while
// read_JPEG stays in front and - with BJ_OUT_REF_MCUS - write_BMP behind.
extern "C" int bj_decode_batch_desc(bj_ctx *c, const bj_image_desc *descs, const uint8_t *const *scans, const size_t *scan_lens,
                                    const int *scan_kinds, int n, int format, uint8_t *const *outs, int *status) {
    if (!c || n < 0 || (n > 0 && (!descs || !scans || !scan_lens || !outs))) return BJ_ERR_ARG;
    if (format != BJ_OUT_RGB8 && format != BJ_OUT_BMP && format != BJ_OUT_REF_MCUS) return BJ_ERR_ARG;
    if (c->async && c->async->pending()) return BJ_ERR_ARG;
    return decode_batch_now(c, CallInput{scans, scan_lens, descs, scan_kinds}, n, format, outs, status);
}

// ------------------------------------------------------------------------------------------------ full path, asynchronous
// bj_submit hands a batch to the context's worker thread and returns; bj_wait blocks until that batch's outputs are
// in host memory.  Jobs run in submission order.  What the reference does with its producer / consumer threads and
// the queue between them (src/decoder_host.cpp:25-38,364-365) a caller gets by submitting batch k+1 (or reading its
// files) while batch k decodes, and writing batch k-1's outputs meanwhile (host/decoder_b200.cpp does exactly that).
struct bj_job {
    const uint8_t *const *files; const size_t *lens; int n, format; uint8_t *const *outs; int *status;
    int rc = BJ_OK;
    bool done = false;
    bj_ctx *ctx = nullptr;
};

void bj::AsyncWorker::run() {
    for (;;) {
        bj_job *j = nullptr;
        {
            std::unique_lock<std::mutex> l(m);
            cv.wait(l, [&] { return stop || !q.empty(); });
            if (q.empty()) return;
            j = q.front();
        }
        const int rc = decode_batch_now(j->ctx, CallInput{j->files, j->lens, nullptr, nullptr}, j->n, j->format, j->outs, j->status);
        {
            std::lock_guard<std::mutex> l(m);
            q.pop_front();
            j->rc = rc; j->done = true;
        }
        done_cv.notify_all();
    }
}

extern "C" int bj_submit(bj_ctx *c, const uint8_t *const *files, const size_t *lens, int n, int format, uint8_t *const *outs, int *status, bj_job **job) {
    if (!c || !job || n < 0 || (n > 0 && (!files || !lens || !outs))) return BJ_ERR_ARG;
    if (format != BJ_OUT_RGB8 && format != BJ_OUT_BMP && format != BJ_OUT_REF_MCUS) return BJ_ERR_ARG;
    *job = nullptr;
    bj_job *j = new (std::nothrow) bj_job{files, lens, n, format, outs, status};
    if (!j) return BJ_ERR_NOMEM;
    j->ctx = c;
    if (!c->async) {
        c->async = new (std::nothrow) AsyncWorker();
        if (!c->async) { delete j; return BJ_ERR_NOMEM; }
        c->async->th = std::thread([w = c->async] { w->run(); });
    }
    { std::lock_guard<std::mutex> l(c->async->m); c->async->q.push_back(j); }
    c->async->cv.notify_one();
    *job = j;
    return BJ_OK;
}

extern "C" int bj_wait(bj_job *j) {
    if (!j || !j->ctx || !j->ctx->async) return BJ_ERR_ARG;
    AsyncWorker *w = j->ctx->async;
    { std::unique_lock<std::mutex> l(w->m); w->done_cv.wait(l, [&] { return j->done; }); }
    const int rc = j->rc;
    delete j;
    return rc;
}
