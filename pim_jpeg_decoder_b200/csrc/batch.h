// Host orchestration of the full path: a batch of JPEG files -> kernels K0..K3 -> pixels.
// Replaces, per image, the producer half of the reference's pipeline (read_JPEG's scan copy + decode_Huffman_data,
// src/decoder_host.cpp:119-181) and its consumer half (pim.copy / pim.exec / pim.copy, :268-312) with one
// asynchronous sequence of kernel launches on a CUDA stream.  Nothing here decodes on the CPU, and the host never
// touches the entropy-coded bytes: it reads the file HEADERS (parse.h, a few hundred bytes per file), builds one small
// record per image and the lookup tables, and hands the file bytes to the GPU - straight from the caller's memory when
// that is page-locked, through a pinned staging copy otherwise.  Where a scan ends, what survives un-stuffing, and
// every per-CTA table are worked out on the device (kernels_huff.cuh: k_unstuff / k_expand_maps).
#pragma once
#include <map>
#include <string>
#include <vector>

#include "bj_host.h"
#include "kernels_huff.cuh"
#include "kernels_idct.cuh"
#include "parse.h"

namespace bj {

struct PinBuf {                       // grow-only pinned host allocation
    void *p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return BJ_OK;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        const size_t want = bytes + bytes / 8 + 4096;
        if (cudaHostAlloc(&p, want, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); p = nullptr; return BJ_ERR_NOMEM; }
        cap = want;
        return BJ_OK;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

constexpr int kSmemLutMax = 3 * (kLutCapDC + kLutCapAC) * 4;
constexpr int kSmemHuffWriteMax = kSmemHuffStage + kSmemLutMax;
constexpr int kSmemHuffSyncMax = kSmemLutMax;
constexpr int kSyncCarveout = 72;      // % of 228 KB: 164 KB of shared memory for 5 CTAs, the rest is L1 (kernels_huff.cuh: kSyncCtas)

inline int batch_kernels_init(Device *dev) {
    if (dev->check(cudaFuncSetAttribute(k_huff_write, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemHuffWriteMax)) != BJ_OK) return BJ_ERR_CUDA;
    if (dev->check(cudaFuncSetAttribute(k_huff_sync, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemHuffSyncMax)) != BJ_OK) return BJ_ERR_CUDA;
    if (dev->check(cudaFuncSetAttribute(k_huff_sync, cudaFuncAttributePreferredSharedMemoryCarveout, kSyncCarveout)) != BJ_OK) return BJ_ERR_CUDA;
    return BJ_OK;
}

}  // namespace bj

struct bj_batch {
    bj::Device *dev = nullptr;
    int n = 0, format = 0;
    int rounds = 3;

    std::vector<bj_image_desc> desc;
    std::vector<int> parse_status;
    std::vector<size_t> out_off, out_size;
    std::vector<uint64_t> file_off;
    std::vector<uint32_t> du_base, ndu;
    std::vector<bj::HuffImg> himg;       // per-image records (kept here between calls: no reallocation in steady state)
    std::vector<bj::ImgDev> idev;

    // host staging (pinned): file bytes; descriptor blob; results
    bj::PinBuf h_files, h_meta, h_res;
    size_t files_bytes = 0, meta_bytes = 0;
    const uint8_t *direct_src = nullptr;   // set: the files are uploaded straight from the caller's (pinned) memory, files_bytes from here
    // offsets inside the descriptor blob (host -> device)
    size_t o_himg = 0, o_idev = 0, o_qtab = 0, o_lutdc = 0, o_lutac = 0, o_lutacs = 0;
    // offsets inside the map buffer (written on the device by k_expand_maps)
    size_t m_tiles = 0, m_blk = 0, m_wblk = 0, m_utile = 0, m_dcc = 0, maps_bytes = 0;
    uint32_t idct_smem = 0;             // dynamic shared memory of k_idct_color: sized for the widest pixel tile of this batch
    uint32_t n_wblk = 0;                // CTAs of the Huffman write pass
    size_t n_slice_slots = 0;
    uint32_t n_idct_tiles = 0, n_blk = 0, n_utile = 0, n_dcc = 0, n_seg_entries = 0, n_sub_slots = 0, lut_smem = 0;
    size_t clean_words = 0, coef_units = 0, out_bytes = 0;
    uint64_t pixels = 0, scan_bytes_max = 0;
    uint32_t nseg_max = 0;              // most restart segments of one image
    uint32_t ref_blocks_max = 0;        // BJ_OUT_REF_MCUS: blocks of the largest image (grid of the padding kernel)

    // device
    bj::DevBuf d_files, d_meta, d_maps, d_look, d_clean, d_seg, d_subseg, d_stin, d_stout, d_tot, d_pre, d_slice, d_quarter, d_blkagg, d_state, d_flags, d_coef, d_dc, d_dcagg, d_out;
    cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // start, un-stuffed, synchronised, written, pixels, copied out
    cudaEvent_t ev_done = nullptr;       // one-call path: recorded behind the copy-out, created for a sleeping wait
    cudaStream_t last_stream = nullptr;
    bool uploaded = false, decoded = false, synced = false;
    bool multi_blk = false;              // some image's sub-sequences span more than one CTA of the synchronisation pass
    bool redone = false;                 // batch_sync had to run extra fix-up rounds: everything after them was computed again
    uint32_t launches = 0, sync_rounds = 0;
    float ms_entropy = 0.f, ms_idct = 0.f, ms_unstuff = 0.f, ms_sync = 0.f, ms_write = 0.f;
    uint64_t d2h_bytes = 0;
    uint32_t d2h_copies = 0;

    bj::HuffImgState *h_state() { return reinterpret_cast<bj::HuffImgState *>(h_res.p); }
    uint32_t *h_flags() { return reinterpret_cast<uint32_t *>(reinterpret_cast<uint8_t *>(h_res.p) + bj::align_up((size_t)n * sizeof(bj::HuffImgState), 64)); }
    template <class T> T *dmeta(size_t off) { return reinterpret_cast<T *>(reinterpret_cast<uint8_t *>(d_meta.p) + off); }
    template <class T> T *hmeta(size_t off) { return reinterpret_cast<T *>(reinterpret_cast<uint8_t *>(h_meta.p) + off); }
    template <class T> T *dmap(size_t off) { return reinterpret_cast<T *>(reinterpret_cast<uint8_t *>(d_maps.p) + off); }

    void release() {
        for (bj::DevBuf *b : {&d_files, &d_meta, &d_maps, &d_look, &d_clean, &d_seg, &d_subseg, &d_stin, &d_stout, &d_tot, &d_pre, &d_slice, &d_quarter, &d_blkagg, &d_state, &d_flags, &d_coef, &d_dc, &d_dcagg, &d_out}) b->release();
        h_files.release(); h_meta.release(); h_res.release();
        for (auto &e : ev) if (e) { cudaEventDestroy(e); e = nullptr; }
        if (ev_done) { cudaEventDestroy(ev_done); ev_done = nullptr; }
    }
};

namespace bj {

constexpr int kMaxRounds = 64;

// (Re)fill a batch object from a list of files: parse the headers, lay out, (stage).  Host work only (plus buffer growth).
//   out_cap   the batch takes images from the front of the list until their decoded bytes pass this (at least one):
//             b->n tells how many.  A few hostile headers (a 1 KB file that declares 65535 x 65535) cannot make a
//             sub-batch of the one-call path arbitrarily large, and an image above ctx->max_image_pixels is refused
//             on its own (BJ_ERR_UNSUPPORTED) like the reference's "Too high resolution" (src/decoder_host.cpp:146-149).
//   descs     (bj_decode_batch_desc) the images come as descriptor + scan bytes instead of files: files[i] / lens[i] are
//             then the scan itself - raw (stuffed, with RSTn; kinds[i] = BJ_SCAN_RAW) or the reference's
//             Header::huffman_data (un-stuffed, markers removed; BJ_SCAN_UNSTUFFED, only without a restart interval:
//             read_JPEG throws the RSTn positions away, SURVEY 0.8) - and nothing is parsed.
inline int batch_assign(bj_batch *b, Device *dev, const uint8_t *const *files, const size_t *lens, int n, int format, size_t out_cap = ~(size_t)0,
                        const bj_image_desc *descs = nullptr, const int *kinds = nullptr) {
    if (format != BJ_OUT_RGB8 && format != BJ_OUT_BMP && format != BJ_OUT_REF_MCUS) return BJ_ERR_ARG;
    const bj_ctx *c = dev->ctx;
    b->dev = dev; b->n = n; b->format = format;
    b->uploaded = b->decoded = b->synced = false;
    b->desc.resize(n); b->parse_status.assign(n, BJ_OK);
    if (dev->check(cudaSetDevice(dev->ordinal)) != BJ_OK) return BJ_ERR_CUDA;
    for (auto &e : b->ev) if (!e && dev->check(cudaEventCreate(&e)) != BJ_OK) return BJ_ERR_CUDA;

    // ---- headers (per image, independent: worker pool).  Nothing behind the SOS header is read.
    std::vector<Geometry> geo(n);
    dev->host_pool.parallel_for(n, 64, [&](int i0, int i1) {
        for (int i = i0; i < i1; i++) {
            bj_image_desc &d = b->desc[i];
            int rc;
            if (descs) {                                                  // a caller-made descriptor: checked before it sizes anything
                d = descs[i];
                d.scan_off = 0; d.scan_len = lens[i];
                rc = !files[i] ? BJ_ERR_ARG : (!desc_is_sane(d) ? BJ_ERR_INVALID_JPEG : BJ_OK);
                for (int j = 0; rc == BJ_OK && j < d.ncomp; j++)
                    if (!d.qt_set[d.qt_id[j]] || !d.dc_set[d.dc_id[j]] || !d.ac_set[d.ac_id[j]]) rc = BJ_ERR_INVALID_JPEG;
                if (rc == BJ_OK && (d.frame_type != 0xC0 || d.scan_ncomp != d.ncomp)) rc = BJ_ERR_UNSUPPORTED;
                if (rc == BJ_OK && kinds && kinds[i] == BJ_SCAN_UNSTUFFED && d.restart_interval != 0) rc = BJ_ERR_UNSUPPORTED;
            } else
                rc = (files[i] && lens[i]) ? parse_header(files[i], lens[i], &d, /*walk_scan=*/false) : BJ_ERR_INVALID_JPEG;
            if (rc == BJ_OK && d.scan_len >= ((size_t)1 << 31)) rc = BJ_ERR_UNSUPPORTED;   // byte counts travel in 31 bits
            if (rc == BJ_OK && (size_t)d.width * d.height > c->max_image_pixels) rc = BJ_ERR_UNSUPPORTED;
            if (rc == BJ_OK) geo[i] = geometry_of(d);
            b->parse_status[i] = rc;
        }
    });
    // ---- how many of the candidates this batch takes
    if (out_cap != ~(size_t)0) {
        size_t acc = 0;
        int m = 0;
        while (m < n) {
            const size_t sz = b->parse_status[m] == BJ_OK ? align_up(output_bytes(b->desc[m], format, c->ref_m), 16) : 0;
            if (m > 0 && acc + sz > out_cap) break;
            acc += sz; m++;
        }
        n = m; b->n = n;
        b->desc.resize(n); b->parse_status.resize(n);
    }
    b->out_off.assign(n, 0); b->out_size.assign(n, 0); b->file_off.assign(n, 0);
    b->du_base.assign(n, 0); b->ndu.assign(n, 0);
    b->himg.resize(n); b->idev.resize(n);

    // ---- where the file bytes are uploaded from.  If the span from the first to the last file lies inside page-locked
    // memory this library knows about (bj_host_alloc / bj_host_register), or the caller says so (option "packed_inputs"
    // = 1), and the files lie close together, the span goes up as it is, straight from the caller's memory: nothing is
    // copied on the host.  Otherwise the files are packed into this batch's pinned staging buffer (worker pool).
    b->direct_src = nullptr;
    uint64_t span_lo = ~0ull, span_hi = 0, span_sum = 0;
    if (c->packed_inputs >= 0 && !descs) {            // (scans handed over one by one are always staged: what precedes them in memory is not ours)
        for (int i = 0; i < n; i++) {
            if (b->parse_status[i] != BJ_OK) continue;
            const uint64_t a = (uint64_t)(uintptr_t)files[i];
            span_lo = std::min(span_lo, a); span_hi = std::max(span_hi, a + lens[i]); span_sum += lens[i];
        }
        // (the upload starts at the 16-byte boundary at or below the first file: that, too, must be page-locked memory)
        if (span_hi > span_lo && span_hi - span_lo <= 2 * span_sum + (1u << 16) &&
            (c->packed_inputs == 1 || pinned_ranges().contains((uintptr_t)(span_lo & ~(uint64_t)15), (uintptr_t)span_hi))) {
            span_lo &= ~(uint64_t)15;
            b->direct_src = reinterpret_cast<const uint8_t *>((uintptr_t)span_lo);
        }
    }

    // ---- sub-sequence length and slices, per image.
    // Explicit (options "subseq_bits", "slices"): the same for every image.  Automatic: nominally 4096 bits - a stream
    // synchronises within about a thousand, so nearly every guess settles inside its own sub-sequence - but shorter
    // when the whole batch would not fill the GPU with threads, and then adjusted per image so that its sub-sequences
    // fill whole CTAs (a nearly empty second CTA costs a cross-CTA fix-up round); the write pass works on whole
    // sub-sequences (1 slice).  An image with restart markers gets sub-sequences that hold a typical restart segment
    // in one piece - segment heads need no speculation at all - and the write pass cuts them into 4 slices (8 when
    // the batch is small), whose entry states the synchronisation pass records.
    const uint32_t fixed_sub = c->subseq_bits ? (uint32_t)c->subseq_bits / 8u : 0u;
    uint32_t fixed_rl = c->slices == 2 ? 1u : c->slices == 4 ? 2u : c->slices == 8 ? 3u : 0u;
    if (fixed_sub) while (fixed_rl && fixed_sub % (1u << fixed_rl)) fixed_rl--;
    constexpr uint64_t kMinSubBytes = 128;              // shortest sub-sequence the automatic layout picks (small batches)
    uint32_t nominal_sub = 512;
    uint64_t total_scan = 0;
    for (int i = 0; i < n; i++) if (b->parse_status[i] == BJ_OK) total_scan += b->desc[i].scan_len;
    if (!fixed_sub) nominal_sub = (uint32_t)std::min<uint64_t>(512u, std::max<uint64_t>(kMinSubBytes, total_scan / ((uint64_t)dev->sm_count * 3072u)));
    auto round_sub = [&](uint32_t len, uint32_t rl) { const uint32_t q = 4u << rl; return (std::max(len, 64u) + q - 1u) / q * q; };
    auto sub_layout_of = [&](uint32_t raw_len, uint32_t nseg, uint32_t *rl) -> uint32_t {
        *rl = c->slices ? fixed_rl : 0u;
        if (fixed_sub) return fixed_sub;
        if (nseg > 1) {
            const uint32_t avg = raw_len / nseg;
            if (avg <= 1024) {
                if (!c->slices) *rl = total_scan < ((uint64_t)16 << 20) ? 3u : 2u;
                return round_sub(std::max(2 * avg, nominal_sub), *rl);
            }
        }
        const uint32_t per_cta = nominal_sub * kHuffThreads;
        const uint32_t m = std::max(1u, (raw_len + per_cta / 2) / per_cta);                  // CTAs for this image
        const uint32_t slots = m * kHuffThreads;                                            // ceil(raw_len / len) + nseg must fit
        if (slots <= nseg + 1) return round_sub(nominal_sub, *rl);
        return round_sub((raw_len + slots - nseg - 1) / (slots - nseg), *rl);
    };

    // ---- layout (serial: prefix sums over the batch, O(images))
    std::vector<HuffImg> &himg = b->himg;
    std::vector<ImgDev> &idev = b->idev;
    std::vector<QTab> qtabs;
    size_t slice_slots = 0;
    std::vector<uint32_t> luts_dc, luts_ac, luts_acs;     // acs: the synchronisation pass' grouped AC tables
    std::map<std::string, int> lut_index[2];
    std::vector<uint16_t> lut_n4[2];                // per pooled table: used size in 16-byte chunks
    size_t fbytes = 0, clean_words = 0, out_bytes = 0, coef_units = 0;
    uint32_t seg_entries = 0, nblk = 0, n_utile = 0, n_wblk = 0, n_dcc = 0, n_tiles = 0;
    int prev = -1;                                  // last valid image: its table slots are reused when the tables match
    b->pixels = 0; b->scan_bytes_max = 0; b->ref_blocks_max = 0; b->nseg_max = 0; b->lut_smem = 0; b->multi_blk = false;
    uint32_t rgb_max = 0;
    auto same_tables = [](const bj_image_desc &a, const bj_image_desc &q) {
        if (a.ncomp != q.ncomp || memcmp(a.dc_id, q.dc_id, 3) || memcmp(a.ac_id, q.ac_id, 3)) return false;
        for (int j = 0; j < a.ncomp; j++) {
            const int di = a.dc_id[j], ai = a.ac_id[j];
            if (memcmp(a.dc_offsets[di], q.dc_offsets[di], 17) || memcmp(a.dc_symbols[di], q.dc_symbols[di], a.dc_offsets[di][16] > 162 ? 162 : a.dc_offsets[di][16]) ||
                memcmp(a.ac_offsets[ai], q.ac_offsets[ai], 17) || memcmp(a.ac_symbols[ai], q.ac_symbols[ai], a.ac_offsets[ai][16] > 162 ? 162 : a.ac_offsets[ai][16])) return false;
        }
        return true;
    };
    for (int i = 0; i < n; i++) {
        bj_image_desc &d = b->desc[i];
        HuffImg &hi = himg[i];
        memset(&hi, 0, sizeof(hi));
        memset(&idev[i], 0, sizeof(ImgDev));
        int rc = b->parse_status[i];
        const Geometry &g = geo[i];
        if (rc == BJ_OK) {
            if (prev >= 0 && same_tables(d, b->desc[prev])) {
                const HuffImg &hp = himg[prev];
                hi.ndc = hp.ndc; hi.nac = hp.nac;
                memcpy(hi.dc_lut, hp.dc_lut, sizeof(hi.dc_lut)); memcpy(hi.ac_lut, hp.ac_lut, sizeof(hi.ac_lut));
                memcpy(hi.dc_slot, hp.dc_slot, sizeof(hi.dc_slot)); memcpy(hi.ac_slot, hp.ac_slot, sizeof(hi.ac_slot));
                memcpy(hi.dc_n4, hp.dc_n4, sizeof(hi.dc_n4)); memcpy(hi.ac_n4, hp.ac_n4, sizeof(hi.ac_n4));
            } else
            // tables -> pools (deduplicated across the batch); per image the distinct ones become staged slots
            for (int ac = 0; ac < 2 && rc == BJ_OK; ac++) {
                std::vector<uint32_t> &pool = ac ? luts_ac : luts_dc;
                const size_t cap = ac ? kLutCapAC : kLutCapDC;
                int slots[3], nslot = 0;
                for (int j = 0; j < 3 && rc == BJ_OK; j++) {
                    const int jj = j < d.ncomp ? j : 0;
                    const uint8_t *off = ac ? d.ac_offsets[d.ac_id[jj]] : d.dc_offsets[d.dc_id[jj]];
                    const uint8_t *sym = ac ? d.ac_symbols[d.ac_id[jj]] : d.dc_symbols[d.dc_id[jj]];
                    std::string key((const char *)off, 17);
                    key.append((const char *)sym, off[16] > 162 ? 162 : off[16]);
                    auto it = lut_index[ac].find(key);
                    int idx;
                    if (it == lut_index[ac].end()) {
                        idx = (int)(pool.size() / cap);
                        pool.resize(pool.size() + cap);
                        const int used = build_lut(off, sym, ac != 0, &pool[(size_t)idx * cap]);
                        if (used < 0) rc = BJ_ERR_UNSUPPORTED;
                        if (ac) {
                            luts_acs.resize(pool.size());
                            build_lut_sync(&pool[(size_t)idx * cap], std::max(used, 0), &luts_acs[(size_t)idx * cap]);
                        }
                        lut_n4[ac].push_back((uint16_t)((std::max(used, 0) + 3) / 4));
                        lut_index[ac][key] = idx;
                        if (idx > 65535) rc = BJ_ERR_UNSUPPORTED;
                    } else idx = it->second;
                    int s = 0;
                    while (s < nslot && slots[s] != idx) s++;
                    if (s == nslot) slots[nslot++] = idx;
                    (ac ? hi.ac_slot : hi.dc_slot)[j] = (uint8_t)s;
                }
                (ac ? hi.nac : hi.ndc) = (uint8_t)nslot;
                for (int s = 0; s < nslot; s++) {
                    (ac ? hi.ac_lut : hi.dc_lut)[s] = (uint16_t)slots[s];
                    (ac ? hi.ac_n4 : hi.dc_n4)[s] = lut_n4[ac][slots[s]];
                }
            }
            uint32_t smem = 0;
            for (int s = 0; s < hi.ndc; s++) smem += hi.dc_n4[s] * 16u;
            for (int s = 0; s < hi.nac; s++) smem += hi.ac_n4[s] * 16u;
            if (smem > b->lut_smem) b->lut_smem = smem;
        }
        b->parse_status[i] = rc;
        b->file_off[i] = b->direct_src ? (uint64_t)(uintptr_t)files[i] - span_lo : fbytes;
        hi.seg_base = seg_entries;
        hi.blk_base = nblk;
        hi.sub_base = nblk * kHuffThreads;
        hi.tile_base = n_utile;
        hi.clean_word0 = (uint32_t)clean_words;
        hi.du_base = (uint32_t)coef_units;
        hi.dcc_base = n_dcc;
        if (rc != BJ_OK) { seg_entries += 2; hi.ndc = hi.nac = 0; continue; }
        fbytes += align_up(lens[i] + 16, 16);
        hi.valid = 1;
        hi.flags = descs ? (uint8_t)((kinds && kinds[i] == BJ_SCAN_UNSTUFFED) ? (kImgClean | kImgExact) : kImgExact) : (uint8_t)0;
        hi.raw_off = b->file_off[i] + d.scan_off;
        hi.raw_len = (uint32_t)d.scan_len;                                   // upper bound: up to the end of the file
        hi.ntile = std::max<uint32_t>(1u, (uint32_t)(((hi.raw_off & 15u) + hi.raw_len + kUnstuffTile - 1) / kUnstuffTile));
        n_utile += hi.ntile;
        hi.nmcu = g.nmcu; hi.ri = d.restart_interval;
        hi.nseg = hi.ri ? (g.nmcu + hi.ri - 1) / hi.ri : 1u;
        b->nseg_max = std::max(b->nseg_max, hi.nseg);
        hi.bpm = (uint8_t)g.bpm; hi.ny = (uint8_t)(d.hs * d.vs); hi.ncomp = d.ncomp;
        hi.ndu = g.ndu;
        {
            uint32_t rl = 0;
            hi.sub_bytes = sub_layout_of(hi.raw_len, hi.nseg, &rl);
            hi.slices_log2 = (uint8_t)rl;
        }
        const uint32_t sub_cap = (uint32_t)((hi.raw_len + hi.sub_bytes - 1) / hi.sub_bytes) + hi.nseg;
        hi.nblk = (sub_cap + kHuffThreads - 1) / kHuffThreads;
        nblk += hi.nblk;
        if (hi.nblk > 1) b->multi_blk = true;
        hi.wblk_base = n_wblk;
        n_wblk += hi.nblk << hi.slices_log2;
        hi.slice_base = (uint32_t)slice_slots;
        slice_slots += ((size_t)hi.nblk * kHuffThreads) << hi.slices_log2;
        hi.ndcc = (g.nmcu + kDcThreads - 1) / kDcThreads;
        n_dcc += hi.ndcc;
        seg_entries += hi.nseg + 1;
        clean_words += hi.raw_len / 4 + 4;
        b->du_base[i] = (uint32_t)coef_units; b->ndu[i] = g.ndu;
        coef_units += g.ndu;
        b->out_size[i] = output_bytes(d, format, c->ref_m);
        b->out_off[i] = out_bytes;
        fill_imgdev(d, g, format, hi.du_base, out_bytes, &idev[i]);
        if (format == BJ_OUT_REF_MCUS) { idev[i].ref_blocks = ref_mcus_chunks(d, c->ref_m) * (uint32_t)(c->ref_m / 4); b->ref_blocks_max = std::max(b->ref_blocks_max, idev[i].ref_blocks); }
        idev[i].dc_sep = 1;
        idev[i].tile0 = n_tiles;
        n_tiles += idct_tile_count(g);
        if (prev >= 0 && same_qtab(d, b->desc[prev])) idev[i].qslot = idev[prev].qslot;
        else { idev[i].qslot = (uint32_t)qtabs.size(); qtabs.emplace_back(); fill_qtab(d, &qtabs.back()); }
        prev = i;
        out_bytes += align_up(b->out_size[i], 16);
        rgb_max = std::max<uint32_t>(rgb_max, std::min<uint32_t>(g.tile_mcus, g.nmx) * d.hs * 8u * d.vs * 8u * 3u);
        b->pixels += (uint64_t)d.width * d.height;
        b->scan_bytes_max += d.scan_len;
        if (coef_units > 0xFFFFFFF0ull || clean_words > 0xFFFFFFF0ull || slice_slots > 0xFFFFFFF0ull) return BJ_ERR_ARG;   // split the batch
    }
    b->idct_smem = kSmemDu + kSmemQ + kRgbFront + std::min<uint32_t>(rgb_max, kRgbMax) + 64;
    b->files_bytes = b->direct_src ? (size_t)(span_hi - span_lo) : fbytes + 64; b->clean_words = clean_words + 96; b->coef_units = coef_units; b->out_bytes = out_bytes;   // (96 words of slack: a damaged unit is read to its end, up to 63 symbols of 27 bits past the data)
    b->n_wblk = n_wblk; b->n_slice_slots = slice_slots;
    b->n_idct_tiles = n_tiles; b->n_blk = nblk; b->n_utile = n_utile;
    b->n_dcc = n_dcc; b->n_seg_entries = seg_entries; b->n_sub_slots = nblk * kHuffThreads;

    // ---- descriptor blob (host -> device): one record per image, the table pools
    size_t o = 0;
    b->o_himg = o;  o = align_up(o + (size_t)n * sizeof(HuffImg), 256);
    b->o_idev = o;  o = align_up(o + (size_t)n * sizeof(ImgDev), 256);
    b->o_qtab = o;  o = align_up(o + qtabs.size() * sizeof(QTab), 256);
    b->o_lutdc = o; o = align_up(o + luts_dc.size() * 4, 256);
    b->o_lutac = o; o = align_up(o + luts_ac.size() * 4, 256);
    b->o_lutacs = o; o = align_up(o + luts_acs.size() * 4, 256);
    b->meta_bytes = o;
    // ---- map buffer (device only: k_expand_maps)
    o = 0;
    b->m_tiles = o; o = align_up(o + (size_t)n_tiles * sizeof(TileDev), 256);
    b->m_blk = o;   o = align_up(o + (size_t)nblk * 4, 256);
    b->m_wblk = o;  o = align_up(o + (size_t)n_wblk * 4, 256);
    b->m_utile = o; o = align_up(o + (size_t)n_utile * 4, 256);
    b->m_dcc = o;   o = align_up(o + (size_t)n_dcc * 4, 256);
    b->maps_bytes = o;
    if (b->h_meta.reserve(b->meta_bytes) || (!b->direct_src && b->h_files.reserve(b->files_bytes)) ||
        b->h_res.reserve(align_up((size_t)n * sizeof(HuffImgState), 64) + kMaxRounds * 4 + 64)) return BJ_ERR_NOMEM;
    if (n) { memcpy(b->hmeta<HuffImg>(b->o_himg), himg.data(), (size_t)n * sizeof(HuffImg)); memcpy(b->hmeta<ImgDev>(b->o_idev), idev.data(), (size_t)n * sizeof(ImgDev)); }
    if (!qtabs.empty()) memcpy(b->hmeta<QTab>(b->o_qtab), qtabs.data(), qtabs.size() * sizeof(QTab));
    if (!luts_dc.empty()) memcpy(b->hmeta<uint32_t>(b->o_lutdc), luts_dc.data(), luts_dc.size() * 4);
    if (!luts_ac.empty()) memcpy(b->hmeta<uint32_t>(b->o_lutac), luts_ac.data(), luts_ac.size() * 4);
    if (!luts_acs.empty()) memcpy(b->hmeta<uint32_t>(b->o_lutacs), luts_acs.data(), luts_acs.size() * 4);
    // ---- stage the file bytes (only when they cannot go up from where they are; per image, independent: worker pool)
    if (!b->direct_src) {
        uint8_t *hf = reinterpret_cast<uint8_t *>(b->h_files.p);
        dev->host_pool.parallel_for(n, 16, [&](int i0, int i1) {
            for (int i = i0; i < i1; i++) {
                if (b->parse_status[i] != BJ_OK) continue;
                memcpy(hf + b->file_off[i], files[i], lens[i]);
                memset(hf + b->file_off[i] + lens[i], 0, align_up(lens[i] + 16, 16) - lens[i]);
            }
        });
    }
    // ---- device buffers
    if (b->d_files.reserve(b->files_bytes + 4096) || b->d_meta.reserve(b->meta_bytes) || b->d_maps.reserve(b->maps_bytes + 16) ||
        b->d_look.reserve((size_t)n_utile * 8 + (size_t)n * 4 + 16) || b->d_clean.reserve(b->clean_words * 4) ||
        b->d_seg.reserve((size_t)(seg_entries + 2) * 4 * 2) || b->d_subseg.reserve((size_t)b->n_sub_slots * 4 + 16) ||
        b->d_stin.reserve((size_t)b->n_sub_slots * 8 + 16) || b->d_stout.reserve((size_t)b->n_sub_slots * 8 + 16) ||
        b->d_tot.reserve((size_t)b->n_sub_slots * 4 + 16) || b->d_pre.reserve((size_t)b->n_sub_slots * 8 + 16) ||
        b->d_slice.reserve(b->n_slice_slots * 16 + 16) || b->d_quarter.reserve((size_t)b->n_sub_slots * 8 * 16 + 16) ||
        b->d_dc.reserve(coef_units * 2 + 64) || b->d_dcagg.reserve((size_t)b->n_dcc * sizeof(DcAgg) + 16) ||
        b->d_blkagg.reserve((size_t)nblk * sizeof(BlkAgg) + 16) ||
        b->d_state.reserve((size_t)n * sizeof(HuffImgState) + 16) || b->d_flags.reserve(kMaxRounds * 4 + 16) ||
        b->d_coef.reserve(coef_units * 128 + 16) || b->d_out.reserve(out_bytes + 64)) return BJ_ERR_NOMEM;
    return BJ_OK;
}

// H2D of the file bytes and the per-image records; the per-CTA maps are then expanded on the device.
inline int batch_upload(bj_batch *b, cudaStream_t s) {
    Device *dev = b->dev;
    if (dev->check(cudaSetDevice(dev->ordinal)) != BJ_OK) return BJ_ERR_CUDA;
    b->last_stream = s;
    if (b->n == 0) { b->uploaded = true; return BJ_OK; }
    int rc = dev->check(cudaMemcpyAsync(b->d_files.p, b->direct_src ? (const void *)b->direct_src : b->h_files.p, b->files_bytes, cudaMemcpyHostToDevice, s));
    if (rc == BJ_OK) rc = dev->check(cudaMemcpyAsync(b->d_meta.p, b->h_meta.p, b->meta_bytes, cudaMemcpyHostToDevice, s));
    if (rc == BJ_OK) {
        k_expand_maps<<<b->n, 256, 0, s>>>(b->dmeta<HuffImg>(b->o_himg), b->dmeta<ImgDev>(b->o_idev), b->dmap<uint32_t>(b->m_utile), b->dmap<uint32_t>(b->m_blk),
                                          b->dmap<uint32_t>(b->m_wblk), b->dmap<uint32_t>(b->m_dcc), b->dmap<TileDev>(b->m_tiles));
        rc = dev->check(cudaGetLastError());
    }
    b->uploaded = rc == BJ_OK;
    return rc;
}

// Launch sync rounds [r0, r1) and everything after them.
inline int batch_launch(bj_batch *b, cudaStream_t s, int r0, int r1) {
    const bj_ctx *c = b->dev->ctx;
    const HuffImg *himg = b->dmeta<HuffImg>(b->o_himg);
    const ImgDev *idev = b->dmeta<ImgDev>(b->o_idev);
    const QTab *qtabs = b->dmeta<QTab>(b->o_qtab);
    const TileDev *tiles = b->dmap<TileDev>(b->m_tiles);
    const uint32_t *blk_img = b->dmap<uint32_t>(b->m_blk), *wblk_img = b->dmap<uint32_t>(b->m_wblk);
    const uint32_t *utile_img = b->dmap<uint32_t>(b->m_utile);
    const uint32_t *dcc_img = b->dmap<uint32_t>(b->m_dcc);
    const uint32_t *luts_dc = b->dmeta<uint32_t>(b->o_lutdc), *luts_ac = b->dmeta<uint32_t>(b->o_lutac), *luts_acs = b->dmeta<uint32_t>(b->o_lutacs);
    uint4 *slices = (uint4 *)b->d_slice.p;
    int16_t *dcp = (int16_t *)b->d_dc.p;
    DcAgg *dcagg = (DcAgg *)b->d_dcagg.p;
    HuffImgState *st = (HuffImgState *)b->d_state.p;
    uint32_t *seg_off = (uint32_t *)b->d_seg.p, *seg_sub0 = seg_off + b->n_seg_entries + 2;
    uint32_t *sub_seg = (uint32_t *)b->d_subseg.p, *flags = (uint32_t *)b->d_flags.p;
    uint32_t *clean = (uint32_t *)b->d_clean.p;
    uint2 *st_in = (uint2 *)b->d_stin.p, *st_out = (uint2 *)b->d_stout.p;
    uint32_t *tot = (uint32_t *)b->d_tot.p;
    uint2 *pre = (uint2 *)b->d_pre.p;
    BlkAgg *agg = (BlkAgg *)b->d_blkagg.p;
    const int n = b->n;
    const size_t lut_smem = b->lut_smem;
    if (r0 == 0) {
        cudaEventRecord(b->ev[0], s);
        if (c->debug_poison) {                                                        // tests: whatever is read later must have been written by this decode
            cudaMemsetAsync(b->d_coef.p, 0xA5, b->coef_units * 128, s);
            cudaMemsetAsync(b->d_dc.p, 0xA5, b->coef_units * 2, s);
            cudaMemsetAsync(b->d_out.p, 0xA5, b->out_bytes, s);
            cudaMemsetAsync(b->d_clean.p, 0xA5, b->clean_words * 4, s);
        }
        cudaMemsetAsync(flags, 0, kMaxRounds * 4, s);
        cudaMemsetAsync(st, 0, (size_t)n * sizeof(HuffImgState), s);                  // (rejected files keep an all-zero state)
        b->launches = 0;
        if (b->n_utile) {
            uint64_t *look = (uint64_t *)b->d_look.p;                                 // look-back words of the tiles + the images' ticket counters behind them
            cudaMemsetAsync(look, 0, (size_t)b->n_utile * 8 + (size_t)n * 4, s);
            k_unstuff<<<b->n_utile, kUnstuffThreads, 0, s>>>((const uint8_t *)b->d_files.p, himg, utile_img, look, (uint32_t *)(look + b->n_utile), st, clean, seg_off);
            b->launches++;
        }
        if (b->nseg_max > 256) k_subseq_table<1024><<<n, 1024, 0, s>>>(himg, st, seg_off, seg_sub0, sub_seg);
        else k_subseq_table<256><<<n, 256, 0, s>>>(himg, st, seg_off, seg_sub0, sub_seg);
        b->launches++;
        b->sync_rounds = 0;
        cudaEventRecord(b->ev[1], s);
    } else {
        // the write pass ran on entry states that had not settled: what it made of the images' states does not count
        k_reset_state<<<(n + 255) / 256, 256, 0, s>>>(st, n);
        b->launches++;
    }
    if (b->n_blk) {
        for (int r = r0; r < r1; r++) {
            k_huff_sync<<<b->n_blk, kHuffThreads, lut_smem, s>>>(himg, st, blk_img, clean, seg_off, seg_sub0, sub_seg, luts_dc, luts_acs, st_in, st_out, tot, pre, slices, (uint4 *)b->d_quarter.p, agg, flags, r);
            b->launches++; b->sync_rounds++;
        }
        cudaEventRecord(b->ev[2], s);
        k_huff_write<<<b->n_wblk, kHuffThreads, kSmemHuffStage + lut_smem, s>>>(himg, st, wblk_img, clean, seg_off, seg_sub0, sub_seg, luts_dc, luts_ac, slices, pre, agg, (int16_t *)b->d_coef.p, dcp);
        b->launches++;
    }
    {
        const int gx = n >= 592 ? 1 : (592 + n - 1) / n;
        k_zero_tail<<<dim3(n, gx > 64 ? 64 : gx), 256, 0, s>>>(himg, st, (int16_t *)b->d_coef.p);
        b->launches++;
    }
    if (b->n_dcc) {
        k_dc_predict<0><<<b->n_dcc, kDcThreads, 0, s>>>(himg, st, dcc_img, dcp, dcagg);
        k_dc_predict<1><<<b->n_dcc, kDcThreads, 0, s>>>(himg, st, dcc_img, dcp, dcagg);
        b->launches += 2;
    }
    if (!b->n_blk) cudaEventRecord(b->ev[2], s);
    cudaEventRecord(b->ev[3], s);
    if (b->n_idct_tiles && b->format == BJ_OUT_REF_MCUS) {
        const unsigned gx = std::min<unsigned>(64u, (b->ref_blocks_max * 12u + 255u) / 256u);
        k_ref_mcus_pad<<<dim3(std::max(gx, 1u), n), 256, 0, s>>>(idev, (uint8_t *)b->d_out.p);
        k_idct_color<true><<<b->n_idct_tiles, kTileThreads, b->idct_smem, s>>>((const int16_t *)b->d_coef.p, dcp, idev, qtabs, tiles, (uint8_t *)b->d_out.p);
        b->launches += 2;
    } else if (b->n_idct_tiles) {
        k_idct_color<false><<<b->n_idct_tiles, kTileThreads, b->idct_smem, s>>>((const int16_t *)b->d_coef.p, dcp, idev, qtabs, tiles, (uint8_t *)b->d_out.p);
        b->launches++;
    }
    cudaEventRecord(b->ev[4], s);
    cudaMemcpyAsync(b->h_state(), st, (size_t)n * sizeof(HuffImgState), cudaMemcpyDeviceToHost, s);
    cudaMemcpyAsync(b->h_flags(), flags, kMaxRounds * 4, cudaMemcpyDeviceToHost, s);
    return b->dev->check(cudaGetLastError());
}

inline int batch_decode(bj_batch *b, cudaStream_t s) {
    const bj_ctx *c = b->dev->ctx;
    if (!b->uploaded) return BJ_ERR_ARG;
    if (b->dev->check(cudaSetDevice(b->dev->ordinal)) != BJ_OK) return BJ_ERR_CUDA;
    b->last_stream = s;
    b->decoded = true; b->synced = false;
    if (b->n == 0) return BJ_OK;
    // round 0 cannot tell whether it settled everything (only rounds > 0 compare across CTAs): at least two - unless no
    // image has more than one CTA: then round 0 is all there is to do (every CTA starts at an image head)
    b->rounds = c->sync_rounds > 0 ? (c->sync_rounds < 2 ? 2 : c->sync_rounds) : 3;
    if (!b->multi_blk) b->rounds = 1;
    return batch_launch(b, s, 0, b->rounds);
}

// Wait for the decode; if the last fix-up round still changed something (a sub-sequence that needed more than a
// whole CTA to synchronise - pathological), run more rounds and redo what depends on them.
inline int batch_sync(bj_batch *b) {
    Device *dev = b->dev;
    if (!b->decoded) return BJ_ERR_ARG;
    if (b->n == 0) { b->synced = true; return BJ_OK; }
    cudaStream_t s = b->last_stream;
    int rc = dev->check(cudaStreamSynchronize(s));
    int r = b->rounds;
    b->redone = false;
    while (rc == BJ_OK && b->n_blk && b->multi_blk && b->h_flags()[r - 1] != 0) {
        b->redone = true;
        if (r + 2 > kMaxRounds) { dev->ctx->set_error("entropy stage did not converge"); return BJ_ERR_CUDA; }
        rc = batch_launch(b, s, r, r + 2);
        if (rc == BJ_OK) rc = dev->check(cudaStreamSynchronize(s));
        r += 2;
    }
    b->rounds = r;
    if (rc == BJ_OK) {
        cudaEventElapsedTime(&b->ms_entropy, b->ev[0], b->ev[3]);
        cudaEventElapsedTime(&b->ms_unstuff, b->ev[0], b->ev[1]);
        cudaEventElapsedTime(&b->ms_sync, b->ev[1], b->ev[2]);        // (only the last group of rounds if extra ones ran)
        cudaEventElapsedTime(&b->ms_write, b->ev[2], b->ev[3]);
        cudaEventElapsedTime(&b->ms_idct, b->ev[3], b->ev[4]);
        b->synced = true;
    }
    return rc;
}

// Enqueue the device->host copies of every decoded image (no host wait).
inline int batch_download_async(bj_batch *b, uint8_t *const *outs, cudaStream_t s) {
    Device *dev = b->dev;
    int rc = BJ_OK;
    b->d2h_bytes = 0; b->d2h_copies = 0;
    // option "packed_outputs": the caller states that host buffers laid out like the device buffer (see
    // bj_batch_output_offset) are one allocation, so runs of images go out as one copy (the <= 15 padding bytes
    // between them are overwritten).  Never inferred from pointer values alone: two separate heap blocks can
    // sit at exactly that distance, with allocator metadata in between.
    int i = 0;
    while (rc == BJ_OK && i < b->n) {
        if (b->parse_status[i] != BJ_OK || !outs[i]) { i++; continue; }
        int k = i;
        size_t end = b->out_off[i] + b->out_size[i];
        while (dev->ctx->packed_outputs && k + 1 < b->n && b->parse_status[k + 1] == BJ_OK && outs[k + 1] &&
               outs[k + 1] == outs[i] + (b->out_off[k + 1] - b->out_off[i])) { k++; end = b->out_off[k] + b->out_size[k]; }
        rc = dev->check(cudaMemcpyAsync(outs[i], (const uint8_t *)b->d_out.p + b->out_off[i], end - b->out_off[i], cudaMemcpyDeviceToHost, s));
        b->d2h_bytes += end - b->out_off[i]; b->d2h_copies++;
        i = k + 1;
    }
    return rc;
}

inline int batch_download(bj_batch *b, uint8_t *const *outs, cudaStream_t s) {
    if (!b->decoded) return BJ_ERR_ARG;
    int rc = BJ_OK;
    if (!b->synced) rc = batch_sync(b);           // the (rare) extra fix-up rounds must be settled before copying out
    if (rc == BJ_OK) rc = batch_download_async(b, outs, s);
    if (rc == BJ_OK) rc = b->dev->check(cudaStreamSynchronize(s));
    return rc;
}

inline int batch_image_status(const bj_batch *b, int i) {
    if (b->parse_status[i] != BJ_OK) return b->parse_status[i];
    if (b->synced) {
        const uint32_t st = const_cast<bj_batch *>(b)->h_state()[i].status;
        if (st == kStatusInvalid) return BJ_ERR_INVALID_JPEG;     // the scan does not end in EOI: read_JPEG sets valid = false
        if (st) return BJ_ERR_CORRUPT_SCAN;
    }
    return BJ_OK;
}

}  // namespace bj
