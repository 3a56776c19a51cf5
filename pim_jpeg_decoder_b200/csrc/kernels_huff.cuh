// K0/K1: entropy stage on sm_100a.  Replaces the host-side, single-threaded, bit-serial Huffman decode of the
// reference (src/jpeg_scanner.cpp:405-520, 707-756) with data-parallel kernels:
//
//   k_unstuff                                             (K0)  raw scan bytes -> un-stuffed big-endian words,
//                                                          restart-segment byte offsets, and WHERE THE SCAN ENDS, in one
//                                                          pass (decoupled look-back between an image's tiles).  The host
//                                                          reads only the file headers; it never walks the entropy-coded bytes
//   k_expand_maps                                               CTA -> image maps and the K2/K3 tile list, from per-image records
//   k_subseq_table                                        (K0d) per image: split every segment into sub-sequences
//   k_huff_sync                                           (K1b) speculative decode of every sub-sequence + fix-up
//                                                          to the fixed point inside a CTA (state only, several
//                                                          symbols per table lookup), entry states of the finer
//                                                          slices the write pass works on, block-level prefix sums
//   k_huff_write                                          (K1a) final decode of every slice from its synchronised
//                                                          entry state, in rounds of up to kWriteSteps symbols per lane;
//                                                          look-back, hand-over to the next unit and the warp-cooperative
//                                                          stores of whole 128-byte units once per round
//   k_zero_tail                                                 units the reference never reached read as zero
//
// All arithmetic/semantics live in huff_core.h (shared with the CPU emulation used by the tests).
#pragma once
#include "bj_dev.h"
#include "huff_core.h"
#include "parse.h"

namespace bj {

constexpr int kHuffThreads = 256;          // sub-sequences per CTA
constexpr int kUnstuffThreads = 256;
constexpr int kUnstuffChunks = 4;          // 16-byte chunks per thread of K0
constexpr int kUnstuffTile = kUnstuffThreads * 16 * kUnstuffChunks;   // raw bytes per CTA of K0

// Per image, written by the host.
struct HuffImg {
    uint64_t raw_off;        // offset of the first scan byte in the batch's file buffer
    uint32_t raw_len;        // UPPER BOUND of the raw scan bytes: everything from the first scan byte to the end of the file
                             // (the scan's true length is found on the device: HuffImgState::raw_len)
    uint32_t clean_word0;    // first word of this image's un-stuffed stream
    uint32_t tile_base, ntile;
    uint32_t seg_base;       // index into seg_off / seg_sub0 (nseg + 1 entries each)
    uint32_t nseg;           // segments expected from the header: ceil(nmcu / RI), 1 without DRI
    uint32_t sub_base;       // first sub-sequence slot (multiple of kHuffThreads)
    uint32_t blk_base, nblk; // CTAs of k_huff_sync / k_huff_write
    uint32_t du_base, ndu;
    uint32_t nmcu, ri;       // ri = restart interval in MCUs (0: none)
    uint32_t dcc_base, ndcc; // CTAs of the DC prediction kernels (kDcThreads MCUs each)
    uint8_t bpm, ny, ncomp, valid;
    uint8_t ndc, nac;        // distinct DC / AC tables of this image = staged slots
    uint16_t dc_lut[3], ac_lut[3];   // pool index of each staged DC / AC slot
    uint8_t dc_slot[3], ac_slot[3];  // per component: staged slot
    uint8_t slices_log2;     // the write pass works on 2^slices_log2 slices of every sub-sequence
    uint8_t flags;           // kImgClean / kImgExact (input handed over as a scan, not as a file: bj_decode_batch_desc)
    uint16_t dc_n4[3], ac_n4[3];     // used size of each staged table in 16-byte chunks (tables are staged packed)
    uint32_t sub_bytes;      // length of this image's sub-sequences (synchronisation pass), a multiple of the slice count
    uint32_t wblk_base;      // first CTA of k_huff_write (nblk << slices_log2 of them)
    uint32_t slice_base;     // first slot of this image in the slice table ((nblk * kHuffThreads) << slices_log2 slots)
};

// Per image, written by the kernels.
struct HuffImgState {
    uint32_t clean_len;      // un-stuffed bytes
    uint32_t nrst;           // RSTn markers found
    uint32_t nseg;           // segments actually decoded: min(nrst + 1, expected); 0 for a file whose scan does not end in EOI
    uint32_t nsub;           // sub-sequences
    uint32_t first_zero;     // first unit (image-local) the reference never reached; >= ndu if none
    uint32_t status;         // 0 ok, 1 corrupt entropy-coded data, 2 invalid file (kStatusInvalid)
    uint32_t raw_len;        // raw scan bytes (stuffed, with RSTn) up to the FF that ends the scan
    uint32_t end_code;       // the byte after that FF (D9 = EOI: the only valid one); 0x100: the file ended first
    uint32_t first_zero0, status0;   // first_zero / status as K0 left them: the write pass updates the two above, and a
                                     // re-launch of the write pass (batch.h: batch_sync) starts from these again
    uint32_t pad_[2];
};
constexpr uint8_t kImgClean = 1;           // the bytes are the reference's Header::huffman_data: already un-stuffed, markers removed - every byte is data
constexpr uint8_t kImgExact = 2;           // raw_len is the scan's exact length: it need not end in a marker
constexpr uint32_t kStatusInvalid = 2u;    // read_JPEG's scan-byte loop would set valid = false (src/jpeg_scanner.cpp:405-433)
constexpr uint32_t kNoEnd = kNoScanEnd;

struct BlkAgg {              // units started in one CTA since its last segment head (or since its start)
    uint32_t n, has_head;
};
struct DcAgg {               // DC difference sums of one chunk of MCUs since its last restart (or since its start)
    uint32_t s0, s1, s2, has_head;
};
constexpr int kDcThreads = 256;

// ------------------------------------------------------------------------------------------------ small helpers
__device__ __forceinline__ uint32_t warp_incl_scan(uint32_t v) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, v, d); if (lane >= d) v += t; }
    return v;
}

// exclusive scan of two counters over the CTA; returns totals through tot_a/tot_b
template <int NT>
__device__ __forceinline__ void block_excl_scan2(uint32_t a, uint32_t b, uint32_t &ea, uint32_t &eb, uint32_t &tot_a,
                                                 uint32_t &tot_b, uint32_t *s_tmp /* 2 * NT/32 + 2 */) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t ia = warp_incl_scan(a), ib = warp_incl_scan(b);
    if (lane == 31) { s_tmp[warp] = ia; s_tmp[NT / 32 + warp] = ib; }
    __syncthreads();
    if (warp == 0) {
        uint32_t wa = lane < NT / 32 ? s_tmp[lane] : 0u, wb = lane < NT / 32 ? s_tmp[NT / 32 + lane] : 0u;
        const uint32_t sa = warp_incl_scan(wa), sb = warp_incl_scan(wb);
        if (lane < NT / 32) { s_tmp[lane] = sa - wa; s_tmp[NT / 32 + lane] = sb - wb; }
        if (lane == 31) { s_tmp[2 * (NT / 32)] = sa; s_tmp[2 * (NT / 32) + 1] = sb; }
    }
    __syncthreads();
    ea = ia - a + s_tmp[warp];
    eb = ib - b + s_tmp[NT / 32 + warp];
    tot_a = s_tmp[2 * (NT / 32)];
    tot_b = s_tmp[2 * (NT / 32) + 1];
    __syncthreads();
}

// ------------------------------------------------------------------------------------------------ K0: un-stuff
// ONE pass over aligned tiles of kUnstuffTile raw bytes (one thread = four consecutive aligned 16-byte chunks of the
// file buffer = four 128-bit loads, classified branch-free four bytes per 32-bit word).  A tile
//   * finds where the scan ends if it ends inside the tile: the first FF followed by something other than 00 / FF /
//     RSTn (src/jpeg_scanner.cpp:405-433) - the host passes only an upper bound of the scan (first scan byte .. end of
//     the file) and never touches the entropy-coded bytes;
//   * counts the bytes that survive and the RSTn markers in front of that point and scans them inside the CTA;
//   * learns what the image's earlier tiles contribute by a DECOUPLED LOOK-BACK: every tile publishes its own counts
//     (one 64-bit word: status, "the scan has ended", surviving bytes, markers), then its first warp reads the words of
//     up to 32 predecessors at a time and adds them up until it meets one that already carries an inclusive prefix.
//     A CTA takes its tile index inside its image from the image's ticket counter, so a tile only ever waits for tiles
//     that have started (one counter per image: a single counter for the whole grid serialises 77 600 atomics);
//   * compacts its surviving bytes in shared memory and stores them as big-endian words at their final place;
//   * the tile in which the scan ends (or, if it never does, the image's last tile) writes the image's state: true scan
//     length, totals, and kStatusInvalid when the scan does not end in EOI - the files read_JPEG rejects.
// The byte before the scan is the SOS header's Ah/Al byte (0 in a baseline file), so the rule "the first byte has no
// FF before it" holds without a special case.
// exclusive scan over the CTA of a packed pair of counters (low 16 bits / high 16 bits; totals stay below 2^16)
template <int NT>
__device__ __forceinline__ uint32_t block_excl_scan_packed(uint32_t v, uint32_t &total, uint32_t *s_tmp /* NT/32 + 1 */) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t inc = warp_incl_scan(v);
    if (lane == 31) s_tmp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        const uint32_t wv = lane < NT / 32 ? s_tmp[lane] : 0u;
        const uint32_t ws = warp_incl_scan(wv);
        if (lane < NT / 32) s_tmp[lane] = ws - wv;
        if (lane == 31) s_tmp[NT / 32] = ws;
    }
    __syncthreads();
    total = s_tmp[NT / 32];
    return inc - v + s_tmp[warp];
}

// The look-back word of a tile: bits 1..0 status (0 nothing yet, 1 the tile's own counts, 2 inclusive prefix of the
// image up to and including the tile), bit 2 "the scan has ended" (in this tile / at or before it), bits 33..3 surviving
// bytes, bits 63..34 RSTn markers.  One 64-bit store publishes it, so data and status arrive together.
constexpr uint64_t kLookOwn = 1, kLookIncl = 2;
__device__ __forceinline__ uint64_t look_pack(uint64_t status, bool ended, uint32_t kept, uint32_t rst) {
    return status | (ended ? 4ull : 0ull) | ((uint64_t)kept << 3) | ((uint64_t)rst << 34);
}
__device__ __forceinline__ uint64_t look_load(const uint64_t *p) {
    uint64_t v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void look_store(uint64_t *p, uint64_t v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// look[] (one word per tile) and ticket[] (one counter per image) are zero when the kernel starts (one memset per decode).
// One thread = kUnstuffChunks consecutive 16-byte chunks (64 bytes), a tile = 16 KB: the fixed costs of a tile - ticket,
// barriers, the look-back's round trips through L2 - are paid once per 16 KB (with 4 KB tiles they were half of the
// kernel's time: 77 600 CTAs that each live only a few microseconds).
constexpr int kUnstuffCtas = 4;          // measured on config 2: 4 CTAs per SM (56 registers) 0.425 ms, 5 (48) 0.449 ms, 6 (40, 8 bytes of spills) 0.434 ms
// Shared-memory staging of the surviving bytes: a thread writes its (up to) 64 bytes one by one, and the 32 threads of a
// warp write 64 bytes apart - 16 of them into the same bank.  XOR-ing the word-in-block bits with the 128-byte block
// index spreads a warp's byte stores over all 32 banks (and keeps the word reads of the store loop conflict free).
__device__ __forceinline__ uint32_t unstuff_swz(uint32_t a) { return a ^ (((a >> 7) & 15u) << 2); }
__global__ void __launch_bounds__(kUnstuffThreads, kUnstuffCtas)
k_unstuff(const uint8_t *__restrict__ files, const HuffImg *__restrict__ imgs, const uint32_t *__restrict__ tile_img,
          uint64_t *__restrict__ look, uint32_t *__restrict__ ticket, HuffImgState *__restrict__ st, uint32_t *__restrict__ clean,
          uint32_t *__restrict__ seg_off) {
    constexpr int NC = kUnstuffChunks;
    __shared__ uint32_t s_tmp[kUnstuffThreads / 32 + 1];
    __shared__ __align__(128) uint8_t s_out[kUnstuffTile + 128];           // surviving byte k of the tile at s_out[unstuff_swz(4 + k)]
    __shared__ uint32_t s_tile, s_end, s_base[3];
    const uint32_t img = tile_img[blockIdx.x];
    const HuffImg &im = imgs[img];
    if (threadIdx.x == 0) { s_tile = atomicAdd(ticket + img, 1u); s_end = kNoEnd; }
    __syncthreads();
    const uint32_t tile = s_tile;                                          // which of the image's tiles this CTA works on
    const uint32_t gtile = im.tile_base + tile;
    const int lane = threadIdx.x & 31;

    // ---- classify this thread's 64 bytes
    const uint64_t a0 = (im.raw_off & ~(uint64_t)15) + (uint64_t)tile * kUnstuffTile + (uint64_t)threadIdx.x * (16 * NC);
    const int64_t r0 = (int64_t)a0 - (int64_t)im.raw_off;                  // scan-relative index of the first byte (may be < 0)
    uint32_t w[4 * NC + 2];                                                // w[0]: the word in front (its top byte counts), w[4 NC + 1]: the word behind
    bool live[NC];
#pragma unroll
    for (int c = 0; c < NC; c++) {
        live[c] = r0 + 16 * c < (int64_t)im.raw_len && r0 + 16 * c + 16 > 0;
        const uint4 v = live[c] ? __ldg(reinterpret_cast<const uint4 *>(files + a0) + c) : make_uint4(0, 0, 0, 0);
        w[4 * c + 1] = v.x; w[4 * c + 2] = v.y; w[4 * c + 3] = v.z; w[4 * c + 4] = v.w;
    }
    // the neighbours' edge bytes: from the adjacent lanes, from memory at the warp's edges
    w[0] = __shfl_up_sync(0xFFFFFFFFu, w[4 * NC], 1);
    w[4 * NC + 1] = __shfl_down_sync(0xFFFFFFFFu, w[1], 1);
    if (lane == 0) w[0] = (live[0] && a0 > 0) ? ((uint32_t)__ldg(files + a0 - 1) << 24) : 0u;
    if (lane == 31) w[4 * NC + 1] = live[NC - 1] ? (uint32_t)__ldg(files + a0 + 16 * NC) : 0u;
    uint32_t keep[NC], rst[NC], end[NC];
    uint32_t my_end = kNoEnd;
#pragma unroll
    for (int c = NC - 1; c >= 0; c--) {
        if (im.flags & kImgClean) { keep[c] = 0xFFFFu; rst[c] = 0u; end[c] = 0u; }
        else classify_words_end(w + 4 * c, keep[c], rst[c], end[c]);
        clip_chunk(r0 + 16 * c, im.raw_len, keep[c], rst[c], end[c]);      // bytes outside [0, raw_len) do not count
        if (end[c]) my_end = (uint32_t)(r0 + 16 * c + (__ffs(end[c]) - 1));
    }
    if (my_end != kNoEnd) atomicMin(&s_end, my_end);
    __syncthreads();
    const uint32_t e = s_end;                                              // where the scan ends, if in this tile
    uint32_t nk = 0, nr = 0;
#pragma unroll
    for (int c = 0; c < NC; c++) {
        const uint32_t m = chunk_mask_before(r0 + 16 * c, e);
        keep[c] &= m; rst[c] &= m;
        nk += __popc(keep[c]); nr += __popc(rst[c]);
    }
    uint32_t tot;
    const uint32_t ex = block_excl_scan_packed<kUnstuffThreads>(nk | (nr << 16), tot, s_tmp);
    const uint32_t ea = ex & 0xFFFFu, eb = ex >> 16, ta = tot & 0xFFFFu, tb = tot >> 16;
    // publish this tile's counts at once: the successors' look-backs find them while this tile compacts
    if (threadIdx.x == 0 && tile > 0) look_store(look + gtile, look_pack(kLookOwn, e != kNoEnd, ta, tb));

    // ---- compact into shared memory (the tile's k-th surviving byte at s_out[4 + k])
    {
        uint32_t pos = 4u + ea;
#pragma unroll
        for (int c = 0; c < NC; c++) {
#pragma unroll
            for (int i = 0; i < 16; i++) {
                if (keep[c] & (1u << i)) s_out[unstuff_swz(pos)] = (uint8_t)(w[4 * c + 1 + (i >> 2)] >> ((i & 3) * 8));
                pos += (keep[c] >> i) & 1u;
            }
        }
    }

    // ---- look-back (first warp): what the image's earlier tiles contribute, and whether the scan has ended in one of them
    if (threadIdx.x < 32) {
        uint32_t pk = 0, pr = 0;
        bool ended = false;
        if (tile > 0) {
            int near = (int)tile - 1;                                      // image-local index of the nearest tile not yet added
            for (;;) {
                const int idx = near - lane;
                uint64_t v = look_pack(kLookIncl, false, 0u, 0u);          // in front of the image's first tile: nothing
                if (idx >= 0) { do { v = look_load(look + im.tile_base + idx); } while ((v & 3ull) == 0ull); }
                const uint32_t incl = __ballot_sync(0xFFFFFFFFu, (v & 3ull) == kLookIncl);
                const int stop = incl ? __ffs(incl) - 1 : 31;              // add lanes 0..stop
                uint32_t k = lane <= stop ? (uint32_t)(v >> 3) & 0x7FFFFFFFu : 0u, r = lane <= stop ? (uint32_t)(v >> 34) : 0u;
                const bool en = lane <= stop && (v & 4ull);
#pragma unroll
                for (int d = 16; d > 0; d >>= 1) { k += __shfl_xor_sync(0xFFFFFFFFu, k, d); r += __shfl_xor_sync(0xFFFFFFFFu, r, d); }
                pk += k; pr += r;
                ended = ended || __any_sync(0xFFFFFFFFu, en);
                if (incl) break;
                near -= 32;
            }
        }
        if (lane == 0) {
            look_store(look + gtile, look_pack(kLookIncl, ended || e != kNoEnd, pk + ta, pr + tb));
            s_base[0] = pk; s_base[1] = pr; s_base[2] = ended ? 1u : 0u;
        }
    }
    __syncthreads();
    const uint2 base = make_uint2(s_base[0], s_base[1]);
    if (s_base[2]) return;                                                 // the scan ended in front of this tile
    if (threadIdx.x == 0 && (e != kNoEnd || tile + 1 == im.ntile)) {       // the image's state
        HuffImgState s;
        s.raw_len = e == kNoEnd ? im.raw_len : e;
        s.end_code = e == kNoEnd ? 0x100u : (uint32_t)__ldg(files + im.raw_off + e + 1);
        // "File ended prematurely" / "Invalid marker during compressed data scan" - unless the caller handed over the scan itself
        const bool invalid = s.end_code != 0xD9u && !(e == kNoEnd && (im.flags & (kImgClean | kImgExact)));
        const uint32_t ca = base.x + ta, cb = base.y + tb;
        s.clean_len = ca; s.nrst = cb;
        s.nseg = invalid ? 0u : min(cb + 1u, im.nseg);
        s.nsub = 0;
        // segments whose marker is missing are never decoded: everything from their first unit on reads as zero
        s.first_zero = invalid ? 0u : ((s.nseg < im.nseg) ? s.nseg * im.ri * im.bpm : 0xFFFFFFFFu);
        s.status = invalid ? kStatusInvalid : ((im.ri != 0 && cb + 1u != im.nseg) ? 1u : 0u);
        s.first_zero0 = s.first_zero; s.status0 = s.status;
        s.pad_[0] = s.pad_[1] = 0;
        st[img] = s;
        seg_off[im.seg_base] = 0;
        if (!invalid) seg_off[im.seg_base + s.nseg] = ca;
    }
    if (nr) {                                         // restart markers: where the next segment starts (rare)
        // (marker k of an image is its segment k's start; markers beyond the expected count are ignored)
        uint32_t sidx = base.y + eb + 1, kept = base.x + ea;
#pragma unroll
        for (int c = 0; c < NC; c++) {
            for (uint32_t mm = rst[c]; mm; mm &= mm - 1) {
                const int i = __ffs(mm) - 1;
                if (sidx < im.nseg) seg_off[im.seg_base + sidx] = kept + __popc(keep[c] & ((1u << i) - 1u));
                sidx++;
            }
            kept += __popc(keep[c]);
        }
    }
    if (ta == 0) return;
    // ---- store: stream byte base.x + k = staged byte k.  Output word j (from the word that holds stream byte base.x)
    // takes the staged bytes 4j - mis .. 4j - mis + 3: two aligned shared words and a funnel shift; the (at most two)
    // words the tile shares with its neighbours are written bytewise.  Stream byte o lands at address o ^ 3.
    const uint32_t mis = base.x & 3u;
    uint32_t *dstw = clean + im.clean_word0 + (base.x >> 2);
    const uint32_t end_b = mis + ta;                  // the tile covers bytes [mis, end_b) of its output words
    const uint32_t nwords = (end_b + 3) >> 2;
    const uint32_t *s32 = reinterpret_cast<const uint32_t *>(s_out);
    for (uint32_t k = threadIdx.x; k < nwords; k += kUnstuffThreads) {
        const uint32_t idx = 4u + 4u * k - mis;       // staged position (in s_out) of the word's first byte
        const uint32_t v = __funnelshift_r(s32[unstuff_swz(idx & ~3u) >> 2], s32[unstuff_swz((idx & ~3u) + 4u) >> 2], (idx & 3u) * 8u);
        if (4 * k >= mis && 4 * k + 4 <= end_b) dstw[k] = __byte_perm(v, 0, 0x0123);
        else {
            uint8_t *db = reinterpret_cast<uint8_t *>(dstw + k);
#pragma unroll
            for (uint32_t b = 0; b < 4; b++)
                if (4 * k + b >= mis && 4 * k + b < end_b) db[b ^ 3u] = (uint8_t)(v >> (8 * b));
        }
    }
}

// CTA -> image maps of the kernels above and below and the tile list of the K2/K3 kernel, expanded on the device from
// the per-image records (the host's layout pass is O(images), not O(CTAs)).  One CTA per image; runs once per layout
// (with the upload), not once per decode.
__global__ void __launch_bounds__(256)
k_expand_maps(const HuffImg *__restrict__ imgs, const ImgDev *__restrict__ idev, uint32_t *__restrict__ tile_img, uint32_t *__restrict__ blk_img,
              uint32_t *__restrict__ wblk_img, uint32_t *__restrict__ dcc_img, TileDev *__restrict__ tiles) {
    const uint32_t img = blockIdx.x;
    const HuffImg &im = imgs[img];
    if (!im.valid) return;
    for (uint32_t k = threadIdx.x; k < im.ntile; k += blockDim.x) tile_img[im.tile_base + k] = img;
    for (uint32_t k = threadIdx.x; k < im.nblk; k += blockDim.x) blk_img[im.blk_base + k] = img;
    for (uint32_t k = threadIdx.x; k < (im.nblk << im.slices_log2); k += blockDim.x) wblk_img[im.wblk_base + k] = img;
    for (uint32_t k = threadIdx.x; k < im.ndcc; k += blockDim.x) dcc_img[im.dcc_base + k] = img;
    const ImgDev &id = idev[img];
    const uint32_t tile_mcus = kTileThreads / id.bpm, per_row = (id.nmx + tile_mcus - 1) / tile_mcus;
    for (uint32_t q = threadIdx.x; q < id.nmy * per_row; q += blockDim.x) {
        const uint32_t my = q / per_row, mx = (q - my * per_row) * tile_mcus;
        TileDev t;
        t.img = img; t.my = (uint16_t)my; t.mx0 = (uint16_t)mx;
        t.nm = (uint16_t)min(tile_mcus, id.nmx - mx);
        t.ndu = (uint16_t)(t.nm * id.bpm);
        t.du0 = id.du_base + (my * id.nmx + mx) * id.bpm;
        tiles[id.tile0 + q] = t;
    }
}

// A re-launch of the write pass (the fix-up had not converged when it first ran: batch.h, batch_sync) starts from the
// state K0 left, not from what the write pass made of it on unsettled entry states.
__global__ void k_reset_state(HuffImgState *__restrict__ st, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { st[i].first_zero = st[i].first_zero0; st[i].status = st[i].status0; }
}

// ------------------------------------------------------------------------------------------------ K0d: sub-sequences
// One CTA per image (of NT threads: 256, or 1024 when an image of the batch has more segments than that).  Segment s of the image covers un-stuffed bytes [seg_off[s], seg_off[s+1]) and is cut into
// max(1, ceil(len / sub_bytes)) sub-sequences; seg_sub0[s] = index of its first one, sub_seg[j] = owner segment.
template <int NT>
__global__ void __launch_bounds__(NT)
k_subseq_table(const HuffImg *__restrict__ imgs, HuffImgState *__restrict__ st, const uint32_t *__restrict__ seg_off,
               uint32_t *__restrict__ seg_sub0, uint32_t *__restrict__ sub_seg) {
    __shared__ uint32_t s_tmp[2 * (NT / 32) + 2];
    __shared__ uint32_t s_first[NT + 1];
    const HuffImg &im = imgs[blockIdx.x];
    const uint32_t sub_bytes = im.sub_bytes;
    const uint32_t nseg = st[blockIdx.x].nseg;
    uint32_t carry = 0;
    for (uint32_t s0 = 0; s0 < nseg; s0 += NT) {
        const uint32_t s = s0 + threadIdx.x;
        uint32_t cnt = 0;
        if (s < nseg) {
            const uint32_t len = seg_off[im.seg_base + s + 1] - seg_off[im.seg_base + s];
            cnt = max(1u, (len + sub_bytes - 1) / sub_bytes);
        }
        uint32_t ex, e2, tot, t2;
        block_excl_scan2<NT>(cnt, 0u, ex, e2, tot, t2, s_tmp);
        s_first[threadIdx.x] = carry + ex;
        if (threadIdx.x == 0) s_first[NT] = carry + tot;
        if (s < nseg) seg_sub0[im.seg_base + s] = carry + ex;
        __syncthreads();
        if (nseg > 1) {
            // fill sub_seg for this chunk's sub-sequences: binary search among the chunk's segment starts
            const uint32_t nchunk = min((uint32_t)NT, nseg - s0);
            for (uint32_t j = s_first[0] + threadIdx.x; j < s_first[NT]; j += NT) {
                uint32_t lo = 0, hi = nchunk;                             // last k with s_first[k] <= j
                while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (s_first[mid] <= j) lo = mid; else hi = mid; }
                sub_seg[im.sub_base + j] = s0 + lo;
            }
        }
        carry += tot;
        __syncthreads();
    }
    if (threadIdx.x == 0) { st[blockIdx.x].nsub = carry; seg_sub0[im.seg_base + nseg] = carry; }
}

// ------------------------------------------------------------------------------------------------ K1 common
struct SubInfo {
    uint32_t seg, k;
    uint32_t start_bit, end_bit, data_end_bit;
    bool head, last;
};

__device__ __forceinline__ SubInfo sub_info(const HuffImg &im, const HuffImgState &is, uint32_t j, const uint32_t *__restrict__ seg_off,
                                            const uint32_t *__restrict__ seg_sub0, const uint32_t *__restrict__ sub_seg) {
    SubInfo u;
    const uint32_t sub_bytes = im.sub_bytes;
    u.seg = is.nseg > 1 ? sub_seg[im.sub_base + j] : 0u;
    const uint32_t j0 = seg_sub0[im.seg_base + u.seg], j1 = seg_sub0[im.seg_base + u.seg + 1];
    u.k = j - j0;
    const uint32_t b0 = seg_off[im.seg_base + u.seg], b1 = seg_off[im.seg_base + u.seg + 1];
    u.start_bit = (b0 + u.k * sub_bytes) * 8u;
    u.end_bit = min(b0 + (u.k + 1u) * sub_bytes, b1) * 8u;
    u.data_end_bit = b1 * 8u;
    u.head = u.k == 0;
    u.last = j + 1 == j1;
    return u;
}

// stage the image's tables into shared memory, packed (DC slots first, then AC slots; only the used part of every
// table), 16 bytes per thread per step.  Returns where they are through `g` (byte offsets) and `luts`.
__device__ __forceinline__ void stage_luts(const HuffImg &im, const uint32_t *__restrict__ lut_dc_pool,
                                           const uint32_t *__restrict__ lut_ac_pool, uint32_t *s_lut, uint4 *s_units /* [16], 256-byte aligned */,
                                           HuffGeom &g, LutMem &luts) {
    uint4 *dst = reinterpret_cast<uint4 *>(s_lut);
    uint32_t off = 0, dc_off[3] = {0, 0, 0}, ac_off[3] = {0, 0, 0};
#pragma unroll
    for (int slot = 0; slot < 3; slot++) {
        if (slot < im.ndc) {
            const uint4 *src = reinterpret_cast<const uint4 *>(lut_dc_pool + (size_t)im.dc_lut[slot] * kLutCapDC);
            const uint32_t n4 = im.dc_n4[slot];
            for (uint32_t i = threadIdx.x; i < n4; i += blockDim.x) dst[off + i] = __ldg(src + i);
            dc_off[slot] = off * 16u;
            off += n4;
        }
    }
#pragma unroll
    for (int slot = 0; slot < 3; slot++) {
        if (slot < im.nac) {
            const uint4 *src = reinterpret_cast<const uint4 *>(lut_ac_pool + (size_t)im.ac_lut[slot] * kLutCapAC);
            const uint32_t n4 = im.ac_n4[slot];
            for (uint32_t i = threadIdx.x; i < n4; i += blockDim.x) dst[off + i] = __ldg(src + i);
            ac_off[slot] = off * 16u;
            off += n4;
        }
    }
    g.bpm = im.bpm; g.ny = im.ny; g.unit_tab = 0;
    const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(s_lut);
#pragma unroll
    for (int j = 0; j < 3; j++) {
        const uint32_t ds = im.dc_slot[j], as = im.ac_slot[j];
        g.dc[j] = sbase + (ds == 0 ? dc_off[0] : ds == 1 ? dc_off[1] : dc_off[2]);
        g.ac[j] = sbase + (as == 0 ? ac_off[0] : as == 1 ? ac_off[1] : ac_off[2]);
    }
    // per unit of the MCU: tables and index of the unit that follows it (huff_core.h: next_unit)
    if (threadIdx.x < g.bpm && threadIdx.x < 16u) {
        const uint32_t c1 = threadIdx.x + 1u == g.bpm ? 0u : threadIdx.x + 1u;
        s_units[threadIdx.x] = make_uint4(dc_of(g, c1), ac_of(g, c1), unit_walk_step(threadIdx.x, c1), c1);
    }
    g.unit_tab = (uint32_t)__cvta_generic_to_shared(s_units);
    asm volatile("mov.u32 %0, %0;" : "+r"(g.unit_tab));                   // a register, not an address rebuilt in the symbol loops
    (void)luts;
}

__device__ __forceinline__ uint32_t pack16(uint32_t lo, uint32_t hi) { return (lo & 0xFFFFu) | (hi << 16); }

// ------------------------------------------------------------------------------------------------ K1b: synchronise
// round 0: every sub-sequence starts from the guess (own first bit, unit 0, DC expected) - exact for segment
//          heads - and the CTA iterates  decode -> hand exit state to the successor  until nothing changes.
//          Work is compacted: only sub-sequences whose entry state changed are decoded again, by the first
//          threads of the CTA.
// round r>0: the first sub-sequence of the CTA takes the exit state of the previous CTA's last one; if that
//          differs from what it used, the CTA re-converges.  flags[r] counts CTAs that changed in round r; the
//          host launches rounds until a round reports 0.
// A decode runs quarter by quarter (eighth by eighth for images with 8 slices) and keeps, per quarter, the state at its
// end and the units started in it (`quarters`, 8 entries per sub-sequence).  From the second decode of a sub-sequence
// on, a decode stops as soon as it meets the trajectory of the previous one: a re-decode whose state at the end of a
// quarter equals the recorded one is done - the rest of its trajectory, its exit state and the later quarters' counts
// are those of the previous decode.  Between quarters the sub-sequences still running are compacted onto the first
// threads, like between the iterations.  At the end the write pass' slice table is filled: slot 0 with the
// sub-sequence's own entry state, the other slices' entry states from the quarter records (a slice always starts at a
// quarter boundary).
struct NoRec {
    __device__ __forceinline__ void operator()(uint32_t, uint32_t, uint32_t, uint32_t) const {}
};
// CTAs per SM the synchronisation pass is compiled for.  Every thread walks its own 128-byte lines of the stream, so
// the L1 has to hold about one line per resident thread or the lines are evicted before their 32 words are used:
// 5 CTAs with the shared-memory carve-out limited to 164 KB (92 KB of L1, batch.h) beat 6 CTAs with 56 KB of L1 by
// a quarter (measured: 6: 2.09 ms, 5: 1.53 ms, 4: 2.16 ms, 3: 2.44 ms on config 2).
constexpr int kSyncCtas = 5;
__global__ void __launch_bounds__(kHuffThreads, kSyncCtas)
k_huff_sync(const HuffImg *__restrict__ imgs, const HuffImgState *__restrict__ ist, const uint32_t *__restrict__ blk_img,
            const uint32_t *__restrict__ clean, const uint32_t *__restrict__ seg_off, const uint32_t *__restrict__ seg_sub0,
            const uint32_t *__restrict__ sub_seg, const uint32_t *__restrict__ lut_dc_pool, const uint32_t *__restrict__ lut_ac_pool,
            uint2 *__restrict__ st_in, uint2 *__restrict__ st_out, uint32_t *__restrict__ sub_tot, uint2 *__restrict__ sub_pre,
            uint4 *__restrict__ slices, uint4 *__restrict__ quarters, BlkAgg *__restrict__ blk_agg, uint32_t *__restrict__ flags, int round) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    uint32_t *s_lut = reinterpret_cast<uint32_t *>(smem_raw);
    __shared__ uint2 s_in[kHuffThreads], s_out[kHuffThreads];
    __shared__ uint32_t s_tot[kHuffThreads];
    __shared__ uint2 s_span[kHuffThreads];                                  // first bit, end bit
    __shared__ __align__(256) uint4 s_units[16];
    __shared__ uint16_t s_work[2][kHuffThreads];
    __shared__ uint32_t s_nwork[2];
    __shared__ uint32_t s_flag;
    __shared__ uint2 s_cur[kHuffThreads];                                   // state at the end of the last quarter done
    __shared__ uint16_t s_plist[2][kHuffThreads];                           // sub-sequences still running in this iteration
    __shared__ uint32_t s_pn[2];
    __shared__ uint32_t s_w[kHuffThreads / 32 + 1];
    __shared__ uint32_t s_wf[kHuffThreads / 32 + 1];

    const uint32_t img = blk_img[blockIdx.x];
    const HuffImg &im = imgs[img];
    const HuffImgState is = ist[img];
    const int tid = threadIdx.x;
    const uint32_t j = (blockIdx.x - im.blk_base) * kHuffThreads + tid;    // image-local sub-sequence
    const uint32_t gj = im.sub_base + j;
    const uint32_t first_j = (blockIdx.x - im.blk_base) * kHuffThreads;
    if (first_j >= is.nsub) return;                                        // whole CTA beyond the image's sub-sequences
    const bool active = j < is.nsub;

    SubInfo u;
    u.head = false; u.end_bit = 0; u.start_bit = 0;
    if (active) u = sub_info(im, is, j, seg_off, seg_sub0, sub_seg);

    if (tid == 0) { s_nwork[0] = 0; s_nwork[1] = 0; s_flag = 0; }
    __syncthreads();
    bool need = false;
    if (round == 0) {
        if (active) { s_in[tid] = make_uint2(u.start_bit, 0u); need = true; }
    } else {
        if (active) { s_in[tid] = st_in[gj]; s_out[tid] = st_out[gj]; s_tot[tid] = sub_tot[gj]; }
        if (tid == 0 && !u.head && j > 0) {
            const uint2 prev = st_out[gj - 1];
            if (prev.x != s_in[0].x || prev.y != s_in[0].y) { s_in[0] = prev; need = true; s_flag = 1; }
        }
    }
    s_span[tid] = make_uint2(u.start_bit, u.end_bit);
    if (need) s_work[0][atomicAdd(&s_nwork[0], 1u)] = (uint16_t)tid;
    __syncthreads();
    if (round > 0 && s_flag == 0) return;                                   // nothing changed at this CTA's entry

    HuffGeom g;
    LutMem luts;
    stage_luts(im, lut_dc_pool, lut_ac_pool, s_lut, s_units, g, luts);
    const uint32_t *__restrict__ words = clean + im.clean_word0;
    const uint32_t slices_log2 = im.slices_log2;
    const uint32_t slice_bits = (im.sub_bytes >> slices_log2) * 8u;
    uint4 *img_slices = slices + im.slice_base;

    const uint32_t ql2 = slices_log2 > 2u ? slices_log2 : 2u;               // quarters (or eighths) per sub-sequence
    const uint32_t qbits = (im.sub_bytes >> ql2) * 8u;
    uint4 *img_quarters = quarters + ((size_t)im.sub_base << 3);

    int cur = 0;
    for (uint32_t iter = 0;; iter++) {
        __syncthreads();
        const uint32_t nw = s_nwork[cur];
        if (nw == 0) break;
        const bool has_prev = round > 0 || iter > 0;                        // every sub-sequence on the list has been decoded before
        for (uint32_t w = tid; w < nw; w += kHuffThreads) s_plist[0][w] = s_work[cur][w];
        if (tid == 0) { s_pn[0] = nw; s_pn[1] = 0; }
        int pc = 0;
        for (uint32_t q = 0; q < (1u << ql2); q++) {
            __syncthreads();
            const uint32_t pn = s_pn[pc];
            if (pn == 0) break;
            for (uint32_t w = tid; w < pn; w += kHuffThreads) {
                const uint32_t item = s_plist[pc][w];
                const uint2 span = s_span[item];
                const uint32_t qs = span.x + q * qbits, qe = min(qs + qbits, span.y);
                const bool last = qe >= span.y;
                const uint2 e = q == 0 ? s_in[item] : s_cur[item];
                HuffState in;
                in.p = e.x; in.cz = e.y;
                uint32_t n;
                NoRec rec;
                const HuffState o = decode_span(words, luts, g, in, qs, qe, qbits, rec, &n);
                uint4 *qr = img_quarters + ((size_t)(first_j + item) << 3) + q;
                uint4 old = make_uint4(0u, 0u, 0u, 0u);
                if (has_prev) old = *qr;
                *qr = make_uint4(o.p, o.cz, n, 0u);
                s_tot[item] = (q == 0 && !has_prev ? 0u : s_tot[item]) + n - old.z;
                if (last) s_out[item] = make_uint2(o.p, o.cz);
                else if (!(has_prev && old.x == o.p && old.y == o.cz)) {            // not yet on the old trajectory: go on
                    s_cur[item] = make_uint2(o.p, o.cz);
                    s_plist[pc ^ 1][atomicAdd(&s_pn[pc ^ 1], 1u)] = (uint16_t)item;
                }
            }
            __syncthreads();
            if (tid == 0) s_pn[pc] = 0;
            pc ^= 1;
        }
        __syncthreads();
        if (tid == 0) s_nwork[cur ^ 1] = 0;
        __syncthreads();
        if (active && tid > 0 && !u.head) {
            const uint2 prev = s_out[tid - 1], mine = s_in[tid];
            if (prev.x != mine.x || prev.y != mine.y) {
                s_in[tid] = prev;
                s_work[cur ^ 1][atomicAdd(&s_nwork[cur ^ 1], 1u)] = (uint16_t)tid;
            }
        }
        cur ^= 1;
    }

    // segmented exclusive scan over the CTA of the units started, restarting at segment heads
    uint32_t v0 = 0, f = 0;
    if (active) { v0 = s_tot[tid]; f = u.head ? 1u : 0u; }
    const uint32_t own0 = v0;
    const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t t0 = __shfl_up_sync(0xFFFFFFFFu, v0, d);
        const uint32_t tf = __shfl_up_sync(0xFFFFFFFFu, f, d);
        if (lane >= d) { if (!f) v0 += t0; f |= tf; }
    }
    if (lane == 31) { s_w[warp] = v0; s_wf[warp] = f; }
    __syncthreads();
    if (tid == 0) {                                                        // 8 warp totals: serial segmented scan
        uint32_t c0 = 0, cf = 0;
        for (int w = 0; w < kHuffThreads / 32; w++) {
            const uint32_t a0 = s_w[w], af = s_wf[w];
            s_w[w] = c0; s_wf[w] = cf;                                     // carry INTO warp w
            if (af) { c0 = a0; cf = 1; } else c0 += a0;
        }
        BlkAgg a;
        a.n = c0; a.has_head = cf;
        blk_agg[blockIdx.x] = a;
    }
    __syncthreads();
    if (active) {
        uint32_t hf = f;
        if (!f) { v0 += s_w[warp]; hf = s_wf[warp]; }
        // exclusive: a head starts from zero; otherwise inclusive minus own
        st_in[gj] = s_in[tid];
        img_slices[(size_t)j << slices_log2] = make_uint4(s_in[tid].x, s_in[tid].y, 0u, 0u);
        if (slices_log2) {                                                 // slice k starts where quarter k * step - 1 ended
            const uint32_t step = 1u << (ql2 - slices_log2);
            const uint4 *qr = img_quarters + ((size_t)j << 3);
            const uint32_t nsl = u.end_bit > u.start_bit ? (u.end_bit - u.start_bit + slice_bits - 1u) / slice_bits : 1u;
            uint32_t cnt = 0;
            for (uint32_t k = 1; k < nsl; k++) {
                uint4 e = qr[0];
                for (uint32_t q = (k - 1u) * step; q < k * step; q++) { e = qr[q]; cnt += e.z; }
                img_slices[((size_t)j << slices_log2) + k] = make_uint4(e.x, e.y, cnt, 0u);
            }
        }
        st_out[gj] = s_out[tid];
        sub_tot[gj] = s_tot[tid];
        sub_pre[gj] = u.head ? make_uint2(0u, 1u) : make_uint2(v0 - own0, hf);   // .y: a head precedes inside this CTA
    }
    if (round > 0 && tid == 0) atomicAdd(&flags[round], 1u);
}

// ------------------------------------------------------------------------------------------------ K1a: write
// One thread = one slice; a CTA's 256 slices are consecutive (kHuffThreads >> slices_log2 sub-sequences of one CTA
// of the synchronisation pass).  A warp works in rounds: every lane takes up to kWriteSteps symbols
// (WriteCursor::step_plain: no checks, no hand-over - the lanes stay together) and stops at the one that completes its
// unit; then the lanes that completed a unit look back over it and hand over to their next unit together
// (WriteCursor::unit_end), and the warp stores those units together.  With the hand-over inside every step (one or two
// lanes of a warp take it in two steps of three) the kernel executed 1.63 G warp-instructions on config 2; in rounds 1.0 G.
// Unit staging in shared memory: thread t owns the 128 bytes at t * 128, its 16-byte chunk q stored at chunk
// position q ^ (t & 7): the 2-byte puts of a warp spread over the banks, and a finished unit leaves as eight
// 128-bit shared loads + eight 128-bit global stores issued by eight LANES (one 128-byte line per instruction).
struct SmemUnitSink {
    uint32_t rowsw;          // shared-memory address of (stage + tid * 128) | ((tid & 7) << 4); rows are 128-byte aligned
    // chunk (zz >> 3) ^ sw, element zz & 7  ==  byte (zz * 2) ^ (sw << 4)
    __device__ __forceinline__ void put(uint32_t zz, int16_t v) {
        asm volatile("st.shared.u16 [%0], %1;" ::"r"(rowsw ^ (zz << 1)), "h"(v) : "memory");
    }
    __device__ __forceinline__ void reset() {            // zero the thread's 128-byte row (rare: a unit is decoded again)
        const uint32_t row = rowsw & ~0x7Fu;
        for (uint32_t k = 0; k < 128u; k += 16u) asm volatile("st.shared.v4.u32 [%0], {%1, %1, %1, %1};" ::"r"(row + k), "r"(0u) : "memory");
    }
};

constexpr int kSmemHuffStage = kHuffThreads * 128;

constexpr int kWriteSteps = 8;         // symbols a lane may take per round of the write pass (look-back, hand-over and unit stores once per round); config 2: one symbol per round with the hand-over inside the step 2.00 ms; rounds of 4 / 6 / 8 symbols 1.589 / 1.550 / 1.556 (profiles/r2_write_round_ab.txt); unrolled, with the leaner bit reader, 5 / 6 / 8: 1.513 / 1.503 / 1.493 (profiles/r2_write_unroll_ab.txt)
constexpr int kWriteCtas = 4;          // shared memory allows 4; telling the compiler buys 52 registers instead of 40 (-2 %)
__global__ void __launch_bounds__(kHuffThreads, kWriteCtas)
k_huff_write(const HuffImg *__restrict__ imgs, HuffImgState *__restrict__ ist, const uint32_t *__restrict__ wblk_img,
             const uint32_t *__restrict__ clean, const uint32_t *__restrict__ seg_off, const uint32_t *__restrict__ seg_sub0,
             const uint32_t *__restrict__ sub_seg, const uint32_t *__restrict__ lut_dc_pool, const uint32_t *__restrict__ lut_ac_pool,
             const uint4 *__restrict__ slices, const uint2 *__restrict__ sub_pre, const BlkAgg *__restrict__ blk_agg,
             int16_t *__restrict__ coef, int16_t *__restrict__ dc_plane) {
    extern __shared__ __align__(128) uint8_t smem_raw[];                   // stage rows must be 128-byte aligned
    uint32_t *s_stage = reinterpret_cast<uint32_t *>(smem_raw);
    uint32_t *s_lut = reinterpret_cast<uint32_t *>(smem_raw + kSmemHuffStage);
    __shared__ uint32_t s_red[kHuffThreads / 32];
    __shared__ int s_h;
    __shared__ __align__(256) uint4 s_units[16];
    __shared__ uint32_t s_zero;                                            // what a finished lane reads as its table (WriteCursor::idle)
    __shared__ uint2 s_slot[kHuffThreads / 32][32];                        // per warp: the lanes that completed a unit in this round and which unit (below)

    const uint32_t img = wblk_img[blockIdx.x];
    const HuffImg &im = imgs[img];
    const HuffImgState is = ist[img];
    const uint32_t slices_log2 = im.slices_log2;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t lw = blockIdx.x - im.wblk_base;                         // this image's write CTA
    const uint32_t lb = lw >> slices_log2;                                 // ... which covers part of this CTA of the synchronisation pass
    const uint32_t slot = (lw & ((1u << slices_log2) - 1u)) * kHuffThreads + tid;   // slice slot within that CTA
    const uint32_t j = lb * kHuffThreads + (slot >> slices_log2);          // image-local sub-sequence
    const uint32_t k = slot & ((1u << slices_log2) - 1u);                  // slice of it
    if (lb * kHuffThreads + ((slot - tid) >> slices_log2) >= is.nsub) return;   // whole CTA beyond the image's sub-sequences
    bool active = j < is.nsub;

    // carry into this CTA: totals of the previous CTAs of the image back to the last one that contains a head
    if (tid == 0) { s_h = 0; s_zero = 0u; }
    __syncthreads();
    {
        int h = -1;
        for (int b = (int)lb - 1 - tid; b >= 0; b -= kHuffThreads)
            if (blk_agg[im.blk_base + b].has_head) { h = b; break; }
        if (h >= 0) atomicMax(&s_h, h);
    }
    __syncthreads();
    uint32_t c0 = 0;
    for (int b = s_h + tid; b < (int)lb; b += kHuffThreads) c0 += blk_agg[im.blk_base + b].n;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) c0 += __shfl_xor_sync(0xFFFFFFFFu, c0, d);
    if (lane == 0) s_red[warp] = c0;
    for (int i = tid; i < 32 * kHuffThreads; i += kHuffThreads) s_stage[i] = 0;
    HuffGeom g;
    LutMem luts;
    stage_luts(im, lut_dc_pool, lut_ac_pool, s_lut, s_units, g, luts);
    __syncthreads();
    c0 = 0;
#pragma unroll
    for (int w = 0; w < kHuffThreads / 32; w++) c0 += s_red[w];

    const uint32_t ndu = im.ndu;
    uint4 *out = reinterpret_cast<uint4 *>(coef + (size_t)im.du_base * 64);
    int16_t *dcp = dc_plane + im.du_base;
    WriteCursor cur;
    cur.first_zero = 0xFFFFFFFFu; cur.du = 0; cur.du_end = 0; cur.fail = 0u; cur.st_du = 0xFFFFFFFFu;
    cur.idle = (uint32_t)__cvta_generic_to_shared(&s_zero);
    asm volatile("mov.u32 %0, %0;" : "+r"(cur.idle));
    SmemUnitSink sink;
    const uint32_t stage_addr = (uint32_t)__cvta_generic_to_shared(s_stage);
    sink.rowsw = (stage_addr + tid * 128) | ((tid & 7) << 4);
    // keep it in a register: recomputing it from the thread index in the symbol loop costs more than it does
    asm volatile("mov.u32 %0, %0;" : "+r"(sink.rowsw));
    bool done = true, last = false;
    if (active) {
        const SubInfo u = sub_info(im, is, j, seg_off, seg_sub0, sub_seg);
        const uint32_t slice_bits = (im.sub_bytes >> slices_log2) * 8u;
        const uint32_t nsl = u.end_bit > u.start_bit ? (u.end_bit - u.start_bit + slice_bits - 1u) / slice_bits : 1u;
        active = k < nsl;
        if (active) {
            const uint4 sl = slices[im.slice_base + ((size_t)j << slices_log2) + k];
            const uint2 pre = sub_pre[im.sub_base + j];
            const uint32_t n_ex = pre.x + (pre.y ? 0u : c0) + sl.z;
            const uint32_t du0 = u.seg * im.ri * im.bpm;
            const uint32_t du_end = (im.ri ? min(im.nmcu, (u.seg + 1u) * im.ri) : im.nmcu) * im.bpm;
            HuffState in;
            in.p = sl.x; in.cz = sl.y;
            last = u.last && k + 1u == nsl;
            const uint32_t ev = cur.open(clean + im.clean_word0, luts, g, in, min(u.start_bit + (k + 1u) * slice_bits, u.end_bit),
                                         u.data_end_bit, du0 + n_ex, du_end);
            done = (ev & kEvDone) != 0u;
        }
    }

    uint32_t warp_stage = stage_addr + (tid & ~31) * 128 + ((lane & 7) << 4);     // + this lane's chunk
    asm volatile("mov.u32 %0, %0;" : "+r"(warp_stage));
    uint4 *out_lane = out + (lane & 7);
    asm volatile("mov.u64 %0, %0;" : "+l"(out_lane));                      // (kept in registers, like warp_stage)
    asm volatile("mov.u64 %0, %0;" : "+l"(dcp));
    // a lane with nothing to do idles like one that has finished; every lane of the warp takes every step
    if (done) {
        if (!active) { cur.bs.base = clean + im.clean_word0; cur.bs.wi = 0u; cur.bs.nx2 = 0u; cur.bs.word_end = kWordS; cur.endS = 0u; cur.dataS = 0xFFFFFFFFu; cur.c = 0u; cur.S0 = 0u; cur.bad = 0u; }
        cur.finish();
    }
    if (!__all_sync(0xFFFFFFFFu, done)) {
        uint2 *slot = s_slot[warp];
        for (;;) {
            // a round: up to kWriteSteps symbols per lane, stopping at the one that completes a unit; then the lanes
            // that completed one look back over it and hand over to their next unit together, and the warp stores those units
            // (bit 6 of S = "the unit is complete" stays set until unit_end has handed over)
            cur.step_plain(luts, sink);
#pragma unroll
            for (int k = 1; k < kWriteSteps && !(cur.S & 0x40u); k++) cur.step_plain(luts, sink);
            const bool fin = (cur.S & 0x40u) != 0u;
            const uint32_t m = __ballot_sync(0xFFFFFFFFu, fin);
            if (m == 0) continue;
            // lanes in m completed unit st_du (or ended on a refused DC symbol: nothing to store, st_du = UINT32_MAX):
            // the k-th of them says so in slot k
            if (fin) {
                cur.unit_end(luts, g, sink);
                slot[__popc(m & ((1u << lane) - 1u))] = make_uint2((uint32_t)lane, cur.st_du);
            }
            __syncwarp();
            const uint32_t nun = (uint32_t)__popc(m);
            for (uint32_t base = 0; base < nun; base += 4u) {              // four units per pass: lanes 0-7, 8-15, 16-23, 24-31
                const uint32_t idx = base + ((uint32_t)lane >> 3);
                if (idx < nun) {
                    const uint2 sl = slot[idx];
                    const uint32_t l = sl.x, du_l = sl.y;
                    const uint32_t x = (l & 7u) << 4;
                    const uint32_t a = (warp_stage + l * 128u) ^ x;        // rows are 128-byte aligned
                    uint4 v;
                    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory");
                    asm volatile("st.shared.v4.u32 [%0], {%1, %1, %1, %1};" ::"r"(a), "r"(0u) : "memory");
                    if (du_l < ndu) {                                      // this lane holds the unit's chunk `lane & 7`
                        if ((lane & 7) == 0) { dcp[du_l] = (int16_t)v.x; v.x &= 0xFFFF0000u; }   // slot 0 = the DC difference
                        __stcs(out_lane + (size_t)du_l * 8, v);
                    }
                }
            }
            __syncwarp();
            if (__all_sync(0xFFFFFFFFu, cur.done != 0u)) break;
        }
    }
    if (active) {
        // the last slice of a segment must have produced the segment's last unit
        if (cur.fail == 0u && last && cur.du < cur.du_end) cur.first_zero = cur.du;
        if (cur.first_zero != 0xFFFFFFFFu) {
            atomicMin(&ist[img].first_zero, cur.first_zero);
            ist[img].status = 1u;
        }
    }
}

// Units from first_zero on were never reached by the reference's decoder: they read as zero.  grid = (nimg, slices).
__global__ void __launch_bounds__(256)
k_zero_tail(const HuffImg *__restrict__ imgs, const HuffImgState *__restrict__ ist, int16_t *__restrict__ coef) {
    const HuffImg &im = imgs[blockIdx.x];
    const uint32_t fz = im.valid ? ist[blockIdx.x].first_zero : 0u;
    if (fz >= im.ndu) return;
    uint4 *p = reinterpret_cast<uint4 *>(coef + ((size_t)im.du_base + fz) * 64);
    const size_t n = (size_t)(im.ndu - fz) * 8;
    for (size_t i = (size_t)blockIdx.y * 256 + threadIdx.x; i < n; i += (size_t)gridDim.y * 256) p[i] = make_uint4(0, 0, 0, 0);
}

// ------------------------------------------------------------------------------------------------ K1c: DC prediction
// The write pass leaves DC DIFFERENCES in a compact plane (one short per unit, decode order).  Two tiny kernels
// turn them into predicted values in place: one thread per MCU sums its differences per component, a segmented
// scan (restarting at every restart interval) runs over the CTA, PHASE 0 publishes the chunk's totals, PHASE 1
// adds the totals of the preceding chunks back to the last restart and rewrites the plane.  Units the reference
// never reached (>= first_zero) read as zero.
template <int PHASE>
__global__ void __launch_bounds__(kDcThreads)
k_dc_predict(const HuffImg *__restrict__ imgs, const HuffImgState *__restrict__ ist, const uint32_t *__restrict__ dcc_img,
             int16_t *__restrict__ dc_plane, DcAgg *__restrict__ dc_agg) {
    __shared__ uint32_t s_w[3][kDcThreads / 32 + 1];
    __shared__ uint32_t s_wf[kDcThreads / 32 + 1];
    __shared__ uint32_t s_red[3][kDcThreads / 32];
    __shared__ int s_h;
    const uint32_t img = dcc_img[blockIdx.x];
    const HuffImg &im = imgs[img];
    const uint32_t fz = ist[img].first_zero;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t lc = blockIdx.x - im.dcc_base;
    const uint32_t m = lc * kDcThreads + tid;
    const bool active = m < im.nmcu;
    HuffGeom g;
    g.bpm = im.bpm; g.ny = im.ny; g.unit_tab = 0;
    int16_t *p = dc_plane + im.du_base + (size_t)m * im.bpm;
    int16_t d[6] = {0, 0, 0, 0, 0, 0};
    uint32_t v0 = 0, v1 = 0, v2 = 0, f = 0;
    if (active) {
#pragma unroll
        for (uint32_t c = 0; c < 6; c++) {
            if (c < g.bpm) {
                d[c] = (m * g.bpm + c < fz) ? p[c] : (int16_t)0;
                const uint32_t k = comp_of(g, c), x = (uint32_t)(uint16_t)d[c];
                if (k == 0) v0 += x; else if (k == 1) v1 += x; else v2 += x;
            }
        }
        f = (m == 0 || (im.ri != 0 && m % im.ri == 0)) ? 1u : 0u;
    }
    const uint32_t own0 = v0, own1 = v1, own2 = v2, head = f;
#pragma unroll
    for (int dd = 1; dd < 32; dd <<= 1) {
        const uint32_t t0 = __shfl_up_sync(0xFFFFFFFFu, v0, dd), t1 = __shfl_up_sync(0xFFFFFFFFu, v1, dd);
        const uint32_t t2 = __shfl_up_sync(0xFFFFFFFFu, v2, dd), tf = __shfl_up_sync(0xFFFFFFFFu, f, dd);
        if (lane >= dd) { if (!f) { v0 += t0; v1 += t1; v2 += t2; } f |= tf; }
    }
    if (lane == 31) { s_w[0][warp] = v0; s_w[1][warp] = v1; s_w[2][warp] = v2; s_wf[warp] = f; }
    if (tid == 0) s_h = 0;
    __syncthreads();
    if (tid == 0) {
        uint32_t c0 = 0, c1 = 0, c2 = 0, cf = 0;
        for (int w = 0; w < kDcThreads / 32; w++) {
            const uint32_t a0 = s_w[0][w], a1 = s_w[1][w], a2 = s_w[2][w], af = s_wf[w];
            s_w[0][w] = c0; s_w[1][w] = c1; s_w[2][w] = c2; s_wf[w] = cf;
            if (af) { c0 = a0; c1 = a1; c2 = a2; cf = 1; } else { c0 += a0; c1 += a1; c2 += a2; }
        }
        if (PHASE == 0) {
            DcAgg a;
            a.s0 = c0; a.s1 = c1; a.s2 = c2; a.has_head = cf;
            dc_agg[blockIdx.x] = a;
        }
    }
    if (PHASE == 0) return;
    // carry from the preceding chunks of this image, back to the last one that contains a restart
    {
        int h = -1;
        for (int b = (int)lc - 1 - tid; b >= 0; b -= kDcThreads)
            if (dc_agg[im.dcc_base + b].has_head) { h = b; break; }
        if (h >= 0) atomicMax(&s_h, h);
    }
    __syncthreads();
    uint32_t c0 = 0, c1 = 0, c2 = 0;
    for (int b = s_h + tid; b < (int)lc; b += kDcThreads) {
        const DcAgg a = dc_agg[im.dcc_base + b];
        c0 += a.s0; c1 += a.s1; c2 += a.s2;
    }
#pragma unroll
    for (int dd = 16; dd > 0; dd >>= 1) {
        c0 += __shfl_xor_sync(0xFFFFFFFFu, c0, dd); c1 += __shfl_xor_sync(0xFFFFFFFFu, c1, dd); c2 += __shfl_xor_sync(0xFFFFFFFFu, c2, dd);
    }
    if (lane == 0) { s_red[0][warp] = c0; s_red[1][warp] = c1; s_red[2][warp] = c2; }
    __syncthreads();
    if (!active) return;
    uint32_t hf = f;
    if (!f) { v0 += s_w[0][warp]; v1 += s_w[1][warp]; v2 += s_w[2][warp]; hf = s_wf[warp]; }
    uint32_t pred[3] = {0, 0, 0};
    if (!head) {
        pred[0] = v0 - own0; pred[1] = v1 - own1; pred[2] = v2 - own2;      // exclusive within the CTA
        if (!hf) {
#pragma unroll
            for (int w = 0; w < kDcThreads / 32; w++) { pred[0] += s_red[0][w]; pred[1] += s_red[1][w]; pred[2] += s_red[2][w]; }
        }
    }
#pragma unroll
    for (uint32_t c = 0; c < 6; c++) {
        if (c < g.bpm) {
            const uint32_t k = comp_of(g, c);
            const uint32_t pr = (k == 0 ? pred[0] : (k == 1 ? pred[1] : pred[2])) + (uint32_t)(uint16_t)d[c];
            if (k == 0) pred[0] = pr; else if (k == 1) pred[1] = pr; else pred[2] = pr;
            p[c] = (m * g.bpm + c < fz) ? (int16_t)(uint16_t)pr : (int16_t)0;
        }
    }
}

}  // namespace bj
