// K2+K3: dequantise + 8x8 IDCT + chroma upsample + YCbCr->RGB + store, fused.  sm_100a.
//
//   k_idct_color : fast layout.  Zig-zag i16 coefficient units in, packed 8-bit pixels out (RGB8 or BMP bytes).
//   k_exec_mcus  : the reference's own `mcus` tile layout in and out, in place = src/decoder_dpu.c as a kernel
//                  (the pim.exec() stand-in of src/decoder_host.cpp:292).
//
// Both: one thread owns one 8x8 unit for dequant + IDCT (all 64 values in registers, no shuffles), units are
// staged through shared memory with 128-bit accesses and an XOR-8 chunk swizzle (bank-conflict free for both the
// unit-major IDCT phase and the row-major colour phase), colour conversion is a second warp-cooperative phase
// whose lanes walk along pixel rows, and pixels leave through 128-bit global stores.
#pragma once
#include "bj_dev.h"
#include "idct_color.cuh"

namespace bj {

constexpr int kSmemDu = kTileThreads * 128;              // 24576 B: coefficient units, then samples, in place
constexpr int kSmemQ = 1024;                             // 3 * kQPitch words, padded
constexpr int kRgbFront = 16;                            // slack in front of the staging tile (the copy-out reads whole words)
constexpr int kRgbMax = 1536 * 8 * 3;                    // widest tile: gray, 192 MCUs x 8 px x 8 rows x 3 B
constexpr int kSmemIdctColor = kSmemDu + kSmemQ + kRgbFront + kRgbMax + 64;
// Scaled output: the compact tile of box averages (at most a quarter of the widest pixel tile) lives at the front of
// s_du, with kRgbFront bytes in front and, behind it, the 20 bytes the copy-out's last-chunk read may reach past a row.
static_assert(kRgbFront + kRgbMax / 4 + 20 <= kSmemDu, "the compact tile of a scaled image fits in s_du");

__device__ __forceinline__ uint4 pack_row(const int (&X)[64], int r) {
    uint4 v;
    v.x = __byte_perm(X[r * 8 + 0], X[r * 8 + 1], 0x5410);
    v.y = __byte_perm(X[r * 8 + 2], X[r * 8 + 3], 0x5410);
    v.z = __byte_perm(X[r * 8 + 4], X[r * 8 + 5], 0x5410);
    v.w = __byte_perm(X[r * 8 + 6], X[r * 8 + 7], 0x5410);
    return v;
}

// The chroma contributions of the samples that feed eight pixels of a row (src/decoder_dpu.c:376-378), with the +128 of
// every channel folded in:  tF = ((kF * F) >> 22) + 128,  tL = ((kL * L) >> 22) + 128,  tG = 128 - ((gF * F) >> 22) -
// ((gL * L) >> 22)  (32-bit wrapping products, arithmetic shifts; the sums are associative mod 2^32).  fw / lw: the chroma
// words of the first / last output channel; with 2:1 horizontal subsampling four samples feed the eight pixels (NS = 4).
// With 2:1 VERTICAL subsampling the same terms serve two pixel rows: they are computed once per row pair.
template <int NS>
__device__ __forceinline__ void chroma_terms_row(const unsigned *fw, const unsigned *lw, unsigned kF, unsigned kL, unsigned gF, unsigned gL,
                                                 int (&tF)[NS], int (&tG)[NS], int (&tL)[NS]) {
#pragma unroll
    for (int ci = 0; ci < NS; ci++) {
        const int f = (ci & 1) ? sext_hi(fw[ci >> 1]) : sext_lo(fw[ci >> 1]);
        const int l = (ci & 1) ? sext_hi(lw[ci >> 1]) : sext_lo(lw[ci >> 1]);
        tF[ci] = ((int)(kF * (unsigned)f) >> 22) + 128;
        tG[ci] = 128 - ((int)(gF * (unsigned)f) >> 22) - ((int)(gL * (unsigned)l) >> 22);
        tL[ci] = ((int)(kL * (unsigned)l) >> 22) + 128;
    }
}
// Eight pixels of one row: luma words yv + the chroma terms above -> unclamped channel values.
template <int NS>
__device__ __forceinline__ void color_row(const uint4 &yv, const int (&tF)[NS], const int (&tG)[NS], const int (&tL)[NS], int (&c0)[8],
                                          int (&c1)[8], int (&c2)[8]) {
    const unsigned yw[4] = {yv.x, yv.y, yv.z, yv.w};
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const int ci = NS == 4 ? (i >> 1) : i;                             // chroma sample of pixel i
        const int yy = (i & 1) ? sext_hi(yw[i >> 1]) : sext_lo(yw[i >> 1]);
        c0[i] = yy + tF[ci];
        c1[i] = yy + tG[ci];
        c2[i] = yy + tL[ci];
    }
}
// 24 bytes of packed, clamped pixels (first, G, last per pixel) into the staging tile
__device__ __forceinline__ void store_rgb24(uint8_t *p, const int (&c0)[8], const int (&c1)[8], const int (&c2)[8]) {
    uint2 *dst = reinterpret_cast<uint2 *>(p);
    dst[0] = make_uint2(pack_sat4(c0[0], c1[0], c2[0], c0[1]), pack_sat4(c1[1], c2[1], c0[2], c1[2]));
    dst[1] = make_uint2(pack_sat4(c2[2], c0[3], c1[3], c2[3]), pack_sat4(c0[4], c1[4], c2[4], c0[5]));
    dst[2] = make_uint2(pack_sat4(c1[5], c2[5], c0[6], c1[6]), pack_sat4(c2[6], c0[7], c1[7], c2[7]));
}
// the same as three 16-byte rows of shorts (R, G, B planes of the reference's block-tiled layout)
__device__ __forceinline__ void store_ref_rows(int16_t *ob, const int (&c0)[8], const int (&c1)[8], const int (&c2)[8]) {
    auto pack8 = [](const int (&c)[8]) {
        return make_uint4(clamp255(c[0]) | (clamp255(c[1]) << 16), clamp255(c[2]) | (clamp255(c[3]) << 16),
                          clamp255(c[4]) | (clamp255(c[5]) << 16), clamp255(c[6]) | (clamp255(c[7]) << 16));
    };
    __stcs(reinterpret_cast<uint4 *>(ob), pack8(c0));
    __stcs(reinterpret_cast<uint4 *>(ob + 256), pack8(c1));
    __stcs(reinterpret_cast<uint4 *>(ob + 512), pack8(c2));
}

// ------------------------------------------------------------------------------------------------ fast layout
// REF_MCUS = false: packed 8-bit pixels (RGB8 or the BMP byte stream).  REF_MCUS = true: the reference's own post-exec
// `mcus` layout - R, G, B as shorts inside the block-tiled buffer that the unchanged write_BMP reads
// (src/bmp_writer.cpp:43-61; layout src/decoder_dpu.c:134-156, destination index src/jpeg_scanner.cpp:733-741): for the
// 8x8 position (pr, pc) of a grid that is W = mcu_width_real positions wide,
//     block = (pr / 2) * ((W + 1) / 2) + pc / 2,  pos = (pr % 2) * 2 + pc % 2,
//     short index = block * 768 + component * 256 + pos * 64 + row * 8 + x
// (the split into MAX_MCU_PER_DPU chunks is the same linear buffer: a chunk is MAX_MCU_PER_DPU / 4 whole blocks).
// Stages 1-3 of one tile of k_idct_color below: the tile's coefficient units are in `s_du` (unit du's 16-byte chunk c
// at chunk position c ^ (du & 7)), the image's quantiser set in `s_q`, the predicted DC values in `s_dc`.
// Stage 1 of one tile: dequantise + IDCT, one thread = one unit, in place in `s_du`.
__device__ __forceinline__ void tile_idct(uint4 *s_du, const uint32_t *s_q, const uint16_t *s_dc, const int ndu, const int hs, const int vs,
                                          const int bpm, const bool dc_sep) {
    const int tid = threadIdx.x;
    // ---- stage 1: one thread = one unit: de-zigzag (with the reference's 48/52 quirk), dequantise, IDCT
    if (tid < ndu) {
        const int du = tid, sw = du & 7;
        const int k = du % bpm, ny = hs * vs;
        const int comp = k < ny ? 0 : k - ny + 1;
        const uint4 *q4 = reinterpret_cast<const uint4 *>(s_q + comp * kQPitch);
        int X[64];
        unsigned raw48 = 0, raw52 = 0;
        const unsigned dcv = s_dc[du];
#pragma unroll
        for (int c = 0; c < 8; c++) {
            uint4 v = s_du[du * 8 + (c ^ sw)];
            if (c == 0 && dc_sep) v.x = (v.x & 0xFFFF0000u) | dcv;
            const uint4 qa = q4[2 * c], qb = q4[2 * c + 1];
            // (w * (q<<16)) mod 2^32 only sees the low 16 bits of w: no unpack needed for the low halves
            X[zz2nat(8 * c + 0)] = (int)(v.x * qa.x);
            X[zz2nat(8 * c + 1)] = (int)((v.x >> 16) * qa.y);
            X[zz2nat(8 * c + 2)] = (int)(v.y * qa.z);
            X[zz2nat(8 * c + 3)] = (int)((v.y >> 16) * qa.w);
            X[zz2nat(8 * c + 4)] = (int)(v.z * qb.x);
            X[zz2nat(8 * c + 5)] = (int)((v.z >> 16) * qb.y);
            X[zz2nat(8 * c + 6)] = (int)(v.w * qb.z);
            X[zz2nat(8 * c + 7)] = (int)((v.w >> 16) * qb.w);
            if (c == 6) { raw48 = v.x & 0xFFFFu; raw52 = v.z & 0xFFFFu; }
        }
        {   // src/headers/common.h:16: index 48 and 52 both land on natural 38 (52 wins when present), 58 stays 0;
            // the quantiser at natural 38 is the one read at index 52 (src/jpeg_scanner.cpp:306,311).
            const unsigned q52 = s_q[comp * kQPitch + 52];
            X[38] = (int)((raw52 != 0 ? raw52 : raw48) * q52);
            X[58] = 0;
        }
        idct8x8(X);
#pragma unroll
        for (int r = 0; r < 8; r++) s_du[du * 8 + (r ^ sw)] = pack_row(X, r);
    }
}

// Stage 3 of one tile: copy-out.  `src`: the tile's packed pixels, `pitch` bytes per row, `ncols` x `rows` pixels whose
// top-left pixel is (x0, y0) of the output image (the full image, or the scaled one); the image record's crop window and
// output layout are in the same coordinates.
__device__ __forceinline__ void tile_copy_out(const uint8_t *src, const int pitch, const int x0, const int y0, const int ncols, const int rows,
                                              const TileDev &t, const ImgDev *__restrict__ im, uint8_t *__restrict__ out) {
    const int tid = threadIdx.x;
    // Each pixel row of the tile is a contiguous byte run in HBM with arbitrary
    // alignment; it is written as 16-byte-aligned 128-bit stores whose payload is funnel-shifted out of the
    // staging tile; only the first/last chunk of a run (and BMP pad bytes) go bytewise.  Only the image's crop window
    // leaves (the whole image unless a region of interest was asked for): tile rows y0 + r in [cy, cy + ch), columns
    // [xs, xe) = the tile's columns inside [cx, cx + cw); pixel (x, y) goes to row y - cy, column x - cx of the output.
    {
        const int cx = (int)im->cx, cy = (int)im->cy, cx_end = cx + (int)im->cw;
        const int xs = max(x0, cx), xe = min(x0 + ncols, cx_end);
        const int r_lo = max(cy - y0, 0), r_hi = min(rows, cy + (int)im->ch - y0);
        const int payload = (xe - xs) * 3;
        const int len = payload + (xe == cx_end ? (int)im->row_pad : 0);   // BMP pad bytes follow the run at the crop's right edge
        const int warp = tid >> 5, lane = tid & 31;
        const long long row_step = (long long)im->row_dir * (long long)im->out_pitch;
        const long long off0 = (long long)im->out_row0 + row_step * (long long)(y0 - cy) + (long long)(xs - cx) * 3;
        const uint8_t *sp0 = src + (xs - x0) * 3;                        // (any byte alignment: the funnel shift below takes it)
        for (int r = r_lo + warp; r < r_hi; r += kTileThreads / 32) {
            uint8_t *g = out + (off0 + row_step * r);
            const uint8_t *sp = sp0 + r * pitch;
            // the run [0, len) = head bytes up to the first 16-byte boundary, nfull whole aligned chunks, ntail bytes
            const int head = min((int)((16u - ((unsigned)(uintptr_t)g & 15u)) & 15u), len);
            const int nfull = (len - head) >> 4;
            const int tail0 = head + 16 * nfull;
            // head and tail bytes in one store: lanes 0-15 a head byte each, lanes 16-31 a tail byte each
            {
                const int idx = lane < 16 ? lane : tail0 + lane - 16;
                const bool ok = lane < 16 ? lane < head : idx < len;
                if (ok) g[idx] = idx < payload ? sp[idx] : (uint8_t)0;
            }
            // body: whole aligned 16-byte chunks.  Those that hold only pixel bytes first (no masking); BMP pad bytes
            // (at most 3 per row) can only lie in the last whole chunk
            const uint8_t *p0 = sp + head;
            const unsigned a = (unsigned)__cvta_generic_to_shared(p0);
            const unsigned sh = (a & 3u) * 8u;
            const unsigned wa = a & ~3u;                                   // shared-memory address of the first word
            uint4 *gp = reinterpret_cast<uint4 *>(g + head);
            const int nbody = min(nfull, max(payload - head, 0) >> 4);
            for (int i = lane; i < nbody; i += 32) {
                uint32_t w0, w1, w2, w3, w4;
                asm volatile("ld.shared.u32 %0, [%5];\n\tld.shared.u32 %1, [%5+4];\n\tld.shared.u32 %2, [%5+8];\n\tld.shared.u32 %3, [%5+12];\n\tld.shared.u32 %4, [%5+16];"
                             : "=r"(w0), "=r"(w1), "=r"(w2), "=r"(w3), "=r"(w4) : "r"(wa + 16u * (unsigned)i));
                uint4 v;
                v.x = __funnelshift_r(w0, w1, sh); v.y = __funnelshift_r(w1, w2, sh);
                v.z = __funnelshift_r(w2, w3, sh); v.w = __funnelshift_r(w3, w4, sh);
                __stcs(gp + i, v);
            }
            if (nbody < nfull && lane == 0) {                              // the chunk with pad bytes (zero) in it
                const int i = nbody;
                const uint32_t *wp = reinterpret_cast<const uint32_t *>(p0 - (a & 3u));
                const uint32_t w0 = wp[4 * i], w1 = wp[4 * i + 1], w2 = wp[4 * i + 2], w3 = wp[4 * i + 3], w4 = wp[4 * i + 4];
                uint32_t vv[4] = {__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh), __funnelshift_r(w3, w4, sh)};
                const int keep = payload - head - 16 * i;                  // data bytes in the chunk, < 16
#pragma unroll
                for (int w = 0; w < 4; w++) {
                    const int kb = keep - 4 * w;
                    vv[w] = kb >= 4 ? vv[w] : (kb <= 0 ? 0u : (vv[w] & (0xFFFFFFFFu >> (32 - 8 * kb))));
                }
                __stcs(gp + i, make_uint4(vv[0], vv[1], vv[2], vv[3]));
            }
        }
        // BMP file header (src/bmp_writer.cpp:26-41) of the cw x ch output, written by the tile that holds pixel (cx, cy):
        // 'B','M', size(4), 0(4), 0x1A(4), 12(4), width(2), height(2), 1(2), 24(2)
        if (im->bgr && t.my == im->my_lo && t.mx0 == im->mx_lo && tid < 26) {
            const unsigned W = im->cw, H = im->ch;
            const unsigned size = 26u + H * W * 3u + im->row_pad * H;
            unsigned v = 0;
            if (tid == 0) v = 'B';
            else if (tid == 1) v = 'M';
            else if (tid < 6) v = size >> ((tid - 2) * 8);
            else if (tid == 10) v = 0x1A;
            else if (tid == 14) v = 12;
            else if (tid == 18) v = W;
            else if (tid == 19) v = W >> 8;
            else if (tid == 20) v = H;
            else if (tid == 21) v = H >> 8;
            else if (tid == 22) v = 1;
            else if (tid == 24) v = 24;
            const long long hdr = (long long)im->out_row0 - (long long)(H - 1) * (long long)im->out_pitch - 26;
            out[hdr + tid] = (uint8_t)v;
        }
    }
}

// Reciprocals of the box sizes n = 1..64 of the reduction below: kBoxRcp.r[n] = ceil(2^31 / n).  For a < 2^15,
// __umulhi(2a, r[n]) = floor(a * r[n] / 2^31) = floor(a / n) exactly (a * (r[n] * n - 2^31) < 2^15 * 64 < 2^31).
struct BoxRcp {
    uint32_t r[65];
    constexpr BoxRcp() : r() {
        for (uint32_t n = 1; n <= 64; n++) r[n] = (uint32_t)((((uint64_t)1 << 31) + n - 1) / n);
    }
};
__constant__ BoxRcp kBoxRcp = BoxRcp();

// Box reduction of one tile (scaled output, s = 1 << SL in {2, 4, 8}): output pixel (X, Y) of the tile is the rounded
// mean, per channel, of the pixels [sX, sX + s) x [sY, sY + s) of the `ncols` x `rows` pixel tile `src` (`pitch` bytes per
// row, top-left pixel (x0, y0) of the full image) that lie inside the image: pixels at x >= width or y >= height (MCU
// padding) count in neither sum nor divisor.  x0, y0, ncols and rows are multiples of 8, so every box lies inside the
// tile.  Into `dst`: (ncols / s) x (rows / s) pixels, 3 * ncols / s bytes per row.
// One item = one quad of 4 horizontally adjacent pixels (three words of `src`) in the s rows of one output row.  Lanes
// take consecutive quads: word addresses 3 apart, which no two lanes of a warp share a bank with.  A quad is 2 output
// pixels at s = 2 and 1 at s = 4; at s = 8 the two lanes of a quad pair add their sums with a shuffle.  The bytes are
// summed two per word in 16-bit lanes (at most 8 * 255 per column, 64 * 255 per box).  Only quads that reach past the
// image's right edge mask bytes out; the rounded division is a multiply by the box size's reciprocal.
template <int SL>
__device__ __forceinline__ void tile_box_reduce(const uint8_t *src, const int pitch, const int ncols, const int rows, const int x0, const int y0,
                                                const ImgDev *__restrict__ im, uint8_t *dst) {
    constexpr int S = 1 << SL;
    const int tid = threadIdx.x;
    const int nq = ncols >> 2, orows = rows >> SL, opitch = (ncols >> SL) * 3;
    const int items = orows * nq;                                    // (nq is even: ncols is a multiple of 8)
    const unsigned inv = 0xFFFFFFFFu / (unsigned)nq + 1u;
    const int wpitch = pitch >> 2;
    const int W = (int)im->width - x0, H = (int)im->height - y0;   // (the image's extent seen from the tile's origin)
    for (int base = 0; base < items; base += kTileThreads) {         // (uniform trip count: the s = 8 shuffle needs every lane)
        const int it = base + tid;
        const int oy = (int)__umulhi((unsigned)it, inv), q = it - oy * nq;
        const int nr = it < items ? min(S, H - (oy << SL)) : 0;      // rows of the box inside the image
        const int nv = W - 4 * q;                                    // pixels of the quad inside the image (4 or more: all)
        uint32_t m[3] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu};
        if (nv < 4) {
#pragma unroll
            for (int j = 0; j < 3; j++) {
                const int kb = 3 * max(nv, 0) - 4 * j;
                m[j] = kb >= 4 ? 0xFFFFFFFFu : (kb <= 0 ? 0u : (0xFFFFFFFFu >> (32 - 8 * kb)));
            }
        }
        uint32_t lo[3] = {0, 0, 0}, hi[3] = {0, 0, 0};               // bytes 4j, 4j + 2 / 4j + 1, 4j + 3 of the quad, column sums
        const uint32_t *wp = reinterpret_cast<const uint32_t *>(src) + (oy << SL) * wpitch + 3 * q;
#pragma unroll
        for (int r = 0; r < S; r++) {
            if (r < nr) {
#pragma unroll
                for (int j = 0; j < 3; j++) {
                    const uint32_t w = wp[r * wpitch + j] & m[j];
                    lo[j] += w & 0x00FF00FFu;
                    hi[j] += (w >> 8) & 0x00FF00FFu;
                }
            }
        }
        // per-pixel channel sums: byte k = 3p + c of the quad
        unsigned S_[12];
#pragma unroll
        for (int j = 0; j < 3; j++) {
            S_[4 * j] = lo[j] & 0xFFFFu; S_[4 * j + 1] = hi[j] & 0xFFFFu; S_[4 * j + 2] = lo[j] >> 16; S_[4 * j + 3] = hi[j] >> 16;
        }
        unsigned v[2][3];
#pragma unroll
        for (int c = 0; c < 3; c++) {
            v[0][c] = S_[c] + S_[3 + c];
            v[1][c] = S_[6 + c] + S_[9 + c];
            if (SL >= 2) v[0][c] += v[1][c];
            if (SL == 3) v[0][c] += __shfl_xor_sync(0xFFFFFFFFu, v[0][c], 1);
        }
        constexpr int NOUT = SL == 1 ? 2 : 1;                        // output pixels of this lane
        const int X = SL == 1 ? 2 * q : (SL == 2 ? q : q >> 1);      // the first one's column in the tile
        const bool mine = SL != 3 || (q & 1) == 0;                   // (s = 8: the even lane of the pair writes)
#pragma unroll
        for (int k = 0; k < NOUT; k++) {
            const int nc = min(S, W - ((X + k) << SL));               // columns of the box inside the image
            if (mine && nr > 0 && nc > 0) {                          // (a box of MCU padding only is never copied out)
                const unsigned n = (unsigned)(nc * nr);
                const unsigned rcp = kBoxRcp.r[n];
                uint8_t *d = dst + oy * opitch + (X + k) * 3;
#pragma unroll
                for (int c = 0; c < 3; c++) d[c] = (uint8_t)__umulhi((v[k][c] + (n >> 1)) << 1, rcp);
            }
        }
    }
}

// Stages 2 and 3 of one tile: colour conversion into the staging tile `s_rgb`, copy-out (REF_MCUS: straight to HBM).
// HS, VS: the luma sampling factors as compile-time constants for three-component images (the index arithmetic of the
// colour stage folds: 4:2:0 and 4:4:4 have their own instances), or 0, 0: whatever the image record says.
// SCALED: images may ask for reduced-size output (ImgDev::scale_log2 > 0); without it the record's scale is not read.
template <bool REF_MCUS, bool SCALED, int HS, int VS>
__device__ __forceinline__ void tile_color_store(const uint4 *s_du, uint8_t *s_rgb, const TileDev &t, const ImgDev *__restrict__ im, const int hs_rt,
                                                 const int vs_rt, const int ncomp_rt, const int bpm_rt, uint8_t *__restrict__ out) {
    const int hs = HS ? HS : hs_rt, vs = HS ? VS : vs_rt, ncomp = HS ? 3 : ncomp_rt, bpm = HS ? HS * VS + 2 : bpm_rt;
    const int tid = threadIdx.x;
    const int nm = t.nm;
    // ---- stage 2: colour.  One item = 8 horizontally adjacent pixels of one row of one luma unit - of TWO rows (2r, 2r + 1)
    // when the image is subsampled 2:1 vertically: both rows take the same chroma row, whose terms are computed once.
    // Consecutive lanes take consecutive segments of the same pixel row(s).  Result: 24 bytes per row into the staging tile.
    const int nseg = nm * hs;             // 8-pixel segments per tile row
    const int rows = vs * 8;
    const int pitch = nseg * 24;
    {
        const unsigned inv = nseg > 1 ? (0xFFFFFFFFu / (unsigned)nseg + 1u) : 0u;
        const int nrow = vs == 2 ? 2 : 1;                                  // pixel rows per item
        const int items = (rows / nrow) * nseg;
        // Output byte order R,G,B or B,G,R: instead of swapping per pixel, swap the roles of the two chroma planes
        // and of their constants once (src/decoder_dpu.c:376-378):  first = y + 128 + ((kF * F) >> 22),
        // last = y + 128 + ((kL * L) >> 22),  G = y + 128 - ((gF * F) >> 22) - ((gL * L) >> 22).
        const bool bgr = im->bgr != 0;
        const unsigned kF = bgr ? 7432306u : 5880414u, kL = bgr ? 5880414u : 7432306u;
        const unsigned gF = bgr ? 1442840u : 2994733u, gL = bgr ? 2994733u : 1442840u;
        const int fdu = bgr ? 0 : 1, ldu = bgr ? 1 : 0;                    // unit offsets of F and L from the Cb unit
        const bool has_f = bgr ? ncomp >= 2 : ncomp >= 3, has_l = bgr ? ncomp >= 3 : ncomp >= 2;
        for (int it = tid; it < items; it += kTileThreads) {
            const int pq = nseg > 1 ? (int)__umulhi((unsigned)it, inv) : it;
            const int s = it - pq * nseg;
            const int py = pq * nrow;                                      // first pixel row of the item
            const int m = hs == 2 ? (s >> 1) : s, bx = hs == 2 ? (s & 1) : 0;
            const int by = py >> 3, r = py & 7;
            const int ydu = m * bpm + by * hs + bx;
            const int cdu = m * bpm + hs * vs;
            const int rc = vs == 2 ? (by * 4 + (r >> 1)) : r;
            uint4 fv = make_uint4(0, 0, 0, 0), lv = make_uint4(0, 0, 0, 0);
            if (has_f) fv = s_du[(cdu + fdu) * 8 + (rc ^ ((cdu + fdu) & 7))];
            if (has_l) lv = s_du[(cdu + ldu) * 8 + (rc ^ ((cdu + ldu) & 7))];
            // destination of the item's first row: the staging tile, or (REF_MCUS) straight to HBM: three 16-byte rows
            // (R, G, B as shorts) of position (pr, pc)
            uint8_t *dst = s_rgb + py * pitch + s * 24;
            int16_t *ob = nullptr;
            if (REF_MCUS) {
                const unsigned pr = (unsigned)t.my * vs + by, pc = ((unsigned)t.mx0 + m) * hs + bx, W = im->nmx * hs;
                const size_t blk = (size_t)(pr >> 1) * ((W + 1u) >> 1) + (pc >> 1);
                ob = reinterpret_cast<int16_t *>(out + im->out_row0) + blk * 768 + ((pr & 1u) * 2u + (pc & 1u)) * 64u + r * 8;
            }
            int c0[8], c1[8], c2[8];
            if (hs == 2) {
                // one unit row feeds two segments (left half / right half), every chroma sample twice
                const unsigned fw[2] = {bx ? fv.z : fv.x, bx ? fv.w : fv.y}, lw[2] = {bx ? lv.z : lv.x, bx ? lv.w : lv.y};
                int tF[4], tG[4], tL[4];
                chroma_terms_row<4>(fw, lw, kF, kL, gF, gL, tF, tG, tL);
#pragma unroll 1
                for (int k = 0; k < nrow; k++) {
                    const uint4 yv = s_du[ydu * 8 + ((r + k) ^ (ydu & 7))];
                    color_row<4>(yv, tF, tG, tL, c0, c1, c2);
                    if (REF_MCUS) store_ref_rows(ob + k * 8, c0, c1, c2);
                    else store_rgb24(dst + k * pitch, c0, c1, c2);
                }
            } else {
                const unsigned fw[4] = {fv.x, fv.y, fv.z, fv.w}, lw[4] = {lv.x, lv.y, lv.z, lv.w};
                int tF[8], tG[8], tL[8];
                chroma_terms_row<8>(fw, lw, kF, kL, gF, gL, tF, tG, tL);
#pragma unroll 1
                for (int k = 0; k < nrow; k++) {
                    const uint4 yv = s_du[ydu * 8 + ((r + k) ^ (ydu & 7))];
                    color_row<8>(yv, tF, tG, tL, c0, c1, c2);
                    if (REF_MCUS) store_ref_rows(ob + k * 8, c0, c1, c2);
                    else store_rgb24(dst + k * pitch, c0, c1, c2);
                }
            }
        }
    }
    if (REF_MCUS) return;
    __syncthreads();

    // ---- stage 3: copy-out of the pixel tile.  Scaled output: each s x s box of it is first averaged into the compact
    // tile, which lives at the front of s_du (free once stage 2 has read it), and the copy-out works on that.  (The
    // compact tile is addressed as an offset from s_rgb, not as a second pointer: with the pointer, ptxas spills two
    // registers across stage 1.)
    const int x0 = t.mx0 * hs * 8, y0 = t.my * vs * 8;
    const int sl = SCALED ? im->scale_log2 : 0;
    int src_off = 0;
    if (SCALED && sl) {
        src_off = kRgbFront - (kSmemDu + kSmemQ + kRgbFront);
        if (sl == 1) tile_box_reduce<1>(s_rgb, pitch, nseg * 8, rows, x0, y0, im, s_rgb + src_off);
        else if (sl == 2) tile_box_reduce<2>(s_rgb, pitch, nseg * 8, rows, x0, y0, im, s_rgb + src_off);
        else tile_box_reduce<3>(s_rgb, pitch, nseg * 8, rows, x0, y0, im, s_rgb + src_off);
        __syncthreads();
    }
    tile_copy_out(s_rgb + src_off, ((nseg * 8) >> sl) * 3, x0 >> sl, y0 >> sl, (nseg * 8) >> sl, rows >> sl, t, im, out);
}

template <bool REF_MCUS, bool SCALED>
__global__ void __launch_bounds__(kTileThreads, 4)
k_idct_color(const int16_t *__restrict__ coef, const int16_t *__restrict__ dc_plane, const ImgDev *__restrict__ imgs,
             const QTab *__restrict__ qtabs, const TileDev *__restrict__ tiles, uint8_t *__restrict__ out) {
    static_assert(!(REF_MCUS && SCALED), "the reference's tile layout has no scaled form");
    extern __shared__ __align__(16) uint8_t smem[];
    uint4 *s_du = reinterpret_cast<uint4 *>(smem);
    uint32_t *s_q = reinterpret_cast<uint32_t *>(smem + kSmemDu);
    uint8_t *s_rgb = smem + kSmemDu + kSmemQ + kRgbFront;
    __shared__ uint16_t s_dc[kTileThreads];

    const int tid = threadIdx.x;
    TileDev t;
    {
        const uint4 tw = __ldg(reinterpret_cast<const uint4 *>(tiles) + blockIdx.x);     // the 16-byte record in one load
        t.img = tw.x; t.my = (uint16_t)tw.y; t.mx0 = (uint16_t)(tw.y >> 16); t.nm = (uint16_t)tw.z; t.ndu = (uint16_t)(tw.z >> 16); t.du0 = tw.w;
    }
    const int ndu = t.ndu;

    // ---- stage 0: this tile's coefficient units (contiguous in HBM) -> smem, coalesced 16 B.  All of a thread's
    // loads are issued before the first store, and nothing here waits for the image record.
    {
        const uint4 *src = reinterpret_cast<const uint4 *>(coef) + (size_t)t.du0 * 8;
        uint4 v[8];
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const int q = tid + k * kTileThreads;
            v[k] = q < ndu * 8 ? __ldcs(src + q) : make_uint4(0, 0, 0, 0);
        }
        // the entropy stage keeps predicted DC values in a separate plane (one short per unit): patched in here
        unsigned dcv = 0;
        const bool dc_sep = dc_plane != nullptr;
        if (dc_sep && tid < ndu) dcv = (unsigned short)__ldg(dc_plane + (size_t)t.du0 + tid);
        s_dc[tid] = (uint16_t)dcv;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const int q = tid + k * kTileThreads;
            const int du = q >> 3, c = q & 7;
            if (q < ndu * 8) s_du[du * 8 + (c ^ (du & 7))] = v[k];
        }
    }
    const ImgDev *__restrict__ im = imgs + t.img;
    const int hs = im->hs, vs = im->vs, ncomp = im->ncomp, bpm = im->bpm;
    {
        const uint32_t *__restrict__ q = &qtabs[im->qslot].q16[0][0];
        for (int i = tid; i < 3 * kQPitch; i += kTileThreads) s_q[i] = __ldg(q + i);
    }
    __syncthreads();

    tile_idct(s_du, s_q, s_dc, ndu, hs, vs, bpm, dc_plane != nullptr);
    __syncthreads();
    if (ncomp == 3 && hs == 2 && vs == 2) tile_color_store<REF_MCUS, SCALED, 2, 2>(s_du, s_rgb, t, im, hs, vs, ncomp, bpm, out);
    else if (ncomp == 3 && hs == 1 && vs == 1) tile_color_store<REF_MCUS, SCALED, 1, 1>(s_du, s_rgb, t, im, hs, vs, ncomp, bpm, out);
    else tile_color_store<REF_MCUS, SCALED, 0, 0>(s_du, s_rgb, t, im, hs, vs, ncomp, bpm, out);
}

// REF_MCUS: what the DPUs leave in the parts of the buffer no pixel lives in - positions of the 2x2-padded grid outside
// the image's own, and the unused blocks at the end of the last chunk: zero coefficients, so R = G = B = 128
// (every DPU runs all its blocks whether used or not, src/decoder_dpu.c:130).  One thread = one (position, component).
__global__ void __launch_bounds__(256)
k_ref_mcus_pad(const ImgDev *__restrict__ imgs, uint8_t *__restrict__ out) {
    const ImgDev &im = imgs[blockIdx.y];
    if (!im.valid) return;
    const unsigned W = im.nmx * im.hs, H = im.nmy * im.vs, bpr = (W + 1u) >> 1;
    const unsigned real_blocks = bpr * ((H + 1u) >> 1);
    int16_t *base = reinterpret_cast<int16_t *>(out + im.out_row0);
    const uint4 v128 = make_uint4(0x00800080u, 0x00800080u, 0x00800080u, 0x00800080u);
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < im.ref_blocks * 12u; i += gridDim.x * blockDim.x) {
        const unsigned blk = i / 12u, pc12 = i - blk * 12u, pos = pc12 & 3u, comp = pc12 >> 2;
        if (blk < real_blocks) {
            const unsigned pr = (blk / bpr) * 2u + (pos >> 1), pcx = (blk % bpr) * 2u + (pos & 1u);
            if (pr < H && pcx < W) continue;                            // a real position: the IDCT kernel writes it
        }
        uint4 *d = reinterpret_cast<uint4 *>(base + (size_t)blk * 768 + comp * 256 + pos * 64);
#pragma unroll
        for (int k = 0; k < 8; k++) d[k] = v128;
    }
}

// ------------------------------------------------------------------------------------------------ compat layout
// 16 blocks (= 16 x 3 components x 4 positions = 192 units) of the reference's `mcus` buffer per CTA.
// Unit (blk, comp, pos) sits at blk*768 + comp*256 + pos*64 shorts (src/decoder_dpu.c:134-156).
__global__ void __launch_bounds__(kTileThreads)
k_exec_mcus(const uint32_t *__restrict__ md_all, int16_t *__restrict__ mcus, int nchunk, int blk_per_chunk, int chunk_len) {
    __shared__ uint4 s_t[kTileThreads * 8];
    const int tid = threadIdx.x;
    const int lb = tid / 12, tt = tid - lb * 12, comp = tt >> 2, pos = tt & 3;
    const int blk = blockIdx.x * 16 + lb;
    const int chunk = blk / blk_per_chunk, bi = blk - chunk * blk_per_chunk;
    const bool in_range = chunk < nchunk;
    const uint32_t *md = md_all + (size_t)(in_range ? chunk : 0) * 276;
    // an idle DPU (all-zero record) processes metadata[19]/4 = 0 blocks (src/decoder_dpu.c:130): leave untouched
    const bool active = in_range && bi < (int)(md[19] / 4);
    int16_t *base = mcus + (size_t)(in_range ? chunk : 0) * chunk_len + (size_t)bi * 768;

    if (active) {
        const uint4 *src = reinterpret_cast<const uint4 *>(base + comp * 256 + pos * 64);
        const unsigned ncomp = md[4];
        const bool deq = (unsigned)comp < ncomp;                         // src/decoder_dpu.c:167: only real components
        const uint4 *q4 = reinterpret_cast<const uint4 *>(md + 20 + 64 * (deq ? (md[7 + comp] & 3u) : 0u));
        int X[64];
#pragma unroll
        for (int c = 0; c < 8; c++) {
            const uint4 v = src[c];
            uint4 qa = make_uint4(1, 1, 1, 1), qb = qa;
            if (deq) { qa = __ldg(q4 + 2 * c); qb = __ldg(q4 + 2 * c + 1); }
            X[8 * c + 0] = (int)(v.x * (qa.x << 16)); X[8 * c + 1] = (int)((v.x >> 16) * (qa.y << 16));
            X[8 * c + 2] = (int)(v.y * (qa.z << 16)); X[8 * c + 3] = (int)((v.y >> 16) * (qa.w << 16));
            X[8 * c + 4] = (int)(v.z * (qb.x << 16)); X[8 * c + 5] = (int)((v.z >> 16) * (qb.y << 16));
            X[8 * c + 6] = (int)(v.w * (qb.z << 16)); X[8 * c + 7] = (int)((v.w >> 16) * (qb.w << 16));
        }
        idct8x8(X);
#pragma unroll
        for (int r = 0; r < 8; r++) s_t[tid * 8 + (r ^ (tid & 7))] = pack_row(X, r);
    }
    __syncthreads();

    // colour: item = (block, position, row); all 3 output components of that row
    for (int it = tid; it < 16 * 4 * 8; it += kTileThreads) {
        const int ib = it >> 5, p = (it >> 3) & 3, r = it & 7;
        const int b2 = blockIdx.x * 16 + ib;
        const int ch2 = b2 / blk_per_chunk, bi2 = b2 - ch2 * blk_per_chunk;
        if (ch2 >= nchunk) continue;
        const uint32_t *m2 = md_all + (size_t)ch2 * 276;
        if (bi2 >= (int)(m2[19] / 4)) continue;
        const unsigned vs = m2[5], hs = m2[6];
        int16_t *ob = mcus + (size_t)ch2 * chunk_len + (size_t)bi2 * 768 + p * 64 + r * 8;
        const int u0 = ib * 12;                                            // unit index of (ib, comp 0, pos 0)
        auto row_of = [&](int unit, int row) { return s_t[unit * 8 + (row ^ (unit & 7))]; };
        const uint4 yv = row_of(u0 + p, r);
        if (!((vs == 1 || vs == 2) && (hs == 1 || hs == 2))) {
            // no branch of convert_colorspace matches (src/decoder_dpu.c:332-355): IDCT output stays
            *reinterpret_cast<uint4 *>(ob) = yv;
            *reinterpret_cast<uint4 *>(ob + 256) = row_of(u0 + 4 + p, r);
            *reinterpret_cast<uint4 *>(ob + 512) = row_of(u0 + 8 + p, r);
            continue;
        }
        // which chroma position / quadrant feeds luma position p (src/decoder_dpu.c:332-355)
        int cpos, vq, hq;
        if (vs == 1 && hs == 1) { cpos = p; vq = 0; hq = 0; }
        else if (vs == 2 && hs == 1) { cpos = p & 1; vq = p >> 1; hq = 0; }
        else if (vs == 1 && hs == 2) { cpos = p & 2; vq = 0; hq = p & 1; }
        else { cpos = 0; vq = p >> 1; hq = p & 1; }
        const int rc = (vs == 2 ? (r >> 1) : r) + 4 * vq;                  // src/decoder_dpu.c:370
        const uint4 cbv = row_of(u0 + 4 + cpos, rc), crv = row_of(u0 + 8 + cpos, rc);
        const unsigned cbw[4] = {cbv.x, cbv.y, cbv.z, cbv.w}, crw[4] = {crv.x, crv.y, crv.z, crv.w};
        const unsigned yw[4] = {yv.x, yv.y, yv.z, yv.w};
        int R[8], G[8], B[8];
#pragma unroll
        for (int x = 0; x < 8; x++) {
            const int cx = (hs == 2 ? (x >> 1) : x) + 4 * hq;
            unsigned cbs = 0, crs = 0;
#pragma unroll
            for (int j = 0; j < 4; j++) if ((cx >> 1) == j) { cbs = cbw[j]; crs = crw[j]; }
            const int cb = (cx & 1) ? sext_hi(cbs) : sext_lo(cbs);
            const int cr = (cx & 1) ? sext_hi(crs) : sext_lo(crs);
            const int yy = (x & 1) ? sext_hi(yw[x >> 1]) : sext_lo(yw[x >> 1]);
            const ChromaTerms t = chroma_terms(cb, cr);
            R[x] = clamp255(yy + t.r); G[x] = clamp255(yy + t.g); B[x] = clamp255(yy + t.b);
        }
        *reinterpret_cast<uint4 *>(ob) = make_uint4(R[0] | (R[1] << 16), R[2] | (R[3] << 16), R[4] | (R[5] << 16), R[6] | (R[7] << 16));
        *reinterpret_cast<uint4 *>(ob + 256) = make_uint4(G[0] | (G[1] << 16), G[2] | (G[3] << 16), G[4] | (G[5] << 16), G[6] | (G[7] << 16));
        *reinterpret_cast<uint4 *>(ob + 512) = make_uint4(B[0] | (B[1] << 16), B[2] | (B[3] << 16), B[4] | (B[5] << 16), B[6] | (B[7] << 16));
    }
}

}  // namespace bj
