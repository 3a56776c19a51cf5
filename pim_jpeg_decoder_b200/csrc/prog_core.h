// Entropy decode of progressive (SOF2) scans, shared by the CUDA kernel (kernels_prog.cuh) and by the host-side
// emulation used in the CPU tests (tests/emu/prog_emu.cpp).  Plain integer code that compiles both as device and as
// host code; the library has no CPU decode path - the host build exists only so the decode can be checked without a GPU.
//
// One WORK ITEM is one restart segment of one scan of one image, decoded sequentially by one thread: a bit reader over
// the stuffed bytes of the file, DC first pass (the item's own prediction) and refinement, AC first pass with EOBRUN,
// AC refinement with correction bits (the decoding procedures of T.81 G.2).  Coefficients land where the
// baseline entropy stage puts them: AC in zig-zag order in the image's units (slot 0 unused), DC in the DC plane, both
// in MCU-interleaved unit order, so the IDCT + colour kernel reads a progressive image exactly like a baseline one.
#pragma once
#include <stdint.h>
#include <string.h>

#ifdef __CUDACC__
#define BJ_PHD __host__ __device__ __forceinline__
#else
#define BJ_PHD inline
#endif

namespace bj {

// One Huffman table: codes of up to 8 bits by one lookup, longer ones by the canonical code ranges (T.81 F.2.2.3).
struct ProgHuff {
    uint16_t look[256];          // (length << 8) | symbol for a code of <= 8 bits that the top 8 bits start with; 0 none
    int32_t maxcode[17];         // per length 9..16: largest code of that length, -1 none
    int32_t valoff[17];          // symbol of code x of length l: val[x + valoff[l]]
    uint8_t val[256];
    uint32_t pad_[2];
};
static_assert(sizeof(ProgHuff) % 16 == 0, "tables are pooled in 16-byte units");

// Host: the table of parse_dht's offsets / symbols (17 + n bytes, parse.h: huff_key).  Codes that do not fit their
// length (an over-subscribed table) never match.
inline void build_prog_huff(const uint8_t *key, size_t key_len, ProgHuff *t) {
    memset(t, 0, sizeof(*t));
    const uint8_t *off = key, *sym = key + 17;
    const unsigned nsym = (unsigned)(key_len - 17);
    for (int l = 0; l < 17; l++) t->maxcode[l] = -1;
    for (unsigned k = 0; k < nsym && k < 256; k++) t->val[k] = sym[k];
    uint32_t code = 0;
    for (int l = 1; l <= 16; l++) {
        const unsigned j0 = off[l - 1], j1 = off[l] < nsym ? off[l] : nsym;
        for (unsigned j = j0; j < j1; j++, code++) {
            if (code >> l) continue;
            if (l <= 8) {
                const uint32_t first = code << (8 - l), cnt = 1u << (8 - l);
                for (uint32_t i = 0; i < cnt; i++) if (!t->look[first + i]) t->look[first + i] = (uint16_t)((l << 8) | sym[j]);
            } else {
                if (t->maxcode[l] < 0) t->valoff[l] = (int32_t)j - (int32_t)code;
                t->maxcode[l] = (int32_t)code;
            }
        }
        code <<= 1;
    }
}

// Per progressive image of a batch.
struct ProgImgDev {
    uint32_t img;                // index of the image in the batch (its HuffImgState)
    uint32_t du_base;            // first unit in the coefficient buffer / DC plane
    uint64_t file_off;           // where the file lies in the batch's file buffer
    uint32_t nmx, nmcu;          // MCUs per row, in all
    uint8_t bpm, ny, hs, vs;     // units per MCU, luma units per MCU, luma sampling
    uint16_t bw[3], bh[3];       // block grid of each component: ceil(Xi / 8) x ceil(Yi / 8)
};

// Per scan: what it codes and where its segments are.
struct ProgScanDev {
    uint32_t pimg;               // its ProgImgDev
    uint32_t seg0, nseg;         // its restart segments: entries [seg0, seg0 + nseg) of the segment table
    uint32_t ri;                 // restart interval (MCUs if interleaved, blocks otherwise); 0: one segment
    uint32_t dc_tab[3], ac_tab;  // pool index of the table of each scan component's DC / of the AC table
    uint8_t ncomp, comp[3];      // components in scan order (frame index)
    uint8_t ss, se, ah, al;
    uint8_t bad;                 // 1: the number of RSTn markers is not the number the restart interval implies
    uint8_t pad_[3];
};

// A segment: its stuffed entropy-coded bytes [lo, hi) relative to the file's first byte.  hi is the FF of the marker
// that ends it (RSTn or the scan's end); a segment that has no marker in the file is empty.
struct ProgSeg {
    uint32_t lo, hi;
};

// ------------------------------------------------------------------------------------------------ bit reader
// Reads the stuffed bytes as they are in the file: FF 00 is a data FF, FF FF a fill byte, FF RSTn (only inside a
// scan without a restart interval, or past the expected markers) is skipped, like the baseline path's un-stuffing.
// Past the segment's end it supplies zeros and remembers that it did: a symbol that takes one of them is damage.
struct ProgBits {
    const uint8_t *p;
    uint32_t q, end;             // next byte, end of the segment
    uint64_t acc;                // bits, MSB first
    int32_t nb;                  // bits in acc
    int32_t real;                // ... of them from the segment (the rest are the zeros behind its end)
    BJ_PHD void open(const uint8_t *file, uint32_t lo, uint32_t hi) { p = file; q = lo; end = hi; acc = 0; nb = 0; real = 0; }
    BJ_PHD void fill() {
        while (nb <= 56) {
            uint32_t b = 0;
            if (q < end) {
                b = p[q];
                if (b == 0xFFu) {
                    const uint32_t m = p[q + 1];
                    if (m != 0x00u) { q += m == 0xFFu ? 1u : 2u; continue; }        // fill byte / RSTn
                    q += 2;
                } else q++;
                real += 8;
            }
            acc |= (uint64_t)b << (56 - nb);
            nb += 8;
        }
    }
    BJ_PHD uint32_t peek16() { fill(); return (uint32_t)(acc >> 48); }
    // false: the bits run past the segment's data
    BJ_PHD bool skip(uint32_t n) { acc <<= n; nb -= (int32_t)n; real -= (int32_t)n; return real >= 0; }
    BJ_PHD bool get(uint32_t n, uint32_t &v) {         // n <= 16
        fill();
        v = n ? (uint32_t)(acc >> (64 - n)) : 0u;
        return skip(n);
    }
    // one Huffman symbol; -1: no such code, or the code runs past the data
    BJ_PHD int32_t symbol(const ProgHuff &t) {
        const uint32_t w = peek16();
        const uint32_t e = t.look[w >> 8];
        if (e) return skip(e >> 8) ? (int32_t)(e & 0xFFu) : -1;
        for (uint32_t l = 9; l <= 16; l++) {
            const int32_t x = (int32_t)(w >> (16 - l));
            if (x <= t.maxcode[l]) return skip(l) ? (int32_t)t.val[(x + t.valoff[l]) & 0xFF] : -1;
        }
        return -1;
    }
};

BJ_PHD int32_t prog_extend(uint32_t v, uint32_t s) { return (s && v < (1u << (s - 1))) ? (int32_t)v - (int32_t)(1u << s) + 1 : (int32_t)v; }

// ------------------------------------------------------------------------------------------------ one work item
// Blocks [b0, b1) of the scan (MCUs of an interleaved scan, blocks of the component's grid in raster order otherwise)
// from the segment's bytes.  `coef` / `dc` are the batch's coefficient buffer and DC plane.  Returns 0, or 1 when the
// item met damaged data (a code not in the table, a DC category above 11 or an AC size above 10, a run past Se, bits past
// the segment's end): it stops there, what it stored before stays.  Every loop is bounded by (b1 - b0) x 64 steps
// whatever EOBRUN the data claims.
struct ProgUnitOf {
    const ProgImgDev &im;
    // unit of block (bx, by) of component j
    BJ_PHD uint32_t operator()(uint32_t j, uint32_t bx, uint32_t by) const {
        const uint32_t h = j ? 1u : im.hs, v = j ? 1u : im.vs;
        const uint32_t m = (by / v) * im.nmx + bx / h;
        const uint32_t u = j ? im.ny + j - 1u : (by % v) * h + bx % h;
        return im.du_base + m * im.bpm + u;
    }
};

BJ_PHD uint32_t prog_decode_item(const ProgScanDev &sc, const ProgImgDev &im, const ProgHuff *tabs, const uint8_t *file,
                                 const ProgSeg &seg, uint32_t b0, uint32_t b1, int16_t *coef, int16_t *dc) {
    ProgBits br;
    br.open(file, seg.lo, seg.hi);
    const ProgUnitOf unit_of{im};
    const bool interleaved = sc.ncomp > 1;
    const uint32_t ss = sc.ss, se = sc.se, al = sc.al;
    int32_t pred[3] = {0, 0, 0};
    uint32_t eobrun = 0;
    const ProgHuff *ac = sc.se ? &tabs[sc.ac_tab] : nullptr;
    for (uint32_t b = b0; b < b1; b++) {
        // the units this block / MCU holds, in scan order
        uint32_t units[6], ucomp[6], nu = 0;
        if (interleaved) {
            const uint32_t mx = b % im.nmx, my = b / im.nmx;
            for (uint32_t i = 0; i < sc.ncomp; i++) {
                const uint32_t j = sc.comp[i], h = j ? 1u : im.hs, v = j ? 1u : im.vs;
                for (uint32_t y = 0; y < v; y++)
                    for (uint32_t x = 0; x < h; x++) { units[nu] = unit_of(j, mx * h + x, my * v + y); ucomp[nu++] = i; }
            }
        } else {
            const uint32_t j = sc.comp[0], bw = im.bw[j];
            units[0] = unit_of(j, b % bw, b / bw); ucomp[0] = 0; nu = 1;
        }
        for (uint32_t n = 0; n < nu; n++) {
            const uint32_t u = units[n];
            int16_t *zz = coef + (size_t)u * 64;
            if (ss == 0) {
                if (sc.ah == 0) {                                       // DC first pass
                    const int32_t s = br.symbol(tabs[sc.dc_tab[ucomp[n]]]);
                    uint32_t v;
                    if (s < 0 || s > 11 || !br.get((uint32_t)s, v)) return 1u;
                    pred[ucomp[n]] += prog_extend(v, (uint32_t)s);
                    dc[u] = (int16_t)(uint16_t)((uint32_t)pred[ucomp[n]] << al);
                } else {                                                // DC refinement: one bit
                    uint32_t v;
                    if (!br.get(1, v)) return 1u;
                    if (v) dc[u] = (int16_t)(uint16_t)((uint16_t)dc[u] | (1u << al));
                }
                continue;
            }
            if (sc.ah == 0) {                                           // AC first pass
                if (eobrun) { eobrun--; continue; }
                for (uint32_t k = ss; k <= se; k++) {
                    const int32_t rs = br.symbol(*ac);
                    if (rs < 0) return 1u;
                    const uint32_t r = (uint32_t)rs >> 4, s = (uint32_t)rs & 15u;
                    if (s) {
                        k += r;
                        uint32_t v;
                        if (k > se || s > 10 || !br.get(s, v)) return 1u;
                        zz[k] = (int16_t)(prog_extend(v, s) * (1 << al));
                    } else if (r == 15) {
                        k += 15;
                        if (k > se) return 1u;
                    } else {
                        uint32_t v = 0;
                        if (r && !br.get(r, v)) return 1u;
                        eobrun = (1u << r) + v - 1u;
                        break;
                    }
                }
                continue;
            }
            // AC refinement
            const int32_t p1 = 1 << al, m1 = -p1;
            uint32_t k = ss;
            if (!eobrun) {
                for (; k <= se; k++) {
                    const int32_t rs = br.symbol(*ac);
                    if (rs < 0) return 1u;
                    int32_t r = rs >> 4, s = rs & 15, nv = 0;
                    if (s) {
                        uint32_t v;
                        if (s != 1 || !br.get(1, v)) return 1u;
                        nv = v ? p1 : m1;
                    } else if (r != 15) {
                        uint32_t v = 0;
                        if (r && !br.get((uint32_t)r, v)) return 1u;
                        eobrun = (1u << r) + v;
                        break;
                    }
                    // skip r zero-history coefficients (correction bits for the non-zero ones on the way), land on the next zero
                    bool placed = false;
                    for (; k <= se; k++) {
                        const int32_t c = zz[k];
                        if (c) {
                            uint32_t v;
                            if (!br.get(1, v)) return 1u;
                            if (v && (c & p1) == 0) zz[k] = (int16_t)(c >= 0 ? c + p1 : c + m1);
                        } else if (--r < 0) { placed = true; break; }
                    }
                    if (!placed) return 1u;                             // a run past Se
                    if (nv) zz[k] = (int16_t)nv;
                }
            }
            if (eobrun) {                                               // the block is inside an end-of-band run
                for (; k <= se; k++) {
                    const int32_t c = zz[k];
                    if (c) {
                        uint32_t v;
                        if (!br.get(1, v)) return 1u;
                        if (v && (c & p1) == 0) zz[k] = (int16_t)(c >= 0 ? c + p1 : c + m1);
                    }
                }
                eobrun--;
            }
        }
    }
    return 0u;
}

// Blocks (or MCUs) of a scan and the range segment k of it covers.
BJ_PHD uint32_t prog_scan_blocks(const ProgScanDev &sc, const ProgImgDev &im) {
    return sc.ncomp > 1 ? im.nmcu : (uint32_t)im.bw[sc.comp[0]] * im.bh[sc.comp[0]];
}
BJ_PHD void prog_seg_blocks(const ProgScanDev &sc, const ProgImgDev &im, uint32_t k, uint32_t &b0, uint32_t &b1) {
    const uint32_t nb = prog_scan_blocks(sc, im);
    if (!sc.ri) { b0 = 0; b1 = nb; return; }
    b0 = k * sc.ri;
    b1 = nb - b0 < sc.ri ? nb : b0 + sc.ri;
}

}  // namespace bj
