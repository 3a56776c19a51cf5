// Host-side JPEG container parse on in-memory bytes (product code; SURVEY.md 8f N1).
// Mirrors the validation of the reference's read_JPEG and its segment readers (src/jpeg_scanner.cpp:6-403):
// a file the reference rejects (header->valid = false) is rejected here with BJ_ERR_INVALID_JPEG, at the same
// condition.  Differences by design: works on a byte range instead of one ifstream::get() per byte, keeps the
// quantisation tables in file order, and does NOT copy/un-stuff the scan (that is kernel K0's job) - it only
// locates it.
#pragma once
#include <stdint.h>
#include <string.h>
#include <algorithm>
#include <string>
#include <vector>
#include "../../include/b200jpeg.h"

namespace bj {

struct Cursor {
    const uint8_t *p;
    size_t n, i;
    bool eof;
    // std::ifstream::get() into a `byte`: past the end reads as 0xFF and latches failure
    unsigned get() { if (i >= n) { eof = true; return 0xFF; } return p[i++]; }
    unsigned get16() { unsigned hi = get(); return (hi << 8) + get(); }
};

struct ParseState {
    bool valid = true;
    bool zero_based = false;
    bool used_in_frame[3] = {false, false, false};
};

// src/jpeg_scanner.cpp:187-285
inline void parse_frame(Cursor &c, bj_image_desc &d, ParseState &st) {
    if (d.ncomp != 0) { st.valid = false; return; }                       // "Multiple SOFs detected"
    const unsigned length = c.get16();
    if (c.get() != 8) { st.valid = false; return; }                       // precision
    d.height = c.get16();
    d.width = c.get16();
    if (d.height == 0 || d.width == 0) { st.valid = false; return; }
    d.mcu_h = (d.height + 7) / 8;  d.mcu_w = (d.width + 7) / 8;
    d.mcu_h_real = d.mcu_h;        d.mcu_w_real = d.mcu_w;
    const unsigned nc = c.get();
    if (nc == 4 || nc == 0) { st.valid = false; return; }                 // CMYK / none
    d.ncomp = (uint8_t)nc;
    for (unsigned i = 0; i < nc; i++) {
        unsigned id = c.get();
        if (id == 0 && i == 0) st.zero_based = true;
        if (st.zero_based) id = (id + 1) & 0xFF;
        if (id == 4 || id == 5 || id == 0 || id > nc) { st.valid = false; return; }
        if (st.used_in_frame[id - 1]) { st.valid = false; return; }
        st.used_in_frame[id - 1] = true;
        const unsigned sf = c.get(), h = sf >> 4, v = sf & 15;
        d.comp_h[id - 1] = (uint8_t)h;  d.comp_v[id - 1] = (uint8_t)v;
        if (id == 1) {
            if ((h != 1 && h != 2) || (v != 1 && v != 2)) { st.valid = false; return; }
            if (h == 2 && d.mcu_w % 2 == 1) d.mcu_w_real += 1;
            if (v == 2 && d.mcu_h % 2 == 1) d.mcu_h_real += 1;
            d.hs = (uint8_t)h;  d.vs = (uint8_t)v;
        } else if (h != 1 || v != 1) { st.valid = false; return; }
        const unsigned q = c.get();
        d.qt_id[id - 1] = (uint8_t)q;
        if (q > 3) { st.valid = false; return; }
    }
    if (length - 8 - 3 * nc != 0) st.valid = false;
}

// src/jpeg_scanner.cpp:287-321
inline void parse_dqt(Cursor &c, bj_image_desc &d, ParseState &st) {
    int length = (int)c.get16() - 2;
    while (length > 0) {
        const unsigned info = c.get();
        length -= 1;
        const unsigned id = info & 15;
        if (id > 3) { st.valid = false; return; }
        d.qt_set[id] = 1;
        if (info >> 4) { for (int k = 0; k < 64; k++) d.qt_zz[id][k] = (uint16_t)c.get16(); length -= 128; }
        else           { for (int k = 0; k < 64; k++) d.qt_zz[id][k] = (uint16_t)c.get();   length -= 64; }
        if (c.eof) { st.valid = false; return; }
    }
    if (length != 0) st.valid = false;
}

// src/jpeg_scanner.cpp:140-185
inline void parse_dht(Cursor &c, bj_image_desc &d, ParseState &st) {
    int length = (int)c.get16() - 2;
    while (length > 0) {
        const unsigned info = c.get(), id = info & 15;
        if (id > 3) { st.valid = false; return; }
        const bool ac = (info >> 4) != 0;
        uint8_t *offsets = ac ? d.ac_offsets[id] : d.dc_offsets[id];
        uint8_t *symbols = ac ? d.ac_symbols[id] : d.dc_symbols[id];
        (ac ? d.ac_set : d.dc_set)[id] = 1;
        offsets[0] = 0;
        unsigned total = 0;
        for (int l = 1; l <= 16; l++) { total += c.get(); offsets[l] = (uint8_t)total; }
        if (total > 162) { st.valid = false; return; }
        for (unsigned k = 0; k < total; k++) symbols[k] = (uint8_t)c.get();
        length -= 17 + (int)total;
        if (c.eof) { st.valid = false; return; }
    }
    if (length != 0) st.valid = false;
}

// src/jpeg_scanner.cpp:6-138
inline void parse_scan_header(Cursor &c, bj_image_desc &d, ParseState &st) {
    if (d.ncomp == 0) { st.valid = false; return; }                       // "SOS detected before SOF"
    const unsigned length = c.get16();
    bool in_scan[3] = {false, false, false};
    const unsigned ns = c.get();
    if (ns == 0) { st.valid = false; return; }
    d.scan_ncomp = (uint8_t)ns;
    for (unsigned i = 0; i < ns; i++) {
        unsigned id = c.get();
        if (st.zero_based) id = (id + 1) & 0xFF;
        if (id == 0 || id > d.ncomp) { st.valid = false; return; }
        if (!st.used_in_frame[id - 1] || in_scan[id - 1]) { st.valid = false; return; }
        in_scan[id - 1] = true;
        const unsigned t = c.get();
        d.dc_id[id - 1] = (uint8_t)(t >> 4);  d.ac_id[id - 1] = (uint8_t)(t & 15);
        if ((t >> 4) > 3 || (t & 15) > 3) { st.valid = false; return; }
    }
    const unsigned ss = c.get(), se = c.get(), ahal = c.get();
    if (d.frame_type == 0xC0 && (ss != 0 || se != 63 || ahal != 0)) { st.valid = false; return; }
    if (d.frame_type == 0xC2) {                                           // :79-106 (progressive is never decoded)
        const unsigned ah = ahal >> 4, al = ahal & 15;
        if (ss > se || se > 63 || (ss == 0 && se != 0) || (ss != 0 && ns != 1) || (ah != 0 && al != ah - 1)) { st.valid = false; return; }
    }
    for (unsigned i = 0; i < d.ncomp; i++) {
        if (!in_scan[i]) continue;
        if (!d.qt_set[d.qt_id[i]]) { st.valid = false; return; }
        if (ss == 0 && !d.dc_set[d.dc_id[i]]) { st.valid = false; return; }
        if (se > 0 && !d.ac_set[d.ac_id[i]]) { st.valid = false; return; }
    }
    if (length - 6 - 2 * ns != 0) st.valid = false;
}

inline void parse_dri(Cursor &c, bj_image_desc &d, ParseState &st) {
    const unsigned l = c.get16();
    d.restart_interval = c.get16();
    if (l != 4) st.valid = false;
}

inline void skip_segment(Cursor &c) {
    const unsigned length = c.get16();
    if (length >= 2) { const size_t adv = length - 2; if (c.i + adv > c.n) { c.i = c.n; c.eof = true; } else c.i += adv; }
}

// Locate the end of the entropy-coded segment (src/jpeg_scanner.cpp:405-433): the first FF that is followed by
// something other than 00 / RSTn / FF.  scan_extent: false if the file ends first; *end = that FF's position, and
// `rst` (if given) receives the positions of the RSTn markers on the way.
inline bool scan_extent(const uint8_t *p, size_t n, size_t start, size_t *end, std::vector<size_t> *rst = nullptr) {
    size_t i = start;
    for (;;) {
        if (i >= n) return false;
        const uint8_t *f = (const uint8_t *)memchr(p + i, 0xFF, n - i);
        if (!f) return false;
        i = (size_t)(f - p);
        if (i + 1 >= n) return false;
        const unsigned m = p[i + 1];
        if (m == 0x00) { i += 2; continue; }
        if (m >= 0xD0 && m <= 0xD7) { if (rst) rst->push_back(i); i += 2; continue; }
        if (m == 0xFF) { i += 1; continue; }
        *end = i;
        return true;
    }
}
// EOI ends the scan; anything else makes the file invalid ("File ended prematurely", "Invalid marker during
// compressed data scan").  Only bj_parse_header (the public, stand-alone restatement of read_JPEG) walks the scan like
// this; the baseline decode path leaves it to the GPU (kernels_huff.cuh: k_unstuff applies the same rule).
inline int find_scan_end(const uint8_t *p, size_t n, size_t start, size_t *end) {
    if (!scan_extent(p, n, start, end)) return BJ_ERR_INVALID_JPEG;
    return p[*end + 1] == 0xD9 ? BJ_OK : BJ_ERR_INVALID_JPEG;
}

// walk_scan = false (the decode path): only the headers are read (a few hundred bytes); scan_len is then an UPPER
// BOUND - everything up to the end of the file - and whether the scan ends properly is decided on the device.
inline int parse_header(const uint8_t *file, size_t len, bj_image_desc *out, bool walk_scan = true) {
    bj_image_desc &d = *out;
    memset(&d, 0, sizeof(d));
    d.hs = d.vs = 1;
    for (int i = 0; i < 3; i++) d.comp_h[i] = d.comp_v[i] = 1;
    Cursor c{file, len, 0, false};
    ParseState st;
    unsigned last = c.get(), cur = c.get();
    if (last != 0xFF || cur != 0xD8) return BJ_ERR_INVALID_JPEG;
    last = c.get();  cur = c.get();
    bool sos = false;
    while (st.valid) {                                                    // src/jpeg_scanner.cpp:371-403
        if (c.eof || last != 0xFF) return BJ_ERR_INVALID_JPEG;
        if (cur == 0xC0 || cur == 0xC2) { d.frame_type = (uint8_t)cur; parse_frame(c, d, st); }
        else if (cur == 0xDB) parse_dqt(c, d, st);
        else if (cur == 0xC4) parse_dht(c, d, st);
        else if (cur == 0xDA) { parse_scan_header(c, d, st); sos = true; break; }
        else if (cur == 0xDD) parse_dri(c, d, st);
        else if ((cur >= 0xE0 && cur <= 0xEF) || cur == 0xFE || (cur >= 0xF0 && cur <= 0xFD) || cur == 0xDC || cur == 0xDE || cur == 0xDF) skip_segment(c);
        else if (cur == 0x01) {}
        else if (cur == 0xFF) { cur = c.get(); continue; }
        // unknown marker: the reference prints a message and carries on (:399)
        last = c.get();  cur = c.get();
    }
    if (!st.valid || !sos || c.eof) return BJ_ERR_INVALID_JPEG;
    d.scan_off = c.i;
    if (walk_scan) {
        size_t end = 0;
        const int rc = find_scan_end(file, len, c.i, &end);
        if (rc != BJ_OK) return rc;
        d.scan_len = end - c.i;
    } else {
        if (c.i >= len) return BJ_ERR_INVALID_JPEG;                        // "File ended prematurely"
        d.scan_len = len - c.i;
    }
    if (d.frame_type != 0xC0) return BJ_ERR_UNSUPPORTED;                  // SOF2: parsed, never decodable (SURVEY 2)
    if (d.scan_ncomp != d.ncomp) return BJ_ERR_UNSUPPORTED;               // non-interleaved scans: reference output is garbage
    return BJ_OK;
}

// ------------------------------------------------------------------------------------------------ progressive files
// The multi-scan walk of an SOF2 file (context option "progressive"): marker by marker to EOI, through every scan.  The
// header segments go through the same readers as above; this is the one place where the host reads entropy-coded
// bytes - scan_extent's memchr for FF - to find where each scan and each of its restart segments lies.
constexpr int kProgMaxScans = 64;

struct ProgScan {
    uint8_t ncomp;               // components in the scan (1 for an AC scan)
    uint8_t comp[3];             // their indices (frame id - 1), in scan order
    uint8_t ss, se, ah, al;
    uint8_t level;               // 1 + the highest level of an earlier scan that touches a coefficient of this one
    uint32_t ri;                 // restart interval: MCUs of an interleaved scan, blocks of a single-component one; 0 none
    std::string dc[3], ac;       // the Huffman tables the scan uses (17 offsets + symbols, as parse_dht keeps them)
    size_t off, end;             // entropy-coded bytes [off, end): end = the FF of the marker that ends the scan
    std::vector<size_t> rst;     // positions of the RSTn markers inside
};

inline std::string huff_key(const uint8_t off[17], const uint8_t *sym) {
    std::string k((const char *)off, 17);
    k.append((const char *)sym, off[16] > 162 ? 162 : off[16]);
    return k;
}

// Returns BJ_OK with *out filled as bj_peek_header fills it (first scan's header fields) and `scans` the scan list, or
// BJ_ERR_INVALID_JPEG for a structural error (no EOI, a marker that may not follow a scan, the T.81 G.1.1.1 rules, an AC
// scan before its component's first DC scan, a refinement of a band with no first pass (or whose Ah is not the band's
// last Al), a first pass of a band that already had one, a table never defined), or BJ_ERR_UNSUPPORTED for more than
// kProgMaxScans scans or a DQT behind the first scan that changes a table a frame component uses.
inline int parse_progressive(const uint8_t *file, size_t len, bj_image_desc *out, std::vector<ProgScan> *scans) {
    bj_image_desc &d = *out;
    memset(&d, 0, sizeof(d));
    d.hs = d.vs = 1;
    for (int i = 0; i < 3; i++) d.comp_h[i] = d.comp_v[i] = 1;
    scans->clear();
    Cursor c{file, len, 0, false};
    ParseState st;
    unsigned last = c.get(), cur = c.get();
    if (last != 0xFF || cur != 0xD8) return BJ_ERR_INVALID_JPEG;
    last = c.get();  cur = c.get();
    int8_t bits[3][64];          // per component and coefficient: Al of the last scan that coded it, -1 none yet
    uint8_t level[3][64];        // ... and that scan's level
    memset(bits, -1, sizeof(bits));
    memset(level, 0, sizeof(level));
    for (;;) {
        if (!st.valid || c.eof || last != 0xFF) return BJ_ERR_INVALID_JPEG;
        const bool after_scan = !scans->empty();
        if (cur == 0xD9) break;
        if (cur == 0xC2 && !after_scan) { d.frame_type = 0xC2; parse_frame(c, d, st); }
        else if (cur == 0xDB) {
            uint16_t qt[4][64];
            uint8_t set[4];
            memcpy(qt, d.qt_zz, sizeof(qt)); memcpy(set, d.qt_set, sizeof(set));
            parse_dqt(c, d, st);
            for (int j = 0; st.valid && after_scan && j < d.ncomp; j++) {
                const int t = d.qt_id[j] & 3;
                if (set[t] && memcmp(qt[t], d.qt_zz[t], sizeof(qt[t]))) return BJ_ERR_UNSUPPORTED;
            }
        }
        else if (cur == 0xC4) parse_dht(c, d, st);
        else if (cur == 0xDD) parse_dri(c, d, st);
        else if (cur == 0xDA) {
            if (d.frame_type != 0xC2) return BJ_ERR_INVALID_JPEG;
            const size_t h0 = c.i;
            parse_scan_header(c, d, st);
            if (!st.valid || c.eof) return BJ_ERR_INVALID_JPEG;
            if ((int)scans->size() == kProgMaxScans) return BJ_ERR_UNSUPPORTED;
            ProgScan s;
            // the header parse_scan_header accepted: length, Ns, Ns x (id, tables), Ss, Se, Ah/Al
            const uint8_t *h = file + h0;
            s.ncomp = h[2];
            for (unsigned i = 0; i < s.ncomp; i++) s.comp[i] = (uint8_t)(((h[3 + 2 * i] + (st.zero_based ? 1u : 0u)) & 0xFF) - 1u);
            s.ss = h[3 + 2 * s.ncomp]; s.se = h[4 + 2 * s.ncomp]; s.ah = h[5 + 2 * s.ncomp] >> 4; s.al = h[5 + 2 * s.ncomp] & 15;
            if (s.al > 13) return BJ_ERR_INVALID_JPEG;                    // (8-bit data: coefficients have at most 11 + 3 bits)
            s.ri = d.restart_interval;
            int lv = 0;
            for (unsigned i = 0; i < s.ncomp; i++) {
                const int j = s.comp[i];
                if (s.ss > 0 && bits[j][0] < 0) return BJ_ERR_INVALID_JPEG;          // AC before the component's first DC scan
                for (int k = s.ss; k <= s.se; k++) {
                    if (s.ah == 0 ? bits[j][k] >= 0 : bits[j][k] != (int)s.ah) return BJ_ERR_INVALID_JPEG;
                    lv = std::max<int>(lv, level[j][k]);
                }
                s.dc[i] = huff_key(d.dc_offsets[d.dc_id[j]], d.dc_symbols[d.dc_id[j]]);
                if (s.se > 0) s.ac = huff_key(d.ac_offsets[d.ac_id[j]], d.ac_symbols[d.ac_id[j]]);
            }
            s.level = (uint8_t)(lv + 1);
            for (unsigned i = 0; i < s.ncomp; i++)
                for (int k = s.ss; k <= s.se; k++) { bits[s.comp[i]][k] = (int8_t)s.al; level[s.comp[i]][k] = s.level; }
            if (scans->empty()) { d.scan_off = c.i; d.scan_len = len - c.i; }
            s.off = c.i;
            if (!scan_extent(file, len, c.i, &s.end, &s.rst)) return BJ_ERR_INVALID_JPEG;   // no EOI
            c.i = s.end;
            const unsigned m = file[s.end + 1];                            // what may follow a scan
            if (!(m == 0xD9 || m == 0xDA || m == 0xC4 || m == 0xDB || m == 0xDD || m == 0xFE || (m >= 0xE0 && m <= 0xEF))) return BJ_ERR_INVALID_JPEG;
            scans->push_back(std::move(s));
        }
        else if ((cur >= 0xE0 && cur <= 0xEF) || cur == 0xFE) skip_segment(c);
        else if (cur == 0xFF) { cur = c.get(); continue; }
        else return BJ_ERR_INVALID_JPEG;                                   // another frame, SOI, DNL, ... inside the file
        last = c.get();  cur = c.get();
    }
    if (scans->empty() || d.ncomp == 0) return BJ_ERR_INVALID_JPEG;
    return BJ_OK;
}

}  // namespace bj
