// TEST INFRASTRUCTURE - host-side emulation of the progressive entropy stage (kernels_prog.cuh).
//
// Compiles the product's shared code (pim_jpeg_decoder_b200/csrc/parse.h: parse_progressive, prog_core.h) with g++ and
// runs what the kernels run: every scan's restart segments as work items, level by level, each decoded by
// prog_decode_item into a coefficient buffer and a DC plane in MCU-interleaved unit order.  It is NOT linked into
// libb200jpeg.so and is only loaded by tests/test_progressive_emu.py.
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <vector>

#include "../../pim_jpeg_decoder_b200/csrc/parse.h"
#include "../../pim_jpeg_decoder_b200/csrc/prog_core.h"

using namespace bj;

// coef: ndu * 64 shorts, zig-zag, DC in slot 0 (as the oracle's coef_zz).  info[0] = scans, info[1] = levels,
// info[2] = work items, info[3] = 1 if an item met damaged data.  Returns parse_progressive's status.
extern "C" int emu_prog_decode(const uint8_t *file, size_t len, int16_t *coef, size_t coef_units, uint32_t *info) {
    bj_image_desc d;
    std::vector<ProgScan> scans;
    const int rc = parse_progressive(file, len, &d, &scans);
    if (rc != BJ_OK) return rc;
    ProgImgDev im{};
    const uint32_t mcu_w = (d.width + 7) / 8, mcu_h = (d.height + 7) / 8;
    im.nmx = (mcu_w + d.hs - 1) / d.hs;
    im.nmcu = im.nmx * ((mcu_h + d.vs - 1) / d.vs);
    im.hs = d.hs; im.vs = d.vs; im.ny = (uint8_t)(d.hs * d.vs);
    im.bpm = (uint8_t)(im.ny + d.ncomp - 1);
    for (int j = 0; j < d.ncomp; j++) {
        const uint32_t h = j ? 1u : d.hs, v = j ? 1u : d.vs;
        im.bw[j] = (uint16_t)(((d.width * h + d.hs - 1) / d.hs + 7) / 8);
        im.bh[j] = (uint16_t)(((d.height * v + d.vs - 1) / d.vs + 7) / 8);
    }
    if ((size_t)im.nmcu * im.bpm > coef_units) return BJ_ERR_ARG;
    std::vector<int16_t> ac((size_t)im.nmcu * im.bpm * 64, 0), dc((size_t)im.nmcu * im.bpm, 0);
    std::vector<ProgHuff> tabs;
    std::map<std::string, uint32_t> idx;
    auto table = [&](const std::string &k) -> uint32_t {
        auto it = idx.find(k);
        if (it != idx.end()) return it->second;
        tabs.emplace_back();
        build_prog_huff((const uint8_t *)k.data(), k.size(), &tabs.back());
        return idx[k] = (uint32_t)tabs.size() - 1;
    };
    uint32_t levels = 0, items = 0, bad = 0;
    for (const ProgScan &s : scans) levels = std::max<uint32_t>(levels, s.level);
    for (uint32_t L = 1; L <= levels; L++) {
        for (const ProgScan &ps : scans) {
            if (ps.level != L) continue;
            ProgScanDev sc{};
            sc.ncomp = ps.ncomp; sc.ss = ps.ss; sc.se = ps.se; sc.ah = ps.ah; sc.al = ps.al; sc.ri = ps.ri;
            for (int j = 0; j < ps.ncomp; j++) { sc.comp[j] = ps.comp[j]; if (ps.ss == 0 && ps.ah == 0) sc.dc_tab[j] = table(ps.dc[j]); }
            if (ps.se) sc.ac_tab = table(ps.ac);
            const uint32_t nb = prog_scan_blocks(sc, im);
            sc.nseg = ps.ri ? (nb + ps.ri - 1) / ps.ri : 1u;
            const size_t R = ps.rst.size();
            if (ps.ri && R + 1 != sc.nseg) bad = 1;
            for (uint32_t k = 0; k < sc.nseg; k++) {
                const size_t lo = k == 0 ? ps.off : (k - 1 < R ? ps.rst[k - 1] + 2 : ps.end);
                const size_t hi = k + 1 == sc.nseg ? ps.end : (k < R ? ps.rst[k] : ps.end);
                ProgSeg seg{(uint32_t)lo, (uint32_t)std::max(lo, hi)};
                uint32_t b0, b1;
                prog_seg_blocks(sc, im, k, b0, b1);
                bad |= prog_decode_item(sc, im, tabs.data(), file, seg, b0, b1, ac.data(), dc.data());
                items++;
            }
        }
    }
    for (size_t u = 0; u < dc.size(); u++) { memcpy(coef + u * 64, &ac[u * 64], 128); coef[u * 64] = dc[u]; }
    info[0] = (uint32_t)scans.size(); info[1] = levels; info[2] = items; info[3] = bad;
    return BJ_OK;
}
