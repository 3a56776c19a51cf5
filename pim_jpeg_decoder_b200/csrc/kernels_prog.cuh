// Progressive (SOF2) entropy stage on sm_100a (context option "progressive").  The host's multi-scan walk
// (parse.h: parse_progressive) gives every scan a LEVEL: scans of one level write disjoint coefficients.  Per batch:
//
//   k_prog_zero_dc     the DC plane of every progressive image is cleared (its units are cleared by k_zero_tail: a
//                      progressive image has first_zero = 0)
//   k_prog_decode      one launch per level over every work item of that level in the batch: one thread decodes one
//                      restart segment of one scan sequentially (prog_core.h: prog_decode_item)
//
// The thread finds its item by a binary search of the level's per-scan prefix of segment counts, so the host lays out
// O(images + scans) records, not one per item.
#pragma once
#include "bj_dev.h"
#include "kernels_huff.cuh"
#include "prog_core.h"

namespace bj {

constexpr int kProgThreads = 128;

__global__ void __launch_bounds__(256)
k_prog_zero_dc(const ProgImgDev *__restrict__ pimgs, int16_t *__restrict__ dc) {
    const ProgImgDev &im = pimgs[blockIdx.x];
    const uint32_t n = im.nmcu * im.bpm;
    for (uint32_t u = threadIdx.x; u < n; u += blockDim.x) dc[im.du_base + u] = 0;
}

// lvl_scans[0, nscans): the scans of this level; lvl_item0: exclusive prefix of their segment counts; nitems in all.
__global__ void __launch_bounds__(kProgThreads)
k_prog_decode(const ProgImgDev *__restrict__ pimgs, const ProgScanDev *__restrict__ scans, const ProgSeg *__restrict__ segs,
              const ProgHuff *__restrict__ tabs, const uint32_t *__restrict__ lvl_scans, const uint32_t *__restrict__ lvl_item0,
              uint32_t nscans, uint32_t nitems, const uint8_t *__restrict__ files, HuffImgState *__restrict__ st,
              int16_t *__restrict__ coef, int16_t *__restrict__ dc) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nitems) return;
    uint32_t lo = 0, hi = nscans;                                          // last j with lvl_item0[j] <= t
    while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (lvl_item0[mid] <= t) lo = mid; else hi = mid; }
    const ProgScanDev sc = scans[lvl_scans[lo]];
    const ProgImgDev im = pimgs[sc.pimg];
    const uint32_t k = t - lvl_item0[lo];
    uint32_t b0, b1;
    prog_seg_blocks(sc, im, k, b0, b1);
    uint32_t bad = (k == 0 && sc.bad) ? 1u : 0u;
    bad |= prog_decode_item(sc, im, tabs, files + im.file_off, segs[sc.seg0 + k], b0, b1, coef, dc);
    if (bad) st[im.img].status = 1u;
}

}  // namespace bj
