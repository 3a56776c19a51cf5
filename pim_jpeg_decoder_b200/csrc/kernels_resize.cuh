// Fixed-size output: bilinear resize of each resized image's scaled crop to its target size.  sm_100a.
//
//   k_resize_bilinear : runs behind k_idct_color, only when some image of the batch has a target size.  Its source is
//                       the RGB8 scaled crop that k_idct_color wrote into the intermediate region of the output buffer;
//                       its output is the final image in the batch's format, written by the same tile_copy_out as the
//                       IDCT + colour kernel's.
#pragma once
#include "bj_dev.h"
#include "kernels_idct.cuh"

namespace bj {

// Source pixels of one staged row: the span of a tile's column taps when the resize reduces by at most 2x
// (resize_plan keeps it there).  A wider span - a stronger reduction - reads its taps from global memory instead.
constexpr int kResizeSpan = 2 * kResizeTileW + 2;

// taps(n_src, n_dst, X) of include/b200jpeg.h: the source index i0 and the weight f in [0, 255] of i0 + 1, from the
// half-pixel-centre position (2X + 1) n_src / (2 n_dst) - 1/2, clamped at 0.  num is up to 2^17 * 2^16: 64 bits.
__device__ __forceinline__ void resize_tap(const uint32_t n_src, const uint32_t n_dst, const uint32_t X, uint32_t *i0, uint32_t *f) {
    const long long num = max((2LL * X + 1) * n_src - (long long)n_dst, 0LL), den = 2LL * n_dst;
    const long long q = num / den;
    *i0 = (uint32_t)q;
    *f = (uint32_t)(((num - q * den) * 256) / den);
}

// One CTA = one output tile of kResizeTileW x kResizeTileH pixels of one resized image.  The shape: a warp's 32 lanes
// take two columns each, so a tile row is 192 bytes, 12 whole 16-byte chunks for the copy-out; 48 rows are eight per
// warp of the kTileThreads-wide CTA that tile_copy_out's row loop is written for.  Each CTA pays a fixed latency (the
// image search, the tap divisions, two barriers), which 48 rows amortise over twice the pixels of 24 (measured: 24 rows
// took 2.04 ms on the config-2 arms of scripts/resize_bench.py).  Staging (9.2 KB), the per-warp source rows (4.7 KB) and
// the taps come to 14.5 KB per CTA; ptxas gives 51 registers, so 6 CTAs per SM.  (Held to 40 registers for 8 CTAs, it
// spills.)
// The CTA finds its image in the prefix of tile counts `tile0` (nrec entries, increasing) by a CTA-wide search: each
// round samples up to kTileThreads entries, so 4096 images take two rounds - no per-tile map is built on the host.
// Each warp makes one output row at a time: it copies the two source rows' span of the tile's column taps into its
// own shared buffer (lanes read consecutive bytes), then each lane interpolates its columns from there.
__global__ void __launch_bounds__(kTileThreads)
k_resize_bilinear(const ResizeDev *__restrict__ recs, const uint32_t *__restrict__ tile0, const int nrec, uint8_t *__restrict__ out) {
    __shared__ uint32_t s_x0[kResizeTileW], s_fx[kResizeTileW], s_y0[kResizeTileH], s_fy[kResizeTileH];
    __shared__ __align__(16) uint8_t s_out[kResizeTileW * 3 * kResizeTileH + 32];          // (+32: the copy-out reads whole words past a row's payload)
    __shared__ uint8_t s_src[kTileThreads / 32][2][kResizeSpan * 3];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t bid = blockIdx.x;
    int lo = 0, hi = nrec;                                   // the last k with tile0[k] <= bid lies in [lo, hi)
    while (hi - lo > 1) {
        const int step = (hi - lo + kTileThreads - 1) / kTileThreads;
        const int k = lo + tid * step;
        const int cnt = __syncthreads_count(k < hi && __ldg(tile0 + k) <= bid);   // (>= 1: tile0[lo] <= bid)
        lo += (cnt - 1) * step;
        hi = min(lo + step, hi);
    }
    const ResizeDev *__restrict__ rz = recs + lo;
    const uint32_t sw = rz->sw, sh = rz->sh, W = rz->out.cw, H = rz->out.ch;
    const uint32_t t = bid - __ldg(tile0 + lo), ty = t / rz->tiles_x, tx = t - ty * rz->tiles_x;
    const int X0 = (int)tx * kResizeTileW, Y0 = (int)ty * kResizeTileH;
    const int ncols = min(kResizeTileW, (int)W - X0), nrows = min(kResizeTileH, (int)H - Y0);
    for (int i = tid; i < kResizeTileW + kResizeTileH; i += kTileThreads) {
        if (i < kResizeTileW) { if (i < ncols) resize_tap(sw, W, X0 + i, &s_x0[i], &s_fx[i]); }
        else if (i - kResizeTileW < nrows) resize_tap(sh, H, Y0 + i - kResizeTileW, &s_y0[i - kResizeTileW], &s_fy[i - kResizeTileW]);
    }
    __syncthreads();
    const uint8_t *src = out + rz->src_off;
    const uint32_t spitch = sw * 3;
    const uint32_t xa = s_x0[0], xb = min(s_x0[ncols - 1] + 1, sw - 1);
    const int span = (int)(xb - xa + 1) * 3;                 // bytes of a source row the tile's columns read
    const bool staged = span <= kResizeSpan * 3;
    const int bgr = rz->out.bgr;
    for (int r = warp; r < nrows; r += kTileThreads / 32) {
        const uint32_t y0 = s_y0[r], y1 = min(y0 + 1, sh - 1), fy = s_fy[r];
        const uint8_t *row0 = src + (size_t)y0 * spitch, *row1 = src + (size_t)y1 * spitch;
        if (staged) {
            uint8_t *b0 = s_src[warp][0], *b1 = s_src[warp][1];
            for (int k = lane; k < span; k += 32) { b0[k] = row0[xa * 3 + k]; b1[k] = row1[xa * 3 + k]; }
            __syncwarp();
            row0 = b0 - xa * 3; row1 = b1 - xa * 3;
        }
        for (int c = lane; c < ncols; c += 32) {
            const uint32_t x0 = s_x0[c], x1 = min(x0 + 1, sw - 1), fx = s_fx[c];
            uint8_t *d = s_out + r * (kResizeTileW * 3) + c * 3;
#pragma unroll
            for (int ch = 0; ch < 3; ch++) {
                const uint32_t top = (256u - fx) * row0[x0 * 3 + ch] + fx * row0[x1 * 3 + ch];
                const uint32_t bot = (256u - fx) * row1[x0 * 3 + ch] + fx * row1[x1 * 3 + ch];
                d[bgr ? 2 - ch : ch] = (uint8_t)(((256u - fy) * top + fy * bot + 32768u) >> 16);
            }
        }
        __syncwarp();                                        // (the warp's source buffer is refilled for its next row)
    }
    __syncthreads();
    TileDev td;                                              // what tile_copy_out reads of it: the tile's position
    td.img = 0; td.my = (uint16_t)ty; td.mx0 = (uint16_t)tx; td.nm = 0; td.ndu = 0; td.du0 = 0;
    tile_copy_out(s_out, kResizeTileW * 3, X0, Y0, ncols, nrows, td, &rz->out, out);
}

}  // namespace bj
