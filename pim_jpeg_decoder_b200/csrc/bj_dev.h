// Structures shared by the host side of the library and its kernels (plain data, lives in HBM).
#pragma once
#include <stdint.h>

namespace bj {

constexpr int kTileThreads = 192;     // K2/K3 CTA size = data units per tile (192 = lcm-friendly for bpm 1,2,3,4,6)
constexpr int kQPitch = 68;           // words between per-component dequant tables in smem (bank skew, 16 B aligned)
constexpr int kResizeTileW = 64;      // k_resize_bilinear: output columns per tile, two per lane of a warp
constexpr int kResizeTileH = 48;      // ... and output rows per tile, eight per warp of the kTileThreads-wide CTA

// Per image: geometry + where its data lives.  Data units ("du") are 64 coefficients = 128 B, zig-zag order,
// stored in decode order (MCU after MCU; inside an MCU: Y units row-major, then Cb, then Cr) - the order of
// the reference's loop nest src/jpeg_scanner.cpp:721-732.
struct ImgDev {
    uint32_t width, height;
    uint32_t nmx, nmy;            // MCUs per row / per column
    uint32_t du_base;             // index of this image's first data unit in the coefficient buffer
    uint32_t out_pitch;           // bytes between consecutive output rows
    uint64_t out_row0;            // byte offset (in the batch output buffer) of pixel (cx, cy), the crop's first
    int32_t  row_dir;             // +1: image row y at out_row0 + (y - cy)*pitch (RGB8); -1: out_row0 - (y - cy)*pitch (BMP, bottom-up)
    uint32_t row_bytes;           // payload bytes per row (cw*3)
    uint32_t row_pad;             // zero bytes after the payload (BMP: cw % 4)
    uint8_t  hs, vs, ncomp, bpm;  // luma sampling, components, data units per MCU
    uint8_t  bgr;                 // 1: B,G,R byte order (BMP)
    uint8_t  valid;
    uint8_t  dc_sep;              // 1: slot 0 of every unit is unused, the DC value comes from the DC plane (informative: the kernel is told by its dc_plane argument)
    uint8_t  scale_log2;          // reduced-size output: each output pixel is the mean of a (1 << scale_log2)^2 box of the full decode
    uint32_t qslot;               // this image's quantiser set in the batch's pool of QTab (deduplicated across the batch)
    uint32_t tile0;               // index of this image's first K2/K3 tile in the batch's tile list
    uint32_t ref_blocks;          // BJ_OUT_REF_MCUS: 2x2-position blocks in this image's output (whole chunks of MAX_MCU_PER_DPU / 4)
    uint32_t cx, cy, cw, ch;      // the pixels that are output (region of interest), in the coordinates of the scaled image:
                                  // [cx, cx + cw) x [cy, cy + ch); the whole (scaled) image by default
    uint16_t mx_lo, mx_hi;        // the MCU columns [mx_lo, mx_hi) and rows [my_lo, my_hi) that hold their full-size pixels
    uint16_t my_lo, my_hi;        // (bj_host.h: set_crop).  The K2/K3 tile list covers exactly these MCUs
};

// K2/K3 tiles per MCU row of the crop window: what the host sizes the tile list with and k_expand_maps fills it with
__host__ __device__ inline uint32_t idct_tiles_per_row(const ImgDev &im) {
    const uint32_t tile_mcus = kTileThreads / im.bpm;
    return ((uint32_t)im.mx_hi - im.mx_lo + tile_mcus - 1) / tile_mcus;
}
__host__ __device__ inline uint32_t idct_tile_count(const ImgDev &im) { return ((uint32_t)im.my_hi - im.my_lo) * idct_tiles_per_row(im); }

// Fixed-size output: one record per image of a batch that is resized (k_resize_bilinear, kernels_resize.cuh).  The
// source is the image's scaled crop, which the IDCT + colour kernel wrote as RGB8 (top-down, sw * 3 bytes per row) into
// the intermediate region of the batch output buffer; the output record is laid out as an image of w x h pixels whose
// crop window is all of it and whose MCU window starts at 0, so that tile_copy_out writes it unchanged and the output
// tile (0, 0) is the one that writes a BMP header.
struct ResizeDev {
    ImgDev out;                   // the final output: width x height = cw x ch = w x h, the format's layout
    uint64_t src_off;             // byte offset of the source's pixel (0, 0) in the batch output buffer
    uint32_t sw, sh;              // source size: the scaled crop's cw x ch
    uint32_t tiles_x;             // output tiles per row (kResizeTileW columns each)
    uint32_t pad_;
};

// One set of quantisation tables as the K2 kernel stages it: per component (quantiser << 16) in ZIG-ZAG (file) order.
struct QTab {
    uint32_t q16[3][kQPitch];
};

// One CTA of the fused dequant/IDCT/colour kernel: `nm` consecutive MCUs of MCU-row `my`, starting at `mx0`.
// 16 bytes, one load; du0 / ndu let the CTA start fetching its coefficient units before it has seen the image record.
struct TileDev {
    uint32_t img;
    uint16_t my, mx0, nm;
    uint16_t ndu;                 // data units of the tile (nm * units per MCU), <= kTileThreads
    uint32_t du0;                 // index of the tile's first data unit in the coefficient buffer / DC plane
};
static_assert(sizeof(TileDev) == 16, "TileDev is loaded as one uint4");

}  // namespace bj
