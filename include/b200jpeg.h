/* b200jpeg.h - C ABI of the B200-native JPEG decode back end (libb200jpeg.so).
 *
 * Drop-in boundary for the MCU-decode hot path of jeun-990806/pim-jpeg-decoder.  Every entry point names the
 * reference interface it replaces (paths relative to the reference tree).  Plain C: pointers and sizes only,
 * no C++ or torch types.  All functions return BJ_OK (0) or a negative bj_status; nothing throws, nothing exits,
 * and there is NO CPU fallback: without a CUDA device every compute entry fails with BJ_ERR_CUDA.
 *
 * Threading: a bj_ctx is single-owner (one consumer thread per context, like the reference's `offloading`
 * thread, src/decoder_host.cpp:213-350).  A context drives a list of GPUs, one host thread each (the first: the
 * caller's): bj_create makes a list of one (one process per GPU, e.g. under torchrun), bj_create_multi a list of
 * several GPUs of the box driven from one process.  Options and counters belong to the context, not to a GPU.
 * Ownership: the caller owns every host pointer it passes; the library owns device and pinned staging memory.
 */
#ifndef B200JPEG_H
#define B200JPEG_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    BJ_OK = 0,
    BJ_ERR_ARG = -1,          /* bad argument */
    BJ_ERR_CUDA = -2,         /* CUDA runtime/driver error (no device, launch failure ...) - see bj_last_error */
    BJ_ERR_NOMEM = -3,
    BJ_ERR_INVALID_JPEG = -4, /* the reference's read_JPEG would set header->valid = false */
    BJ_ERR_UNSUPPORTED = -5,  /* valid for the reference's parser but not decodable by its baseline path (SOF2) */
    BJ_ERR_CORRUPT_SCAN = -6  /* entropy-coded data inconsistent (the reference's decode_Huffman_data returns false) */
} bj_status;

typedef struct bj_ctx bj_ctx;

/* ---------------------------------------------------------------------------------------------------------
 * Context.  Replaces: `auto pim = DpuSet::allocate(DPU_ALLOCATE_ALL)` + `pim.load(DPU_BINARY)`
 * (src/decoder_host.cpp:32,268).  `device` is the CUDA ordinal (LOCAL_RANK in a one-process-per-GPU job). */
int bj_create(bj_ctx **ctx, int device);
/* All GPUs from ONE process, like `DpuSet::allocate(DPU_ALLOCATE_ALL)` takes every DPU of the machine
 * (src/decoder_host.cpp:32-33).  ndev <= 0: every visible device; devices == NULL: ndev devices spread evenly over the
 * visible ones (0, count/ndev, 2 count/ndev ...: neighbouring ordinals often share a PCIe uplink).  On any context,
 * bj_decode_batch / bj_submit deal the image list to its GPUs sub-batch by sub-batch from one shared cursor (images are
 * independent: no collective); bj_exec_mcus splits its DPUs into equal contiguous shares; the staged and stage-level
 * entries run on the first device; bj_exec_mcus_device refuses a context of more than one device. */
int bj_create_multi(bj_ctx **ctx, const int *devices, int ndev);
int bj_device_count(const bj_ctx *ctx);
void bj_destroy(bj_ctx *ctx);
const char *bj_status_string(int status);
const char *bj_last_error(const bj_ctx *ctx);   /* text of the last CUDA error seen by this context */
int bj_device_sm_count(const bj_ctx *ctx);

/* Pinned host memory for caller buffers (fast PCIe path).  Replaces nothing (UPMEM copies from pageable
 * std::vector, src/decoder_host.cpp:25-30); optional. */
void *bj_host_alloc(size_t bytes);
void bj_host_free(void *p);
/* Page-lock memory the caller already owns (cudaHostRegister) and tell the library about it.  Input files that lie
 * inside memory from bj_host_alloc / bj_host_register are uploaded straight from there (no staging copy on the host). */
int bj_host_register(void *p, size_t bytes);
int bj_host_unregister(void *p);

/* ---------------------------------------------------------------------------------------------------------
 * COMPAT ENTRY = the DPU program.  Replaces the sequence
 *     pim.copy("metadata_buffer", batch.metadata); pim.copy("mcus", batch.mcus);   src/decoder_host.cpp:276-277
 *     pim.exec();                                                                    src/decoder_host.cpp:292
 *     pim.copy(batch.mcus, "mcus");                                                  src/decoder_host.cpp:308
 * i.e. src/decoder_dpu.c:82-390 run on `nchunk` DPUs.
 *   metadata : [nchunk][276] u32, record layout of src/decoder_host.cpp:156-178 / src/decoder_dpu.c:112-132
 *   mcus     : [nchunk][64*M*3] i16 in/out, layout [block][component][position][64] (src/decoder_dpu.c:134-156);
 *              M = metadata[19] of the first non-idle chunk (MAX_MCU_PER_DPU, Makefile:2)
 * In: Huffman-decoded, de-zigzagged coefficients.  Out: R,G,B as i16 in the same tiles.  Bit-exact, in place.
 * The _device variant takes device pointers and a cudaStream_t (as void*) and does not synchronise. */
int bj_exec_mcus(bj_ctx *ctx, const uint32_t *metadata, int16_t *mcus, int nchunk);
int bj_exec_mcus_device(bj_ctx *ctx, const uint32_t *d_metadata, int16_t *d_mcus, int nchunk, int M, void *stream);

/* ---------------------------------------------------------------------------------------------------------
 * Image descriptor: POD mirror of the reference's `Header` (src/headers/jpeg.h:146-179) for a baseline file.
 * Filled by bj_parse_header (a restatement of read_JPEG's marker walk on in-memory bytes,
 * src/jpeg_scanner.cpp:6-403) or by the caller from a `Header*` it already has (see INTEGRATION.md). */
typedef struct {
    uint32_t width, height;
    uint32_t mcu_w, mcu_h;            /* Header::mcu_width/height: ceil(w/8), ceil(h/8) */
    uint32_t mcu_w_real, mcu_h_real;  /* Header::mcu_width_real/height_real */
    uint32_t restart_interval;        /* in MCUs, 0 = none */
    uint8_t ncomp;                    /* 1..3 */
    uint8_t hs, vs;                   /* Header::h/v_sampling_factor (luma) */
    uint8_t frame_type;               /* 0xC0 baseline / 0xC2 progressive */
    uint8_t comp_h[3], comp_v[3];     /* ColorComponent::h/v_sampling_factor */
    uint8_t qt_id[3], dc_id[3], ac_id[3];
    uint8_t qt_set[4], dc_set[4], ac_set[4];
    uint8_t scan_ncomp;               /* Header::components_in_scan */
    uint16_t qt_zz[4][64];            /* quantisation tables in FILE (zig-zag) order; the reference's quirky
                                         de-zigzag (src/headers/common.h:9-18) is applied inside the kernels */
    uint8_t dc_offsets[4][17], dc_symbols[4][162];   /* HuffmanTable::offsets/symbols, src/headers/jpeg.h:129-134 */
    uint8_t ac_offsets[4][17], ac_symbols[4][162];
    uint64_t scan_off;                /* offset of the first entropy-coded byte in the file */
    uint64_t scan_len;                /* raw scan bytes (stuffed, with RSTn) up to, not including, the EOI marker */
} bj_image_desc;

/* Replaces: read_JPEG (src/jpeg_scanner.cpp:345-436) minus the byte-at-a-time scan copy.
 * BJ_ERR_INVALID_JPEG exactly where the reference sets valid=false; BJ_ERR_UNSUPPORTED for SOF2 or a scan that
 * does not interleave all frame components (the reference cannot decode those either, SURVEY.md section 2). */
int bj_parse_header(const uint8_t *file, size_t len, bj_image_desc *desc);
/* The same without the walk over the entropy-coded bytes: only the headers are read (what the decode entries do
 * internally - they find the end of the scan on the GPU).  scan_len is then an UPPER BOUND (everything up to the end of
 * the file), and a file whose scan does not end in EOI is only found out by the decode (per-image BJ_ERR_INVALID_JPEG).
 * Enough to size output buffers with bj_output_size. */
int bj_peek_header(const uint8_t *file, size_t len, bj_image_desc *desc);

/* Output layouts of the full path. */
typedef enum {
    BJ_OUT_RGB8 = 0,   /* top-down packed R,G,B bytes, width*height*3 */
    BJ_OUT_BMP = 1,    /* the exact file bytes write_BMP produces (src/bmp_writer.cpp:19-67): 26-byte header,
                          bottom-up B,G,R rows, width%4 zero bytes after every row */
    BJ_OUT_REF_MCUS = 2 /* the reference's own `mcus` buffers after pim.exec() + pim.copy(batch.mcus, "mcus")
                          (src/decoder_host.cpp:292,308): R,G,B as int16 in the [block][component][position][64] tile
                          layout (src/decoder_dpu.c:134-156), nchunks x 64*MAX_MCU_PER_DPU*3 shorts per image, every
                          short of every chunk as the DPUs leave it (unused tiles 128) - what the UNCHANGED write_BMP
                          (src/bmp_writer.cpp:19-67) takes.  MAX_MCU_PER_DPU: option "ref_max_mcu_per_dpu" (default 100) */
} bj_out_format;
size_t bj_output_size(const bj_image_desc *desc, int format);          /* BJ_OUT_REF_MCUS: for MAX_MCU_PER_DPU = 100 */
/* BJ_OUT_REF_MCUS for any MAX_MCU_PER_DPU (a multiple of 4): bytes of the image's chunks; *nchunks = how many
 * (need_dpus of src/decoder_host.cpp:125-128). */
size_t bj_ref_mcus_size(const bj_image_desc *desc, int max_mcu_per_dpu, int *nchunks);

/* ---------------------------------------------------------------------------------------------------------
 * FULL PATH, one call.  Replaces, per image, decode_Huffman_data (src/jpeg_scanner.cpp:707-756) + the DPU
 * program + write_BMP's pixel gathering:  compressed file bytes in host memory -> decoded pixels in host memory.
 *   files[i], lens[i] : the complete JPEG file i
 *   outs[i]           : caller buffer of bj_output_size() bytes (discover with bj_parse_header), may be pinned
 *   status[i]         : per-image bj_status (optional).  An invalid image is skipped like the reference does
 *                       (src/decoder_host.cpp:120-123) and does not fail the batch.
 * Internally: sub-batches double-buffered over pinned staging on CUDA streams; blocks until outs are written. */
int bj_decode_batch(bj_ctx *ctx, const uint8_t *const *files, const size_t *lens, int n, int format,
                    uint8_t *const *outs, int *status);

/* FULL PATH behind the UNCHANGED scanner.  Replaces decode_Huffman_data(header, MCU_buffer, dpu_offset) + pim.copy /
 * pim.exec / pim.copy (src/decoder_host.cpp:181, :268-312) for a host that keeps read_JPEG in front: it fills one
 * bj_image_desc per `Header` (field for field, see INTEGRATION.md) and hands over the scan bytes -
 *   BJ_SCAN_UNSTUFFED  Header::huffman_data as read_JPEG leaves it (FF00 un-stuffed, RSTn removed, src/jpeg_scanner.cpp:
 *                      405-433).  Only for restart_interval == 0: read_JPEG throws the RSTn positions away, and with them
 *                      the segment boundaries (per-image BJ_ERR_UNSUPPORTED otherwise)
 *   BJ_SCAN_RAW        the scan as it is in the file (stuffed, with RSTn), with or without the EOI behind it
 * scan_kinds == NULL: all BJ_SCAN_RAW.  desc->scan_off / scan_len are ignored.  With format BJ_OUT_REF_MCUS the outputs
 * are the `mcus` buffers the unchanged write_BMP reads. */
typedef enum { BJ_SCAN_RAW = 0, BJ_SCAN_UNSTUFFED = 1 } bj_scan_kind;
int bj_decode_batch_desc(bj_ctx *ctx, const bj_image_desc *descs, const uint8_t *const *scans, const size_t *scan_lens,
                         const int *scan_kinds, int n, int format, uint8_t *const *outs, int *status);

/* FULL PATH, asynchronous.  bj_submit hands the batch to the context's worker thread and returns at once; bj_wait blocks
 * until that batch's outputs are in host memory, returns what bj_decode_batch would have returned and releases the job.
 * Jobs run in submission order.  All arrays (files, lens, outs, status) must stay valid until bj_wait returns.  This is
 * the reference's producer / consumer overlap (two threads and a queue, src/decoder_host.cpp:25-38,364-365): submit
 * batch k+1 - or read its files - while batch k decodes, write batch k-1's BMPs meanwhile.  While jobs are pending the
 * context may only be used through bj_submit / bj_wait. */
typedef struct bj_job bj_job;
int bj_submit(bj_ctx *ctx, const uint8_t *const *files, const size_t *lens, int n, int format,
              uint8_t *const *outs, int *status, bj_job **job);
int bj_wait(bj_job *job);

/* FULL PATH, staged (device-resident batch) - what bj_decode_batch is made of, and what bench.py times with the
 * inputs already in HBM. */
typedef struct bj_batch bj_batch;
int bj_batch_create(bj_ctx *ctx, const uint8_t *const *files, const size_t *lens, int n, int format, bj_batch **out);
int bj_batch_upload(bj_batch *b, void *stream);                 /* H2D: file bytes + descriptors          */
int bj_batch_decode(bj_batch *b, void *stream);                 /* enqueue all kernels; input and output stay in HBM */
int bj_batch_sync(bj_batch *b);                                 /* wait; settles the (rare) extra Huffman fix-up rounds */
int bj_batch_download(bj_batch *b, uint8_t *const *outs, void *stream);   /* D2H into caller buffers, then sync */
/* Where image i sits in the batch's device output buffer.  A caller that lays its host buffers out the same way
 * (outs[i] = base + offset_i) and sets option "packed_outputs" gets one large copy instead of one per image.
 * Returns the image's parse status. */
int bj_batch_output_offset(const bj_batch *b, int i, size_t *offset, size_t *bytes);
int bj_batch_status(const bj_batch *b, int *status /*[n]*/);
void bj_batch_destroy(bj_batch *b);

/* Introspection for tests and the benchmark. */
typedef struct {
    uint64_t pixels;            /* decoded pixels (valid images) */
    uint64_t scan_bytes;        /* raw entropy-coded bytes */
    uint64_t data_units;        /* 8x8 units = 128 B of coefficients each */
    uint64_t out_bytes;
    uint64_t h2d_bytes, d2h_bytes;
    uint32_t subsequences;      /* Huffman decode threads */
    uint32_t sync_rounds;       /* fix-up rounds the last bj_batch_decode needed */
    uint32_t launches;          /* kernels launched by the last bj_batch_decode */
    float ms_entropy, ms_idct;  /* CUDA-event time of the two stages of the last bj_batch_decode */
    float ms_unstuff, ms_sync, ms_write;   /* ms_entropy split: K0 (un-stuff + tables), K1 fix-up rounds, K1 write pass */
    uint64_t clean_bytes;       /* entropy-coded bytes after un-stuffing / marker removal */
} bj_batch_info;
int bj_batch_get_info(const bj_batch *b, bj_batch_info *info);
int bj_batch_device_output(const bj_batch *b, int i, void **dptr, size_t *bytes);
/* zig-zag i16 units (slot 0 of every unit unused) + the plane of predicted DC values, one i16 per unit */
int bj_batch_device_coefficients(const bj_batch *b, int i, void **dptr, size_t *bytes, void **dc_dptr);

/* Stage-level entry for known-answer tests: dequant + IDCT + upsample + colour only, on caller-supplied
 * coefficients (zig-zag order, DC un-differenced, MCU-interleaved unit order = what the entropy stage emits).
 * Replaces: the DPU program on the fast layout. */
int bj_stage_idct_color(bj_ctx *ctx, const bj_image_desc *desc, const int16_t *coef_zz, int format, uint8_t *out);

/* Stage-level entry for known-answer tests: un-stuffing + Huffman decode only (kernels K0/K1).  Output = what
 * decode_Huffman_data (src/jpeg_scanner.cpp:707-756) produces, but in zig-zag order and MCU-interleaved unit order
 * (ndu * 64 shorts).  *status = BJ_OK or BJ_ERR_CORRUPT_SCAN. */
int bj_stage_entropy(bj_ctx *ctx, const uint8_t *file, size_t len, int16_t *coef_zz, size_t capacity_bytes, int *status);

/* Tunables (0 = default):
 *   "subseq_bits"      sub-sequence size of the Huffman synchronisation pass in bits (multiple of 32, >= 128);
 *                      0 = chosen per image (2400-4096 bits, so that an image's sub-sequences fill whole CTAs;
 *                      a typical restart segment in one piece)
 *   "slices"           pieces of a sub-sequence the Huffman write pass works on (1, 2, 4 or 8; default 1: the write
 *                      pass works on whole sub-sequences)
 *   "sync_rounds"      launches of the fix-up kernel before convergence is first checked
 *   "sub_batch_bytes"  compressed bytes per sub-batch of bj_decode_batch
 *   "sub_batch_ramp"   0: all sub-batches the same size (default 1: the first two are 1/8 and 1/3 of it, so that the
 *                      copy-out starts early)
 *   "host_threads"     worker threads for the per-image host work of bj_decode_batch, the caller included
 *   "packed_inputs"    where the file bytes are uploaded from.  0 (default): straight from the caller's memory when the
 *                      files of a sub-batch lie close together inside memory from bj_host_alloc / bj_host_register,
 *                      through a pinned staging copy otherwise;  1: the caller states that the files lie in ONE
 *                      page-locked allocation the library does not know (e.g. cudaHostAlloc) - only set it when that
 *                      is true, pageable memory would make the upload synchronous;  -1: always stage
 *   "ref_max_mcu_per_dpu"  BJ_OUT_REF_MCUS: the MAX_MCU_PER_DPU the reading host was compiled with (Makefile:2; default
 *                      100, a multiple of 4)
 *   "max_image_pixels" images with more pixels get BJ_ERR_UNSUPPORTED (default 2^28), like the reference's "Too high
 *                      resolution" (src/decoder_host.cpp:146-149): a tiny file cannot claim tens of GB of buffers
 *   "sub_batch_out_bytes"  decoded bytes per sub-batch of bj_decode_batch (default 1 GiB)
 *   "debug_poison"     1: coefficient, DC, stream and output buffers are filled with 0xA5 before every decode (tests:
 *                      every byte that is read or returned must have been written by that decode)
 *   "packed_outputs"   1: output pointers that follow bj_batch_output_offset's layout (outs[i] = base + offset_i,
 *                      for the one-call path: offsets restart at 0 in every sub-batch) belong to ONE allocation,
 *                      so runs of images are copied out in one transfer, padding bytes included */
int bj_set_option(bj_ctx *ctx, const char *name, long value);
/* Counters of the last call: "exec_ms" (kernel time of bj_exec_mcus - the reference's "DPU execution" profile line,
 * src/decoder_host.cpp:291-294), "decode_batch_sub_batches", "decode_batch_launches", "decode_batch_h2d_bytes",
 * "decode_batch_d2h_bytes", "decode_batch_d2h_copies", "decode_batch_host_ms" (header parse + layout [+ staging copy]),
 * "decode_batch_wait_ms" (caller blocked on the GPU), "host_threads", "devices", and the kernel time per stage summed
 * over the sub-batches - the reference's per-stage "Profiles" lines (src/decoder_host.cpp:379-394) -
 * "decode_batch_ms_unstuff", "decode_batch_ms_sync", "decode_batch_ms_write", "decode_batch_ms_idct";
 * "decode_batch_direct_uploads" (sub-batches whose files went up straight from the caller's page-locked memory).
 * "total_<counter>" (total_sub_batches, total_launches, total_h2d_bytes, total_d2h_bytes, total_host_ms, total_wait_ms,
 * total_d2h_copies, total_ms_unstuff, total_ms_sync, total_ms_write, total_ms_idct, total_direct_uploads): the same
 * summed over every bj_decode_batch / bj_submit job since the context was created.
 * For a context of several GPUs: byte and launch counts are sums, times the maximum over the devices.
 * Environment: B200JPEG_TRACE=1 prints one line per sub-batch of bj_decode_batch (host prepare, kernels, copy-out). */
int bj_get_stat(const bj_ctx *ctx, const char *name, double *value);

/* Version / build info. */
const char *bj_build_info(void);

#ifdef __cplusplus
}
#endif
#endif /* B200JPEG_H */
