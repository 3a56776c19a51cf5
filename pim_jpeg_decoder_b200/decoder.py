"""Host side of the hot path, mirroring the reference's interface (src/decoder_host.cpp) over the C ABI.

    reference                                              here
    -----------------------------------------------------  ---------------------------------------------------
    DpuSet::allocate + load            (:32, :268)         Decoder(device)
    pim.copy / pim.exec / pim.copy     (:276-308)          Decoder.exec_mcus(metadata, mcus)      [compat layout]
    read_JPEG                          (jpeg_scanner:345)  parse_header(bytes)
    decode_Huffman_data + exec + write_BMP gather          Decoder.decode(files, fmt) / Batch     [fast layout]
    (a crop of each image: rois=, see roi_output_size; at 1/2, 1/4 or 1/8 size: scales=, see scaled_output_size;
    resized to a fixed size: sizes=, see resized_output_size and resize_plan)
    main(argv): sort by size, decode, write <name>.bmp     decode_files(paths)
"""
import ctypes as C
import os

import numpy as np

from . import _lib as L


def parse_header(data):
    """read_JPEG on in-memory bytes (minus the scan copy).  Returns (status, ImageDesc)."""
    d = L.ImageDesc()
    buf = np.frombuffer(data, dtype=np.uint8)
    st = L.lib().bj_parse_header(buf.ctypes.data_as(C.c_void_p), len(data), C.byref(d))
    return st, d


def _sizing_header(data):
    """The descriptor that sizes a file's output: bj_parse_header's, or for a progressive (SOF2) file - which
    bj_parse_header calls invalid at the end of its first scan, and which the decode entries take with the context option
    "progressive" - bj_peek_header's (the size functions read only the frame)."""
    st, d = parse_header(data)
    if st != L.BJ_OK:
        p = L.ImageDesc()
        buf = np.frombuffer(data, dtype=np.uint8)
        if L.lib().bj_peek_header(buf.ctypes.data_as(C.c_void_p), len(data), C.byref(p)) == L.BJ_ERR_UNSUPPORTED and p.frame_type == 0xC2:
            return L.BJ_OK, p
    return st, d


def _roi_table(rois, n):
    """rois: None (whole images) or n rows of (x, y, w, h) - an (n, 4) array or anything numpy makes one of; a row of
    zeros is the whole image.  -> (keepalive uint32 array or None, pointer for the C ABI)"""
    if rois is None:
        return None, None
    a = np.ascontiguousarray(rois, dtype=np.uint32).reshape(n, 4)
    return a, a.ctypes.data_as(C.c_void_p)


def _scale_table(scales, n):
    """scales: None (full size), one int for every image, or n of them - each 1, 2, 4 or 8 (any other value is refused per
    image by the library).  -> (keepalive uint8 array or None, pointer for the C ABI)"""
    if scales is None:
        return None, None
    v = np.broadcast_to(np.asarray(scales), (n,))
    if v.dtype.kind not in "iuf":
        raise TypeError(f"scales must be numbers, not {v.dtype}")
    # a value that is not a whole number in 1..8 would wrap or truncate to some other scale in the uint8 cast: it goes
    # to the library as 0, which refuses that image (BJ_ERR_ARG) like any other scale it does not have
    ok = (v >= 1) & (v <= 8) & (v == np.floor(v)) if v.dtype.kind == "f" else (v >= 1) & (v <= 8)
    a = np.ascontiguousarray(np.where(ok, v, 0).astype(np.uint8))
    return a, a.ctypes.data_as(C.c_void_p)


def _size_table(sizes, n):
    """sizes: None (no resize), one (w, h) for every image, or an (n, 2) array of them - each two whole numbers in
    1..65535, or (0, 0) for no resize.  -> (keepalive uint32 (n, 2) array or None, pointer for the C ABI)"""
    if sizes is None:
        return None, None
    v = np.asarray(sizes)
    if v.dtype.kind not in "iuf":
        raise TypeError(f"sizes must be numbers, not {v.dtype}")
    v = np.broadcast_to(v, (n, 2)) if v.shape == (2,) else v.reshape(n, 2)
    # a pair that is not two whole numbers in 1..65535 (nor (0, 0)) would wrap or truncate to some other size in the
    # uint32 cast: it goes to the library as (1, 0), which refuses that image (BJ_ERR_ARG)
    whole = (v == np.floor(v)) if v.dtype.kind == "f" else np.ones(v.shape, dtype=bool)
    ok = ((v >= 1) & (v <= 65535) & whole).all(axis=1) | (v == 0).all(axis=1)
    a = np.ascontiguousarray(np.where(ok[:, None], v, np.array([1, 0])).astype(np.uint32))
    return a, a.ctypes.data_as(C.c_void_p)


def roi_output_size(desc, roi, fmt=L.BJ_OUT_RGB8):
    """Output bytes of the image `desc` (ImageDesc) cropped to `roi` ((x, y, w, h), a Roi, or None for the whole image);
    0 if the ROI does not fit the image, and for BJ_OUT_REF_MCUS."""
    if roi is not None and not isinstance(roi, L.Roi):
        roi = L.Roi(*(int(v) for v in roi))
    return L.lib().bj_roi_output_size(C.byref(desc), C.byref(roi) if roi is not None else None, fmt)


def scaled_output_size(desc, roi, scale, fmt=L.BJ_OUT_RGB8):
    """Output bytes of the image `desc` at 1/scale of its size (scale 1, 2, 4 or 8) cropped to `roi`, a rectangle of the
    scaled image ((x, y, w, h), a Roi, or None for all of it); 0 if the scale or the ROI is refused, and for
    BJ_OUT_REF_MCUS."""
    if roi is not None and not isinstance(roi, L.Roi):
        roi = L.Roi(*(int(v) for v in roi))
    return L.lib().bj_scaled_output_size(C.byref(desc), C.byref(roi) if roi is not None else None, int(scale), fmt)


def resized_output_size(desc, roi, scale, size, fmt=L.BJ_OUT_RGB8):
    """Output bytes of the image `desc` at 1/scale, cropped to `roi` (a rectangle of the scaled image, as for
    scaled_output_size) and resized to `size` ((w, h), a Size, or None / (0, 0) for no resize); 0 for anything the
    library refuses, and for BJ_OUT_REF_MCUS."""
    if roi is not None and not isinstance(roi, L.Roi):
        roi = L.Roi(*(int(v) for v in roi))
    if size is not None and not isinstance(size, L.Size):
        size = L.Size(*(int(v) for v in size))
    return L.lib().bj_resized_output_size(C.byref(desc), C.byref(roi) if roi is not None else None, int(scale),
                                          C.byref(size) if size is not None else None, fmt)


def resize_plan(width, height, box, size):
    """The request that turns the box (x, y, w, h) of a width x height image (None: all of it) into a (tw, th) output:
    returns (scale, roi) for the scales= and rois= arguments.  The scale s is the largest of 8, 4, 2, 1 with
    w >= s * tw and h >= s * th, so the bilinear stage reduces by less than 2x unless the box is more than 16 times the
    target; the ROI is the box rounded outward onto the image scaled by 1/s (x // s, ceil((x + w) / s) - x // s, the
    same for y), which always fits the scaled image."""
    tw, th = (int(v) for v in size)
    x, y, w, h = (0, 0, int(width), int(height)) if box is None else (int(v) for v in box)
    if tw < 1 or th < 1 or w < 1 or h < 1 or x < 0 or y < 0 or x + w > width or y + h > height:
        raise ValueError(f"resize_plan: box {box} of a {width}x{height} image to {size}")
    s = next((s for s in (8, 4, 2) if w >= s * tw and h >= s * th), 1)
    xs, ys = x // s, y // s
    return s, (xs, ys, -(-(x + w) // s) - xs, -(-(y + h) // s) - ys)


class PinnedBuffer:
    """Page-locked host memory from bj_host_alloc, exposed as a numpy uint8 array."""

    def __init__(self, nbytes):
        self.nbytes = int(nbytes)
        self.ptr = L.lib().bj_host_alloc(max(self.nbytes, 1))
        if not self.ptr:
            raise MemoryError(f"bj_host_alloc({nbytes}) failed")
        self.array = np.ctypeslib.as_array((C.c_uint8 * max(self.nbytes, 1)).from_address(self.ptr))[: self.nbytes]

    def free(self):
        if self.ptr:
            self.array = None
            L.lib().bj_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def _file_arrays(files):
    """list of bytes / uint8 arrays -> (keepalive arrays, char** , size_t*)"""
    arrs = [f if isinstance(f, np.ndarray) else np.frombuffer(f, dtype=np.uint8) for f in files]
    n = len(arrs)
    ptrs = (C.c_void_p * max(n, 1))(*[a.__array_interface__["data"][0] for a in arrs])
    lens = (C.c_size_t * max(n, 1))(*[a.size for a in arrs])
    return arrs, ptrs, lens


class Batch:
    """A device-resident batch (bj_batch): upload -> decode -> download, each asynchronous on the context's stream.
    rois: None, or one (x, y, w, h) crop per image (see roi_output_size); scales: None, or a scale denominator for every
    image or one per image (see scaled_output_size; a ROI is then a rectangle of the scaled image); sizes: None, or a
    (w, h) target size for every image or one per image (see resized_output_size)."""

    def __init__(self, dec, files, fmt=L.BJ_OUT_RGB8, rois=None, scales=None, sizes=None):
        self.dec = dec
        self.n = len(files)
        self._keep, ptrs, lens = _file_arrays(files)
        _, rp = _roi_table(rois, self.n)
        _, sp = _scale_table(scales, self.n)
        _, zp = _size_table(sizes, self.n)
        self.h = C.c_void_p()
        L.check(L.lib().bj_batch_create_resized(dec.ctx, ptrs, lens, rp, sp, zp, self.n, fmt, C.byref(self.h)), "bj_batch_create_resized", dec.ctx)
        self.offsets, self.sizes, self.parse_status = [], [], []
        for i in range(self.n):
            off, nb = C.c_size_t(), C.c_size_t()
            st = L.lib().bj_batch_output_offset(self.h, i, C.byref(off), C.byref(nb))
            self.parse_status.append(st)
            self.offsets.append(off.value)
            self.sizes.append(nb.value)
        self.total_out = max((o + s for o, s in zip(self.offsets, self.sizes)), default=0)

    def upload(self, stream=None):
        """stream: a cudaStream_t as an integer (e.g. torch.cuda.Stream().cuda_stream); None = the context's own."""
        L.check(L.lib().bj_batch_upload(self.h, stream), "bj_batch_upload", self.dec.ctx)

    def decode(self, stream=None):
        L.check(L.lib().bj_batch_decode(self.h, stream), "bj_batch_decode", self.dec.ctx)

    def sync(self):
        L.check(L.lib().bj_batch_sync(self.h), "bj_batch_sync", self.dec.ctx)

    def download(self, out=None, only=None):
        """Copy decoded images to the host.  `out`: uint8 array of total_out bytes (e.g. PinnedBuffer.array) laid
        out like the device buffer; `only`: indices to copy (default all).  Returns per-image views (None = skipped)."""
        if out is None:
            out = np.zeros(self.total_out, dtype=np.uint8)
        base = out.ctypes.data
        want = set(range(self.n)) if only is None else set(only)
        ok = [st == L.BJ_OK and i in want for i, st in enumerate(self.parse_status)]
        ptrs = (C.c_void_p * max(self.n, 1))(*[base + o if k else None for o, k in zip(self.offsets, ok)])
        L.check(L.lib().bj_batch_download(self.h, ptrs, None), "bj_batch_download", self.dec.ctx)
        return [out[o:o + s] if k else None for o, s, k in zip(self.offsets, self.sizes, ok)]

    def status(self):
        st = (C.c_int * max(self.n, 1))()
        L.check(L.lib().bj_batch_status(self.h, st), "bj_batch_status")
        return list(st)[: self.n]

    def info(self):
        info = L.BatchInfo()
        L.check(L.lib().bj_batch_get_info(self.h, C.byref(info)), "bj_batch_get_info")
        return info

    def device_output(self, i):
        p, nb = C.c_void_p(), C.c_size_t()
        L.check(L.lib().bj_batch_device_output(self.h, i, C.byref(p), C.byref(nb)), "bj_batch_device_output")
        return p.value, nb.value

    def destroy(self):
        if self.h:
            L.lib().bj_batch_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass


class Job:
    """A batch handed to bj_submit: wait() blocks until its outputs are in host memory and returns the status array."""

    def __init__(self, dec, handle, keep, status, n):
        self.dec, self.h, self._keep, self._status, self.n = dec, handle, keep, status, n

    def wait(self):
        if self.h is not None:
            h, self.h = self.h, None
            L.check(L.lib().bj_wait(h), "bj_wait", self.dec.ctx)
        return self._status[: self.n]


class Decoder:
    """One context.  Decoder(device) drives one GPU (one process per GPU, the torchrun way); Decoder(devices=[...])
    - or devices="all" - drives several GPUs of the box from this one process (bj_create_multi), the way the
    reference's single process takes every DPU (src/decoder_host.cpp:32-33)."""

    def __init__(self, device=0, devices=None):
        self.ctx = C.c_void_p()
        if devices is None:
            st = L.lib().bj_create(C.byref(self.ctx), device)
            what = "bj_create"
        elif isinstance(devices, str):
            st = L.lib().bj_create_multi(C.byref(self.ctx), None, 0)
            what = "bj_create_multi"
        else:
            arr = (C.c_int * len(devices))(*devices)
            st = L.lib().bj_create_multi(C.byref(self.ctx), arr, len(devices))
            what = "bj_create_multi"
        if st != L.BJ_OK:
            self.ctx = None
            raise L.BjError(st, what + " (this back end has no CPU fallback)")
        self.device = device
        self.device_count = L.lib().bj_device_count(self.ctx)

    def close(self):
        if self.ctx:
            L.lib().bj_destroy(self.ctx)
            self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, name, value):
        L.check(L.lib().bj_set_option(self.ctx, name.encode(), int(value)), f"bj_set_option({name})")

    def stat(self, name):
        v = C.c_double()
        L.check(L.lib().bj_get_stat(self.ctx, name.encode(), C.byref(v)), f"bj_get_stat({name})")
        return v.value

    # ---- compat entry: the DPU program on the reference's own buffers (in place)
    def exec_mcus(self, metadata, mcus):
        md = np.ascontiguousarray(metadata, dtype=np.uint32).reshape(-1, 276)
        out = np.ascontiguousarray(mcus, dtype=np.int16).copy()
        L.check(L.lib().bj_exec_mcus(self.ctx, md.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p), md.shape[0]),
                "bj_exec_mcus", self.ctx)
        return out

    # ---- stage entries (known-answer tests)
    def stage_entropy(self, data):
        st, d = parse_header(data)
        if st != L.BJ_OK:
            raise L.BjError(st, "bj_parse_header")
        nmx = (d.mcu_w + d.hs - 1) // d.hs
        nmy = (d.mcu_h + d.vs - 1) // d.vs
        bpm = sum(d.comp_h[j] * d.comp_v[j] for j in range(d.ncomp))
        coef = np.full((nmx * nmy * bpm, 64), 0x5A5A, dtype=np.int16)
        buf = np.frombuffer(data, dtype=np.uint8)
        status = C.c_int(0)
        L.check(L.lib().bj_stage_entropy(self.ctx, buf.ctypes.data_as(C.c_void_p), len(data), coef.ctypes.data_as(C.c_void_p),
                                         coef.nbytes, C.byref(status)), "bj_stage_entropy", self.ctx)
        return coef, status.value

    def stage_idct_color(self, desc, coef_zz, fmt=L.BJ_OUT_RGB8):
        co = np.ascontiguousarray(coef_zz, dtype=np.int16)
        out = np.zeros(L.lib().bj_output_size(C.byref(desc), fmt), dtype=np.uint8)
        L.check(L.lib().bj_stage_idct_color(self.ctx, C.byref(desc), co.ctypes.data_as(C.c_void_p), fmt, out.ctypes.data_as(C.c_void_p)),
                "bj_stage_idct_color", self.ctx)
        return out

    # ---- full path, one call (host buffers in, host buffers out)
    def decode(self, files, fmt=L.BJ_OUT_RGB8, outs=None, rois=None, scales=None, sizes=None):
        """Returns (list of uint8 arrays or None for rejected files, list of per-image status).  rois: None, or one
        (x, y, w, h) crop per image (see roi_output_size); scales: None, or a scale denominator (1, 2, 4, 8) for every
        image or one per image (see scaled_output_size); sizes: None, or a (w, h) target size for every image or one
        per image (see resized_output_size).  An image whose scale, ROI or size is refused gets BJ_ERR_ARG."""
        n = len(files)
        keep, ptrs, lens = _file_arrays(files)
        ra, rp = _roi_table(rois, n)
        sa, sp = _scale_table(scales, n)
        za, zp = _size_table(sizes, n)
        if outs is None:
            outs = []
            for i, f in enumerate(files):
                st, d = _sizing_header(f)
                size = 0
                if st == L.BJ_OK and ra is None and sa is None and za is None:
                    size = L.lib().bj_output_size(C.byref(d), fmt)          # (BJ_OUT_REF_MCUS included: it has no crop, scale or size)
                elif st == L.BJ_OK:
                    size = resized_output_size(d, None if ra is None else ra[i], 1 if sa is None else sa[i], None if za is None else za[i], fmt)
                outs.append(np.zeros(size, dtype=np.uint8) if size else None)
        optrs = (C.c_void_p * max(n, 1))(*[o.__array_interface__["data"][0] if o is not None else None for o in outs])
        status = (C.c_int * max(n, 1))()
        L.check(L.lib().bj_decode_batch_resized(self.ctx, ptrs, lens, rp, sp, zp, n, fmt, optrs, status), "bj_decode_batch_resized", self.ctx)
        st = list(status)[:n]
        return [o if s in (L.BJ_OK, L.BJ_ERR_CORRUPT_SCAN) else None for o, s in zip(outs, st)], st


    def decode_desc(self, descs, scans, kinds=None, fmt=L.BJ_OUT_REF_MCUS):
        """bj_decode_batch_desc: the caller holds parsed headers (ImageDesc, e.g. filled from the reference's `Header`) and
        the scan bytes.  Returns (list of arrays - int16 for BJ_OUT_REF_MCUS, uint8 otherwise -, list of status)."""
        n = len(descs)
        arr = (L.ImageDesc * max(n, 1))(*descs)
        keep, ptrs, lens = _file_arrays(scans)
        m = C.c_int(0)
        sizes = [L.lib().bj_ref_mcus_size(C.byref(d), 100, C.byref(m)) if fmt == L.BJ_OUT_REF_MCUS else L.lib().bj_output_size(C.byref(d), fmt) for d in descs]
        outs = [np.zeros(s, dtype=np.uint8) for s in sizes]
        optrs = (C.c_void_p * max(n, 1))(*[o.__array_interface__["data"][0] for o in outs])
        kp = (C.c_int * max(n, 1))(*kinds) if kinds is not None else None
        status = (C.c_int * max(n, 1))()
        L.check(L.lib().bj_decode_batch_desc(self.ctx, arr, ptrs, lens, kp, n, fmt, optrs, status), "bj_decode_batch_desc", self.ctx)
        if fmt == L.BJ_OUT_REF_MCUS:
            outs = [o.view(np.int16) for o in outs]
        return outs, list(status)[:n]

    def decode_packed(self, src, src_off, src_len, dst, dst_off, fmt=L.BJ_OUT_RGB8, rois=None, scales=None, sizes=None):
        """bj_decode_batch for a batch-pipeline caller: the n files sit in ONE host buffer `src` (uint8 array, ideally
        a PinnedBuffer) at byte offsets `src_off` with lengths `src_len`; image i is written to `dst[dst_off[i]:]`
        (bj_output_size bytes, or bj_scaled_output_size with `rois`: an (n, 4) uint32 array of (x, y, w, h) crops, and
        `scales`: a scale denominator for every image or one per image; bj_resized_output_size with `sizes`: one (w, h)
        for every image or an (n, 2) array - with one size for all, dst can be one [n, h, w, 3] array).  The pointer tables are built with vector
        arithmetic, so the host-side cost per call does not grow with a Python loop over images.  Returns the
        per-image status as an int32 array."""
        n = len(src_off)
        ip = (np.asarray(src_off, dtype=np.uint64) + np.uint64(src.__array_interface__["data"][0]))
        il = np.ascontiguousarray(src_len, dtype=np.uint64)
        op = (np.asarray(dst_off, dtype=np.uint64) + np.uint64(dst.__array_interface__["data"][0]))
        ra, rp = _roi_table(rois, n)
        sa, sp = _scale_table(scales, n)
        za, zp = _size_table(sizes, n)
        status = np.zeros(max(n, 1), dtype=np.int32)
        L.check(L.lib().bj_decode_batch_resized(self.ctx, ip.ctypes.data_as(C.c_void_p), il.ctypes.data_as(C.c_void_p), rp, sp, zp, n, fmt,
                                                op.ctypes.data_as(C.c_void_p), status.ctypes.data_as(C.c_void_p)), "bj_decode_batch_resized", self.ctx)
        return status[:n]


    def submit_packed(self, src, src_off, src_len, dst, dst_off, fmt=L.BJ_OUT_RGB8, rois=None, scales=None, sizes=None):
        """decode_packed without waiting (bj_submit): returns a Job; job.wait() gives the status array."""
        n = len(src_off)
        ip = (np.asarray(src_off, dtype=np.uint64) + np.uint64(src.__array_interface__["data"][0]))
        il = np.ascontiguousarray(src_len, dtype=np.uint64)
        op = (np.asarray(dst_off, dtype=np.uint64) + np.uint64(dst.__array_interface__["data"][0]))
        ra, rp = _roi_table(rois, n)
        sa, sp = _scale_table(scales, n)
        za, zp = _size_table(sizes, n)
        status = np.zeros(max(n, 1), dtype=np.int32)
        h = C.c_void_p()
        L.check(L.lib().bj_submit_resized(self.ctx, ip.ctypes.data_as(C.c_void_p), il.ctypes.data_as(C.c_void_p), rp, sp, zp, n, fmt,
                                          op.ctypes.data_as(C.c_void_p), status.ctypes.data_as(C.c_void_p), C.byref(h)), "bj_submit_resized", self.ctx)
        return Job(self, h, (ip, il, op, ra, sa, za, src, dst), status, n)


def lpt_shards(costs, world_size):
    """Deal a stream of images over `world_size` ranks: longest processing time first - sort by cost (compressed size,
    the reference's sort key, src/decoder_host.cpp:46-61) descending and give each image to the rank with the least
    work so far.  Returns world_size index lists (each in ascending index order)."""
    import heapq
    order = sorted(range(len(costs)), key=lambda i: (-costs[i], i))
    heap = [(0, r) for r in range(world_size)]
    out = [[] for _ in range(world_size)]
    for i in order:
        load, r = heapq.heappop(heap)
        out[r].append(i)
        heapq.heappush(heap, (load + costs[i], r))
    return [sorted(o) for o in out]


def shard_by_size(sizes, world_size):
    """Deal images to ranks: sort ascending by compressed size (the reference sorts its inputs the same way,
    src/decoder_host.cpp:46-61,360), then round-robin.  Images are independent, so there is no collective on the
    data path.  Returns world_size index lists."""
    order = sorted(range(len(sizes)), key=lambda i: (sizes[i], i))
    return [order[r::world_size] for r in range(world_size)]


def decode_files(paths, device=0, rank=0, world_size=1, decoder=None):
    """The reference CLI's behaviour (src/decoder_host.cpp:352-394): every input gets `<name>.bmp` next to it
    (:328-330); unreadable / invalid files are reported and skipped (:120-123).  With world_size > 1 each rank
    takes its shard.  Returns {path: status}."""
    paths = list(paths)
    sizes = [os.path.getsize(p) if os.path.exists(p) else 0 for p in paths]
    mine = shard_by_size(sizes, world_size)[rank]
    dec = decoder or Decoder(device)
    files = []
    for i in mine:
        try:
            with open(paths[i], "rb") as f:
                files.append(f.read())
        except OSError:
            files.append(b"")
    outs, status = dec.decode(files, L.BJ_OUT_BMP)
    result = {}
    for i, o, st in zip(mine, outs, status):
        result[paths[i]] = st
        if o is None:
            print(f"Error - {paths[i]}: {L.lib().bj_status_string(st).decode()}")
            continue
        stem, dot, _ = paths[i].rpartition(".")
        with open((stem if dot else paths[i]) + ".bmp", "wb") as f:
            f.write(o.tobytes())
    return result
