"""A context of one device is the same whichever entry made it: bj_create(0) and bj_create_multi([0]) decode the same
mixed batch (damaged files included) to the same bytes, statuses and counters, and refuse the same option values."""
import ctypes as C
import hashlib
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

COUNTERS = ["sub_batches", "launches", "h2d_bytes", "d2h_bytes", "host_ms", "wait_ms", "d2h_copies",
            "ms_unstuff", "ms_sync", "ms_write", "ms_idct", "direct_uploads"]
COUNTS = ["sub_batches", "launches", "h2d_bytes", "d2h_bytes", "d2h_copies", "direct_uploads"]


def _files(golden, golden_dir):
    names = sorted(golden) * 3
    return names, [open(os.path.join(golden_dir, golden[n]["file"]), "rb").read() for n in names]


def _out_size(bj, data):
    """What a decode may write for a file: sized from its headers alone (a scan's end is found on the device)."""
    d = bj.ImageDesc()
    buf = np.frombuffer(data, dtype=np.uint8)
    ok = bj.lib().bj_peek_header(buf.ctypes.data_as(C.c_void_p), len(data), C.byref(d)) == 0
    return bj.lib().bj_output_size(C.byref(d), bj.BJ_OUT_BMP) if ok else 0


def _decode_twice(bj, dec, files):
    """Two calls on small sub-batches: pageable inputs into one buffer per image, then pinned inputs into one packed
    output buffer.  Returns (outputs, statuses, decode_batch_* counters) of each call and the total_* counters."""
    dec.set_option("sub_batch_bytes", 1 << 16)
    calls = []
    outs, status = dec.decode(files, bj.BJ_OUT_BMP)
    calls.append(([o.tobytes() if o is not None else None for o in outs], status,
                  {k: dec.stat("decode_batch_" + k) for k in COUNTERS}))
    sizes = [_out_size(bj, f) for f in files]
    dst_off = np.concatenate([[0], np.cumsum([(s + 15) // 16 * 16 for s in sizes])]).astype(np.int64)
    src = bj.PinnedBuffer(sum(len(f) for f in files))
    dst = bj.PinnedBuffer(int(dst_off[-1]) + 16)
    try:
        src_off = np.concatenate([[0], np.cumsum([len(f) for f in files])[:-1]]).astype(np.int64)
        for f, o in zip(files, src_off):
            src.array[o:o + len(f)] = np.frombuffer(f, dtype=np.uint8)
        dec.set_option("packed_outputs", 1)
        st = dec.decode_packed(src.array, src_off, [len(f) for f in files], dst.array, dst_off[:-1], bj.BJ_OUT_BMP)
        calls.append(([dst.array[o:o + n].tobytes() if s == 0 else None for o, n, s in zip(dst_off, sizes, st)], list(st),
                      {k: dec.stat("decode_batch_" + k) for k in COUNTERS}))
    finally:
        src.free()
        dst.free()
    return calls, {k: dec.stat("total_" + k) for k in COUNTERS}


def test_single_device_context_either_way(golden, golden_dir):
    import pim_jpeg_decoder_b200 as bj
    names, files = _files(golden, golden_dir)
    single, multi = bj.Decoder(0), bj.Decoder(devices=[0])
    try:
        assert single.stat("devices") == multi.stat("devices") == 1
        assert single.device_count == multi.device_count == 1
        assert single.stat("host_threads") == multi.stat("host_threads")
        runs = [_decode_twice(bj, d, files) for d in (single, multi)]
        for calls, totals in runs:
            assert calls[1][2]["direct_uploads"] > 0 and calls[0][2]["direct_uploads"] == 0
            for k in COUNTERS:                       # totals: the sum of the two calls since the context was made
                assert totals[k] == calls[0][2][k] + calls[1][2][k], k
            for outs, status, _ in calls:
                for n, o, s in zip(names, outs, status):
                    if golden[n].get("invalid"):
                        assert s == bj.BJ_ERR_INVALID_JPEG and o is None, n
                    else:
                        assert s == 0 and hashlib.sha256(o).hexdigest() == golden[golden[n]["expect"]]["bmp_sha256"], n
        (calls_s, _), (calls_m, _) = runs
        for (outs_s, st_s, cnt_s), (outs_m, st_m, cnt_m) in zip(calls_s, calls_m):
            assert st_s == st_m and outs_s == outs_m
            assert cnt_s["sub_batches"] > 3
            for k in COUNTS:
                assert cnt_s[k] == cnt_m[k], k
        for dec in (single, multi):
            for name, value in [("subseq_bits", 100), ("slices", 3), ("host_threads", 0), ("sync_phased", 0), ("idct_tma", 1)]:
                with pytest.raises(bj.BjError):
                    dec.set_option(name, value)
    finally:
        single.close()
        multi.close()
