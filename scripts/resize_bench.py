#!/usr/bin/env python
"""Fixed-size output on the config-2 batch (4096 x 500x375 4:2:0), RGB8, 224 x 224 per image, four arms in one process:

    host      today's pipeline: roi_bench.rrc_rois boxes decoded at full size (bj_decode_batch_roi), then resized to
              224 x 224 on the host with the same integer bilinear (resize_ref.bilinear, numpy, one image at a time)
    rrc_plan  the same boxes resized in the library, resize_plan choosing the scale and the ROI
    rrc_s1    the same at s = 1 (the box itself, no prescale)
    whole     whole images resized to 224 x 224 in the library

Per arm, one JSON line: device-resident ms per step (staged Batch, host clock around bj_batch_decode + bj_batch_sync),
end-to-end ms per step (decode_packed from pinned host buffers into one pinned [n, 224, 224, 3] array, or the arm's
crops for `host`), the host resize's ms per batch for `host` (the work this feature removes), the copy-out bytes and the
D2H floor from a pinned 1 GB copy in the same run, and the k_resize_bilinear kernel time from a separate torch.profiler
run with its bytes/s over (source bytes read + output bytes written).  The arms alternate (--reps rounds of --steps
steps after one round of warm-up; the host resize runs --host-steps times).  Then 16 seeded images of every arm are
checked against bilinear(crop(box_scale(whole decode, s))).  The GPU's name and power limit are read in the same run.

    python scripts/resize_bench.py [--steps 10] [--reps 3] [--host-steps 2] [--out FILE] [--trace-dir DIR]
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "scripts"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)

import numpy as np  # noqa: E402

import bench  # noqa: E402  (workload_specs / generate; its main() is guarded)
from resize_ref import bilinear  # noqa: E402
from roi_bench import H, W, gpu_identity, rrc_rois  # noqa: E402
from scale_bench import box_scale  # noqa: E402

TW, TH = 224, 224


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--host-steps", type=int, default=2)
    ap.add_argument("--out", default="")
    ap.add_argument("--trace-dir", default="")
    args = ap.parse_args()

    specs, desc = bench.workload_specs("config2", 4096, 1024, 0)
    blobs = bench.generate(specs, min(32, os.cpu_count() or 1))     # CPU, before CUDA comes up
    n = len(blobs)

    import torch
    import pim_jpeg_decoder_b200 as bj
    fmt = bj.BJ_OUT_RGB8
    ident = gpu_identity()
    ident["torch_device"] = torch.cuda.get_device_name(0)
    dec = bj.Decoder(0)
    st, d = bj.parse_header(blobs[0])
    assert st == 0 and (d.width, d.height) == (W, H)

    boxes = rrc_rois(n)
    plans = [bj.resize_plan(W, H, b, (TW, TH)) for b in boxes]
    arms = {
        "host": {"rois": boxes, "scales": None, "sizes": None},
        "rrc_plan": {"rois": np.array([r for _, r in plans], dtype=np.uint32), "scales": np.array([s for s, _ in plans], dtype=np.uint8), "sizes": (TW, TH)},
        "rrc_s1": {"rois": boxes, "scales": None, "sizes": (TW, TH)},
        "whole": {"rois": None, "scales": None, "sizes": (TW, TH)},
    }
    pin_in, in_off, in_len = bench.pack_pinned(bj, blobs)
    for name, a in arms.items():
        sizes = np.array([bj.resized_output_size(d, None if a["rois"] is None else a["rois"][i], 1 if a["scales"] is None else a["scales"][i],
                                                 a["sizes"], fmt) for i in range(n)], dtype=np.uint64)
        assert sizes.all(), name
        offs = np.concatenate([[0], np.cumsum((sizes + 15) // 16 * 16)]).astype(np.uint64)
        a["out_sizes"], a["offs"] = sizes, offs[:-1]
        a["pin_out"] = bj.PinnedBuffer(int(offs[-1]) + 16)
        a["batch"] = bj.Batch(dec, blobs, fmt, rois=a["rois"], scales=a["scales"], sizes=a["sizes"])
        a["batch"].upload()
        # source bytes the resize reads: the scaled crops (what k_idct_color writes for it)
        a["src_bytes"] = 0 if a["sizes"] is None else sum(
            bj.scaled_output_size(d, None if a["rois"] is None else a["rois"][i], 1 if a["scales"] is None else a["scales"][i], fmt) for i in range(n))
        a.update(res_ms=[], e2e_ms=[], e2e_stats=[], stage=[], host_ms=[])

    # the copy-out's floor: one pinned 1 GB device -> host copy
    src = torch.empty(1 << 30, dtype=torch.uint8, device="cuda")
    dst = torch.empty(1 << 30, dtype=torch.uint8, pin_memory=True)
    d2h_gbs = 0.0
    for _ in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize()
        d2h_gbs = max(d2h_gbs, (1 << 30) / (time.perf_counter() - t0) / 1e9)
    del src, dst

    dec.set_option("packed_outputs", 1)
    stat_names = ["host_ms", "wait_ms", "d2h_bytes", "sub_batches", "ms_idct", "ms_resize"]

    def host_resize(a, out):
        for i in range(n):
            x, y, w, h = (int(v) for v in a["rois"][i])
            c = a["pin_out"].array[int(a["offs"][i]):int(a["offs"][i]) + int(a["out_sizes"][i])].reshape(h, w, 3)
            out[i] = bilinear(c, TW, TH)

    def run_arm(a, record):
        b = a["batch"]
        for _ in range(args.steps):
            t0 = time.perf_counter()
            b.decode()
            b.sync()                                                  # ends in a device synchronise
            t1 = time.perf_counter()
            i = b.info()
            if record:
                a["res_ms"].append(1e3 * (t1 - t0))
                a["stage"].append((i.ms_entropy, i.ms_idct))
        for _ in range(args.steps):
            t0 = time.perf_counter()
            status = dec.decode_packed(pin_in.array, in_off, in_len, a["pin_out"].array, a["offs"], fmt, rois=a["rois"], scales=a["scales"], sizes=a["sizes"])
            t1 = time.perf_counter()
            if status.any():
                raise SystemExit(f"resize_bench: {int((status != 0).sum())} images failed")
            if record:
                a["e2e_ms"].append(1e3 * (t1 - t0))
                a["e2e_stats"].append([dec.stat("decode_batch_" + k) for k in stat_names])

    for rep in range(args.reps + 1):                                  # round 0 is the warm-up
        for name in arms:
            run_arm(arms[name], rep > 0)
    host_out = np.zeros((n, TH, TW, 3), np.uint8)
    for _ in range(args.host_steps):
        t0 = time.perf_counter()
        host_resize(arms["host"], host_out)
        arms["host"]["host_ms"].append(1e3 * (time.perf_counter() - t0))

    # k_resize_bilinear's kernel time: torch.profiler over the staged decode of each resizing arm, a run of its own
    kern = {}
    from torch.profiler import ProfilerActivity, profile
    for name, a in arms.items():
        if a["sizes"] is None:
            continue
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.steps):
                a["batch"].decode()
                a["batch"].sync()
        ev = [e for e in prof.events() if "k_resize_bilinear" in e.name]
        us = [e.device_time for e in ev] if ev and hasattr(ev[0], "device_time") else [e.cuda_time for e in ev]
        kern[name] = {"launches": len(us), "ms_median": float(np.median(us)) / 1e3 if us else None}
        if args.trace_dir:
            os.makedirs(args.trace_dir, exist_ok=True)
            with open(os.path.join(args.trace_dir, f"resize_{name}_kernels.txt"), "w") as f:
                f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=20))

    dec.set_option("packed_outputs", 0)
    lines = []
    for name, a in arms.items():
        b = a["batch"]
        b.download()
        info = b.info()
        es = np.mean(np.array(a["e2e_stats"]), axis=0)
        out_bytes = int(a["out_sizes"].sum())
        line = {"arm": name, "images": n, "workload": desc, "format": "RGB8", "target": [TW, TH], "steps": args.steps, "reps": args.reps,
                "scales_used": {int(s): int(c) for s, c in zip(*np.unique(a["scales"] if a["scales"] is not None else np.ones(n, np.uint8), return_counts=True))},
                "resident": {"ms_per_step": float(np.median(a["res_ms"])), "ms_entropy": float(np.mean([s[0] for s in a["stage"]])),
                             "ms_idct": float(np.mean([s[1] for s in a["stage"]])),
                             "timer": "host clock around bj_batch_decode + bj_batch_sync, median step"},
                "e2e": {"ms_per_step": float(np.median(a["e2e_ms"])), "host_prepare_ms": es[0], "host_wait_ms": es[1], "d2h_bytes_per_step": int(es[2]),
                        "sub_batches": int(es[3]), "ms_idct_summed": es[4], "ms_resize_summed": es[5],
                        "d2h_floor_ms": es[2] / (d2h_gbs * 1e9) * 1e3,
                        "timer": "host clock around the blocking decode_packed call (pinned in, pinned out, packed_outputs=1), median step"},
                "copy_out_bytes": out_bytes, "d2h_bytes_staged": int(info.d2h_bytes), "pinned_d2h_gbs": d2h_gbs, **ident}
        if name == "host":
            hm = float(np.median(a["host_ms"]))
            line["host_resize_ms_per_batch"] = hm
            line["host_resize_note"] = f"numpy integer bilinear, one image at a time, one thread, median of {args.host_steps} batches"
            line["e2e_plus_host_resize_ms"] = line["e2e"]["ms_per_step"] + hm
        else:
            k = kern[name]
            moved = a["src_bytes"] + out_bytes
            line["k_resize_bilinear"] = {"ms": k["ms_median"], "launches_profiled": k["launches"], "source_bytes": int(a["src_bytes"]),
                                         "output_bytes": out_bytes,
                                         "gb_s": moved / (k["ms_median"] * 1e-3) / 1e9 if k["ms_median"] else None,
                                         "timer": "torch.profiler CUDA activity, separate run, median over steps"}
        lines.append(line)
        print(json.dumps(line), flush=True)

    # parity: 16 seeded images of every arm == bilinear(crop(box_scale(whole decode, s), roi)); whole decode from the library
    rng = np.random.default_rng(16)
    pick = sorted(int(i) for i in rng.choice(n, size=16, replace=False))
    whole, wst = dec.decode([blobs[i] for i in pick], fmt)
    assert all(s == 0 for s in wst)
    mism = {}
    for name, a in arms.items():
        m = 0
        for j, i in enumerate(pick):
            full = whole[j].reshape(H, W, 3)
            s = 1 if a["scales"] is None else int(a["scales"][i])
            x, y, w, h = (0, 0, W, H) if a["rois"] is None else (int(v) for v in a["rois"][i])
            want = bilinear(box_scale(full, s)[y:y + h, x:x + w], TW, TH)
            got = host_out[i] if name == "host" else a["pin_out"].array[int(a["offs"][i]):int(a["offs"][i]) + int(a["out_sizes"][i])].reshape(TH, TW, 3)
            m += not np.array_equal(got, want)
        mism[name] = m
    check = {"check": "16 seeded images per arm (last end-to-end step) == bilinear(crop(box_scale(whole decode, s), roi), 224, 224)",
             "images": pick, "mismatches": mism}
    lines.append(check)
    print(json.dumps(check), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            for ln in lines:
                f.write(json.dumps(ln) + "\n")
    for a in arms.values():
        a["batch"].destroy()
        a["pin_out"].free()
    pin_in.free()
    dec.close()
    if any(mism.values()):
        raise SystemExit(f"resize_bench: mismatches {mism}")


if __name__ == "__main__":
    main()
