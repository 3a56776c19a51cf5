#!/usr/bin/env python
"""Reduced-size decode on the config-2 batch (4096 x 500x375 4:2:0), RGB8, five arms in one process:

    whole   whole images at full size (scales=None: the path every other entry takes)
    s2      every image at 1/2 (250x188)
    s4      every image at 1/4 (125x94)
    s8      every image at 1/8 (63x47)
    rrc_s2  the random-resized-crop boxes of roi_bench.rrc_rois, mapped to the image at 1/2:
            x' = x // 2, y' = y // 2, w' = ceil((x + w) / 2) - x', h' = ceil((y + h) / 2) - y'

Per arm, one JSON line: device-resident ms per step with the stage times of bj_batch_get_info (staged path,
bj_batch_create_scaled; ms_idct is the IDCT + colour kernel), end-to-end ms per step (decode_packed from pinned host
buffers to pinned host buffers), images/s, the bytes copied out and the copy-out floor from a pinned 1 GB D2H measured in
the same run, and the GPU's name and power limit read in the same run.  The arms alternate (--reps rounds of --steps steps
each, after one round of warm-up).  Then 16 seeded images of each scaled arm are checked against box_scale of the same
images' whole decode.

    python scripts/scale_bench.py [--steps 10] [--reps 3] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import numpy as np  # noqa: E402

import bench  # noqa: E402  (workload_specs / generate; its main() is guarded)
from roi_bench import H, W, gpu_identity, rrc_rois  # noqa: E402


def box_scale(rgb, s):
    """Per channel, the rounded mean of each s x s box of rgb [H, W, 3], boxes cut short at the right and bottom edges."""
    h, w = rgb.shape[:2]
    ho, wo = -(-h // s), -(-w // s)
    acc = np.zeros((ho * s, wo * s, 3), np.uint32)
    acc[:h, :w] = rgb
    cnt = np.zeros((ho * s, wo * s), np.uint32)
    cnt[:h, :w] = 1
    S = acc.reshape(ho, s, wo, s, 3).sum((1, 3))
    N = cnt.reshape(ho, s, wo, s).sum((1, 3))[..., None]
    return ((S + N // 2) // N).astype(np.uint8)


def rrc_rois_scaled(n, s=2):
    """roi_bench's random-resized-crop boxes as rectangles of the image at 1/s: the boxes of the scaled image that cover them."""
    r = rrc_rois(n).astype(np.int64)
    x, y = r[:, 0] // s, r[:, 1] // s
    w, h = -(-(r[:, 0] + r[:, 2]) // s) - x, -(-(r[:, 1] + r[:, 3]) // s) - y
    return np.stack([x, y, w, h], axis=1).astype(np.uint32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default="")
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
    arms = {"whole": (None, None), "s2": (None, 2), "s4": (None, 4), "s8": (None, 8), "rrc_s2": (rrc_rois_scaled(n), 2)}

    pin_in, in_off, in_len = bench.pack_pinned(bj, blobs)
    state = {}
    for name, (rois, s) in arms.items():
        sizes = np.array([bj.scaled_output_size(d, None if rois is None else rois[i], s or 1, fmt) for i in range(n)], dtype=np.uint64)
        assert sizes.all(), name
        offs = np.concatenate([[0], np.cumsum((sizes + 15) // 16 * 16)]).astype(np.uint64)
        b = bj.Batch(dec, blobs, fmt, rois=rois, scales=s)
        b.upload()
        state[name] = {"rois": rois, "scale": s, "sizes": sizes, "offs": offs[:-1], "out_px": int(sizes.sum()) // 3, "batch": b,
                       "pin_out": bj.PinnedBuffer(int(offs[-1]) + 16), "res_ms": [], "stage": [], "e2e_ms": [], "e2e_stats": []}

    # what the copy-out can do at best: one pinned 1 GB device -> host copy
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
    stat_names = ["host_ms", "wait_ms", "d2h_bytes", "h2d_bytes", "sub_batches", "ms_idct"]

    def run_arm(s, record):
        b = s["batch"]
        for _ in range(args.steps):
            t0 = time.perf_counter()
            b.decode()
            b.sync()                                                  # ends in a device synchronise
            t1 = time.perf_counter()
            i = b.info()
            if record:
                s["res_ms"].append(1e3 * (t1 - t0))
                s["stage"].append((i.ms_unstuff, i.ms_sync, i.ms_write, i.ms_idct))
        for _ in range(args.steps):
            t0 = time.perf_counter()
            status = dec.decode_packed(pin_in.array, in_off, in_len, s["pin_out"].array, s["offs"], fmt, rois=s["rois"], scales=s["scale"])
            t1 = time.perf_counter()
            if status.any():
                raise SystemExit(f"scale_bench: {int((status != 0).sum())} images failed")
            if record:
                s["e2e_ms"].append(1e3 * (t1 - t0))
                s["e2e_stats"].append([dec.stat("decode_batch_" + k) for k in stat_names])

    for rep in range(args.reps + 1):                                  # round 0 is the warm-up
        for name in arms:
            run_arm(state[name], rep > 0)

    # the staged download: one copy per image (packed_outputs off), so d2h_bytes is the sum of the outputs
    dec.set_option("packed_outputs", 0)
    lines = []
    pixels = n * W * H
    for name, s in state.items():
        b = s["batch"]
        b.download()
        info = b.info()
        res = float(np.median(s["res_ms"]))
        e2e = float(np.median(s["e2e_ms"]))
        stage = np.mean(np.array(s["stage"]), axis=0)
        es = np.mean(np.array(s["e2e_stats"]), axis=0)
        line = {"arm": name, "scale": s["scale"] or 1, "images": n, "workload": desc, "format": "RGB8", "steps": args.steps, "reps": args.reps,
                "out_pixels": s["out_px"], "out_fraction": s["out_px"] / pixels,
                "resident": {"ms_per_step": res, "images_per_s": n / res * 1e3, "decoded_gpix_s": pixels / res / 1e6,
                             "ms_unstuff": stage[0], "ms_sync": stage[1], "ms_write": stage[2], "ms_idct": stage[3],
                             "timer": "host clock around bj_batch_decode + bj_batch_sync, median step"},
                "e2e": {"ms_per_step": e2e, "images_per_s": n / e2e * 1e3, "decoded_gpix_s": pixels / e2e / 1e6, "host_prepare_ms": es[0],
                        "host_wait_ms": es[1], "d2h_bytes_per_step": int(es[2]), "h2d_bytes_per_step": int(es[3]), "sub_batches": int(es[4]),
                        "ms_idct_summed_over_sub_batches": es[5], "d2h_floor_ms": es[2] / (d2h_gbs * 1e9) * 1e3,
                        "timer": "host clock around the blocking decode_packed call (pinned in, pinned out, packed_outputs=1), median step"},
                "d2h_bytes": int(info.d2h_bytes), "sum_scaled_output_size": int(s["sizes"].sum()),
                "d2h_equals_sum_scaled_output_size": int(info.d2h_bytes) == int(s["sizes"].sum()),
                "out_bytes": int(info.out_bytes), "pinned_d2h_gbs": d2h_gbs, **ident}
        lines.append(line)
        print(json.dumps(line), flush=True)

    # parity: the scaled outputs of 16 seeded images == box_scale of the same images' whole decode, cropped
    rng = np.random.default_rng(16)
    pick = sorted(int(i) for i in rng.choice(n, size=16, replace=False))
    whole = state["whole"]
    mism = 0
    for name in ("s2", "s4", "s8", "rrc_s2"):
        s = state[name]
        for i in pick:
            full = whole["pin_out"].array[int(whole["offs"][i]):int(whole["offs"][i]) + int(whole["sizes"][i])].reshape(H, W, 3)
            small = box_scale(full, s["scale"])
            x, y, w, h = (0, 0, small.shape[1], small.shape[0]) if s["rois"] is None else (int(v) for v in s["rois"][i])
            got = s["pin_out"].array[int(s["offs"][i]):int(s["offs"][i]) + int(s["sizes"][i])]
            mism += not np.array_equal(got, small[y:y + h, x:x + w].reshape(-1))
    check = {"check": "scaled outputs of 16 seeded images (every scaled arm, last end-to-end step) == box_scale of their whole decode, cropped",
             "images": pick, "mismatches": mism}
    lines.append(check)
    print(json.dumps(check), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            for ln in lines:
                f.write(json.dumps(ln) + "\n")
    for s in state.values():
        s["batch"].destroy()
        s["pin_out"].free()
    pin_in.free()
    dec.close()
    if mism:
        raise SystemExit(f"scale_bench: {mism} scaled outputs differ from box_scale of the whole decode")


if __name__ == "__main__":
    main()
