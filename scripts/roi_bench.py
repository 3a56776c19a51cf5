#!/usr/bin/env python
"""Region-of-interest decode on the config-2 batch (4096 x 500x375 4:2:0), three arms in one process:

    whole   whole images (rois=None: the path every other entry takes)
    centre  a centre crop of 224x224 per image
    rrc     random-resized-crop boxes: area 8-100 % of the image, aspect 3/4-4/3 (numpy, fixed seed; the box only,
            no resize), like a training data loader's

Per arm, one JSON line: device-resident ms per step with the stage times of bj_batch_get_info (staged path,
bj_batch_create_roi), end-to-end ms per step (decode_packed from pinned host buffers to pinned host buffers), images/s,
output and decoded Gpixel/s, the bytes copied out, and the GPU's name and power limit read in the same run.  The arms
alternate (--reps rounds of --steps steps each, after one round of warm-up).  Then 16 seeded images of each crop arm
are checked against the crop of the same images' whole decode.

    python scripts/roi_bench.py [--steps 10] [--reps 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import bench  # noqa: E402  (workload_specs / generate; its main() is guarded)

W, H = 500, 375


def centre_rois(n, size=224):
    return np.tile(np.array([(W - size) // 2, (H - size) // 2, size, size], dtype=np.uint32), (n, 1))


def rrc_rois(n, seed=0, scale=(0.08, 1.0), ratio=(3 / 4, 4 / 3)):
    """The box of torchvision's RandomResizedCrop: 10 tries at a random area and log-uniform aspect, else the whole image."""
    rng = np.random.default_rng(seed)
    out = np.zeros((n, 4), dtype=np.uint32)
    for i in range(n):
        box = (0, 0, W, H)
        for _ in range(10):
            area = W * H * rng.uniform(*scale)
            aspect = np.exp(rng.uniform(np.log(ratio[0]), np.log(ratio[1])))
            w, h = int(round(np.sqrt(area * aspect))), int(round(np.sqrt(area / aspect)))
            if 0 < w <= W and 0 < h <= H:
                box = (int(rng.integers(0, W - w + 1)), int(rng.integers(0, H - h + 1)), w, h)
                break
        out[i] = box
    return out


def gpu_identity():
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        name, power, clk = (x.strip() for x in r.stdout.strip().split(","))
        return {"gpu": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:                                          # (reported, not hidden: the numbers need the card)
        return {"gpu": None, "power_limit": None, "error": str(e)}


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
    arms = {"whole": None, "centre": centre_rois(n), "rrc": rrc_rois(n)}

    pin_in, in_off, in_len = bench.pack_pinned(bj, blobs)
    state = {}
    for name, rois in arms.items():
        sizes = np.array([bj.roi_output_size(d, None if rois is None else rois[i], fmt) for i in range(n)], dtype=np.uint64)
        offs = np.concatenate([[0], np.cumsum((sizes + 15) // 16 * 16)]).astype(np.uint64)
        out_px = int(sizes.sum()) // 3
        b = bj.Batch(dec, blobs, fmt, rois=rois)
        b.upload()
        state[name] = {"rois": rois, "sizes": sizes, "offs": offs[:-1], "out_px": out_px, "batch": b,
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
            status = dec.decode_packed(pin_in.array, in_off, in_len, s["pin_out"].array, s["offs"], fmt, rois=s["rois"])
            t1 = time.perf_counter()
            if status.any():
                raise SystemExit(f"roi_bench: {int((status != 0).sum())} images failed")
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
        line = {"arm": name, "images": n, "workload": desc, "format": "RGB8", "steps": args.steps, "reps": args.reps,
                "out_pixels": s["out_px"], "out_fraction": s["out_px"] / pixels,
                "resident": {"ms_per_step": res, "images_per_s": n / res * 1e3, "output_gpix_s": s["out_px"] / res / 1e6,
                             "decoded_gpix_s": pixels / res / 1e6, "ms_unstuff": stage[0], "ms_sync": stage[1], "ms_write": stage[2],
                             "ms_idct": stage[3], "timer": "host clock around bj_batch_decode + bj_batch_sync, median step"},
                "e2e": {"ms_per_step": e2e, "images_per_s": n / e2e * 1e3, "output_gpix_s": s["out_px"] / e2e / 1e6,
                        "decoded_gpix_s": pixels / e2e / 1e6, "host_prepare_ms": es[0], "host_wait_ms": es[1],
                        "d2h_bytes_per_step": int(es[2]), "h2d_bytes_per_step": int(es[3]), "sub_batches": int(es[4]),
                        "ms_idct_summed_over_sub_batches": es[5], "d2h_floor_ms": es[2] / (d2h_gbs * 1e9) * 1e3,
                        "timer": "host clock around the blocking decode_packed call (pinned in, pinned out, packed_outputs=1), median step"},
                "d2h_bytes": int(info.d2h_bytes), "sum_roi_output_size": int(s["sizes"].sum()),
                "d2h_equals_sum_roi_output_size": int(info.d2h_bytes) == int(s["sizes"].sum()),
                "out_bytes": int(info.out_bytes), "pinned_d2h_gbs": d2h_gbs, **ident}
        lines.append(line)
        print(json.dumps(line), flush=True)

    # parity: the ROI outputs of 16 seeded images == the crops of the same images' whole decode
    rng = np.random.default_rng(16)
    pick = sorted(int(i) for i in rng.choice(n, size=16, replace=False))
    whole = state["whole"]
    mism = 0
    for name in ("centre", "rrc"):
        s = state[name]
        for i in pick:
            full = whole["pin_out"].array[int(whole["offs"][i]):int(whole["offs"][i]) + int(whole["sizes"][i])].reshape(H, W, 3)
            x, y, w, h = (int(v) for v in s["rois"][i])
            got = s["pin_out"].array[int(s["offs"][i]):int(s["offs"][i]) + int(s["sizes"][i])]
            mism += not np.array_equal(got, full[y:y + h, x:x + w].reshape(-1))
    check = {"check": "ROI outputs of 16 seeded images (both crop arms, last end-to-end step) == crops of their whole decode",
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
        raise SystemExit(f"roi_bench: {mism} ROI outputs differ from the crops of the whole decode")


if __name__ == "__main__":
    main()
