#!/usr/bin/env python
"""Progressive (SOF2) decode on the config-2 seeds (500x375 4:2:0 q90), each encoded by Pillow as a progressive file and
as its baseline twin, RGB8, five arms alternating in one process:

    baseline     the 4096 baseline twins
    progressive  the 4096 progressive files
    mixed        50/50: even seeds progressive, odd seeds baseline
    prog_rst     the progressive files written with a restart marker every --rst MCUs (more work items per scan)
    latency_4k   one 3840x2160 progressive image

Per arm, one JSON line: device-resident ms per step (staged Batch: host clock around bj_batch_decode + bj_batch_sync),
the progressive stage's ms and launches (decode_batch_ms_progressive, decode_batch_launches of the one-call path),
end-to-end ms per step (bj_decode_batch into preallocated host buffers), host ms per batch (decode_batch_host_ms: header
parse, the progressive files' scan walk, layout, staging), and the longest work item's entropy-coded bytes (one restart
segment of one scan: the critical path of a level).  Then 16 seeded images of every arm are checked against the GPU's
decode of their twins.  The GPU's name and power limit are read in the same run.

    python scripts/progressive_bench.py [--steps 5] [--reps 3] [--n 4096] [--rst 8] [--out FILE]
"""
import argparse
import concurrent.futures as cf
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "scripts"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)

import numpy as np  # noqa: E402

from roi_bench import gpu_identity  # noqa: E402


def _twins(args):
    import jpeg_synth as js
    import prog_synth as ps
    w, h, seed, rst = args
    return ps.pil_twins(js.synth_rgb(w, h, seed), 90, 2, rst)


def longest_item(data):
    """entropy-coded bytes of the longest restart segment of any scan of a progressive file"""
    best, i = 0, 2
    while True:
        i = data.find(b"\xFF\xDA", i)
        if i < 0:
            return best
        s = i + 2 + ((data[i + 2] << 8) | data[i + 3])
        j, seg0 = s, s
        while True:
            j = data.index(b"\xFF", j)
            m = data[j + 1]
            if m == 0x00 or m == 0xFF:
                j += 1 if m == 0xFF else 2
                continue
            best = max(best, j - seg0)
            if 0xD0 <= m <= 0xD7:
                j += 2
                seg0 = j
                continue
            break
        i = j


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--n", type=int, default=4096)
    ap.add_argument("--rst", type=int, default=8)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    ident = gpu_identity()
    specs = [(500, 375, i, 0) for i in range(a.n)]
    with cf.ProcessPoolExecutor(max_workers=min(32, os.cpu_count() or 1)) as ex:
        pairs = list(ex.map(_twins, specs, chunksize=64))
        rst_pairs = list(ex.map(_twins, [(500, 375, i, a.rst) for i in range(a.n)], chunksize=64))
    big = _twins((3840, 2160, 7, 0))
    import pim_jpeg_decoder_b200 as bj
    dec = bj.Decoder(0)
    dec.set_option("progressive", 1)
    arms = {
        "baseline": ([t for _, t in pairs], [t for _, t in pairs]),
        "progressive": ([p for p, _ in pairs], [t for _, t in pairs]),
        "mixed": ([p if i % 2 == 0 else t for i, (p, t) in enumerate(pairs)], [t for _, t in pairs]),
        "prog_rst": ([p for p, _ in rst_pairs], [t for _, t in rst_pairs]),
        "latency_4k": ([big[0]], [big[1]]),
    }
    outs = {k: [np.empty(500 * 375 * 3 if k != "latency_4k" else 3840 * 2160 * 3, np.uint8) for _ in f] for k, (f, _) in arms.items()}
    batches = {k: bj.Batch(dec, f, 0) for k, (f, _) in arms.items()}
    for b in batches.values():
        b.upload()
    res = {k: {"dev_ms": [], "e2e_ms": [], "prog_ms": [], "host_ms": [], "launches": None} for k in arms}
    for rep in range(a.reps + 1):                       # round 0 warms up every arm
        for k, (files, _) in arms.items():
            b = batches[k]
            t0 = time.perf_counter()
            for _ in range(a.steps):
                b.decode(); b.sync()
            dev = (time.perf_counter() - t0) * 1e3 / a.steps
            t0 = time.perf_counter()
            pr, hm = 0.0, 0.0
            for _ in range(a.steps):
                _, st = dec.decode(files, 0, outs=outs[k])
                pr += dec.stat("decode_batch_ms_progressive"); hm += dec.stat("decode_batch_host_ms")
            e2e = (time.perf_counter() - t0) * 1e3 / a.steps
            assert all(s == 0 for s in st), k
            if rep:
                r = res[k]
                r["dev_ms"].append(round(dev, 3)); r["e2e_ms"].append(round(e2e, 3))
                r["prog_ms"].append(round(pr / a.steps, 3)); r["host_ms"].append(round(hm / a.steps, 3))
                r["launches"] = dec.stat("decode_batch_launches")
    # parity: 16 seeded images per arm against the decode of their twins
    rng = np.random.default_rng(0)
    lines = []
    for k, (files, twins) in arms.items():
        pick = sorted(set(rng.integers(0, len(files), size=16).tolist()))
        got, _ = dec.decode([files[i] for i in pick], 0)
        want, _ = dec.decode([twins[i] for i in pick], 0)
        ok = sum(int(np.array_equal(g, w)) for g, w in zip(got, want))
        longest = max(longest_item(f) for f in files if f[2:].find(b"\xFF\xC2") >= 0) if any(b"\xFF\xC2" in f for f in files) else 0
        r = res[k]
        line = dict(arm=k, images=len(files), **{m: r[m] for m in ("dev_ms", "e2e_ms", "prog_ms", "host_ms", "launches")},
                    longest_item_bytes=longest, parity=f"{ok}/{len(pick)}", **ident)
        lines.append(line)
        print(json.dumps(line), flush=True)
    for b in batches.values():
        b.destroy()
    dec.close()
    if a.out:
        with open(a.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
