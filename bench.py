#!/usr/bin/env python
"""Benchmark of the B200 JPEG decode back end (contract: see the task statement / DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload config2|config3|config4|config5|compat] [--batch B]
    python bench.py --workload config5 --stream 65536      # BASELINE configs[4]: one stream dealt over the ranks (strong scaling)
    python bench.py --impl reference ...        # the reference's own CPU implementation on the host cores

A "step" = one pass of the hot path (un-stuff, Huffman decode, dequantise, IDCT, upsample, colour, BMP bytes)
over one batch of synthetic JPEGs.  Default workload = BASELINE.json configs[1]: 4096 baseline 4:2:0 q=90 JPEGs of
500x375.  `value` = Mpixel/s with the compressed batch already resident in HBM (CUDA events on the launching
stream, max over ranks); `e2e` = the same through the one-call C ABI with host buffers (H2D + D2H inside).
One process per GPU; images are sharded by rank, there is no collective on the data path (scaling = weak).
"""
import argparse
import concurrent.futures as cf
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

METRIC = "decoded_mpixel_per_s"
UNIT = "Mpixel/s"

MIX = [((500, 375), 0.40), ((375, 500), 0.15), ((640, 480), 0.15), ((224, 224), 0.10), ((1024, 768), 0.10),
       ((1920, 1080), 0.07), ((3840, 2160), 0.03)]


def _strip_comments(text):
    """C/C++ source without comments and with runs of white space collapsed (string literals are kept as they are)."""
    out, i, n = [], 0, len(text)
    while i < n:
        c = text[i]
        if c == '"' or c == "'":
            j = i + 1
            while j < n and text[j] != c:
                j += 2 if text[j] == "\\" else 1
            out.append(text[i:j + 1]); i = j + 1
        elif text.startswith("//", i):
            j = text.find("\n", i)
            i = n if j < 0 else j
        elif text.startswith("/*", i):
            j = text.find("*/", i + 2)
            i = n if j < 0 else j + 2
            out.append(" ")
        else:
            out.append(c); i += 1
    return " ".join("".join(out).split())


def kernel_sources_sha(root=None):
    """Identifies the DEVICE code a profile was taken from (profiles/ncu_traffic.json carries the same key): the kernel
    files and the headers they share with nothing but the emulator, comments and white space removed (a reworded comment
    does not change what a kernel moves through DRAM); host-only files (batch.h, bj_host.h, parse.h) do not either."""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(root or ROOT, "pim_jpeg_decoder_b200", "csrc")
    for f in ("kernels_huff.cuh", "kernels_idct.cuh", "idct_color.cuh", "huff_core.h", "bj_dev.h"):
        h.update(_strip_comments(open(os.path.join(d, f), "r", encoding="utf-8").read()).encode())
    return h.hexdigest()[:16]


def stream_pool_specs(unique):
    """The pool of BASELINE configs[4] (SURVEY 8d): `unique` files, sizes drawn with default_rng(5) from the fixed mix;
    the same on every rank - the stream is ONE list that the ranks share out."""
    rng = np.random.default_rng(5)
    sizes = rng.choice(len(MIX), size=unique, p=[m[1] for m in MIX])
    return [(MIX[s][0][0], MIX[s][0][1], 5_000_000 + i, 2, False, 0) for i, s in enumerate(sizes)]


def workload_specs(name, batch, unique, rank):
    """-> (list of (w, h, seed, subsampling, gray, restart_blocks), description)"""
    base = rank * 1_000_003
    if name == "config2":
        u = min(unique, batch)
        pool = [(500, 375, base + i, 2, False, 0) for i in range(u)]
        return [pool[i % u] for i in range(batch)], f"{batch} x 500x375 4:2:0 q=90 baseline JPEG ({u} unique seeds, cycled)"
    if name == "config3":
        return [(3840, 2160, base, 2, False, 8)] * batch, f"{batch} x 3840x2160 4:2:0 q=90 restart interval 8 MCUs"
    if name == "config4":
        one = [(3840, 2160, base + 1, 0, False, 0), (3840, 2160, base + 2, 2, True, 0)]
        return [one[i % 2] for i in range(batch)], f"{batch} x 3840x2160 (4:4:4 and gray alternating), no restart markers"
    if name == "config5":
        rng = np.random.default_rng(5 + rank)
        u = min(unique, batch)
        sizes = rng.choice(len(MIX), size=u, p=[m[1] for m in MIX])
        pool = [(MIX[s][0][0], MIX[s][0][1], base + i, 2, False, 0) for i, s in enumerate(sizes)]
        return [pool[i % u] for i in range(batch)], f"{batch} mixed-size 4:2:0 q=90 JPEGs ({u} unique, cycled; SURVEY 8d mix)"
    raise SystemExit(f"unknown workload {name}")


def _gen(spec):
    import jpeg_synth as js
    w, h, seed, sub, gray, ri = spec
    return js.synth_jpeg(w, h, seed, subsampling=sub, gray=gray, restart_blocks=ri)


def generate(specs, workers):
    uniq = sorted(set(specs))
    if workers > 1 and len(uniq) > 8:
        with cf.ProcessPoolExecutor(max_workers=workers) as ex:        # before any CUDA initialisation (fork)
            data = list(ex.map(_gen, uniq, chunksize=max(1, len(uniq) // (workers * 4))))
    else:
        data = [_gen(s) for s in uniq]
    table = dict(zip(uniq, data))
    return [table[s] for s in specs]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the timed region runs (profiling guide's clocks line)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index, interval_ms=100):
        self.index = index
        self.rows = []
        self.proc = None
        self.interval_ms = interval_ms

    def start(self):
        if self.interval_ms <= 0:
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", str(self.interval_ms)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
            t0 = time.perf_counter()                # NVML start-up can stall the GPU for seconds: wait it out here,
            while not self.rows and time.perf_counter() - t0 < 20:    # not inside a timed step
                time.sleep(0.05)
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()

    def summary(self, windows):
        rows = [r for t, r in self.rows if any(a <= t <= b for a, b in windows)] or [r for _, r in self.rows]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        try:
            sm = sorted(float(r[0]) for r in rows)
            mx = max(float(r[1]) for r in rows)
        except ValueError:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": len(rows)}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) > 3 + k and r[3 + k].lower().startswith("active") for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": mx, "reasons": reasons, "samples": len(rows)}


# ------------------------------------------------------------------------------------------------ reference arm

def reference_binary():
    p = os.path.join(ROOT, "oracle", "_ref", "decoder")
    return p if os.path.exists(p) else None


def _ref_run(args):
    files, nr_dpus = args
    env = dict(os.environ, ORACLE_NR_DPUS=str(nr_dpus))
    t = time.perf_counter()
    subprocess.run([reference_binary()] + files, env=env, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, check=True)
    return time.perf_counter() - t


def _port_run(files):
    import oracle_lib as ol
    t = time.perf_counter()
    for f in files:
        data = open(f, "rb").read()
        r = ol.Restated(data, 0)
        with open(f[:-4] + ".bmp", "wb") as o:
            o.write(r.bmp.tobytes())
    return time.perf_counter() - t


class CpuReference:
    """The reference's own CPU implementation of the path: its unmodified sources (decoder_host.cpp,
    jpeg_scanner.cpp, decoder_dpu.c, bmp_writer.cpp) compiled against the functional UPMEM stand-in
    (oracle/_ref/decoder), one process per host core on a slice of the file list (the reference itself has no
    multi-core mode: 2 threads per process).  Falls back to the C restatement ("port") if the binary is absent."""

    def __init__(self, blobs, pixels):
        self.cores = os.cpu_count() or 1
        self.kind = "reference" if reference_binary() else "port"
        # what ran, for the JSON lines: the reference CLI runs 2 threads per process, the restatement one
        self.program = "the reference CLI (oracle/_ref/decoder)" if self.kind == "reference" else "the C restatement (oracle/librestate.so)"
        self.threads = " x 2 threads" if self.kind == "reference" else ""
        base ="/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
        self.dir = tempfile.mkdtemp(prefix="bjref_", dir=base)
        self.files = []
        for i, b in enumerate(blobs):
            p = os.path.join(self.dir, f"img{i:05d}.jpg")
            with open(p, "wb") as f:
                f.write(b)
            self.files.append(p)
        self.pixels = pixels
        big = max(len(b) for b in blobs) > (1 << 20)
        self.nr_dpus = 2560 if big else 64        # results do not depend on it (SURVEY 0.9); 64 is the faster choice for small images

    def step(self):
        nproc = max(1, min(self.cores, len(self.files)))
        slices = [self.files[i::nproc] for i in range(nproc)]
        t = time.perf_counter()
        with cf.ThreadPoolExecutor(max_workers=nproc) as ex:
            if self.kind == "reference":
                list(ex.map(_ref_run, [(s, self.nr_dpus) for s in slices]))
            else:
                with cf.ProcessPoolExecutor(max_workers=nproc) as px:
                    list(px.map(_port_run, slices))
        return time.perf_counter() - t

    def close(self):
        shutil.rmtree(self.dir, ignore_errors=True)


def pixels_of(specs):
    return sum(s[0] * s[1] for s in specs)


# ------------------------------------------------------------------------------------------------ --dump-outputs

DUMP_IMAGES = 16           # images of the batch whose outputs are written (a fixed, seeded choice)
DUMP_VALUES = 15 << 20     # float32 values in all: 60 MiB, below the 64 MB the dump may take


def dump_selection(n):
    """Indices of the images --dump-outputs writes: the same for the same batch size on every run."""
    rng = np.random.default_rng(0)
    return sorted(int(i) for i in rng.choice(n, size=min(n, DUMP_IMAGES), replace=False))


def download_selected(batch, first, wanted):
    """{index in the whole batch: BMP bytes} of the wanted images that lie in `batch` (images first .. first + n - 1)."""
    mine = [i - first for i in wanted if first <= i < first + batch.n]
    if not mine:
        return {}
    views = batch.download(only=mine)
    return {first + j: views[j].copy() for j in mine}


def write_dump(dirname, arrays):
    """arrays: {name: integer array} -> dirname/<name>.npy as float32 (exact for int16 / uint8 values).  An array larger
    than its share of DUMP_VALUES is written as a seeded sample: its values at sorted random positions, which depend only
    on its size, so that two builds of the project write comparable samples."""
    os.makedirs(dirname, exist_ok=True)
    share = DUMP_VALUES // max(1, len(arrays))
    for name, a in arrays.items():
        if a.size > share:
            pos = np.sort(np.random.default_rng(a.size).choice(a.size, size=share, replace=False))
            a = a.reshape(-1)[pos]
        np.save(os.path.join(dirname, name + ".npy"), a.astype(np.float32))


def run_reference(args, rank, world):
    if rank != 0:
        return
    n = args.ref_sample or (128 if args.workload in ("config2", "config5") else 2) * (os.cpu_count() or 1)
    specs, desc = workload_specs(args.workload, n, min(n, args.unique), 0)
    blobs = generate(specs, args.gen_workers)
    ref = CpuReference(blobs, pixels_of(specs))
    try:
        for _ in range(args.warmup):
            ref.step()
        times = [ref.step() for _ in range(args.steps)]
        if args.dump_outputs:
            write_dump(args.dump_outputs, {f"bmp_{i:05d}": np.fromfile(ref.files[i][:-4] + ".bmp", dtype=np.uint8)
                                           for i in dump_selection(len(ref.files))})
    finally:
        ref.close()
    total = sum(times)
    mpx = ref.pixels * args.steps / total / 1e6
    sample = f"{n} images of the workload per step ({desc}), {min(ref.cores, n)} processes{ref.threads} of {ref.program}, files on tmpfs, BMP written"
    line = {"impl": "reference", "metric": METRIC, "value": mpx, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32/int16",
            "data": "synthetic", "images_per_s": n * args.steps / total,
            "config": {"workload": desc, "sample_images_per_step": n},
            "cpu_baseline": {"value": mpx, "unit": UNIT, "cores": ref.cores, "kind": ref.kind, "sample": sample},
            "e2e": {"value": mpx, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ GPU arm

def bind_to_gpu_numa_node(index):
    """Run this process (and what it allocates: the pinned staging buffers, first touch) on the cores next to its
    GPU, so that the PCIe copies do not cross the socket interconnect.  Best effort: no NVML, no change."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        pynvml.nvmlShutdown()
    except Exception:
        pass


def twin_spec(spec):
    """Restart-parity rule (DESIGN.md section 4): a subsampled image with restart markers must equal the reference's
    decode of its restart-free twin (same pixels, quality, tables)."""
    w, h, seed, sub, gray, ri = spec
    return (w, h, seed, sub, gray, 0) if (ri and sub != 0 and not gray) else spec


def sha_file(path):
    import hashlib
    with open(path, "rb") as f:
        return hashlib.sha256(f.read()).hexdigest()


def pack_pinned(bj, blobs):
    total = sum(len(b) for b in blobs)
    pin = bj.PinnedBuffer(total + 16)
    off, o = np.zeros(len(blobs), dtype=np.uint64), 0
    for i, b in enumerate(blobs):
        pin.array[o:o + len(b)] = np.frombuffer(b, dtype=np.uint8)
        off[i] = o
        o += len(b)
    return pin, off, np.array([len(b) for b in blobs], dtype=np.uint64)


def out_sizes(bj, blobs, specs):
    cache, sizes = {}, []
    for b, sp in zip(blobs, specs):
        key = sp[:2] + sp[3:5]                 # BMP size depends on the dimensions only
        if key not in cache:
            st, d = bj.parse_header(b)
            cache[key] = bj.lib().bj_output_size(d, bj.BJ_OUT_BMP)
        sizes.append(cache[key])
    return sizes


def d2h_probe(torch, dist, world, hview, nb):
    """Pinned copy-out rate with EVERY rank copying at the same time (barrier in front of each repetition): what the
    host can take back from all its GPUs at once.  -> (this rank alone-ish best GB/s, aggregate GB/s over all ranks)."""
    dbuf = torch.empty(nb, dtype=torch.uint8, device="cuda")
    best_single, best_agg = 0.0, 0.0
    for rep in range(4):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        hview.copy_(dbuf, non_blocking=True)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        t = torch.tensor([dt], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        best_single = max(best_single, nb / dt / 1e9)
        best_agg = max(best_agg, world * nb / float(t.item()) / 1e9)
    a, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); dbuf.copy_(hview, non_blocking=True); b2.record(); torch.cuda.synchronize()
    h2d = nb / (a.elapsed_time(b2) * 1e-3) / 1e9
    del dbuf
    return best_single, best_agg, h2d


def run_compat(args, rank, local_rank, world):
    """--workload compat: Level 0 of INTEGRATION.md - bj_exec_mcus, the literal stand-in for pim.exec() on the
    reference's own metadata/mcus buffers (src/decoder_host.cpp:276-308) - against the reference's DPU program
    (src/decoder_dpu.c through oracle/_ref/libref.so) on the host cores."""
    import oracle_lib as ol
    import torch
    import pim_jpeg_decoder_b200 as bj
    torch.cuda.set_device(local_rank)
    nimg = args.batch or 64
    specs, _ = workload_specs("config2", nimg, min(nimg, 32), rank)
    blobs = generate(specs, max(1, args.gen_workers))
    uniq = {}
    for sp, b in zip(specs, blobs):
        if sp not in uniq:
            uniq[sp] = ol.Restated(b, 0)
    md = np.concatenate([uniq[sp].metadata for sp in specs])
    pre = np.concatenate([uniq[sp].mcus_pre for sp in specs])
    post = np.concatenate([uniq[sp].mcus_post for sp in specs])
    nchunk = md.shape[0]
    px = pixels_of(specs)
    dec = bj.Decoder(local_rank)
    got = dec.exec_mcus(md, pre)
    if not np.array_equal(got, post):
        raise SystemExit("bench compat: bj_exec_mcus differs from the oracle")
    for _ in range(max(args.warmup, 3)):
        dec.exec_mcus(md, pre)
    t0 = time.perf_counter()
    kern_ms = 0.0
    for _ in range(args.steps):
        got = dec.exec_mcus(md, pre)
        kern_ms += dec.stat("exec_ms")
    wall = time.perf_counter() - t0
    dec.close()
    if args.dump_outputs and rank == 0:
        write_dump(args.dump_outputs, {"mcus": got})
    cpu = None
    if ol.ref_available():
        t0 = time.perf_counter()
        reps = 0
        while reps < 3 and time.perf_counter() - t0 < 10:
            ol.ref_exec_mcus(md, pre)
            reps += 1
        dt = (time.perf_counter() - t0) / reps
        cpu = {"value": px / dt / 1e6, "unit": UNIT, "cores": 1, "kind": "reference",
               "sample": f"the reference's DPU program (decoder_dpu.c, 11 tasklets run in turn) on {nchunk} chunks, one host thread, {reps} passes"}
    chunk_bytes = 64 * 100 * 3 * 2
    line = {"metric": METRIC, "value": px * args.steps / (kern_ms * 1e-3) / 1e6, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": kern_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32/int16 fixed point",
            "data": "synthetic", "config": {"workload": f"compat: bj_exec_mcus on {nchunk} DPU chunks ({nimg} x 500x375 4:2:0), the reference's mcus/metadata layout, in place"},
            "roofline": {"bound": "hbm", "kernel": "k_exec_mcus", "achieved": 2.0 * nchunk * chunk_bytes / (kern_ms / args.steps * 1e-3) / 1e9,
                         "peak": 6540.2, "unit": "GB/s", "frac": 2.0 * nchunk * chunk_bytes / (kern_ms / args.steps * 1e-3) / 1e9 / 6540.2, "traffic": None},
            "e2e": {"value": px * args.steps / wall / 1e6, "unit": UNIT, "h2d_bytes_per_step": int(md.nbytes + pre.nbytes), "d2h_bytes_per_step": int(pre.nbytes),
                    "timer": "host wall clock around bj_exec_mcus (pageable numpy buffers in and out, like the reference's std::vector)"},
            "cpu_baseline": cpu, "gpu_launches": args.steps, "parity": {"checked": nchunk, "mismatches": 0, "against": "oracle restatement of the DPU program, whole buffers"}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10,
                    help="timed steps of every decode pass that reports a value: device-resident (one and several streams), one-call "
                         "(unless --e2e-steps), compat, reference.  Baselines run a fixed length: the CPU arm beside the GPU run (up to 12 "
                         "passes or 10 s), the CLI leg (3 runs) and, with several ranks, rank 0's one-call pass alone (2 passes)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="config2")
    ap.add_argument("--batch", type=int, default=0, help="images per GPU per step (default: 4096 for config2/5, 16 for config3/4; BASELINE states configs 3 and 4 as single images: --batch 1 / 2)")
    ap.add_argument("--stream", type=int, default=0, help="config5 only: ONE stream of this many images (pool of --unique files cycled), dealt over the ranks by compressed size (LPT): strong scaling")
    ap.add_argument("--unique", type=int, default=1024, help="distinct synthetic images generated per rank (cycled to fill the batch)")
    ap.add_argument("--subseq-bits", type=int, default=0, help="sub-sequence length of the Huffman synchronisation pass (0 = library default: per image, about 4096 bits)")
    ap.add_argument("--slices", type=int, default=0, help="slices of a sub-sequence the Huffman write pass works on (0 = library default: 1)")
    ap.add_argument("--sync-rounds", type=int, default=0)
    ap.add_argument("--sync-phased", type=int, default=-1, help="1/0: Huffman synchronisation pass with / without early stop of re-decodes (-1 = library default)")
    ap.add_argument("--sync-preroll", type=int, default=-1, help="bits of pre-roll of the Huffman synchronisation pass' first guess (-1 = library default)")
    ap.add_argument("--streams", type=int, default=2, help="device-resident value: decode the batch as this many independent parts on as many CUDA streams (1: one stream; the per-stage times always come from a one-stream pass)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="timed steps of the one-call path (0 = --steps)")
    ap.add_argument("--sub-batch-mb", type=int, default=0, help="compressed MB per sub-batch of the one-call path (0 = library default)")
    ap.add_argument("--host-threads", type=int, default=0, help="host worker threads of the one-call path (0 = library default)")
    ap.add_argument("--no-ramp", action="store_true", help="one-call path: all sub-batches the same size")
    ap.add_argument("--staged-inputs", action="store_true", help="one-call path: force the pinned staging copy of the input files (default: they are uploaded straight from the pinned input buffer)")
    ap.add_argument("--ref-sample", type=int, default=0)
    ap.add_argument("--gen-workers", type=int, default=min(32, os.cpu_count() or 1))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cli", action="store_true", help="skip the CLI-to-CLI leg (decoder_b200 vs the reference CLI on the same tmpfs files)")
    ap.add_argument("--clock-sample-ms", type=int, default=100, help="nvidia-smi polling interval while the timed regions run (0 = no sampling: for A/B only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what the last one computed (rank 0) to DIR/<name>.npy as float32: the BMP bytes of "
                         f"a fixed, seeded choice of {DUMP_IMAGES} images (bmp_<index in the batch>; --workload compat: the mcus buffers), "
                         "larger ones as a seeded sample of their bytes, at most 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 0)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.workload == "compat":
        run_compat(args, rank, local_rank, world)
        return

    # which GPU this rank drives.  With more GPUs visible than ranks, neighbouring ordinals often hang off the same PCIe
    # switch and share its uplink for the copy-out (measured on an 8-GPU box: GPUs 0+1 together 72 GB/s, one alone 57,
    # profiles/r2_d2h_probe_8gpu.txt); spreading the ranks over the visible devices gives each its own path to the host.
    # B200JPEG_BENCH_SPREAD=0 keeps device = LOCAL_RANK.
    device, dev_stride = local_rank, 1
    if world > 1 and os.environ.get("B200JPEG_BENCH_SPREAD", "1") != "0":
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = pynvml.nvmlDeviceGetCount()
            pynvml.nvmlShutdown()
            cvd = os.environ.get("CUDA_VISIBLE_DEVICES")
            if cvd:
                visible = len([x for x in cvd.split(",") if x.strip()])
            if visible >= 2 * world and int(os.environ.get("LOCAL_WORLD_SIZE", world)) == world:
                dev_stride = visible // world
                device = local_rank * dev_stride
        except Exception:
            pass
    bind_to_gpu_numa_node(device)
    workers = max(1, args.gen_workers // max(1, world))
    stream = args.stream if args.workload == "config5" else 0
    if stream:
        # ONE stream for the whole job (BASELINE configs[4]): pool cycled, dealt over the ranks by compressed size
        pool_specs = stream_pool_specs(args.unique)
        pool = generate(pool_specs, workers)
        import pim_jpeg_decoder_b200 as bj0
        costs = [len(pool[i % len(pool)]) for i in range(stream)]
        mine = bj0.lpt_shards(costs, world)[rank]
        specs = [pool_specs[i % len(pool)] for i in mine]
        blobs = [pool[i % len(pool)] for i in mine]
        desc = (f"ONE stream of {stream} mixed-size 4:2:0 q=90 JPEGs (pool of {len(pool)} unique files cycled {stream // len(pool)}x; SURVEY 8d mix), "
                f"dealt over {world} rank(s) by compressed size (LPT)")
        batch_n = len(blobs)
        total_px = sum(pool_specs[i % len(pool)][0] * pool_specs[i % len(pool)][1] for i in range(stream))
        total_images = stream
    else:
        batch_n = args.batch or (4096 if args.workload in ("config2", "config5") else 16)
        specs, desc = workload_specs(args.workload, batch_n, args.unique, rank)
        blobs = generate(specs, workers)                          # CPU, before CUDA comes up
        total_px = pixels_of(specs) * world
        total_images = batch_n * world
    px = pixels_of(specs)

    import torch
    import torch.distributed as dist
    import pim_jpeg_decoder_b200 as bj
    torch.cuda.set_device(device)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # stdout carries exactly one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", device))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(v):
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    dec = bj.Decoder(device)                                  # raises without a GPU: no CPU fallback exists
    if args.subseq_bits:
        dec.set_option("subseq_bits", args.subseq_bits)
    if args.slices:
        dec.set_option("slices", args.slices)
    if args.sync_rounds:
        dec.set_option("sync_rounds", args.sync_rounds)
    if args.sync_phased >= 0:
        dec.set_option("sync_phased", args.sync_phased)
    if args.sync_preroll >= 0:
        dec.set_option("sync_preroll_bits", args.sync_preroll)
    sampler = ClockSampler(device, args.clock_sample_ms)
    sampler.start()
    windows = []

    # ---- (1) device-resident: compressed batch already in HBM when the clock starts.  A stream is cut into resident
    # chunks of <= 4096 images, decoded one after the other (each uploaded before its clock starts).
    cuda_stream = torch.cuda.Stream()
    sp = cuda_stream.cuda_stream
    chunk = 4096 if stream else max(1, len(blobs))
    chunks = [(i, min(i + chunk, len(blobs))) for i in range(0, len(blobs), chunk)] or [(0, 0)]
    stage_ms = {"unstuff": 0.0, "sync": 0.0, "write": 0.0, "idct": 0.0}
    agg = {"scan_bytes": 0, "clean_bytes": 0, "data_units": 0, "subsequences": 0, "out_bytes": 0}
    launches = 0
    ms_total = 0.0
    first_hash = None
    steps = args.steps
    # the reported value comes from the multi-stream pass (1b) when there is one, else from this pass: --dump-outputs
    # writes the outputs of that pass' last step
    nstreams = 1 if stream else max(1, min(args.streams, len(blobs)))
    dump_idx = dump_selection(len(blobs)) if args.dump_outputs and rank == 0 else []
    dumped = {}
    barrier()
    t_wall0 = time.perf_counter()
    for ci, (c0, c1) in enumerate(chunks):
        batch = bj.Batch(dec, blobs[c0:c1], bj.BJ_OUT_BMP)
        batch.upload(sp)
        for _ in range(max(args.warmup, 1) if ci == 0 else 1):
            batch.decode(sp)
            batch.sync()
        bad = [s for s in batch.status() if s != 0]
        if bad:
            raise SystemExit(f"bench: {len(bad)} images did not decode cleanly: {bad[:4]}")
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if not stream:
            barrier()
            t_wall0 = time.perf_counter()
        ev0.record(cuda_stream)
        for _ in range(steps):
            batch.decode(sp)
            batch.sync()
            i = batch.info()
            stage_ms["unstuff"] += i.ms_unstuff; stage_ms["sync"] += i.ms_sync; stage_ms["write"] += i.ms_write; stage_ms["idct"] += i.ms_idct
        ev1.record(cuda_stream)
        torch.cuda.synchronize()
        ms_total += ev0.elapsed_time(ev1)
        info = batch.info()
        launches += info.launches * steps
        for k in agg:
            agg[k] += getattr(info, k)
        if rank == 0 and ci == 0:
            import hashlib
            first = batch.download(only=[0])[0]
            first_hash = hashlib.sha256(first.tobytes()).hexdigest()
        if nstreams == 1:
            dumped.update(download_selected(batch, c0, dump_idx))
        batch.destroy()
    barrier()
    windows.append((t_wall0, time.perf_counter()))
    ms_serial = allmax(ms_total)
    ms_max = ms_serial

    # ---- (1b) the same batch as S independent parts on S CUDA streams (public staged API, one bj_batch per part): the
    # kernels of different parts overlap on the GPU - the Huffman kernels are latency bound, the IDCT kernel issue bound,
    # so they fill each other's gaps.  This is the whole-job device-resident throughput; the per-stage times above come
    # from the one-stream pass, where a kernel has the GPU to itself.
    if nstreams > 1:
        streams = [torch.cuda.Stream() for _ in range(nstreams)]
        cut = [len(blobs) * i // nstreams for i in range(nstreams + 1)]
        parts = []
        for i in range(nstreams):
            bpart = bj.Batch(dec, blobs[cut[i]:cut[i + 1]], bj.BJ_OUT_BMP)
            bpart.upload(streams[i].cuda_stream)
            parts.append(bpart)

        def pstep():
            for bpart, st_ in zip(parts, streams):
                bpart.decode(st_.cuda_stream)
            for bpart in parts:
                bpart.sync()

        for _ in range(max(args.warmup, 1)):
            pstep()
        barrier()
        ev0 = torch.cuda.Event(enable_timing=True)
        ends = [torch.cuda.Event(enable_timing=True) for _ in streams]
        t_wall0 = time.perf_counter()
        ev0.record(streams[0])
        for st_ in streams[1:]:
            st_.wait_event(ev0)
        for _ in range(steps):
            pstep()
        for st_, e_ in zip(streams, ends):
            e_.record(st_)
        torch.cuda.synchronize()
        ms_par = max(ev0.elapsed_time(e_) for e_ in ends)
        barrier()
        windows.append((t_wall0, time.perf_counter()))
        if rank == 0:
            import hashlib
            assert hashlib.sha256(parts[0].download(only=[0])[0].tobytes()).hexdigest() == first_hash, "multi-stream and one-stream decodes disagree"
        launches = sum(bpart.info().launches for bpart in parts) * steps
        for p, bpart in enumerate(parts):
            dumped.update(download_selected(bpart, cut[p], dump_idx))
            bpart.destroy()
        ms_max = allmax(ms_par)

    # ---- (2) end to end through the one-call C ABI: host buffers in, host buffers out
    e2e = None
    parity = None
    pin_out = None
    if not args.no_e2e:
        pin_in, in_off, in_len = pack_pinned(bj, blobs)
        sizes = out_sizes(bj, blobs, specs)
        padded = np.array([(s + 15) // 16 * 16 for s in sizes], dtype=np.uint64)
        # a stream's outputs go to a ring of <= 8 GB (they are consumed as they come); a batch's outputs all stay
        ring = min(int(padded.sum()), 8 << 30) if stream else int(padded.sum())
        pin_out = bj.PinnedBuffer(ring + 16)
        calls = []                                            # [(i0, i1, out offsets)] : one bj_decode_batch per call
        i0 = 0
        while i0 < len(blobs):
            i1, acc = i0, 0
            while i1 < len(blobs) and acc + int(padded[i1]) <= ring:
                acc += int(padded[i1]); i1 += 1
            offs = np.concatenate([[0], np.cumsum(padded[i0:i1])]).astype(np.uint64)[:-1]
            calls.append((i0, i1, offs))
            i0 = i1
        dec.set_option("packed_outputs", 1)
        # the input files sit in ONE pinned buffer from bj_host_alloc: the library uploads them straight from there
        # (no staging copy, no host pass over the compressed bytes); --staged-inputs forces the copy for A/B
        dec.set_option("packed_inputs", -1 if args.staged_inputs else 0)
        if args.sub_batch_mb:
            dec.set_option("sub_batch_bytes", args.sub_batch_mb << 20)
        # host worker threads of this rank: its share of the box's cores (the library's own default, min(4, cores/2),
        # does not know about the other ranks), one core left to the calling thread
        share = len(os.sched_getaffinity(0)) // max(1, world)
        host_threads = args.host_threads or (max(1, min(4, share - 1)) if world > 1 else 0)
        if host_threads:
            dec.set_option("host_threads", host_threads)
        if args.no_ramp:
            dec.set_option("sub_batch_ramp", 0)
        # what the link gives: one large pinned copy each way, all ranks at the same time
        nb = min(ring, 1 << 30)
        hview = torch.from_numpy(pin_out.array[:nb])
        d2h_single, d2h_agg, h2d_single = d2h_probe(torch, dist, world, hview, nb)

        def one_pass():
            st_all = []
            for (a, b, offs) in calls:
                st_all.append(dec.decode_packed(pin_in.array, in_off[a:b], in_len[a:b], pin_out.array, offs, bj.BJ_OUT_BMP))
            return st_all

        k2 = args.e2e_steps or steps
        e2e_single = None
        if world > 1:                                         # rank 0 alone first: the denominator of the e2e scaling efficiency
            if rank == 0:
                one_pass()
                t0 = time.perf_counter()
                for _ in range(2):
                    one_pass()
                e2e_single = px * 2 / (time.perf_counter() - t0) / 1e6
            barrier()
        if stream:                                            # a stream's warm-up is its first call (buffers reach their size)
            a, b, offs = calls[0]
            dec.decode_packed(pin_in.array, in_off[a:b], in_len[a:b], pin_out.array, offs, bj.BJ_OUT_BMP)
        for _ in range(max(1, min(args.warmup, 2)) if not stream else 0):
            one_pass()
        barrier()
        stat_names = ["decode_batch_host_ms", "decode_batch_wait_ms", "decode_batch_h2d_bytes", "decode_batch_d2h_bytes", "decode_batch_sub_batches",
                      "decode_batch_d2h_copies", "decode_batch_direct_uploads", "decode_batch_launches"]
        acc = dict.fromkeys(stat_names, 0.0)
        step_ms = []
        t0 = time.perf_counter()
        for _ in range(k2):
            ts = time.perf_counter()
            for (a, b, offs) in calls:
                st = dec.decode_packed(pin_in.array, in_off[a:b], in_len[a:b], pin_out.array, offs, bj.BJ_OUT_BMP)
                if st.any():
                    raise SystemExit("bench e2e: images failed to decode")
                for nme in stat_names:
                    acc[nme] += dec.stat(nme)
            step_ms.append(1e3 * (time.perf_counter() - ts))
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        windows.append((t0, t1))
        e2e_s = allmax(t1 - t0)
        if rank == 0 and len(calls) == 1:
            import hashlib
            assert hashlib.sha256(pin_out.array[:sizes[0]].tobytes()).hexdigest() == first_hash, "e2e and device-resident paths disagree"
        d2h_per_step = acc["decode_batch_d2h_bytes"] / k2
        floor_ms = 1e3 * d2h_per_step / (d2h_agg / world * 1e9) if d2h_agg else None
        e2e_value = total_px * k2 / e2e_s / 1e6
        e2e = {"value": e2e_value, "unit": UNIT, "images_per_s": total_images * k2 / e2e_s,
               "ms_per_step": 1e3 * e2e_s / k2, "steps": k2, "rank0_step_ms": [round(x, 2) for x in step_ms],
               "h2d_bytes_per_step": int(acc["decode_batch_h2d_bytes"] / k2), "d2h_bytes_per_step": int(d2h_per_step),
               "sub_batches_per_step": int(acc["decode_batch_sub_batches"] / k2), "d2h_copies_per_step": int(acc["decode_batch_d2h_copies"] / k2),
               "direct_uploads_per_step": int(acc["decode_batch_direct_uploads"] / k2), "calls_per_step": len(calls),
               "host_threads": int(dec.stat("host_threads")),
               "host_prepare_ms_per_step": acc["decode_batch_host_ms"] / k2, "host_wait_gpu_ms_per_step": acc["decode_batch_wait_ms"] / k2,
               "pcie_pinned_copy": {"d2h_gbs": d2h_single, "h2d_gbs": h2d_single},
               # the copy-out bounds this path (3 B per pixel go back over PCIe): its floor with every rank copying at once
               "aggregate_d2h_gbs": d2h_agg, "d2h_floor_ms_per_step": floor_ms, "frac_of_floor": (floor_ms / (1e3 * e2e_s / k2)) if floor_ms else None,
               "single_rank_value": e2e_single, "e2e_efficiency": (e2e_value / (world * e2e_single)) if e2e_single and not stream else None,
               "timer": "host wall clock around the blocking bj_decode_batch call(s) (pinned host buffers in and out), max over ranks; "
                        "aggregate_d2h_gbs: all ranks copying out at once behind a barrier"}
        pin_in.free()

    # ---- (3) the reference on this box's host cores, bounded sample (rank 0, N=1 only): passes over the first
    # 128 x cores images of the batch until about 10 s of wall time (= 10 s x cores of CPU work) have been spent.
    # The BMP files it writes are the parity check of this run: the GPU's BMP bytes of the same images must be identical
    # (for a subsampled image with restart markers: the reference's decode of its restart-free twin, DESIGN.md section 4).
    cpu = None
    cli = None
    rule = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        n = args.ref_sample or (256 if args.workload in ("config2", "config5") else 2) * (os.cpu_count() or 1)
        n = min(n, len(blobs), 4096)
        ref = CpuReference(blobs[:n], pixels_of(specs[:n]))
        try:
            t, passes = 0.0, 0
            while passes < 12 and t < 10.0:
                t += ref.step()
                passes += 1
            cpu = {"value": ref.pixels * passes / t / 1e6, "unit": UNIT, "cores": ref.cores, "kind": ref.kind, "images_per_s": n * passes / t,
                   "sample": f"first {n} images of the batch, {passes} passes, {min(ref.cores, n)} processes{ref.threads} of {ref.program} on tmpfs (BMP written), {t:.2f} s"}
            # ---- parity against what the reference just wrote
            if pin_out is not None:
                want = {}
                twins = [twin_spec(sp) for sp in specs[:n]]
                if any(tw != sp for tw, sp in zip(twins, specs[:n])):
                    rule = ("restart-parity rule: subsampled images with restart markers are compared with the reference's decode of the restart-free twin "
                            "(the reference's own restart handling is wrong for subsampled files, SURVEY 0.7)")
                    tw_uniq = sorted(set(twins))
                    tw_blobs = dict(zip(tw_uniq, generate(tw_uniq, 1)))
                    tref = CpuReference([tw_blobs[tw] for tw in twins], 0)
                    tref.step()
                    want = {i: sha_file(f[:-4] + ".bmp") for i, f in enumerate(tref.files)}
                    tref.close()
                else:
                    want = {i: sha_file(f[:-4] + ".bmp") for i, f in enumerate(ref.files)}
                import hashlib
                a0, b0, offs0 = calls[0]
                nchk = min(n, b0 - a0)
                mism = [i for i in range(nchk) if hashlib.sha256(pin_out.array[int(offs0[i]):int(offs0[i]) + sizes[i]].tobytes()).hexdigest() != want[i]]
                parity = {"checked": nchk, "mismatches": len(mism), "against": f"the BMP files {ref.program} wrote in this run", "rule": rule}
            # ---- CLI to CLI on the same tmpfs files: decoder_b200 (file -> BMP file, one process, every visible GPU)
            cli_bin = os.path.join(ROOT, "pim_jpeg_decoder_b200", "host", "_build", "decoder_b200")
            if not args.no_cli and os.path.exists(cli_bin) and ref.kind == "reference":
                dec.close()
                dec = None
                refs = {f: sha_file(f[:-4] + ".bmp") for f in ref.files} if rule is None else None
                for f in ref.files:
                    os.remove(f[:-4] + ".bmp")
                tc, cli_out = [], ""
                for _ in range(3):
                    t0 = time.perf_counter()
                    cli_out = subprocess.run([cli_bin] + ref.files, capture_output=True, text=True, check=True, env=dict(os.environ, B200JPEG_DEVICES="1")).stdout
                    tc.append(time.perf_counter() - t0)
                bad = sum(1 for f in ref.files if refs is not None and sha_file(f[:-4] + ".bmp") != refs[f])
                startup = 0.0
                for ln in cli_out.splitlines():
                    if "Start-up" in ln:
                        startup = float(ln.split(":")[-1].strip().rstrip("s"))
                cli = {"b200": {"value": ref.pixels / min(tc) / 1e6, "unit": UNIT, "seconds": min(tc), "runs": tc, "startup_s": startup,
                                "value_without_startup": ref.pixels / max(min(tc) - startup, 1e-9) / 1e6,
                                "what": "decoder_b200 <files>: process start, CUDA context, file read, decode on one GPU, BMP files written (tmpfs)"},
                       "reference": {"value": cpu["value"], "unit": UNIT, "what": "the reference CLI, one process per host core on a slice of the same files"},
                       "ratio": (ref.pixels / min(tc) / 1e6) / cpu["value"], "images": n,
                       "b200_profiles": [ln.strip() for ln in cli_out.split("Profiles:")[-1].splitlines() if ln.strip()],
                       "bmp_files_identical": (bad == 0) if refs is not None else None}
        finally:
            ref.close()
    if pin_out is not None:
        pin_out.free()
    sampler.stop()
    if dec is not None:
        dec.close()
    if dumped:
        write_dump(args.dump_outputs, {f"bmp_{i:05d}": b for i, b in sorted(dumped.items())})

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except OSError:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "6650 GB/s (of fallback)"
    # algorithmic bytes per launch (DESIGN.md "Roofline"): per kernel group of ONE step on ONE GPU (rank 0)
    clean = float(agg["clean_bytes"])
    units = float(agg["data_units"])
    nsub = float(agg["subsequences"])
    scan = float(agg["scan_bytes"])
    outb = float(agg["out_bytes"])
    alg = {
        "unstuff": 1.0 * scan + clean,                                # raw bytes read once + clean bytes written
        "sync": clean + (28.0 + 16.0 * (args.slices or 1) + 64.0) * nsub,    # stream read once + per-sub-sequence states/totals + slice entry states + 4 quarter records written
        "write": clean + 128.0 * units,                               # stream read once + every coefficient unit written once
        "idct": 128.0 * units + outb,                                 # coefficients read once + pixels written once
    }
    stages = {}
    for k in stage_ms:
        t = stage_ms[k] / steps
        stages[k] = {"ms": t, "alg_bytes": alg[k], "achieved_gbs": alg[k] / (t * 1e-3) / 1e9 if t > 0 else None,
                     "frac": (alg[k] / (t * 1e-3) / 1e9 / peak) if t > 0 else None}
    stages["sync"]["compressed_gbs"] = scan / (stages["sync"]["ms"] * 1e-3) / 1e9 if stages["sync"]["ms"] else None
    ent_ms = stages["unstuff"]["ms"] + stages["sync"]["ms"] + stages["write"]["ms"]
    dom = max(stage_ms, key=lambda k: stage_ms[k])
    # DRAM traffic per launch group: from the committed ncu --set full capture, valid only for the kernel sources and
    # the workload it was taken with (else null: a stale constant must not ride along)
    traffic, traffic_src = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            tj = json.load(f)
        if tj.get("kernel_sources_sha") == kernel_sources_sha() and tj.get("workload") == args.workload and not stream and batch_n == tj.get("images"):
            traffic = tj.get(dom)
            traffic_src = f"profiles/ncu_traffic.json: ncu --set full capture of {tj.get('capture')}, same kernel sources ({tj.get('kernel_sources_sha')})"
        else:
            traffic_src = "profiles/ncu_traffic.json was taken with other kernel sources or another workload: not reported"
    except (OSError, ValueError):
        pass
    kname = {"unstuff": "k_unstuff+k_subseq_table", "sync": "k_huff_sync (all rounds)",
             "write": "k_huff_write (+k_zero_tail, k_dc_predict)", "idct": "k_idct_color"}
    roofline = {"bound": "hbm", "kernel": kname[dom], "achieved": stages[dom]["achieved_gbs"], "peak": peak, "unit": "GB/s",
                "frac": stages[dom]["frac"], "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "note": "Huffman kernels are latency/issue bound, not HBM bound: the fraction is reported against HBM as SURVEY 8d prescribes"}
    total_s = ms_max * 1e-3
    images_rank0 = len(blobs)
    line = {
        "metric": METRIC, "value": total_px * steps / total_s / 1e6, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": max(args.warmup, 1),
        "ms_per_step": ms_max / steps, "ms_per_image": ms_max / steps / max(1, images_rank0), "higher_is_better": True, "scaling": "strong" if stream else "weak", "vs_baseline": None,
        "dtype": "int32/int16 fixed point (u8 pixels)", "data": "synthetic",
        "images_per_s": total_images * steps / total_s,
        "config": {"workload": desc, "images_per_gpu_per_step": images_rank0, "output": "BMP bytes (bit-exact to the reference's write_BMP)",
                   "l2": "per-step working set (coefficients + pixels) is far larger than the 126 MB L2; no explicit flush" if px > 40e6 else
                         "working set of one step is smaller than the 126 MB L2 and stays there between steps (single-image latency case); inputs are re-read from HBM-resident buffers",
                   "subseq_bits": args.subseq_bits or "per image (library default)", "slices": args.slices or "per image (library default)",
                   "streams": nstreams, "value_one_stream": total_px * steps / (ms_serial * 1e-3) / 1e6, "ms_per_step_one_stream": ms_serial / steps,
                   "devices": f"rank r drives GPU {dev_stride} x r" if dev_stride > 1 else "rank r drives GPU r",
                   "sharding": "ONE list dealt over the ranks by compressed size (LPT), no collective on the data path" if stream else "by image, no collective on the data path",
                   "restart_parity_rule": rule or ("files with restart markers that are subsampled follow the restart-parity rule (DESIGN.md section 4)" if args.workload == "config3" else None)},
        "roofline": roofline, "stages": stages,
        "entropy": {"ms": ent_ms, "compressed_gbs": scan / (ent_ms * 1e-3) / 1e9 if ent_ms else None},
        # the whole decode as one box (SURVEY 8d): compressed bytes in + 3 B/px out; the coefficient round trip is overhead, not credit
        "whole_decode": {"alg_bytes": scan + outb,
                         "achieved_gbs": (scan + outb) / (ms_total / steps * 1e-3) / 1e9,
                         "frac": (scan + outb) / (ms_total / steps * 1e-3) / 1e9 / peak},
        "cpu_baseline": cpu, "e2e": e2e, "cli_e2e": cli, "parity": parity, "gpu_launches": int(launches),
        "clocks": sampler.summary(windows),
        "first_bmp_sha256": first_hash,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    if parity and parity["mismatches"]:
        raise SystemExit(f"bench: {parity['mismatches']} of {parity['checked']} images differ from the reference's BMP files")


if __name__ == "__main__":
    main()
