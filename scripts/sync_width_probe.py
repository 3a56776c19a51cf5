"""CPU probe: how often a re-decode of the synchronisation pass fails to merge inside its own sub-sequence, at the
sub-sequence length a config-2 image gets from a 256-wide and from a 128-wide CTA of k_huff_sync.

Drives the entropy-stage emulator (tests/emu/huff_emu.cpp) over config-2 images from the bench generator and seeds
(500x375 4:2:0 q=90, seeds 0..n-1) and records its per-round histogram: round r counts the sub-sequences decoded in
Jacobi round r (round 0: every one; round 1: nearly every one, its entry guess was wrong; round 2 on: the successors
of re-decodes that did not merge).  The sub-sequence length per image follows the automatic layout of batch.h for a
full config-2 batch: one CTA of NT sub-sequences per image, so ceil(raw_len / (NT - 1)) bytes, rounded up to a
multiple of 4 times the slice count.

    python scripts/sync_width_probe.py [n_images]          (default 48)
"""
import ctypes as C
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import jpeg_synth as js          # noqa: E402
import oracle_lib as ol          # noqa: E402


def load_emu(tmp):
    so = os.path.join(tmp, "libhuffemu.so")
    subprocess.run(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-o", so, os.path.join(ROOT, "tests", "emu", "huff_emu.cpp")], check=True)
    lib = C.CDLL(so)
    lib.emu_entropy.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    lib.emu_set_round_hist.argtypes = [C.c_void_p]
    return lib


def sub_bytes_of(raw_len, nt, slices_log2):
    q = 4 << slices_log2
    return (max((raw_len + nt - 2) // (nt - 1), 64) + q - 1) // q * q


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 48
    files = [js.synth_jpeg(500, 375, i, subsampling=2) for i in range(n)]
    with tempfile.TemporaryDirectory() as tmp:
        lib = load_emu(tmp)
        print(f"{n} config-2 images (500x375 4:2:0 q=90, bench seeds 0..{n - 1}); emulator Jacobi rounds, whole image")
        for nt, rl in ((256, 0), (128, 1)):
            tot = np.zeros(64, dtype=np.uint64)
            sub_sizes = []
            for data in files:
                raw_len = ol.Restated(data, 0).h.scan_len
                sub = sub_bytes_of(raw_len, nt, rl)
                sub_sizes.append(sub)
                hist = np.zeros(64, dtype=np.uint32)
                lib.emu_set_round_hist(ol._ptr(hist))
                coef = np.zeros(((500 + 15) // 16) * ((375 + 15) // 16) * 6 * 64, dtype=np.int16)
                info = np.zeros(4, dtype=np.uint32)
                rc = lib.emu_entropy(ol._ptr(np.frombuffer(data, dtype=np.uint8)), len(data), sub >> rl, 1 << rl, ol._ptr(coef), ol._ptr(info))
                lib.emu_set_round_hist(None)
                assert rc == 0 and info[3] == 0
                tot += hist
            nsub = int(tot[0])
            print(f"\nCTA width {nt}: sub-sequences of {min(sub_sizes)}..{max(sub_sizes)} B (mean {np.mean(sub_sizes):.0f} B, "
                  f"{8 * np.mean(sub_sizes):.0f} bits) x {1 << rl} slice(s); {nsub} sub-sequences")
            for r in range(64):
                if tot[r] == 0:
                    break
                print(f"  round {r}: {int(tot[r]):7d} decoded  {100.0 * tot[r] / nsub:6.2f} % of sub-sequences")
            print(f"  re-decodes of round 1 that do not merge (round 2 / round 1): {100.0 * tot[2] / max(tot[1], 1):.2f} %")
            print(f"  decode-equivalents: {tot.sum() / nsub:.3f} (whole re-decodes, no early stop)")


if __name__ == "__main__":
    main()
