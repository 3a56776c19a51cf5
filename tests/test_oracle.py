"""CPU tests: the oracle restatement (oracle/restate.c) is pinned to the reference.

Two anchors: (1) tests/golden/golden.json - SHA-256 of the BMP, the post-Huffman buffer and the post-exec buffer
that the REAL reference code produced for every fixture (made by tests/golden/make_golden.py);
(2) tests/golden/reference_vectors.json - what the reference's DPU program computed on seeded random buffers, and,
when oracle/_ref/libref.so is present, the real reference code itself, run live on the same buffers.
"""
import hashlib
import os

import numpy as np
import pytest

import oracle_lib as ol


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _names(golden_path=os.path.join(os.path.dirname(__file__), "golden", "golden.json")):
    import json
    with open(golden_path) as f:
        return sorted(json.load(f).keys())


@pytest.mark.parametrize("name", _names())
def test_restatement_reproduces_reference_hashes(name, golden, golden_dir):
    e = golden[name]
    data = open(os.path.join(golden_dir, e["file"]), "rb").read()
    r = ol.Restated(data, restart_mode=1)  # 1 = bug-compatible restart rule, jpeg_scanner.cpp:723
    if e.get("invalid"):
        assert not r.valid
        return
    assert r.valid
    assert (r.h.width, r.h.height, r.h.ncomp, r.h.hs, r.h.vs) == (e["width"], e["height"], e["ncomp"], e["hs"], e["vs"])
    assert r.nchunk == e["nchunks"]
    assert sha(r.metadata[0]) == e["metadata_sha256"]
    assert sha(r.mcus_pre) == e["mcus_pre_sha256"]
    assert sha(r.mcus_post) == e["mcus_post_sha256"]
    assert sha(r.bmp) == e["bmp_sha256"]
    assert int(r.huff_rc == 0) == e["huffman_ok"]


def test_bundled_image_golden_hash(golden):
    # SURVEY.md section 0 fact 10: the reference's BMP for its own bundled image
    assert golden["ilsvrc_444"]["bmp_sha256"] == "11ab0c81cfc918410245c5ff0923f787219521073c094cbfd7e763f4b3444c1f"


@pytest.mark.parametrize("name", [n for n in _names() if n.endswith("_ri4")])
def test_restart_parity_rule(name, golden, golden_dir):
    """Subsampled + DRI: T.81-correct restart handling must give the reference's decode of the restart-free twin."""
    e = golden[name]
    twin = golden[e["expect"]]
    assert twin["file"] != e["file"]
    data = open(os.path.join(golden_dir, e["file"]), "rb").read()
    r = ol.Restated(data, restart_mode=0)
    assert r.huff_rc == 0
    assert sha(r.bmp) == twin["bmp_sha256"]
    assert sha(r.bmp) != e["bmp_sha256"]  # ... and the reference's own decode of the DRI file is different


@pytest.mark.parametrize("name", [n for n in _names() if "_ri" in n and not n.endswith("_ri4")])
def test_restart_modes_agree_when_not_subsampled(name, golden, golden_dir):
    e = golden[name]
    data = open(os.path.join(golden_dir, e["file"]), "rb").read()
    assert sha(ol.Restated(data, 0).bmp) == e["bmp_sha256"]


def _random_exec_case(rng, vs, hs, ncomp, nchunk, full_range):
    md = np.zeros((nchunk, 276), dtype=np.uint32)
    md[:, 4] = ncomp
    md[:, 5] = vs
    md[:, 6] = hs
    for j in range(ncomp):
        md[:, 7 + j] = min(j, 1)
    md[:, 19] = ol.M
    md[:, 20:20 + 128] = rng.integers(1, 256 if not full_range else 65536, size=128, dtype=np.uint32)
    lim = 32768 if full_range else 64
    mcus = rng.integers(-lim, lim, size=(nchunk, ol.CHUNK)).astype(np.int16)
    if not full_range:
        mcus[rng.random(size=mcus.shape) > 0.2] = 0
    return md, mcus


EXEC_SHAPES = [(1, 1, 3), (2, 1, 3), (1, 2, 3), (2, 2, 3), (1, 1, 1), (2, 2, 1), (0, 0, 0)]


def exec_case(vs, hs, ncomp, full_range):
    """-> (key in reference_vectors.json, metadata, mcus): three chunks of seeded random input for the DPU program."""
    rng = np.random.default_rng(vs * 100 + hs * 10 + ncomp + (1000 if full_range else 0))
    md, mcus = _random_exec_case(rng, vs, hs, ncomp, 3, full_range)
    if ncomp == 0:
        md[:] = 0  # idle DPU: nothing runs, buffer unchanged
    return f"{vs},{hs},{ncomp},{int(full_range)}", md, mcus


@pytest.mark.parametrize("vs,hs,ncomp", EXEC_SHAPES)
@pytest.mark.parametrize("full_range", [False, True])
def test_exec_restatement_vs_live_reference(vs, hs, ncomp, full_range):
    """The DPU program (dequant, IDCT, colour) on random buffers, incl. values that wrap 16 and 32 bits: the
    restatement against what the reference's program computed on the same buffers (tests/golden/reference_vectors.json),
    and against the reference itself where oracle/_ref/libref.so is built."""
    key, md, mcus = exec_case(vs, hs, ncomp, full_range)
    want = ol.reference_vectors()["exec_mcus"][key]
    assert ol.sha256(md, mcus) == want["input_sha256"], "the seeded inputs are not the ones the reference was run on"
    got = ol.restate_exec_mcus(md, mcus)
    assert ol.sha256(got) == want["output_sha256"]
    if ol.ref_available():
        assert np.array_equal(got, ol.ref_exec_mcus(md, mcus))


def test_idct_dc_only():
    """A DC-only tile is flat: value ((dc*181>>5)*... ) - checks rs_idct8 wiring with a hand-computed case."""
    lib = ol.restate()
    inp = np.array([64, 0, 0, 0, 0, 0, 0, 0], dtype=np.int32)
    out = np.zeros(8, dtype=np.int32)
    lib.rs_idct8(ol._ptr(inp), ol._ptr(out))
    assert (out == ((64 * 181) >> 5) >> 4).all()
