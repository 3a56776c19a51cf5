"""Generates tests/golden/reference_vectors.json: what the reference computes on the seeded inputs of
test_oracle.py::test_exec_restatement_vs_live_reference (its DPU program on random buffers, values that wrap 16 and 32
bits included) and test_abi.py::test_parse_header_validity_matches_the_reference_on_damaged_files (read_JPEG's verdict
and sizes on 640 damaged files).

    python tests/golden/make_reference_vectors.py                      # from oracle/_ref/libref.so (make -C oracle ref)
    python tests/golden/make_reference_vectors.py --from-restatement   # see below

--from-restatement records the same values from oracle/restate.c and bj_parse_header.  That is only valid at a commit
where both tests pass against the live reference, which compares them with it bit for bit.  The committed file was made
this way from the code of commit 19db0c8, where both tests ran against the live reference and passed; oracle/restate.c,
the header parser and both tests' inputs were unchanged when it was written.
"""
import ctypes as C
import json
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import oracle_lib as ol  # noqa: E402
import test_abi  # noqa: E402
import test_oracle  # noqa: E402


def main():
    live = "--from-restatement" not in sys.argv[1:]
    if live and not ol.ref_available():
        raise SystemExit("oracle/_ref/libref.so is not built (make -C oracle ref REF=<reference sources>)")
    out = {"exec_mcus": {}, "parse_header_damaged": {}}
    for full_range in (False, True):
        for vs, hs, ncomp in test_oracle.EXEC_SHAPES:
            key, md, mcus = test_oracle.exec_case(vs, hs, ncomp, full_range)
            post = ol.ref_exec_mcus(md, mcus) if live else ol.restate_exec_mcus(md, mcus)
            out["exec_mcus"][key] = {"input_sha256": ol.sha256(md, mcus), "output_sha256": ol.sha256(post)}
    files = list(test_abi.damaged_files())
    results = []
    if live:
        with tempfile.TemporaryDirectory() as td:
            path = os.path.join(td, "m.jpg")
            for data in files:
                with open(path, "wb") as f:
                    f.write(data)
                info = ol.RefInfo()
                valid = ol.ref().ref_probe(path.encode(), C.byref(info)) > 0
                results.append([int(valid)] + ([info.width, info.height, info.ncomp, info.h_samp, info.v_samp, info.restart_interval] if valid else []))
    else:
        import pim_jpeg_decoder_b200 as bj
        for data in files:
            st, d = bj.parse_header(data)
            results.append([int(st in (bj.BJ_OK, bj.BJ_ERR_UNSUPPORTED))] +
                           ([d.width, d.height, d.ncomp, d.hs, d.vs, d.restart_interval] if st == bj.BJ_OK else []))
    out["parse_header_damaged"] = {"inputs_sha256": ol.sha256(*[np.frombuffer(f, dtype=np.uint8) for f in files]),
                                   "results": results}
    with open(ol.REFERENCE_VECTORS, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote", ol.REFERENCE_VECTORS, "from", "the reference" if live else "the restatement")


if __name__ == "__main__":
    main()
