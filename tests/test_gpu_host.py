"""GPU tests of decoder_b200, the CLI above the C ABI (pim_jpeg_decoder_b200/host) on the full GPU path
(bj_decode_batch), bit-exact against the hashes the reference itself produced (tests/golden/golden.json).  The other
two host programs there, decoder_compat and decoder_hybrid, link the reference's own sources and are built only where
those are present."""
import hashlib
import os
import shutil
import subprocess

import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
HOST = os.path.join(ROOT, "pim_jpeg_decoder_b200", "host")


def _copy(names, golden, golden_dir, tmp_path):
    paths = []
    for n in names:
        p = str(tmp_path / golden[n]["file"])
        shutil.copy(os.path.join(golden_dir, golden[n]["file"]), p)
        paths.append(p)
    return paths


def _sha(path):
    return hashlib.sha256(open(path, "rb").read()).hexdigest()


def _valid_names(golden):
    return sorted(k for k, v in golden.items() if not v.get("invalid"))


def test_decoder_b200_cli(golden, golden_dir, tmp_path):
    subprocess.run(["make", "-s", "-C", HOST, os.path.join(HOST, "_build", "decoder_b200")], check=True)
    exe = os.path.join(HOST, "_build", "decoder_b200")
    names = _valid_names(golden) + ["bad_not_jpeg", "bad_truncated"]
    paths = _copy(names, golden, golden_dir, tmp_path)
    out = subprocess.run([exe] + paths + [str(tmp_path / "missing.jpg")], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "Profiles:" in out.stdout
    for n, p in zip(names, paths):
        if golden[n].get("invalid"):
            assert f"{p}: Error - Invalid JPEG" in out.stdout and not os.path.exists(p[:-4] + ".bmp")
        else:
            assert _sha(p[:-4] + ".bmp") == golden[golden[n]["expect"]]["bmp_sha256"], n
    assert "missing.jpg: Error - Invalid JPEG" in out.stdout


def test_decoder_b200_pipeline_of_many_groups(golden, golden_dir, tmp_path):
    """Groups of 5 images: the reader thread, the GPU jobs (bj_submit / bj_wait) and the writer thread overlap over ~8
    groups that rotate through 4 sets of pinned buffers; every device of the box is used (bj_create_multi)."""
    exe = os.path.join(HOST, "_build", "decoder_b200")
    names = _valid_names(golden) + ["bad_not_jpeg", "bad_truncated"]
    paths = _copy(names, golden, golden_dir, tmp_path)
    env = dict(os.environ, B200JPEG_GROUP_IMAGES="5")
    out = subprocess.run([exe] + paths, env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "Huffman synchronisation kernels" in out.stdout and "IDCT + colour conversion kernel" in out.stdout
    groups = int(out.stdout.split(" - Total ")[1].split(" groups")[0])
    assert groups >= len(names) // 5
    for n, p in zip(names, paths):
        if golden[n].get("invalid"):
            assert not os.path.exists(p[:-4] + ".bmp")
        else:
            assert _sha(p[:-4] + ".bmp") == golden[golden[n]["expect"]]["bmp_sha256"], n


def test_decoder_b200_sharded_by_rank(golden, golden_dir, tmp_path):
    """Two 'ranks' (processes) on the same GPU each take their share of the sorted list; together they cover it."""
    exe = os.path.join(HOST, "_build", "decoder_b200")
    names = _valid_names(golden)[:12]
    paths = _copy(names, golden, golden_dir, tmp_path)
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", LOCAL_RANK="0")
        assert subprocess.run([exe] + paths, env=env, capture_output=True, text=True, timeout=600).returncode == 0
    for n, p in zip(names, paths):
        assert _sha(p[:-4] + ".bmp") == golden[golden[n]["expect"]]["bmp_sha256"], n
