"""The JSON number formatter (csrc/json_format.cuh) built host-side with nvcc against Python's float.__repr__, its Ryu
tables against their defining formula, the row-size bound of the result writer, and the refusals of
avdf_format_results (no launch)."""
import ctypes
import json
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "audio_visual_deepfake_detection_b200", "csrc", "json_format.cuh")


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    exe = str(tmp_path_factory.mktemp("jf") / "json_format_driver")
    subprocess.run([nvcc, "-O2", "-std=c++17", os.path.join(ROOT, "tests", "json_format_driver.cu"), "-o", exe], check=True,
                   capture_output=True)
    return exe


def check(driver, tmp_path, bits):
    bits = np.ascontiguousarray(bits, dtype=np.uint32)
    src, dst = tmp_path / "in.u32", tmp_path / "out.txt"
    bits.tofile(src)
    subprocess.run([driver, str(src), str(dst)], check=True)
    got = dst.read_text()
    with np.errstate(invalid="ignore"):
        want = json.dumps(bits.view(np.float32).astype(np.float64).tolist())
    if got != want:
        g, w = got[1:-1].split(", "), want[1:-1].split(", ")
        bad = [(hex(int(bits[i])), g[i], w[i]) for i in range(min(len(g), len(w))) if g[i] != w[i]]
        pytest.fail("%d mismatches, first: %s" % (len(bad), bad[:8]))


def exponent_block(e8):
    return (np.uint32(e8) << np.uint32(23)) | np.arange(1 << 23, dtype=np.uint32)


@pytest.mark.parametrize("value", [0.2, 1e-4, 1e16, "max", "subnormal"])
def test_all_mantissas_of_an_exponent(driver, tmp_path, value):
    if value == "max":
        e8 = 254
    elif value == "subnormal":
        e8 = 0
    else:
        e8 = int(np.float32(value).view(np.uint32)) >> 23
    b = exponent_block(e8)
    check(driver, tmp_path, np.concatenate([b, b | np.uint32(1 << 31)]) if value in ("subnormal", 0.2) else b)


def test_every_exponent_random_mantissas_and_specials(driver, tmp_path):
    rng = np.random.default_rng(1)
    e = np.repeat(np.arange(256, dtype=np.uint32), 4096)
    bits = (rng.integers(0, 2, e.size, dtype=np.uint32) << 31) | (e << 23) | rng.integers(0, 1 << 23, e.size, dtype=np.uint32)
    special = np.array([0, 0x80000000, 0x7f800000, 0xff800000, 0x7fc00000, 0xffc00000, 0x7f800001], np.uint32)
    check(driver, tmp_path, np.concatenate([special, bits]))


def test_random_bit_patterns(driver, tmp_path):
    rng = np.random.default_rng(2)
    for _ in range(5):
        check(driver, tmp_path, rng.integers(0, 1 << 32, 2_000_000, dtype=np.uint64).astype(np.uint32))


def test_tables_match_their_formula():
    text = open(HEADER).read()

    def rows(name):
        body = text.split("#define %s \\\n" % name)[1].split("\n\n")[0]
        return [int(lo, 16) | (int(hi, 16) << 64) for lo, hi in re.findall(r"\{(0x[0-9a-f]+)ull, (0x[0-9a-f]+)ull\}", body)]

    def pow5bits(e):
        return ((e * 1217359) >> 19) + 1
    inv, pw = rows("AVDF_RYU_POW5_INV"), rows("AVDF_RYU_POW5")
    assert inv == [(1 << (pow5bits(q) - 1 + 125)) // 5 ** q + 1 for q in range(21)]
    want = []
    for i in range(64):
        sh = pow5bits(i) - 125
        want.append(5 ** i >> sh if sh >= 0 else 5 ** i << -sh)
    assert pw == want


def longest_numbers(n):
    """n distinct fp32 values whose text has the maximal 23 bytes."""
    rng = np.random.default_rng(4)
    out = []
    while len(out) < n:
        v = (-(rng.random(4096) + 1) * 1e-30).astype(np.float32).astype(np.float64).tolist()
        out += [x for x in v if len(repr(x)) == 23]
    return out[:n]


@pytest.mark.parametrize("K", [1, 7, 100])
def test_row_bound_holds_the_longest_rows(K):
    from audio_visual_deepfake_detection_b200.libs.utils.result_writer import row_bytes_max
    from audio_visual_deepfake_detection_b200.native import FORMAT_PREDICTIONS, FORMAT_RECORDS
    x = longest_numbers(3 * K + 1)
    vid = "aé\"\\\x01/x.mp4"
    id_bytes = len(json.dumps(vid, ensure_ascii=False).encode())
    item = {"video_id": vid, "video_cls": [x[0]], "scores": x[1:K + 1], "segments": [[x[K + 1 + 2 * j], x[K + 2 + 2 * j]] for j in range(K)]}
    two = json.dumps([item, item], ensure_ascii=False, indent=4).encode()
    row = (len(two) - 4) // 2 + 1                    # one item with its ",\n" separator
    assert row <= row_bytes_max(FORMAT_RECORDS, K, id_bytes) <= row + 40
    pred = {vid: [[x[j], x[K + j], x[2 * K + j]] for j in range(K)], vid + "2": [[x[j], x[K + j], x[2 * K + j]] for j in range(K)]}
    two = json.dumps(pred, sort_keys=True, ensure_ascii=False, indent=4).encode()
    row = (len(two) - 4 - 1) // 2 + 1
    assert row <= row_bytes_max(FORMAT_PREDICTIONS, K, id_bytes) <= row + 70


def test_format_results_refuses_bad_arguments():
    from audio_visual_deepfake_detection_b200 import native as nv
    from audio_visual_deepfake_detection_b200.libs.utils.result_writer import row_bytes_max
    L = nv.lib()
    fake = 1 << 40                                   # never dereferenced: every case below is refused before any launch
    ws = L.avdf_format_results_workspace_bytes(16)
    assert ws > 0

    def args(**kw):
        a = nv.FormatArgs()
        a.mode, a.K, a.records, a.n_records, a.order, a.n_pos = nv.FORMAT_RECORDS, 4, fake, 16, fake, 16
        a.ids, a.id_off, a.id_bytes_max, a.pos_begin, a.n_rows, a.min_score = fake, fake, 10, 0, 16, 0.2
        a.out, a.out_capacity, a.out_bytes = fake, 16 * row_bytes_max(nv.FORMAT_RECORDS, 4, 10), fake
        a.workspace, a.workspace_bytes = fake & ~255, ws
        for k, v in kw.items():
            setattr(a, k, v)
        return a
    cases = [dict(records=None), dict(order=None), dict(ids=None), dict(id_off=None), dict(out=None), dict(out_bytes=None),
             dict(workspace=None), dict(K=0), dict(K=-3), dict(mode=2), dict(n_rows=0), dict(pos_begin=10),
             dict(n_rows=1, out_capacity=row_bytes_max(nv.FORMAT_RECORDS, 4, 10) - 1),
             dict(out_capacity=16 * row_bytes_max(nv.FORMAT_RECORDS, 4, 10) - 1), dict(workspace_bytes=ws - 1),
             dict(workspace=(fake & ~255) + 8), dict(min_score=float("nan")), dict(id_bytes_max=-1),
             dict(mode=nv.FORMAT_PREDICTIONS, out_capacity=16 * row_bytes_max(nv.FORMAT_PREDICTIONS, 4, 10) - 1)]
    for kw in cases:
        assert L.avdf_format_results(ctypes.byref(args(**kw)), None) == -1, kw
        assert L.avdf_last_error()
    assert L.avdf_format_results(None, None) == -1
