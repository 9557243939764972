"""Result files written on the GPU (csrc/results.cu, libs/utils/result_writer.py) against the bytes Python's json writes:
the numbers against float.__repr__, data_left.json against json.dump of the result_item lists, prediction.json /
prediction.txt against merge_results, and the files of inference_one_epoch / inference_sharded / inference.py --merge."""
import json
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest
import torch

from audio_visual_deepfake_detection_b200.libs.utils import merge_results
from audio_visual_deepfake_detection_b200.libs.utils.infer_utils import result_item
from audio_visual_deepfake_detection_b200.libs.utils.result_writer import write_predictions, write_result_records
from audio_visual_deepfake_detection_b200.libs.utils.sharding import unpack_records

pytestmark = pytest.mark.gpu

ODD_IDS = ["", 'q"uote', "back\\slash", "ctl\x01\x1f\t\n", "été/видео/動画.mp4", "emoji \U0001F600", "plain/000.mp4"]


def records(rng, n_rows, K, counts):
    rec = np.zeros((n_rows, 3 + 3 * K), np.float32)
    rec[:, 0] = np.arange(n_rows)
    rec[:, 1] = counts
    rec[:, 2] = rng.standard_normal(n_rows).astype(np.float32) * 4
    rec[:, 3:3 + K] = rng.random((n_rows, K), dtype=np.float32)
    rec[:, 3 + K:] = rng.random((n_rows, 2 * K), dtype=np.float32) * 33
    return torch.from_numpy(rec)


def dumped(items):
    return json.dumps(items, ensure_ascii=False, indent=4).encode("utf-8")


def test_numbers_match_repr(tmp_path):
    """>= 2^24 stratified bit patterns: every exponent and sign with random mantissas, and decimals of 1 - 17 significant
    digits rounded to fp32; checked in slices of 2^22 numbers (one file each) to bound host memory."""
    rng = np.random.default_rng(0)
    e = np.repeat(np.arange(256, dtype=np.uint32), 1 << 16)
    bits = (rng.integers(0, 2, e.size, dtype=np.uint32) << 31) | (e << 23) | rng.integers(0, 1 << 23, e.size, dtype=np.uint32)
    dec = []
    for d in range(1, 18):
        m = rng.integers(10 ** (d - 1), 10 ** d, 1 << 15, dtype=np.int64).astype(np.float64)
        dec.append((m * 10.0 ** rng.integers(-45, 39 - d, m.size)).astype(np.float32).view(np.uint32))
    special = np.array([0, 0x80000000, 0x7f800000, 0xff800000, 0x7fc00000, 1, 0x80000001, 0x7f7fffff], np.uint32)
    bits = np.concatenate([bits, *dec, special])
    assert bits.size >= 1 << 24
    K = 1000
    for s0 in range(0, bits.size, 1 << 22):
        part = bits[s0:s0 + (1 << 22)]
        n_rows = -(-part.size // (3 * K))
        flat = np.zeros(n_rows * 3 * K, np.uint32)
        flat[:part.size] = part
        rec = np.zeros((n_rows, 3 + 3 * K), np.uint32)
        rec[:, 1] = np.float32(K).view(np.uint32)
        rec[:, 3:] = flat.reshape(n_rows, 3 * K)
        path = tmp_path / "numbers.json"
        write_result_records(str(path), ["v%d" % i for i in range(n_rows)], torch.from_numpy(rec.view(np.float32)).cuda(), K)
        body = re.sub(r'"video_id": "v\d+",', "", path.read_text())
        got = re.findall(r"-?[0-9][0-9.e+\-]*|NaN|-?Infinity", body)
        vals = rec.view(np.float32)
        with np.errstate(invalid="ignore"):
            want_vals = np.concatenate([vals[:, 2:3], vals[:, 3:]], axis=1).reshape(-1).astype(np.float64)
        want = json.dumps(want_vals.tolist())[1:-1].split(", ")
        assert len(got) == len(want)
        bad = [i for i, (g, w) in enumerate(zip(got, want)) if g != w]
        assert not bad, [(got[i], want[i]) for i in bad[:10]]


@pytest.mark.parametrize("K", [1, 7, 100])
def test_record_list_bytes(tmp_path, K):
    rng = np.random.default_rng(K)
    n = 40
    counts = np.concatenate([[0, 1, K, 0, 1], rng.integers(0, K + 1, n - 5)])
    rec = records(rng, n, K, counts)
    ids = [(ODD_IDS[i] if i < len(ODD_IDS) else "id%03d/x.mp4" % i) for i in range(n)]
    by = unpack_records(rec, K)
    want = dumped([result_item(ids[j], by[j]) for j in range(n)])
    # ring order: a permutation with -1 pad rows, positions pick their rows through `order`
    perm = rng.permutation(n)
    ring = torch.zeros((n + 5, rec.shape[1]))
    ring[:, 0] = -1
    ring[:n] = rec[perm]
    ring = ring[torch.from_numpy(rng.permutation(n + 5))]
    order = torch.full((n,), -1, dtype=torch.int32)
    idx = ring[:, 0]
    order[idx[idx >= 0].long()] = torch.nonzero(idx >= 0).reshape(-1).int()
    for chunk in (1 << 26, None):
        path = tmp_path / "dl.json"
        from audio_visual_deepfake_detection_b200.libs.utils.result_writer import row_bytes_max
        cb = chunk or row_bytes_max(0, K, max(len(json.dumps(i, ensure_ascii=False).encode()) for i in ids)) * 3
        write_result_records(str(path), ids, ring.cuda(), K, order.cuda(), chunk_bytes=cb)
        assert path.read_bytes() == want
    for m in (0, 1):
        write_result_records(str(tmp_path / "m.json"), ids[:m], rec[:m].cuda(), K)
        assert (tmp_path / "m.json").read_bytes() == dumped([result_item(ids[j], by[j]) for j in range(m)])


def test_invalid_rows_raise(tmp_path):
    from audio_visual_deepfake_detection_b200.native import AvdfError
    rec = records(np.random.default_rng(1), 4, 3, [1, 2, 3, 4])           # n = 4 > K
    with pytest.raises(AvdfError):
        write_result_records(str(tmp_path / "x.json"), list("abcd"), rec.cuda(), 3)


def merged_files(tmp_path, name, ids, rec, K, files=None):
    """merge_results over json.dump-written result files of the same records."""
    src = tmp_path / (name + "_src")
    src.mkdir()
    by = unpack_records(rec, K)
    files = files or [("data_left.json", list(range(len(ids))))]
    for fname, rows in files:
        with open(src / fname, "w", encoding="utf-8") as f:
            json.dump([result_item(ids[r], by[r]) for r in rows], f, ensure_ascii=False, indent=4)
    merge_results([str(src)], str(tmp_path / (name + "_ref")))
    return [(tmp_path / (name + "_ref") / f).read_bytes() for f in ("prediction.json", "prediction.txt")]


def test_prediction_bytes(tmp_path):
    rng = np.random.default_rng(3)
    K, n = 20, 60
    rec = records(rng, n, K, rng.integers(0, K + 1, n))
    rec[0, 3:3 + K] = 0.1                                          # every segment filtered out
    rec[1, 3:3 + K] = 0.2                                          # == 0.2 (fp32) and the next fp32 above it
    rec[1, 4] = float(np.nextafter(np.float32(0.2), np.float32(1)))
    rec[1, 1] = 5
    rec[2, 1] = 0
    ids = ["z%02d" % (i % 45) for i in range(n)]                   # duplicates: first occurrence wins
    ids[3:3 + len(ODD_IDS)] = ODD_IDS
    ids[20] = "Ä-key"
    ids[21] = "a-key"
    want = merged_files(tmp_path, "p", ids, rec, K)
    out = tmp_path / "gpu"
    write_predictions(str(out), ids, rec.cuda(), K, chunk_bytes=4096)
    assert [(out / f).read_bytes() for f in ("prediction.json", "prediction.txt")] == want
    # every video filtered out, and no videos
    rec[:, 3:3 + K] = 0.0
    want = merged_files(tmp_path, "q", ids, rec, K)
    write_predictions(str(tmp_path / "gq"), ids, rec.cuda(), K)
    assert [(tmp_path / "gq" / f).read_bytes() for f in ("prediction.json", "prediction.txt")] == want
    write_predictions(str(tmp_path / "e"), [], rec[:0].cuda(), K)
    assert (tmp_path / "e" / "prediction.json").read_bytes() == b"{}" and (tmp_path / "e" / "prediction.txt").read_bytes() == b""


def _model_and_data(tmp_path, durs):
    from test_datasets_results import _cli_setup, dataset_kwargs
    from audio_visual_deepfake_detection_b200.libs.datasets import make_inference_dataset
    from audio_visual_deepfake_detection_b200.libs.modeling import make_meta_arch
    root, folders, cfg_path, full, sd = _cli_setup(tmp_path, durs)
    ds = make_inference_dataset("deepfake_video_audioEmoBYOLA_inference", False, ["test"], 3, **dataset_kwargs(folders))
    model = make_meta_arch(full["model_name"], **full["model"], max_batch=4)
    model.load_state_dict(sd)
    model.to("cuda").eval()
    return root, cfg_path, full, sd, ds, model


def test_end_to_end_files(tmp_path):
    from audio_visual_deepfake_detection_b200.libs.datasets import make_data_loader
    from audio_visual_deepfake_detection_b200.libs.utils import inference_one_epoch, inference_sharded
    durs = [4.03, 5.5, 7.42, 9.04, 6.2, 11.0, 4.7, 23.5]
    root, cfg_path, full, sd, ds, model = _model_and_data(tmp_path, durs)
    seen = []

    class Spy:
        def eval(self):
            model.eval()

        def __call__(self, vl):
            out = model(vl)
            seen.append([result_item(v["video_id"], o) for v, o in zip(vl, out)])
            return out
    loader = make_data_loader(ds, False, None, 2, 0)
    last = inference_one_epoch(loader, Spy(), -1, output_folder=str(tmp_path / "a"), dump_every=2)
    windows = [sum(seen[i:i + 2], []) for i in range(0, len(seen), 2)]
    names = ["data_left%d.json" % (2 * k) for k in range(1, len(windows))] + ["data_left.json"]
    for name, items in zip(names, windows):
        assert (tmp_path / "a" / name).read_bytes() == dumped(items)
    assert last == windows[-1]
    assert sorted(os.listdir(tmp_path / "a")) == sorted(names)
    for kw, tag in (({}, "b"), ({"window": 10.0, "hop": 5.0}, "c")):
        res = inference_sharded(ds, model, str(tmp_path / tag), batch_size=4, **kw)
        assert (tmp_path / tag / "data_left.json").read_bytes() == dumped(res)


def test_cli_merge_and_stale_file(tmp_path):
    durs = [4.03, 5.5, 7.42, 9.04, 6.2]
    root, cfg_path, full, sd, ds, model = _model_and_data(tmp_path, durs)
    ckpt = str(tmp_path / "run" / "epoch_010.pth.tar")
    os.makedirs(os.path.dirname(ckpt))
    torch.save({"epoch": 10, "state_dict_ema": sd}, ckpt)
    out_dir = tmp_path / "run" / "3"
    stale = [{"video_id": "stale/clip.mp4", "video_cls": [2.0], "scores": [0.9], "segments": [[1.0, 2.0]]},
             {"video_id": "id000/clip.mp4", "video_cls": [-3.0], "scores": [], "segments": []}]
    for extra, stale_file in (([], False), ([], True), (["--window", "6"], False)):
        if out_dir.exists():
            shutil.rmtree(out_dir)
        if stale_file:
            out_dir.mkdir(parents=True)
            with open(out_dir / "data_left.0.json", "w", encoding="utf-8") as f:   # sorts before data_left.json
                json.dump(stale, f, ensure_ascii=False, indent=4)
        r = subprocess.run([sys.executable, os.path.join(root, "inference.py"), cfg_path, "3", ckpt, "-b", "4", "--merge", *extra],
                           capture_output=True, text=True, cwd=root, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        ref = tmp_path / "ref"
        if ref.exists():
            shutil.rmtree(ref)
        shutil.copytree(out_dir, ref / "in", ignore=shutil.ignore_patterns("prediction*"))
        merge_results([str(ref / "in")], str(ref / "out"))
        for f in ("prediction.json", "prediction.txt"):
            assert (out_dir / f).read_bytes() == (ref / "out" / f).read_bytes(), (extra, stale_file, f)
        if stale_file:
            assert "stale/clip.mp4" in json.load(open(out_dir / "prediction.json"))
