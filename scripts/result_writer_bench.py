"""Result-file writing on the GPU vs. Python's json (libs/utils/result_writer.py).

    python scripts/result_writer_bench.py [--videos 343233] [--out-dir DIR] [--json profiles/result_writer_bench.json]

Workload: the AV-Deepfake1M test list size (343,233 videos), K = 100, synthetic records: scores uniform fp32 in (0, 1),
segments in [0, 33] s, AV-Deepfake1M-like ids; two count mixes (all 100 segments; counts drawn 0 - 100). Reports
  - device formatting time of the whole list (CUDA events around back-to-back avdf_format_results calls, median of 7,
    warm), records (data_left.json) and predictions (prediction.json) modes;
  - write_result_records / write_predictions wall time into --out-dir (host clock around synchronised calls, median of
    3), bytes written and GB/s: this includes the device -> host copies and the file system;
  - the Python writers (json.dump of result_item lists, merge_results) on the first 1,000 videos only, not extrapolated,
    and SHA-256 equality of both writers' files on that subset;
  - the card name and power limit, read in the same run.
"""
import argparse
import hashlib
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from audio_visual_deepfake_detection_b200 import ops  # noqa: E402
from audio_visual_deepfake_detection_b200.native import FORMAT_PREDICTIONS, FORMAT_RECORDS  # noqa: E402
from audio_visual_deepfake_detection_b200.libs.utils import merge_results  # noqa: E402
from audio_visual_deepfake_detection_b200.libs.utils.infer_utils import result_item  # noqa: E402
from audio_visual_deepfake_detection_b200.libs.utils.result_writer import (CHUNK_BYTES, _id_blob, prediction_order,  # noqa: E402
                                                                           row_bytes_max, write_predictions, write_result_records)
from audio_visual_deepfake_detection_b200.libs.utils.sharding import unpack_records  # noqa: E402

K = 100


def synth(n, mix, seed):
    g = torch.Generator().manual_seed(seed)
    rec = torch.zeros((n, 3 + 3 * K), dtype=torch.float32)
    rec[:, 0] = torch.arange(n, dtype=torch.float32)
    rec[:, 1] = K if mix == "full" else torch.randint(0, K + 1, (n,), generator=g).float()
    rec[:, 2] = torch.randn(n, generator=g) * 3
    s = torch.rand((n, K), generator=g)
    rec[:, 3:3 + K] = torch.where(s > 0, s, torch.full_like(s, 0.5))
    rec[:, 3 + K:] = torch.rand((n, 2 * K), generator=g) * 33
    ids = ["test/id%05d/%08x/real_video_fake_audio.mp4" % (i // 7, (i * 2654435761) & 0xffffffff) for i in range(n)]
    return ids, rec


def device_time(mode, ids, rec, order, min_score=0.2, reps=7):
    """Formats the whole list in CHUNK_BYTES chunks on one stream, CUDA events around it."""
    dev = rec.device
    blob, off, id_max = _id_blob(ids, dev)
    row_max = row_bytes_max(mode, K, id_max)
    per = min(len(ids), CHUNK_BYTES // row_max)
    buf = torch.empty(per * row_max, dtype=torch.uint8, device=dev)
    cnt = torch.empty(1, dtype=torch.int64, device=dev)
    ws = None
    total = torch.zeros(1, dtype=torch.int64, device=dev)

    def once():
        nonlocal ws
        total.zero_()
        for p0 in range(0, len(ids), per):
            ws = ops.format_results(mode, rec, K, order, blob, off, id_max, p0, min(per, len(ids) - p0), buf, cnt,
                                    min_score=min_score, workspace=ws)
            total.add_(cnt)
    once()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        once()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1) / 1e3)
    return statistics.median(ts), int(total.item()), len(range(0, len(ids), per))


def wall(fn, reps=3):
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts)


def sha(path):
    with open(path, "rb") as f:
        return hashlib.sha256(f.read()).hexdigest()


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()[0]
        name, limit = [x.strip() for x in out.split(",")]
        return name, limit
    except Exception as exc:  # noqa: BLE001
        return torch.cuda.get_device_name(0), "unknown (%s)" % exc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--videos", type=int, default=343233)
    ap.add_argument("--python-videos", type=int, default=1000)
    ap.add_argument("--out-dir", default=None)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the benchmark measures the GPU writer"
    name, limit = card()
    out_dir = args.out_dir or tempfile.mkdtemp(prefix="result_writer_bench_")
    os.makedirs(out_dir, exist_ok=True)
    res = {"gpu": name, "power_limit": limit, "videos": args.videos, "K": K, "chunk_bytes": CHUNK_BYTES, "mixes": {}}
    for mix in ("full", "random"):
        ids, rec_h = synth(args.videos, mix, 0 if mix == "full" else 1)
        rec = rec_h.cuda()
        order = torch.arange(len(ids), dtype=torch.int32, device=rec.device)
        r = {}
        t, nbytes, chunks = device_time(FORMAT_RECORDS, ids, rec, order)
        r["device_format_records_s"], r["records_json_bytes"], r["records_chunks"] = round(t, 5), nbytes + 4, chunks
        keys, rows = prediction_order(ids, order)
        t, nbytes, _ = device_time(FORMAT_PREDICTIONS, keys, rec, rows)
        r["device_format_predictions_s"], r["prediction_json_bytes"] = round(t, 5), nbytes + 4
        path = os.path.join(out_dir, "data_left.json")
        t = wall(lambda: write_result_records(path, ids, rec, K))
        size = os.path.getsize(path)
        r["write_result_records_s"], r["write_result_records_bytes"], r["write_result_records_GBps"] = round(t, 4), size, round(size / t / 1e9, 3)
        pdir = os.path.join(out_dir, "pred")
        t = wall(lambda: write_predictions(pdir, ids, rec, K))
        size = os.path.getsize(os.path.join(pdir, "prediction.json")) + os.path.getsize(os.path.join(pdir, "prediction.txt"))
        r["write_predictions_s"], r["write_predictions_bytes"], r["write_predictions_GBps"] = round(t, 4), size, round(size / t / 1e9, 3)
        # the Python writers on the first videos only (not extrapolated)
        m = args.python_videos
        sub_ids, sub = ids[:m], rec_h[:m]
        py_dir, gpu_dir = os.path.join(out_dir, "py"), os.path.join(out_dir, "gpu")
        for d in (py_dir, gpu_dir):
            shutil.rmtree(d, ignore_errors=True)
            os.makedirs(d)
        t0 = time.perf_counter()
        by = unpack_records(sub, K)
        items = [result_item(sub_ids[j], by[j]) for j in range(m)]
        with open(os.path.join(py_dir, "data_left.json"), "w", encoding="utf-8") as f:
            json.dump(items, f, ensure_ascii=False, indent=4)
        t_py_rec = time.perf_counter() - t0
        t0 = time.perf_counter()
        merge_results([py_dir], py_dir)
        t_py_pred = time.perf_counter() - t0
        write_result_records(os.path.join(gpu_dir, "data_left.json"), sub_ids, sub.cuda(), K)
        write_predictions(gpu_dir, sub_ids, sub.cuda(), K)
        r["python_subset_videos"] = m
        r["python_subset_note"] = "first %d videos only, not extrapolated" % m
        r["python_json_dump_records_s"], r["python_merge_results_s"] = round(t_py_rec, 4), round(t_py_pred, 4)
        r["sha256_equal"] = {f: sha(os.path.join(py_dir, f)) == sha(os.path.join(gpu_dir, f))
                             for f in ("data_left.json", "prediction.json", "prediction.txt")}
        res["mixes"][mix] = r
        print(mix, json.dumps(r), flush=True)
    if not args.out_dir:
        shutil.rmtree(out_dir, ignore_errors=True)
    line = json.dumps(res)
    print(line)
    if args.json:
        with open(args.json, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
