"""Result files written from the device records: `data_left*.json` and `prediction.json` / `prediction.txt`, byte for byte
what `json.dump` writes today (infer_utils.inference_one_epoch / inference_sharded, results.merge_results), with the
JSON text made by the GPU (csrc/results.cu, avdf_format_results) instead of Python's pure-Python indent encoder.

Rows are the fixed-size records of libs/utils/sharding.py (fp32 [R, 3 + 3K] on a CUDA device); `order[i]` is the row of
the i-th listed video and `ids[i]` its id. The host quotes each id with json's own string encoder and uploads them as
one blob; the device formats chunks of rows that fit `chunk_bytes` while the previous chunk goes device -> pinned host
buffer -> file (two buffers of each). There is no CPU fallback: without CUDA the writers raise AvdfError.
"""
import collections
import os
from json.encoder import encode_basestring

import numpy as np
import torch

from ... import ops
from ...native import FORMAT_PREDICTIONS, FORMAT_RECORDS, AvdfError
from .results import video_probability

NUM_MAX = 23                 # longest text of one number (json_format.cuh AVDF_JSON_NUM_MAX)
CHUNK_BYTES = 64 << 20


def row_bytes_max(mode, K, id_bytes):
    """Longest text of one output position (csrc/results.cu row_bytes_max): the buffer of a chunk of n rows must hold n
    of these."""
    N = NUM_MAX
    if mode == FORMAT_RECORDS:
        return (2 + 26 + id_bytes + 37 + N + 31 + 31 + K * (13 + N + 1) + 33
                + K * (31 + N + 18 + N + 14 + 1) + 16)
    return 2 + 4 + id_bytes + 3 + 64 + K * (23 + 3 * N + 2 * 14 + 10 + 1) + 6


def _device(records):
    if not torch.cuda.is_available():
        raise AvdfError("result_writer formats on sm_100a kernels only; no CUDA device is visible (no CPU fallback)")
    if not records.is_cuda or records.dtype != torch.float32 or records.dim() != 2:
        raise AvdfError("records must be a 2-D fp32 CUDA tensor")
    return records.device


def _id_blob(ids, device):
    enc = [encode_basestring(s).encode("utf-8") for s in ids]
    lens = np.fromiter((len(e) for e in enc), dtype=np.int64, count=len(enc))
    off = np.zeros(len(enc) + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    blob = bytearray(b"".join(enc) or b"\0")
    return (torch.frombuffer(blob, dtype=torch.uint8).to(device), torch.from_numpy(off).to(device),
            int(lens.max()) if len(enc) else 0)


def _order(order, n_rows, n, device):
    if order is None:
        if n != n_rows:
            raise ValueError("without `order`, ids must name every row (%d ids, %d rows)" % (n, n_rows))
        return torch.arange(n, dtype=torch.int32, device=device)
    order = torch.as_tensor(order).to(device=device, dtype=torch.int32).contiguous()
    if order.numel() != n:
        raise ValueError("order has %d entries for %d ids" % (order.numel(), n))
    return order


def _write(path, mode, ids, records, K, order, brackets, min_score, chunk_bytes):
    """Streams the text of positions 0 .. len(ids) - 1 into `path` between `brackets` ("[]" or "{}")."""
    device = records.device
    if records.shape[1] != 3 + 3 * K:
        raise ValueError("records have width %d, K = %d needs %d" % (records.shape[1], K, 3 + 3 * K))
    n = len(ids)
    with open(path, "wb") as f:
        if n == 0:
            f.write(brackets.encode())
            return
        with torch.cuda.device(device):
            blob, off, id_max = _id_blob(ids, device)
            row_max = row_bytes_max(mode, K, id_max)
            if chunk_bytes < row_max:
                raise ValueError("chunk_bytes = %d cannot hold one row (%d bytes)" % (chunk_bytes, row_max))
            per = min(n, chunk_bytes // row_max, (1 << 31) - 1)
            cap = per * row_max
            dbuf = [torch.empty(cap, dtype=torch.uint8, device=device) for _ in range(2)]
            hbuf = [torch.empty(cap, dtype=torch.uint8, pin_memory=True) for _ in range(2)]
            dcnt = torch.empty(2, dtype=torch.int64, device=device)
            hcnt = torch.empty(2, dtype=torch.int64, pin_memory=True)
            main, side = torch.cuda.current_stream(device), torch.cuda.Stream(device)
            formatted = [torch.cuda.Event() for _ in range(2)]
            copied = [torch.cuda.Event() for _ in range(2)]
            pending = collections.deque()

            def flush():
                b, rows = pending.popleft()
                copied[b].synchronize()
                nbytes = int(hcnt[b])
                if nbytes < 0:
                    raise AvdfError("avdf_format_results: a row index, segment count or id length is out of range")
                f.write(memoryview(hbuf[b].numpy())[:nbytes])

            f.write(brackets[0].encode() + b"\n")
            ws = None
            for i, p0 in enumerate(range(0, n, per)):
                b, rows = i & 1, min(per, n - p0)
                if len(pending) == 2:        # buffers b are free once chunk i - 2 is in the file
                    flush()
                ws = ops.format_results(mode, records, K, order, blob, off, id_max, p0, rows, dbuf[b], dcnt[b:b + 1],
                                        min_score=min_score, workspace=ws)
                formatted[b].record(main)
                side.wait_event(formatted[b])
                with torch.cuda.stream(side):
                    hcnt[b:b + 1].copy_(dcnt[b:b + 1], non_blocking=True)
                    hbuf[b][:rows * row_max].copy_(dbuf[b][:rows * row_max], non_blocking=True)
                    copied[b].record(side)
                pending.append((b, rows))
            while pending:
                flush()
            f.write(b"\n" + brackets[1].encode())


def write_result_records(path, ids, records, K, order=None, chunk_bytes=CHUNK_BYTES):
    """`json.dump([result_item(ids[i], row order[i]) ...], f, ensure_ascii=False, indent=4)` into `path`, byte for byte.
    records: fp32 CUDA [R, 3 + 3K]; order: int32 rows (default: every row in order)."""
    device = _device(records)
    _write(path, FORMAT_RECORDS, ids, records, K, _order(order, records.shape[0], len(ids), device), "[]", 0.0, chunk_bytes)


def prediction_order(ids, order):
    """The (id, row) pairs of prediction.json: first occurrence of each id wins, sorted by id (merge_results)."""
    first = {}
    for i, vid in enumerate(ids):
        first.setdefault(vid, i)
    keys = sorted(first)
    pick = torch.tensor([first[k] for k in keys], dtype=torch.long, device=order.device)
    return keys, order[pick].contiguous() if keys else order[:0]


def write_predictions(out_dir, ids, records, K, min_score=0.2, snap=0.9, order=None, chunk_bytes=CHUNK_BYTES):
    """prediction.txt and prediction.json of merge_results over the result records listed as (ids[i], row order[i]), in
    the order merge_results would read them: byte for byte the files merge_results writes from the same records."""
    device = _device(records)
    order = _order(order, records.shape[0], len(ids), device)
    keys, rows = prediction_order(ids, order)
    os.makedirs(out_dir, exist_ok=True)
    cls = records[rows.long(), 2].double().cpu().tolist() if keys else []
    probs = [[k, str(video_probability(c, snap))] for k, c in zip(keys, cls)]
    with open(os.path.join(out_dir, "prediction.txt"), "w") as fo:
        fo.write("\n".join(";".join(i) for i in probs))
    _write(os.path.join(out_dir, "prediction.json"), FORMAT_PREDICTIONS, keys, records, K, rows, "{}", min_score, chunk_bytes)
