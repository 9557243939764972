"""Inference driver with the reference's interface (libs/utils/train_utils.py:510-596
`inference_one_epoch`, :22-40 `fix_random_seed`, `valid_one_epoch`). Training utilities (optimizer,
scheduler, EMA, checkpoint saving) are outside the accelerated path."""
import os
import pickle
import random
import time

import numpy as np
import torch

from ...native import AvdfError
from .result_writer import write_result_records
from .sharding import record_width


class AverageMeter(object):
    def __init__(self):
        self.val = self.avg = self.sum = 0.0
        self.count = 0

    def update(self, val, n=1):
        self.val = val
        self.sum += val * n
        self.count += n
        self.avg = self.sum / self.count


def fix_random_seed(seed, include_cuda=True):
    gen = torch.manual_seed(seed)
    np.random.seed(seed)
    random.seed(seed)
    os.environ["PYTHONHASHSEED"] = str(seed)
    if include_cuda and torch.cuda.is_available():
        torch.cuda.manual_seed_all(seed)
    return gen


def result_item(video_id, out):
    """The JSON record of train_utils.py:577-591."""
    n = out["segments"].shape[0]
    return {"video_id": video_id, "video_cls": out["video_cls"].numpy().tolist(),
            "scores": out["scores"].numpy().tolist() if n else [],
            "segments": out["segments"].numpy().tolist() if n else []}


def pack_outputs(outputs):
    """Model output dicts (segments [n, 2], scores [n], video_cls [1], fp32) -> (records fp32 [len, 3 + 3K], K) in the
    layout of sharding.pack_records with K = the largest n (at least 1) and index 0; one scatter per field."""
    n = torch.tensor([int(o["scores"].shape[0]) for o in outputs], dtype=torch.long)
    K = max(1, int(n.max())) if len(outputs) else 1
    rec = torch.zeros((len(outputs), record_width(K)), dtype=torch.float32)
    if not outputs:
        return rec, K
    rec[:, 1] = n.float()
    rec[:, 2] = torch.cat([o["video_cls"].reshape(-1)[:1] for o in outputs]).float()
    valid = torch.arange(K)[None, :] < n[:, None]
    rec[:, 3:3 + K][valid] = torch.cat([o["scores"].reshape(-1) for o in outputs]).float()
    rec[:, 3 + K:].view(len(outputs), K, 2)[valid] = torch.cat([o["segments"].reshape(-1, 2) for o in outputs]).float()
    return rec, K


def one_epoch_records(val_loader, model, output_folder, dump_every=5000):
    """The loop of inference_one_epoch: runs `model(video_list)` over the loader and writes `data_left<iter>.json` every
    `dump_every` iterations plus a final `data_left.json` through the GPU writer. Returns the files written, in order, as
    (file name, ids, records on the device, K), and the model outputs of the last dump window."""
    model.eval()
    os.makedirs(output_folder, exist_ok=True)
    device = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else None
    files, ids, outs = [], [], []

    def dump(name):
        rec, K = pack_outputs(outs)
        if device is None:
            raise AvdfError("inference_one_epoch writes its results on sm_100a kernels; no CUDA device is visible")
        rec = rec.to(device)
        write_result_records(os.path.join(output_folder, name), ids, rec, K)
        files.append((name, list(ids), rec, K))
    for iter_idx, video_list in enumerate(val_loader, 0):
        if iter_idx > 0 and iter_idx % dump_every == 0:
            dump(f"data_left{iter_idx}.json")
            ids, outs = [], []
        with torch.no_grad():
            output = model(video_list)
        for vid_idx in range(len(output)):
            ids.append(video_list[vid_idx]["video_id"])
            outs.append(output[vid_idx])
    if len(outs) > 0:
        dump("data_left.json")
    return files, list(zip(ids, outs))


def inference_one_epoch(val_loader, model, curr_epoch, ext_score_file=None, evaluator=None, output_folder=None,
                        tb_writer=None, print_freq=20, subset="test", max_avg_nr_proposal=100, dataset_name="",
                        dump_every=5000):
    """Runs `model(video_list)` over the loader and writes `data_left<iter>.json` every `dump_every`
    iterations plus a final `data_left.json` (train_utils.py:546-595), with the bytes json.dump writes (the text is
    formatted on the GPU, libs/utils/result_writer.py). Returns the records of the last dump window (the reference
    returns None; callers ignore it)."""
    assert (evaluator is not None) or (output_folder is not None)
    _, last = one_epoch_records(val_loader, model, output_folder, dump_every)
    return [result_item(vid, out) for vid, out in last]


def valid_one_epoch(val_loader, model, curr_epoch, ext_score_file=None, evaluator=None, output_file=None, tb_writer=None,
                    print_freq=20):
    """The reference's validation loop: runs `model(video_list)` over the loader, collects every segment into the
    evaluator's dict form (video-id, t-start, t-end, label, score) and returns the evaluator's average mAP
    (libs/utils/metrics.py ANETdetection, on the GPU). Without an evaluator the dict is pickled to `output_file` and
    0.0 is returned. ext_score_file (the reference's external classification scores, postprocess_results) is not
    supported."""
    assert (evaluator is not None) or (output_file is not None)
    if ext_score_file is not None:
        raise NotImplementedError("ext_score_file (postprocess_results with external classification scores) is not supported")
    batch_time = AverageMeter()
    model.eval()
    results = {"video-id": [], "t-start": [], "t-end": [], "label": [], "score": []}
    start = time.time()
    for iter_idx, video_list in enumerate(val_loader, 0):
        with torch.no_grad():
            output = model(video_list)
            for vid_idx in range(len(output)):
                n = output[vid_idx]["segments"].shape[0]
                if n > 0:
                    results["video-id"].extend([output[vid_idx]["video_id"]] * n)
                    results["t-start"].append(output[vid_idx]["segments"][:, 0])
                    results["t-end"].append(output[vid_idx]["segments"][:, 1])
                    results["label"].append(output[vid_idx]["labels"])
                    results["score"].append(output[vid_idx]["scores"])
        if (iter_idx != 0) and iter_idx % print_freq == 0:
            torch.cuda.synchronize()
            batch_time.update((time.time() - start) / print_freq)
            start = time.time()
            print("Test: [{0:05d}/{1:05d}]\tTime {batch_time.val:.2f} ({batch_time.avg:.2f})".format(
                iter_idx, len(val_loader), batch_time=batch_time))
    for k, dt in (("t-start", torch.float32), ("t-end", torch.float32), ("label", torch.long), ("score", torch.float32)):
        results[k] = torch.cat(results[k]).cpu().numpy() if results[k] else torch.zeros(0, dtype=dt).numpy()
    if evaluator is not None:
        _, mAP, _ = evaluator.evaluate(results, verbose=True)
    else:
        with open(output_file, "wb") as f:
            pickle.dump(results, f)
        mAP = 0.0
    if tb_writer is not None:
        tb_writer.add_scalar("validation/mAP", mAP, curr_epoch)
    return mAP


def sharded_records(dataset, model, output_folder, batch_size=32, rank=0, world=1, print_freq=0, window=None, hop=None):
    """The work of inference_sharded up to its file: streams this rank's shard, all-gathers the records and writes
    `data_left.json` on rank 0 from the gathered device records. Returns (ids in dataset order, records, order, K) on
    rank 0 (order[j] = the record row of video j), None elsewhere."""
    from .sharding import gather_records, shard_indices
    model.eval()
    n = len(dataset)
    mine = shard_indices(n, rank, world)
    K = int(model.test_max_seg_num)
    if model.test_nms_method == "none":
        raise NotImplementedError("nms_method 'none' returns a variable number of segments: use inference_one_epoch per shard")
    runner = model.runner()
    ring, counter = runner.enable_records(max(1, len(mine)))

    def batches():
        for i in range(0, len(mine), batch_size):
            chunk = []
            for j in mine[i:i + batch_size]:
                item = dict(dataset[j])
                item["index"] = j
                chunk.append(item)
            yield chunk
    if window is None:
        outs = model.stream(batches())
    else:
        fs, nf = getattr(dataset, "feat_stride", 1), getattr(dataset, "num_frames", 1)
        outs = (runner.run_windows(chunk, window, hop, fs, nf) for chunk in batches())
    done = 0
    try:
        for out in outs:
            done += len(out)
            if print_freq and rank == 0 and (done // batch_size) % print_freq == 0:
                print("Test: [{0:05d}/{1:05d}]".format(done, len(mine)))
        torch.cuda.synchronize(ring.device)
        assert int(counter.item()) == len(mine), (int(counter.item()), len(mine))
        rec = gather_records(ring[:len(mine)], n, world)
    finally:
        runner.enable_records(None)
    if rank != 0:
        return None
    index = rec[:, 0]
    valid = index >= 0
    order = torch.full((n,), -1, dtype=torch.int32, device=rec.device)
    order[index[valid].long()] = torch.nonzero(valid).reshape(-1).int()
    assert int(valid.sum()) == n and bool((order >= 0).all()), (int(valid.sum()), n)
    ids = [dataset.data_list[j]["id"] for j in range(n)]
    os.makedirs(output_folder, exist_ok=True)
    write_result_records(f"{output_folder}/data_left.json", ids, rec, K, order)
    return ids, rec, order, K


def inference_sharded(dataset, model, output_folder, batch_size=32, rank=0, world=1, print_freq=0, window=None, hop=None):
    """Multi-GPU form of inference_one_epoch: one process per GPU (torchrun), rank r takes videos r, r + world, ... of the
    dataset (the reference splits its list into 7 files run as 7 processes, libs/datasets/deepfake_video_audio.py:420-431,
    inference.py:116-124); each rank streams its shard through `model.stream` (pinned staging, H2D, CUDA graph), the
    postprocess kernel appends one fixed-size record per video to a device ring, and ONE all-gather of those records
    (NCCL) is the path's only exchange. Rank 0 writes `data_left.json` in dataset order from the gathered device records
    (the text is formatted on the GPU, libs/utils/result_writer.py), exactly the bytes inference_one_epoch writes for the
    same list. Returns the records on rank 0, None elsewhere.

    window / hop (seconds): recordings longer than `window` run as overlapping windows merged on the GPU
    (model.forward_streams(..., window, hop)); still one record per recording. Per-window metadata uses the dataset's
    feat_stride / num_frames."""
    from .sharding import unpack_records
    res = sharded_records(dataset, model, output_folder, batch_size, rank, world, print_freq, window, hop)
    if res is None:
        return None
    ids, rec, _, K = res
    by_index = unpack_records(rec, K)
    assert len(by_index) == len(ids), (len(by_index), len(ids))
    return [result_item(ids[j], by_index[j]) for j in range(len(ids))]
