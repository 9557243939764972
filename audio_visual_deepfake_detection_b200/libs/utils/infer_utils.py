"""Inference driver with the reference's interface (libs/utils/train_utils.py:510-596
`inference_one_epoch`, :22-40 `fix_random_seed`, `valid_one_epoch`). Training utilities (optimizer,
scheduler, EMA, checkpoint saving) are outside the accelerated path."""
import json
import os
import pickle
import random
import time

import numpy as np
import torch


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


def inference_one_epoch(val_loader, model, curr_epoch, ext_score_file=None, evaluator=None, output_folder=None,
                        tb_writer=None, print_freq=20, subset="test", max_avg_nr_proposal=100, dataset_name="",
                        dump_every=5000):
    """Runs `model(video_list)` over the loader and writes `data_left<iter>.json` every `dump_every`
    iterations plus a final `data_left.json` (train_utils.py:546-595). Returns the records of the last dump
    window (the reference returns None; callers ignore it)."""
    assert (evaluator is not None) or (output_folder is not None)
    model.eval()
    os.makedirs(output_folder, exist_ok=True)
    batch_results = []
    for iter_idx, video_list in enumerate(val_loader, 0):
        if iter_idx > 0 and iter_idx % dump_every == 0:
            with open(f"{output_folder}/data_left{iter_idx}.json", "w", encoding="utf-8") as f:
                json.dump(batch_results, f, ensure_ascii=False, indent=4)
            batch_results = []
        with torch.no_grad():
            output = model(video_list)
        for vid_idx in range(len(output)):
            batch_results.append(result_item(video_list[vid_idx]["video_id"], output[vid_idx]))
    if len(batch_results) > 0:
        with open(f"{output_folder}/data_left.json", "w", encoding="utf-8") as f:
            json.dump(batch_results, f, ensure_ascii=False, indent=4)
    return batch_results


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


def inference_sharded(dataset, model, output_folder, batch_size=32, rank=0, world=1, print_freq=0, window=None, hop=None):
    """Multi-GPU form of inference_one_epoch: one process per GPU (torchrun), rank r takes videos r, r + world, ... of the
    dataset (the reference splits its list into 7 files run as 7 processes, libs/datasets/deepfake_video_audio.py:420-431,
    inference.py:116-124); each rank streams its shard through `model.stream` (pinned staging, H2D, CUDA graph), the
    postprocess kernel appends one fixed-size record per video to a device ring, and ONE all-gather of those records
    (NCCL) is the path's only exchange. Rank 0 writes `data_left.json` in dataset order, exactly the records
    inference_one_epoch writes for the same list. Returns the records on rank 0, None elsewhere.

    window / hop (seconds): recordings longer than `window` run as overlapping windows merged on the GPU
    (model.forward_streams(..., window, hop)); still one record per recording. Per-window metadata uses the dataset's
    feat_stride / num_frames."""
    from .sharding import gather_records, shard_indices, unpack_records
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
    by_index = unpack_records(rec, K)
    assert len(by_index) == n, (len(by_index), n)
    results = [result_item(dataset.data_list[j]["id"], by_index[j]) for j in range(n)]
    os.makedirs(output_folder, exist_ok=True)
    with open(f"{output_folder}/data_left.json", "w", encoding="utf-8") as f:
        json.dump(results, f, ensure_ascii=False, indent=4)
    return results
