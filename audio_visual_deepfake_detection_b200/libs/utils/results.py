"""Final result files of the challenge submission (SURVEY.md 8f-2): the logic of generate_results.ipynb cells 1-2.

merge_results(folders) reads every `data*.json` / `*.json` written by inference_one_epoch (one folder per shard),
de-duplicates video ids (first occurrence wins, like the notebook) and produces
  prediction.txt   `video_id;prob` with prob = sigmoid(video_cls), snapped to 1.0 above 0.9 (cell 1)
  prediction.json  {video_id: [[score, start, end], ...]} keeping only segments with score > 0.2, `[[0,0,0]]` when none
                   survive (cell 2; this is the 0.2 score filter of the north star)
"""
import glob
import json
import math
import os


def video_probability(video_cls, snap=0.9):
    x = float(video_cls[0] if isinstance(video_cls, (list, tuple)) else video_cls)
    p = 1.0 / (1.0 + math.exp(-x))
    return 1.0 if p > snap else p


def filter_segments(scores, segments, min_score=0.2):
    out = [[s, seg[0], seg[1]] for s, seg in zip(scores, segments) if s > min_score]
    return out if out else [[0, 0, 0]]


def iter_result_records(folders, pattern="*.json"):
    """The result records of every `pattern` file (sorted by name) of every folder, in that order, skipping `prediction*`
    files; a video id seen before is skipped (first occurrence wins, like the notebook)."""
    seen = set()
    for folder in folders:
        for path in sorted(glob.glob(os.path.join(folder, pattern))):
            if os.path.basename(path).startswith("prediction"):
                continue
            with open(path, "r", encoding="utf-8") as f:
                data = json.load(f)
            for item in data:
                vid = item["video_id"]
                if vid in seen:
                    continue
                seen.add(vid)
                yield item


def merge_results(folders, out_dir=None, min_score=0.2, snap=0.9):
    probs, segs = [], {}
    for item in iter_result_records(folders):
        vid = item["video_id"]
        probs.append([vid, str(video_probability(item["video_cls"], snap))])
        segs[vid] = filter_segments(item["scores"], item["segments"], min_score)
    probs.sort(key=lambda x: x[0])
    if out_dir is not None:
        os.makedirs(out_dir, exist_ok=True)
        with open(os.path.join(out_dir, "prediction.txt"), "w") as fo:
            fo.write("\n".join(";".join(i) for i in probs))
        with open(os.path.join(out_dir, "prediction.json"), "w", encoding="utf-8") as f:
            json.dump(segs, f, sort_keys=True, ensure_ascii=False, indent=4)
    return probs, segs
