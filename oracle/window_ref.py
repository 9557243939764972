"""Host restatement of the sliding-window path (libs/modeling/windows.py + csrc/window.cu): slice every window out of
the recording on the host as a W-second item of its own, and merge the per-window results with the reference's
batched_nms (oracle/nms_ref.py).

TEST INFRASTRUCTURE — see oracle/model_ref.py's header for who may import it.
"""
import numpy as np
import torch

import nms_ref
from audio_visual_deepfake_detection_b200.libs.modeling.windows import window_plan

STREAMS = ("video", "byola", "emo")


def slice_windows(rec, window, hop=None):
    """rec {video_id, duration, streams} -> (list of (s_k, W-second item with contiguous copies of its rows), single)
    where single is True when the recording is its own (only) window."""
    names = [n for n in STREAMS if n in rec["streams"]]
    lens = [rec["streams"][n].shape[0] if n in rec["streams"] else None for n in STREAMS]
    plan = window_plan(rec["duration"], lens, window, hop)
    if len(plan) == 1:
        return [(0.0, rec)], True
    out = []
    for k, (s, rng) in enumerate(plan):
        streams = {n: np.ascontiguousarray(rec["streams"][n][a:a + m]) for n, (a, m) in zip(STREAMS, rng) if n in names}
        out.append((s, {"video_id": "%s@%d" % (rec["video_id"], k), "duration": float(window), "streams": streams}))
    return out, False


def merge(results, starts, test_cfg):
    """Per-window results (dicts of forward_streams, ascending window order) + window starts (seconds) -> one merged
    result: shift in fp32, class-agnostic batched_nms over the union in window order, max window logit."""
    segs = np.concatenate([(np.float32(s) + r["segments"].numpy().astype(np.float32)).reshape(-1, 2)
                           for s, r in zip(starts, results)]).astype(np.float32)
    scores = np.concatenate([r["scores"].numpy().astype(np.float32) for r in results])
    vcls = max(float(r["video_cls"][0]) for r in results)
    tc = test_cfg
    voting = 0.0 if tc["multiclass_nms"] else tc["voting_thresh"]
    s, p, _ = nms_ref.batched_nms(torch.from_numpy(segs), torch.from_numpy(scores), torch.zeros(len(scores), dtype=torch.long),
                                  tc["iou_threshold"], tc["min_score"], tc["max_seg_num"], use_soft_nms=tc["nms_method"] == "soft",
                                  multiclass=False, sigma=tc["nms_sigma"], voting_thresh=voting)
    return {"segments": s.reshape(-1, 2), "scores": p, "video_cls": torch.tensor([vcls], dtype=torch.float32)}


def run(model, recs, window, hop=None):
    """The composition oracle: every recording through model.forward_streams window by window (host-sliced), merged
    on the host."""
    tc = {k: getattr(model, "test_" + k) for k in ("iou_threshold", "min_score", "max_seg_num", "nms_method", "nms_sigma",
                                                      "voting_thresh", "multiclass_nms")}
    out = []
    for rec in recs:
        wins, single = slice_windows(rec, window, hop)
        res = model.forward_streams([w for _, w in wins])
        out.append(res[0] if single else merge(res, [s for s, _ in wins], tc))
    return out
