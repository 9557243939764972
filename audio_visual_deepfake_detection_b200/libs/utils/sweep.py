"""Post-processing sweeps: one forward pass, many test_cfg settings scored against ground truth, all on the GPU.

The nine post-processing settings of test_cfg (nms_method, iou_threshold, min_score, nms_sigma, voting_thresh,
pre_nms_thresh, pre_nms_topk, duration_thresh, max_seg_num; multiclass_nms as the model reads it) never touch the
network: they only change the last launch of a pass. Here the pass runs once with its dense outputs kept on the device
(engine.DenseStore), then avdf_postprocess_sweep decodes, suppresses and writes result rows for up to 64 settings per
launch, and every setting's rows are scored by the GPU evaluators (metrics.ANETdetection.evaluate_rows, and
eval_proposal.average_recall_from_rows). Each setting's results are exactly what a model built with that test_cfg
returns from the same weights.

    res = sweep_postprocess(model, items, [{"nms_method": "soft", "min_score": 0.1}, ...], "gt.json", split="dev")
    res.results[i]        # {"setting", "mAP", "average_mAP", "mRecall"[, "AR@AN", "auc"]}
    res.records(i)        # setting i's results as the model's list of dicts (video_id, segments, scores, labels, video_cls)

Command line (loads state_dict_ema and the config's inference dataset like inference.py):
    python -m audio_visual_deepfake_detection_b200.libs.utils.sweep CFG CKPT --gt GT --split dev \\
        --set nms_method=hard,soft --set iou_threshold=0.1,0.3 ... [--out sweep.json]
"""
import argparse
import itertools
import json
import math

import numpy as np
import torch

from ... import native as nv
from ... import ops
from ...native import AvdfError
from ..modeling.engine import DenseStore
from .Evaluation.eval_proposal import AR_AT, area_under_curve, average_recall_from_rows
from .metrics import DEFAULT_TIOU, ANETdetection, RowsLayout

SETTING_KEYS = ("nms_method", "iou_threshold", "min_score", "nms_sigma", "voting_thresh", "pre_nms_thresh", "pre_nms_topk",
                "duration_thresh", "max_seg_num", "multiclass_nms")
_INT_KEYS = ("pre_nms_topk", "max_seg_num")
MAX_PER_LAUNCH = 64


def _parse_value(key, text):
    if key == "nms_method":
        return text
    if key == "multiclass_nms":
        if text.lower() in ("true", "1", "yes"):
            return True
        if text.lower() in ("false", "0", "no"):
            return False
        raise ValueError("multiclass_nms takes true / false, not %r" % text)
    return int(text) if key in _INT_KEYS else float(text)


def parse_set(arg):
    """'key=v1,v2,...' -> (key, [values]) with the type test_cfg uses for that key."""
    if "=" not in arg:
        raise ValueError("--set takes key=v1,v2,..., got %r" % arg)
    key, vals = arg.split("=", 1)
    key = key.strip()
    if key not in SETTING_KEYS:
        raise ValueError("%r is not a post-processing setting (one of %s)" % (key, ", ".join(SETTING_KEYS)))
    values = [_parse_value(key, v.strip()) for v in vals.split(",") if v.strip()]
    if not values:
        raise ValueError("--set %s has no values" % key)
    return key, values


def grid(sets):
    """Cartesian product of [(key, [values]), ...] as a list of dicts; the last key varies fastest."""
    keys = [k for k, _ in sets]
    if len(set(keys)) != len(keys):
        raise ValueError("a setting is given twice: %s" % keys)
    return [dict(zip(keys, combo)) for combo in itertools.product(*[v for _, v in sets])]


def full_setting(base, setting, num_classes=1):
    """A complete, checked setting: `setting` over the test_cfg `base`. Raises AvdfError for what the sweep refuses."""
    unknown = [k for k in setting if k not in SETTING_KEYS]
    if unknown:
        raise ValueError("not post-processing settings: %s" % unknown)
    s = {k: base[k] for k in SETTING_KEYS}
    s.update(setting)
    if s["nms_method"] not in ("hard", "soft"):
        raise AvdfError("nms_method %r: a sweep runs hard or soft NMS ('none' returns every candidate)" % (s["nms_method"],))
    if s["multiclass_nms"] and num_classes > 1:
        raise AvdfError("multiclass NMS with more than one class is not on the accelerated path")
    for k in SETTING_KEYS:
        if k not in ("nms_method", "multiclass_nms") and not math.isfinite(float(s[k])):
            raise AvdfError("%s = %r is not finite" % (k, s[k]))
    if not (1 <= int(s["max_seg_num"]) <= nv.MAX_SEGS):
        raise AvdfError("max_seg_num must be 1..%d, got %r" % (nv.MAX_SEGS, s["max_seg_num"]))
    if s["nms_method"] == "soft" and not float(s["nms_sigma"]) > 0:
        raise AvdfError("soft NMS needs nms_sigma > 0, got %r" % (s["nms_sigma"],))
    if int(s["pre_nms_topk"]) < 0:
        raise AvdfError("pre_nms_topk must be >= 0")
    return s


def c_setting(s):
    """A full setting -> the kernel's table entry (what engine.postprocess passes for that test_cfg)."""
    return nv.SweepSetting(float(s["pre_nms_thresh"]), int(s["pre_nms_topk"]), float(s["duration_thresh"]),
                           float(s["iou_threshold"]), float(s["min_score"]), float(s["nms_sigma"]),
                           0.0 if s["multiclass_nms"] else float(s["voting_thresh"]), int(s["max_seg_num"]),
                           1 if s["nms_method"] == "soft" else 0)


def sweep_rows(store, settings, device=None):
    """Result rows of every stored video under `settings` (full settings, any number): fp32 [S, N, 3 + 3K] on the device,
    K = the largest max_seg_num, rows in the store's video order."""
    if not settings:
        raise AvdfError("the settings grid is empty")
    N = len(store)
    K = max(int(s["max_seg_num"]) for s in settings)
    dev = device or (store.chunks[0]["logits"].device if store.chunks else torch.device("cuda", torch.cuda.current_device()))
    rows = torch.empty((len(settings), N, 3 + 3 * K), dtype=torch.float32, device=dev)
    table = [c_setting(s) for s in settings]
    ws = None
    for c in store.chunks:
        n = c["n"]
        valid = torch.from_numpy(c["valid"][:n]).to(dev)
        pos = torch.from_numpy(c["pos"][:n]).to(dev)
        meta = [c["meta"][i, :n] for i in range(4)]
        for s0 in range(0, len(table), MAX_PER_LAUNCH):
            part = table[s0:s0 + MAX_PER_LAUNCH]
            ws = ops.postprocess_sweep(c["logits"][:n], c["offsets"][:n], valid, level_len=c["level_len"],
                                       level_stride=c["level_stride"], settings=part, out_rows=rows[s0:s0 + len(part)],
                                       vid_meta=meta, vid_cls=c["vcls"][:n], vid_index=pos, workspace=ws)
    return rows


def rows_to_records(ids, rows):
    """One setting's rows [N, 3 + 3K] -> the model's list of dicts, in store order."""
    r = rows.cpu()
    K = (r.shape[1] - 3) // 3
    counts = r[:, 1].to(torch.int64).tolist()
    segs = r[:, 3 + K:].reshape(-1, K, 2)
    empty_labels = torch.zeros(K, dtype=torch.long)
    return [{"video_id": vid, "segments": segs[b, :n].clone(), "scores": r[b, 3:3 + n].clone(), "labels": empty_labels[:n],
             "video_cls": r[b, 2:3].clone()} for b, (vid, n) in enumerate(zip(ids, counts))]


def collect_dense(model, items_or_dataset, batch_size=None):
    """One forward pass over raw-stream or feats items (a list or a dataset) with the dense outputs kept."""
    store = DenseStore()
    bs = batch_size or model.max_batch
    batch = []

    def flush():
        if batch:
            if "streams" in batch[0] and "feats" not in batch[0]:
                model.forward_streams(batch, dense=store)
            else:
                model(batch, dense=store)
            batch.clear()
    for i in range(len(items_or_dataset)):
        batch.append(items_or_dataset[i])
        if len(batch) == bs:
            flush()
    flush()
    return store


class SweepResult:
    def __init__(self, settings, results, store):
        self.settings, self.results, self.store = settings, results, store

    def records(self, i):
        """Setting i's results as the model's list of dicts (one post-processing launch over the kept outputs)."""
        return rows_to_records(self.store.ids, sweep_rows(self.store, [self.settings[i]])[0])

    def table(self):
        order = sorted(range(len(self.results)), key=lambda i: -self.results[i]["average_mAP"])
        keys = [k for k in SETTING_KEYS if len({json.dumps(s[k]) for s in self.settings}) > 1] or ["nms_method"]
        head = "  ".join("%14s" % k for k in keys) + "  avg-mAP(%)" + ("     AUC(%)" if "auc" in self.results[0] else "")
        lines = [head]
        for i in order:
            r = self.results[i]
            line = "  ".join("%14s" % (r["setting"][k],) for k in keys) + "  %10.2f" % (100 * r["average_mAP"])
            if "auc" in r:
                line += "  %9.2f" % r["auc"]
            lines.append(line)
        return "\n".join(lines)


def sweep_postprocess(model, items_or_dataset, settings, gt, split=None, tiou_thresholds=DEFAULT_TIOU, top_k=(1, 5),
                      proposals=False, max_bytes=1 << 30, max_avg_nr_proposals=100.0, batch_size=None):
    """Score every post-processing setting in `settings` (dicts over SETTING_KEYS; missing keys come from the model's
    test_cfg) on one forward pass over `items_or_dataset` (raw-stream or feats items, a dataset, or a filled DenseStore).
    gt: ground-truth file or DataFrame (metrics.load_gt formats). Settings run in groups whose rows fit `max_bytes`; a
    group is evaluated and freed before the next. Returns a SweepResult."""
    base = {k: getattr(model, "test_" + k) for k in SETTING_KEYS}
    full = [full_setting(base, s, model.num_classes) for s in settings]
    if not full:
        raise AvdfError("the settings grid is empty")
    store = items_or_dataset if isinstance(items_or_dataset, DenseStore) else collect_dense(model, items_or_dataset, batch_size)
    det = ANETdetection(gt, split=split, tiou_thresholds=tiou_thresholds, top_k=top_k)
    layout = RowsLayout(det.ground_truth, store.ids)
    results = []
    N = max(1, len(store))
    i = 0
    while i < len(full):
        j, K = i, 0
        while j < len(full):
            K2 = max(K, int(full[j]["max_seg_num"]))
            if j > i and (j + 1 - i) * N * (3 + 3 * K2) * 4 > max_bytes:
                break
            K, j = K2, j + 1
        rows = sweep_rows(store, full[i:j])
        for s in range(j - i):
            mAP, avg, mRecall = det.evaluate_rows(rows[s], K, layout)
            r = {"setting": full[i + s], "mAP": [float(x) for x in mAP], "average_mAP": float(avg),
                 "mRecall": [[float(x) for x in row] for row in mRecall]}
            if proposals:
                _, avg_recall, ppv = average_recall_from_rows(det.ground_truth, rows[s], K, layout,
                                                              max_avg_nr_proposals=max_avg_nr_proposals, tiou_thresholds=tiou_thresholds)
                r["AR@AN"] = {}
                for an in AR_AT:
                    k = int(round(an * 100.0 / ppv[-1])) - 1
                    if 0 <= k < 100 and abs(ppv[k] - an) <= 1e-9 * an:
                        r["AR@AN"][an] = float(avg_recall[k])
                r["auc"] = area_under_curve(avg_recall, ppv)
            results.append(r)
        del rows
        i = j
    return SweepResult(full, results, store)


def main(argv=None):
    from ..core import load_config
    from ..datasets import make_inference_dataset
    from ..modeling import make_meta_arch
    ap = argparse.ArgumentParser(description="score post-processing settings on one forward pass (all on the GPU)")
    ap.add_argument("config")
    ap.add_argument("ckpt")
    ap.add_argument("--gt", required=True, help="ActivityNet-format JSON or AV-Deepfake1M metadata JSON")
    ap.add_argument("--split", default=None, help="ground-truth subset to score against")
    ap.add_argument("--sub-index", type=int, default=0, help="inference list of the dataset (as inference.py)")
    ap.add_argument("--set", action="append", default=[], metavar="KEY=V1,V2", help="values of one setting (repeatable)")
    ap.add_argument("--tiou", type=float, nargs="+", default=list(DEFAULT_TIOU))
    ap.add_argument("--top-k", type=int, nargs="+", default=[1, 5])
    ap.add_argument("--proposals", action="store_true", help="also AR@AN and AUC")
    ap.add_argument("-b", "--batch", type=int, default=32)
    ap.add_argument("--max-bytes", type=float, default=float(1 << 30), help="device bytes of result rows per group")
    ap.add_argument("--out", default=None, help="write every setting's numbers as JSON")
    args = ap.parse_args(argv)
    settings = grid([parse_set(s) for s in args.set]) if args.set else [{}]
    cfg = load_config(args.config)
    dataset = make_inference_dataset(cfg["dataset_name"], False, cfg["test_split"], args.sub_index, **cfg["dataset"])
    model = make_meta_arch(cfg["model_name"], **cfg["model"], max_batch=args.batch)
    checkpoint = torch.load(args.ckpt, map_location="cpu")
    model.load_state_dict(checkpoint["state_dict_ema"])
    del checkpoint
    model.to(torch.device(cfg["devices"][0])).eval()
    res = sweep_postprocess(model, dataset, settings, args.gt, split=args.split, tiou_thresholds=args.tiou, top_k=args.top_k,
                            proposals=args.proposals, max_bytes=int(args.max_bytes), batch_size=args.batch)
    print(res.table())
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"tiou_thresholds": [float(t) for t in args.tiou], "top_k": args.top_k, "videos": len(res.store),
                       "results": res.results}, f, indent=1)
    return res


if __name__ == "__main__":
    main()
