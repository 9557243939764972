"""Detection evaluation with the reference's API (ActionFormer / UMMAFormer libs/utils/metrics.py `ANETdetection`): mAP per
tIoU threshold and Recall@kx, computed by the sm_100a kernels of csrc/eval.cu (avdf_eval_detection).

    det = ANETdetection("gt.json", split="test", tiou_thresholds=np.linspace(0.5, 0.95, 10))
    mAP, average_mAP, mRecall = det.evaluate(preds)

`preds` is the reference's dict (`video-id`, `t-start`, `t-end`, `label`, `score`), a DataFrame with those columns, or the
result records `inference_one_epoch` writes (`data_left*.json`: one {video_id, scores, segments} item per video, label 0).
The host builds, per class, the CSR of the videos that have GT or predictions of that class (one device call per class,
like libs/utils/nms.py's multiclass path); matching, sorting and the AP scan run on the GPU. There is no CPU fallback.

Ties the reference leaves to numpy's sort are fixed here: equal scores rank by smaller input index, and a prediction tries
equal-tIoU GT rows of its video from the larger GT index down (what argsort()[::-1] gives for <= 16 rows).

Command line, over folders of result records (the same de-duplication as results.merge_results):
    python -m audio_visual_deepfake_detection_b200.libs.utils.metrics --gt FILE [--split S] FOLDER...
"""
import argparse
import json
import os

import numpy as np
import torch

from ... import ops
from ...native import AvdfError

DEFAULT_TIOU = np.linspace(0.5, 0.95, 10)       # db_attributes["tiou_thresholds"] of the deepfake datasets


def _device():
    if not torch.cuda.is_available():
        raise AvdfError("libs.utils.metrics runs on sm_100a kernels only; no CUDA device is visible (no CPU fallback)")
    return torch.device("cuda", torch.cuda.current_device())


def _frame(vids, starts, stops, labels):
    import pandas as pd
    return pd.DataFrame({"video-id": vids, "t-start": np.asarray(starts, dtype=np.float64),
                         "t-end": np.asarray(stops, dtype=np.float64), "label": np.asarray(labels, dtype=np.int64)})


def load_gt_seg_from_json(json_file, split=None, label="label", label_offset=0):
    """ActivityNet-format ground truth (`database -> video id -> {subset, annotations: [{segment, <label>}]}`) ->
    DataFrame (video-id, t-start, t-end, label). `split` keeps the videos whose `subset` equals it (case-insensitive).
    label=None reads no label (every row gets 0): the class-agnostic proposal task, whose labels may be names."""
    with open(json_file, "r", encoding="utf8") as f:
        json_db = json.load(f)["database"]
    vids, starts, stops, labels = [], [], [], []
    for k, v in json_db.items():
        if (split is not None) and v["subset"].lower() != split.lower():
            continue
        for event in v["annotations"]:
            vids.append(k)
            starts.append(float(event["segment"][0]))
            stops.append(float(event["segment"][1]))
            if label is None:
                label_id = 0
            elif isinstance(event[label], (tuple, list)):
                label_id = 0              # the reference's folding of a label tuple with label_offset
                for i, x in enumerate(event[label][::-1]):
                    label_id += label_offset ** i + int(x)
            else:
                label_id = int(event[label])
            labels.append(label_id)
    return _frame(vids, starts, stops, labels)


def load_gt_seg_from_metadata(metadata, split=None):
    """AV-Deepfake1M / LAV-DF metadata (`[{"file", "fake_segments", ...}]`, a path or the loaded list) -> the same table:
    one row per fake segment, label 0, video id = `file`; real videos contribute no rows. `split` keeps the entries whose
    `split` field equals it (entries without the field are kept)."""
    if isinstance(metadata, (str, os.PathLike)):
        with open(metadata, "r", encoding="utf8") as f:
            metadata = json.load(f)
    vids, starts, stops = [], [], []
    for item in metadata:
        if split is not None and "split" in item and str(item["split"]).lower() != split.lower():
            continue
        for seg in item.get("fake_segments") or []:
            vids.append(item["file"])
            starts.append(float(seg[0]))
            stops.append(float(seg[1]))
    return _frame(vids, starts, stops, [0] * len(vids))


def load_gt(ant_file, split=None, label="label", label_offset=0):
    """Either ground-truth format, told apart by the JSON's top level (object with `database` / list)."""
    with open(ant_file, "r", encoding="utf8") as f:
        db = json.load(f)
    if isinstance(db, list):
        return load_gt_seg_from_metadata(db, split=split)
    return load_gt_seg_from_json(ant_file, split=split, label=label, label_offset=label_offset)


def _np(x, dtype):
    if isinstance(x, torch.Tensor):
        x = x.detach().cpu().numpy()
    elif isinstance(x, (list, tuple)) and len(x) and isinstance(x[0], (np.ndarray, torch.Tensor)):
        x = np.concatenate([_np(v, dtype) for v in x])
    return np.asarray(x, dtype=dtype).reshape(-1)


def prediction_columns(preds):
    """preds (dict / DataFrame / result records) -> (video ids [M] object, rows per id [M] int64, t-start, t-end, label,
    score [N]); the rows of id i are rows sum(rows[:i]) .. + rows[i] when they come grouped (result records), else every
    row is its own entry (rows all 1)."""
    if isinstance(preds, list):                                   # result records
        vids = np.array([it["video_id"] for it in preds], dtype=object)
        rows = np.array([len(it["scores"]) for it in preds], dtype=np.int64)
        score = np.fromiter((s for it in preds for s in it["scores"]), dtype=np.float64, count=int(rows.sum()))
        se = np.fromiter((t for it in preds for seg in it["segments"] for t in seg[:2]), dtype=np.float64, count=2 * int(rows.sum()))
        return vids, rows, se[0::2].copy(), se[1::2].copy(), np.zeros(score.size, dtype=np.int64), score
    cols = preds
    if hasattr(preds, "columns"):                                 # DataFrame
        cols = {k: preds[k].values for k in ("video-id", "t-start", "t-end", "label", "score")}
    vids = np.asarray(list(cols["video-id"]), dtype=object)
    score = _np(cols["score"], np.float64)
    return (vids, np.ones(vids.size, dtype=np.int64), _np(cols["t-start"], np.float64), _np(cols["t-end"], np.float64),
            _np(cols["label"], np.int64), score)


def video_codes(vids, rows, gt):
    """One code per video id: prediction ids first (in order of appearance, so grouped records stay in order), then the
    ids only GT rows have. -> (code per prediction row, code per GT row, number of codes)."""
    import pandas as pd
    codes, _ = pd.factorize(np.concatenate([vids, gt["video-id"].values.astype(object)]))
    n_codes = int(codes.max()) + 1 if codes.size else 0
    return np.repeat(codes[:vids.size], rows), codes[vids.size:], n_codes


def video_csr(p_code, g_code, n_codes, gt_videos_only=False):
    """Prediction rows and GT rows (video codes p_code, g_code) -> the CSR of the videos that have GT rows or predictions
    (gt_videos_only: GT rows), in code order: (p_rows, order, pred_off int64 [V+1], g_rows, gt_off int32 [V+1]).
    p_rows / g_rows index the inputs in CSR order; predictions of the other videos are left out. The kept rows keep their
    order inside each video; order is their regrouping permutation (None when they already come grouped)."""
    present = np.zeros(n_codes, dtype=bool)
    present[g_code] = True
    p_rows = np.arange(p_code.size)
    if gt_videos_only:
        p_rows = p_rows[present[p_code]]
    else:
        present[p_code] = True
    local = np.cumsum(present) - 1
    n_video = int(present.sum())
    p_loc = local[p_code[p_rows]]
    order = None if (p_loc.size < 2 or (np.diff(p_loc) >= 0).all()) else np.argsort(p_loc, kind="stable")
    if order is not None:
        p_rows, p_loc = p_rows[order], p_loc[order]
    g_loc = local[g_code]
    g_rows = np.argsort(g_loc, kind="stable")
    pred_off = np.zeros(n_video + 1, dtype=np.int64)
    pred_off[1:] = np.cumsum(np.bincount(p_loc, minlength=n_video))
    gt_off = np.zeros(n_video + 1, dtype=np.int32)
    gt_off[1:] = np.cumsum(np.bincount(g_loc, minlength=n_video))
    return p_rows, order, pred_off, g_rows, gt_off


class ANETdetection(object):
    """The reference's evaluator. ant_file: ActivityNet-format JSON or AV-Deepfake1M metadata JSON (or a ground-truth
    DataFrame from one of the loaders). num_workers is accepted for compatibility and unused."""

    def __init__(self, ant_file, split=None, tiou_thresholds=np.linspace(0.1, 0.5, 5), top_k=(1, 5), label="label",
                 label_offset=0, num_workers=8, dataset_name=None):
        self.tiou_thresholds = np.asarray(tiou_thresholds, dtype=np.float64).reshape(-1)
        self.top_k = tuple(int(k) for k in top_k)
        self.ap = None
        self.recall = None
        self.num_workers = num_workers
        self.split = split
        if hasattr(ant_file, "columns"):
            self.dataset_name = dataset_name or "ground_truth"
            gt = ant_file.copy()
        else:
            self.dataset_name = dataset_name if dataset_name is not None else os.path.basename(ant_file).replace(".json", "")
            gt = load_gt(ant_file, split=split, label=label, label_offset=label_offset)
        for c in ("t-start", "t-end"):
            if np.isnan(gt[c].values.astype(np.float64)).any():
                raise ValueError("ground truth has NaN segment bounds")
        self.activity_index = {j: i for i, j in enumerate(sorted(gt["label"].unique()))}
        gt["label"] = gt["label"].map(lambda x: self.activity_index.get(x, x))
        self.ground_truth = gt

    def evaluate(self, preds, verbose=True):
        """-> (mAP [n_thr], average_mAP, mRecall [n_thr, n_topk]); per-class values stay in self.ap [n_thr, n_cls] and
        self.recall [n_thr, n_topk, n_cls]."""
        self.ap, self.recall, _ = self.evaluate_classes(preds)
        mAP = self.ap.mean(axis=1)
        mRecall = self.recall.mean(axis=2)
        average_mAP = mAP.mean()
        if verbose:
            print(self.table(mAP, average_mAP, mRecall))
        return mAP, average_mAP, mRecall

    def table(self, mAP, average_mAP, mRecall):
        block = "[RESULTS] Action detection results on {:s}.".format(self.dataset_name)
        for tiou, tiou_mAP, tiou_mRecall in zip(self.tiou_thresholds, mAP, mRecall):
            block += "\n|tIoU = {:.2f}: ".format(tiou)
            block += "mAP = {:>4.2f} (%) ".format(tiou_mAP * 100)
            for idx, k in enumerate(self.top_k):
                block += "Recall@{:d}x = {:>4.2f} (%) ".format(k, tiou_mRecall[idx] * 100)
        return block + "\nAverage-mAP: {:>4.2f} (%)".format(average_mAP * 100)

    def evaluate_classes(self, preds, want_tp=False):
        """-> (ap [n_thr, n_cls], recall [n_thr, n_topk, n_cls], tp_mask): tp_mask (want_tp) is a uint16 array over the
        prediction rows in input order, bit t = TP at threshold t within the row's class."""
        dev = _device()
        vids, rows, t0, t1, label, score = prediction_columns(preds)
        if np.isnan(t0).any() or np.isnan(t1).any() or np.isnan(score).any():
            raise ValueError("predictions contain NaN")
        if label.size:                  # a label that is no GT label value is kept as it is (the reference's replace())
            u, inv = np.unique(label, return_inverse=True)
            label = np.array([self.activity_index.get(int(x), int(x)) for x in u], dtype=np.int64)[inv.reshape(-1)]
        gt = self.ground_truth
        p_code, g_code, n_codes = video_codes(vids, rows, gt)
        g_lab = gt["label"].values.astype(np.int64)
        g_se = np.stack([gt["t-start"].values, gt["t-end"].values], 1).astype(np.float64)
        n_thr, n_k, n_cls = len(self.tiou_thresholds), len(self.top_k), len(self.activity_index)
        ap = np.zeros((n_thr, n_cls))
        recall = np.zeros((n_thr, n_k, n_cls))
        tp_all = np.zeros(score.size, dtype=np.uint16) if want_tp else None
        ws = None
        for c in range(n_cls):
            gsel = np.nonzero(g_lab == c)[0]
            psel = np.nonzero(label == c)[0]
            p_rows, order, pred_off, g_rows, gt_off = video_csr(p_code[psel], g_code[gsel], n_codes)
            psel = psel[p_rows]
            # rows not grouped by video: the CSR regroups them, equal scores keep the input order
            rank = None if order is None else torch.from_numpy(order.astype(np.int32)).to(dev)
            seg = np.stack([t0[psel], t1[psel]], 1)
            tp = torch.empty(psel.size, dtype=torch.uint16, device=dev) if want_tp else None
            if ws is None:
                ws = torch.empty(ops.nv.lib().avdf_eval_workspace_bytes(score.size, n_codes), dtype=torch.uint8, device=dev)
            a, h, _ = ops.eval_detection(torch.from_numpy(pred_off).to(dev), torch.from_numpy(seg).to(dev),
                                         torch.from_numpy(score[psel]).to(dev), torch.from_numpy(gt_off).to(dev),
                                         torch.from_numpy(np.ascontiguousarray(g_se[gsel[g_rows]])).to(dev),
                                         self.tiou_thresholds, self.top_k, tp_mask=tp, pred_rank=rank, workspace=ws)
            ap[:, c] = a.cpu().numpy()
            recall[:, :, c] = h.cpu().numpy() / float(gsel.size)
            if want_tp:
                tp_all[psel] = tp.view(torch.int16).cpu().numpy().view(np.uint16)
        return ap, recall, tp_all


def main(argv=None):
    from .results import iter_result_records
    ap = argparse.ArgumentParser(description="mAP / Recall@kx of result records (data_left*.json) against a ground truth")
    ap.add_argument("--gt", required=True, help="ActivityNet-format JSON or AV-Deepfake1M metadata JSON")
    ap.add_argument("--split", default=None)
    ap.add_argument("--tiou", type=float, nargs="+", default=list(DEFAULT_TIOU))
    ap.add_argument("--top-k", type=int, nargs="+", default=[1, 5])
    ap.add_argument("--label", default="label")
    ap.add_argument("folders", nargs="+")
    args = ap.parse_args(argv)
    records = list(iter_result_records(args.folders, pattern="data_left*.json"))
    det = ANETdetection(args.gt, split=args.split, tiou_thresholds=args.tiou, top_k=args.top_k, label=args.label)
    mAP, average_mAP, mRecall = det.evaluate(records, verbose=True)
    print(json.dumps({"dataset": det.dataset_name, "tiou_thresholds": [float(t) for t in det.tiou_thresholds],
                      "top_k": list(det.top_k), "mAP": [float(x) for x in mAP], "average_mAP": float(average_mAP),
                      "mRecall": [[float(x) for x in r] for r in mRecall], "videos": len(records),
                      "predictions": int(sum(len(r["scores"]) for r in records))}))
    return mAP, average_mAP, mRecall


if __name__ == "__main__":
    main()
