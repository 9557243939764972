"""CPU oracle of the detection evaluator: a literal pandas restatement of ActionFormer's ANETdetection
(libs/utils/metrics.py: segment_iou, compute_average_precision_detection, compute_topkx_recall_detection,
interpolated_prec_rec, evaluate), which UMMAFormer inherits. For tests only: it keeps the reference's row-by-row
`iterrows` matching loop. It deviates only where the reference leaves ties unspecified:
  * predictions: score descending, equal scores by smaller input index (np.lexsort((arange, -score)));
  * GT rows of a video: tIoU descending, equal tIoU by larger GT index (numpy's argsort()[::-1] for <= 16 rows).
"""
import numpy as np
import pandas as pd


def segment_iou(target_segment, candidate_segments):
    tt1 = np.maximum(target_segment[0], candidate_segments[:, 0])
    tt2 = np.minimum(target_segment[1], candidate_segments[:, 1])
    segments_intersection = (tt2 - tt1).clip(0)
    segments_union = (candidate_segments[:, 1] - candidate_segments[:, 0]) + (target_segment[1] - target_segment[0]) - segments_intersection
    return segments_intersection.astype(float) / segments_union


def k_segment_iou(target_segments, candidate_segments):
    return np.stack([segment_iou(t, candidate_segments) for t in target_segments])


def interpolated_prec_rec(prec, rec):
    mprec = np.hstack([[0], prec, [0]])
    mrec = np.hstack([[0], rec, [1]])
    for i in range(len(mprec) - 1)[::-1]:
        mprec[i] = max(mprec[i], mprec[i + 1])
    idx = np.where(mrec[1::] != mrec[0:-1])[0] + 1
    return np.sum((mrec[idx] - mrec[idx - 1]) * mprec[idx])


def score_order(scores):
    scores = np.asarray(scores, dtype=np.float64)
    return np.lexsort((np.arange(len(scores)), -scores))


def compute_average_precision_detection(ground_truth, prediction, tiou_thresholds=np.linspace(0.5, 0.95, 10)):
    """-> (ap [n_thr], tp [n_thr, n_pred] in INPUT order of `prediction`)."""
    ap = np.zeros(len(tiou_thresholds))
    tp_in = np.zeros((len(tiou_thresholds), len(prediction)))
    if prediction.empty:
        return ap, tp_in
    npos = float(len(ground_truth))
    lock_gt = np.ones((len(tiou_thresholds), len(ground_truth))) * -1
    sort_idx = score_order(prediction["score"].values)
    prediction = prediction.loc[sort_idx].reset_index(drop=True)
    tp = np.zeros((len(tiou_thresholds), len(prediction)))
    fp = np.zeros((len(tiou_thresholds), len(prediction)))
    ground_truth_gbvn = ground_truth.groupby("video-id")
    for idx, this_pred in prediction.iterrows():
        try:
            ground_truth_videoid = ground_truth_gbvn.get_group(this_pred["video-id"])
        except Exception:
            fp[:, idx] = 1
            continue
        this_gt = ground_truth_videoid.reset_index()
        tiou_arr = segment_iou(this_pred[["t-start", "t-end"]].values.astype(np.float64),
                               this_gt[["t-start", "t-end"]].values.astype(np.float64))
        # tIoU descending, equal tIoU: larger GT index first
        tiou_sorted_idx = np.lexsort((-np.arange(len(tiou_arr)), -tiou_arr))
        for tidx, tiou_thr in enumerate(tiou_thresholds):
            for jdx in tiou_sorted_idx:
                if tiou_arr[jdx] < tiou_thr:
                    fp[tidx, idx] = 1
                    break
                if lock_gt[tidx, int(this_gt.loc[jdx]["index"])] >= 0:
                    continue
                tp[tidx, idx] = 1
                lock_gt[tidx, int(this_gt.loc[jdx]["index"])] = idx
                break
            if fp[tidx, idx] == 0 and tp[tidx, idx] == 0:
                fp[tidx, idx] = 1
    tp_cumsum = np.cumsum(tp, axis=1).astype(float)
    fp_cumsum = np.cumsum(fp, axis=1).astype(float)
    recall_cumsum = tp_cumsum / npos
    precision_cumsum = tp_cumsum / (tp_cumsum + fp_cumsum)
    for tidx in range(len(tiou_thresholds)):
        ap[tidx] = interpolated_prec_rec(precision_cumsum[tidx, :], recall_cumsum[tidx, :])
    tp_in[:, sort_idx] = tp
    return ap, tp_in


def compute_topkx_recall_detection(ground_truth, prediction, tiou_thresholds=np.linspace(0.5, 0.95, 10), top_k=(1, 5)):
    if prediction.empty:
        return np.zeros((len(tiou_thresholds), len(top_k)))
    n_gts = 0
    n_tps = np.zeros((len(tiou_thresholds), len(top_k)))
    ground_truth_gbvn = ground_truth.groupby("video-id")
    prediction_gbvn = prediction.groupby("video-id")
    for videoid, _ in prediction_gbvn.groups.items():
        try:
            ground_truth_videoid = ground_truth_gbvn.get_group(videoid)
        except Exception:
            continue
        prediction_videoid = prediction_gbvn.get_group(videoid)
        this_gt = ground_truth_videoid.reset_index()
        this_pred = prediction_videoid.reset_index()
        score_sort_idx = score_order(this_pred["score"].values)
        top_kx_idx = score_sort_idx[:max(top_k) * len(this_gt)]
        tiou_arr = k_segment_iou(this_pred[["t-start", "t-end"]].values.astype(np.float64)[top_kx_idx],
                                 this_gt[["t-start", "t-end"]].values.astype(np.float64))
        for tidx, tiou_thr in enumerate(tiou_thresholds):
            for kidx, k in enumerate(top_k):
                tiou = tiou_arr[:k * len(this_gt)]
                n_tps[tidx, kidx] += ((tiou >= tiou_thr).sum(axis=0) > 0).sum()
    n_gts = len(ground_truth)
    return n_tps / n_gts


def evaluate(ground_truth, preds, tiou_thresholds, top_k=(1, 5)):
    """ground_truth / preds: DataFrames (video-id, t-start, t-end, label[, score]) with RAW labels.
    -> (ap [n_thr, n_cls], recall [n_thr, n_topk, n_cls], tp {class index: [n_thr, n_pred of class] input order},
        class rows {class index: row positions of the class in preds})."""
    activity_index = {j: i for i, j in enumerate(sorted(ground_truth["label"].unique()))}
    ground_truth = ground_truth.copy()
    preds = preds.copy().reset_index(drop=True)
    ground_truth["label"] = ground_truth["label"].map(lambda x: activity_index.get(x, x))
    preds["label"] = preds["label"].map(lambda x: activity_index.get(x, x))
    n_cls = len(activity_index)
    ap = np.zeros((len(tiou_thresholds), n_cls))
    recall = np.zeros((len(tiou_thresholds), len(top_k), n_cls))
    tps, rows = {}, {}
    for cidx in range(n_cls):
        gt_c = ground_truth[ground_truth["label"] == cidx].reset_index(drop=True)
        sel = np.nonzero(preds["label"].values == cidx)[0]
        p_c = preds.loc[sel].reset_index(drop=True)
        ap[:, cidx], tps[cidx] = compute_average_precision_detection(gt_c, p_c, tiou_thresholds)
        recall[:, :, cidx] = compute_topkx_recall_detection(gt_c, p_c, tiou_thresholds, top_k)
        rows[cidx] = sel
    return ap, recall, tps, rows
