"""CPU oracle of the proposal evaluator: a literal pandas restatement of ActivityNet's eval_proposal.py
(segment_iou, wrapper_segment_iou, average_recall_vs_avg_nr_proposals, and the AUC of ANETproposal.evaluate). For tests
only: it keeps the reference's per-video `get_group` loop and its threshold x budget `count_nonzero` loop. It deviates
only where the reference leaves ties unspecified: equal scores inside a video keep their input order
(np.lexsort((arange, -score)) instead of argsort()[::-1]).
"""
import numpy as np


def segment_iou(target_segment, candidate_segments):
    tt1 = np.maximum(target_segment[0], candidate_segments[:, 0])
    tt2 = np.minimum(target_segment[1], candidate_segments[:, 1])
    segments_intersection = (tt2 - tt1).clip(0)
    segments_union = (candidate_segments[:, 1] - candidate_segments[:, 0]) + (target_segment[1] - target_segment[0]) - segments_intersection
    return segments_intersection.astype(float) / segments_union


def wrapper_segment_iou(target_segments, candidate_segments):
    n, m = candidate_segments.shape[0], target_segments.shape[0]
    tiou = np.empty((n, m))
    for i in range(m):
        tiou[:, i] = segment_iou(target_segments[i, :], candidate_segments)
    return tiou


def average_recall_vs_avg_nr_proposals(ground_truth, proposals, max_avg_nr_proposals=None,
                                       tiou_thresholds=np.linspace(0.5, 0.95, 10)):
    """ground_truth: DataFrame (video-id, t-start, t-end); proposals: DataFrame (video-id, t-start, t-end, score).
    -> (recall [n_thr, 100], avg_recall [100], proposals_per_video [100])."""
    video_lst = ground_truth["video-id"].unique()
    if not max_avg_nr_proposals:
        max_avg_nr_proposals = float(proposals.shape[0]) / video_lst.shape[0]
    ratio = max_avg_nr_proposals * float(video_lst.shape[0]) / proposals.shape[0]
    ground_truth_gbvn = ground_truth.groupby("video-id")
    proposals_gbvn = proposals.groupby("video-id")
    score_lst = []
    total_nr_proposals = 0
    for videoid in video_lst:
        ground_truth_videoid = ground_truth_gbvn.get_group(videoid)
        this_video_ground_truth = ground_truth_videoid.loc[:, ["t-start", "t-end"]].values
        try:
            proposals_videoid = proposals_gbvn.get_group(videoid)
        except KeyError:
            score_lst.append(np.zeros((this_video_ground_truth.shape[0], 1)))
            continue
        this_video_proposals = proposals_videoid.loc[:, ["t-start", "t-end"]].values
        if this_video_proposals.shape[0] == 0:
            score_lst.append(np.zeros((this_video_ground_truth.shape[0], 1)))
            continue
        scores = proposals_videoid["score"].values
        sort_idx = np.lexsort((np.arange(len(scores)), -scores))
        this_video_proposals = this_video_proposals[sort_idx, :]
        nr_proposals = np.minimum(int(this_video_proposals.shape[0] * ratio), this_video_proposals.shape[0])
        total_nr_proposals += nr_proposals
        this_video_proposals = this_video_proposals[:nr_proposals, :]
        tiou = wrapper_segment_iou(this_video_proposals, this_video_ground_truth)
        score_lst.append(tiou)

    pcn_lst = np.arange(1, 101) / 100.0 * (max_avg_nr_proposals * float(video_lst.shape[0]) / total_nr_proposals)
    matches = np.empty((video_lst.shape[0], pcn_lst.shape[0]))
    positives = np.empty(video_lst.shape[0])
    recall = np.empty((tiou_thresholds.shape[0], pcn_lst.shape[0]))
    for ridx, tiou in enumerate(tiou_thresholds):
        for i, score in enumerate(score_lst):
            positives[i] = score.shape[0]
            true_positives_tiou = score >= tiou
            pcn_proposals_per_video = np.minimum((score.shape[1] * pcn_lst).astype(int), score.shape[1])
            for j, nr_proposals in enumerate(pcn_proposals_per_video):
                matches[i, j] = np.count_nonzero((true_positives_tiou[:, :nr_proposals]).sum(axis=1))
        recall[ridx, :] = matches.sum(axis=0) / positives.sum()
    avg_recall = recall.mean(axis=0)
    proposals_per_video = pcn_lst * (float(total_nr_proposals) / video_lst.shape[0])
    return recall, avg_recall, proposals_per_video


def auc(avg_recall, proposals_per_video):
    """ANETproposal.evaluate's printed AUC, in percent."""
    area_under_curve = np.trapezoid(avg_recall, proposals_per_video)
    return 100.0 * float(area_under_curve) / proposals_per_video[-1]
