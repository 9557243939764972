"""Proposal evaluation with the API of ActivityNet's eval_proposal.py (`ANETproposal`,
`average_recall_vs_avg_nr_proposals`): average recall over tIoU thresholds against the average number of proposals per
video (the AR-AN curve) and the area under it. The task is class-agnostic: labels are ignored.

    prop = ANETproposal("gt.json", records, subset="test", max_avg_nr_proposals=100, verbose=True)
    prop.evaluate()     # sets prop.recall [n_thr, 100], prop.avg_recall [100], prop.proposals_per_video [100]

Ground truth: ActivityNet-format JSON, AV-Deepfake1M metadata JSON (metrics.load_gt, the same split rule) or a DataFrame.
Proposals: an ActivityNet `results` JSON (path or loaded dict), a DataFrame (video-id, t-start, t-end, score) or the result
records `inference_one_epoch` writes (data_left*.json). Matching runs on the GPU (csrc/eval.cu, avdf_eval_proposal); the
host builds the CSR of the videos that have GT rows, the proposals walked per video and the 100 curve points, and turns
the device's integer match counts into recall. There is no CPU fallback.

As upstream, the proposal count that sets the budget includes the proposals of videos without GT rows (in AV-Deepfake1M:
the real videos). Upstream leaves equal scores inside a video to numpy's argsort()[::-1]; here they are walked in input
order. Where upstream divides by zero (no GT rows, no proposals, a budget that keeps no proposal) this raises ValueError.
`check_status` is accepted and never downloads anything: the blocked-video list is empty.

Command line, over folders of result records:
    python -m audio_visual_deepfake_detection_b200.libs.utils.Evaluation.eval_proposal --gt FILE [--split S] \\
        [--max-avg-nr-proposals 100] [--tiou T ...] FOLDER...
"""
import argparse
import json
import os

import numpy as np
import torch

from .... import ops
from ..metrics import _device, _np, load_gt, prediction_columns, video_codes, video_csr

GROUND_TRUTH_FIELDS = ["database", "taxonomy", "version"]
PROPOSAL_FIELDS = ["results", "version", "external_data"]
DEFAULT_TIOU = np.linspace(0.5, 0.95, 10)
AR_AT = (1, 5, 10, 20, 50, 100)


def _proposal_columns(proposals):
    """-> (video ids [M], rows per id [M], t-start, t-end, score [N]) of any accepted proposal input."""
    if isinstance(proposals, dict) and "results" in proposals:
        vids, t0, t1, score = [], [], [], []
        for vid, items in proposals["results"].items():
            for it in items:
                vids.append(vid)
                t0.append(float(it["segment"][0]))
                t1.append(float(it["segment"][1]))
                score.append(float(it["score"]))
        proposals = {"video-id": vids, "t-start": t0, "t-end": t1, "score": score}
    if not isinstance(proposals, list):
        get = (lambda k: proposals[k].values) if hasattr(proposals, "columns") else (lambda k: proposals[k])
        cols = {k: get(k) for k in ("video-id", "t-start", "t-end", "score")}
        cols["label"] = np.zeros(_np(cols["score"], np.float64).size, dtype=np.int64)
        proposals = cols
    vids, rows, t0, t1, _, score = prediction_columns(proposals)
    return vids, rows, t0, t1, score


def area_under_curve(avg_recall, proposals_per_video):
    """ANETproposal.evaluate's AUC in percent: 100 * trapz(avg_recall, proposals_per_video) / proposals_per_video[-1]."""
    trapz = getattr(np, "trapezoid", None) or np.trapz
    return 100.0 * float(trapz(avg_recall, proposals_per_video)) / proposals_per_video[-1]


def average_recall_vs_avg_nr_proposals(ground_truth, proposals, max_avg_nr_proposals=None,
                                       tiou_thresholds=DEFAULT_TIOU):
    """ground_truth: DataFrame (video-id, t-start, t-end); proposals: see the module docstring.
    -> (recall [n_thr, 100], avg_recall [100], proposals_per_video [100])."""
    thr = np.asarray(tiou_thresholds, dtype=np.float64).reshape(-1)
    vids, rows, t0, t1, score = _proposal_columns(proposals)
    if np.isnan(t0).any() or np.isnan(t1).any() or np.isnan(score).any():
        raise ValueError("proposals contain NaN")
    p_code, g_code, n_codes = video_codes(vids, rows, ground_truth)
    p_rows, _, prop_off, g_rows, gt_off = video_csr(p_code, g_code, n_codes, gt_videos_only=True)
    n_video, n_prop = gt_off.size - 1, score.size
    if n_video == 0:
        raise ValueError("the ground truth has no rows: average recall is undefined")
    if n_prop == 0:
        raise ValueError("there are no proposals: the average number of proposals is undefined")
    if not max_avg_nr_proposals:
        max_avg_nr_proposals = float(n_prop) / n_video
    if max_avg_nr_proposals < 0:
        raise ValueError("max_avg_nr_proposals must not be negative")
    ratio = max_avg_nr_proposals * float(n_video) / n_prop
    n_p = np.diff(prop_off)
    keep = np.minimum((n_p * ratio).astype(np.int64), n_p)
    total = int(keep.sum())
    if total == 0:
        raise ValueError("max_avg_nr_proposals keeps no proposal of any video with ground truth")
    pcn = np.arange(1, 101) / 100.0 * (max_avg_nr_proposals * float(n_video) / total)

    dev = _device()
    g_se = np.stack([ground_truth["t-start"].values, ground_truth["t-end"].values], 1).astype(np.float64)[g_rows]
    seg = np.stack([t0[p_rows], t1[p_rows]], 1)
    matches, _ = ops.eval_proposal(torch.from_numpy(prop_off).to(dev), torch.from_numpy(seg).to(dev),
                                   torch.from_numpy(score[p_rows]).to(dev), torch.from_numpy(keep.astype(np.int32)).to(dev),
                                   torch.from_numpy(gt_off).to(dev), torch.from_numpy(np.ascontiguousarray(g_se)).to(dev),
                                   thr, pcn)
    recall = matches.cpu().numpy().astype(np.float64) / float(g_code.size)
    avg_recall = recall.mean(axis=0)
    proposals_per_video = pcn * (float(total) / n_video)
    return recall, avg_recall, proposals_per_video


class ANETproposal(object):
    """The ActivityNet proposal evaluator. ground_truth_filename: a GT file or DataFrame; proposal_filename: an
    ActivityNet results JSON, a DataFrame or result records. The *_fields are checked on ActivityNet-format JSON files."""

    def __init__(self, ground_truth_filename=None, proposal_filename=None, ground_truth_fields=GROUND_TRUTH_FIELDS,
                 proposal_fields=PROPOSAL_FIELDS, tiou_thresholds=DEFAULT_TIOU, max_avg_nr_proposals=None,
                 subset="validation", verbose=False, check_status=True):
        if ground_truth_filename is None:
            raise IOError("Please input a valid ground truth file.")
        if proposal_filename is None:
            raise IOError("Please input a valid proposal file.")
        self.subset = subset
        self.tiou_thresholds = np.asarray(tiou_thresholds, dtype=np.float64).reshape(-1)
        self.max_avg_nr_proposals = max_avg_nr_proposals
        self.verbose = verbose
        self.gt_fields = ground_truth_fields
        self.pred_fields = proposal_fields
        self.recall = None
        self.avg_recall = None
        self.proposals_per_video = None
        self.check_status = check_status
        self.blocked_videos = []
        self.ground_truth = self._import_ground_truth(ground_truth_filename)
        self.proposal = self._import_proposal(proposal_filename)
        if self.verbose:
            print("[INIT] Loaded annotations from {} subset.".format(subset))
            print("\tNumber of ground truth instances: {}".format(len(self.ground_truth)))
            print("\tNumber of proposals: {}".format(_proposal_columns(self.proposal)[4].size))
            print("\tFixed threshold for tiou score: {}".format(self.tiou_thresholds))

    def _import_ground_truth(self, ground_truth_filename):
        if hasattr(ground_truth_filename, "columns"):
            gt = ground_truth_filename.copy()
        else:
            with open(ground_truth_filename, "r", encoding="utf8") as f:
                data = json.load(f)
            if isinstance(data, dict) and not all(field in data for field in self.gt_fields):
                raise IOError("Please input a valid ground truth file.")
            gt = load_gt(ground_truth_filename, split=self.subset, label=None)
        for c in ("t-start", "t-end"):
            if np.isnan(gt[c].values.astype(np.float64)).any():
                raise ValueError("ground truth has NaN segment bounds")
        return gt

    def _import_proposal(self, proposal_filename):
        if isinstance(proposal_filename, (str, os.PathLike)):
            with open(proposal_filename, "r", encoding="utf8") as f:
                proposal_filename = json.load(f)
            if not isinstance(proposal_filename, list) and not all(field in proposal_filename for field in self.pred_fields):
                raise IOError("Please input a valid proposal file.")
        return proposal_filename

    def evaluate(self):
        """Sets self.recall [n_thr, 100], self.avg_recall [100] and self.proposals_per_video [100]; prints the AUC when
        verbose."""
        recall, avg_recall, proposals_per_video = average_recall_vs_avg_nr_proposals(
            self.ground_truth, self.proposal, max_avg_nr_proposals=self.max_avg_nr_proposals,
            tiou_thresholds=self.tiou_thresholds)
        if self.verbose:
            print("[RESULTS] Performance on ActivityNet proposal task.")
            print("\tArea Under the AR vs AN curve: {}%".format(area_under_curve(avg_recall, proposals_per_video)))
        self.recall = recall
        self.avg_recall = avg_recall
        self.proposals_per_video = proposals_per_video


def main(argv=None):
    from ..results import iter_result_records
    ap = argparse.ArgumentParser(description="AR@AN and AUC of result records (data_left*.json) against a ground truth")
    ap.add_argument("--gt", required=True, help="ActivityNet-format JSON or AV-Deepfake1M metadata JSON")
    ap.add_argument("--split", default=None)
    ap.add_argument("--max-avg-nr-proposals", type=float, default=100.0,
                    help="proposal budget per video (0: all proposals, upstream's default)")
    ap.add_argument("--tiou", type=float, nargs="+", default=list(DEFAULT_TIOU))
    ap.add_argument("folders", nargs="+")
    args = ap.parse_args(argv)
    records = list(iter_result_records(args.folders, pattern="data_left*.json"))
    prop = ANETproposal(args.gt, records, ground_truth_fields=["database"], tiou_thresholds=args.tiou,
                        max_avg_nr_proposals=args.max_avg_nr_proposals, subset=args.split, verbose=True)
    prop.evaluate()
    auc = area_under_curve(prop.avg_recall, prop.proposals_per_video)
    ar = {}
    for an in AR_AT:                 # the curve points at these budgets (every one of them when the budget is 100)
        j = int(round(an * 100.0 / prop.proposals_per_video[-1])) - 1
        if 0 <= j < 100 and abs(prop.proposals_per_video[j] - an) <= 1e-9 * an:
            ar["AR@%d" % an] = float(prop.avg_recall[j])
            print("AR@{:d} = {:>4.2f} (%)".format(an, 100 * prop.avg_recall[j]))
    print("AUC = {:>4.2f} (%)".format(auc))
    print(json.dumps({"ground_truth": os.path.basename(args.gt), "split": args.split,
                      "tiou_thresholds": [float(t) for t in prop.tiou_thresholds],
                      "max_avg_nr_proposals": args.max_avg_nr_proposals, **ar, "auc": auc,
                      "avg_recall": [float(x) for x in prop.avg_recall],
                      "proposals_per_video": [float(x) for x in prop.proposals_per_video], "videos": len(records),
                      "proposals": int(sum(len(r["scores"]) for r in records))}))
    return prop.recall, prop.avg_recall, prop.proposals_per_video, auc


if __name__ == "__main__":
    main()
