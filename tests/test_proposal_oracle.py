"""CPU checks of the proposal evaluator: the pandas oracle (oracle/anet_proposal_ref.py) reproduces a hand-derived answer,
the C entry point rejects bad arguments before touching CUDA, the cases where the reference divides by zero raise
ValueError, and evaluate() has no CPU fallback."""
import ctypes
import json

import numpy as np
import pandas as pd
import pytest
import torch

import anet_proposal_ref as ref
from audio_visual_deepfake_detection_b200 import native
from audio_visual_deepfake_detection_b200.libs.utils import ANETproposal, average_recall_vs_avg_nr_proposals

# video c has proposals and no GT; first-hit ranks: a-GT0 rank 0 (tIoU 1.0), a-GT1 rank 1 (0.8), b rank 1 (1.0)
PKA_THR = np.array([0.5, 0.75, 0.9])
PKA_GT = [("a", 0.0, 10.0), ("a", 20.0, 30.0), ("b", 5.0, 6.0)]
PKA_PROP = [("a", 0, 10, .9), ("a", 21, 29, .8), ("a", 1, 11, .7), ("a", 40, 50, .3), ("b", 4, 6.5, .6), ("b", 5, 6, .5),
            ("c", 0, 5, .95), ("c", 1, 2, .1)]
# max_avg_nr_proposals -> ({(threshold index, point j): recall}, AUC % to 4 decimals)
PKA = {None: ({(0, 24): 1 / 3, (0, 49): 2 / 3, (0, 74): 1.0, (2, 99): 2 / 3}, 49.5556),
       2: ({(0, 99): 2 / 3}, 26.5),
       100: ({(0, 0): 1 / 3, (1, 0): 1 / 3, (2, 0): 1 / 3, (0, 24): 1.0, (1, 24): 1.0, (2, 24): 2 / 3}, 87.3889)}


def proposal_known_answer_frames():
    gt = pd.DataFrame({"video-id": [g[0] for g in PKA_GT], "t-start": [g[1] for g in PKA_GT], "t-end": [g[2] for g in PKA_GT],
                       "label": [0] * len(PKA_GT)})
    pr = pd.DataFrame({"video-id": [p[0] for p in PKA_PROP], "t-start": [float(p[1]) for p in PKA_PROP],
                       "t-end": [float(p[2]) for p in PKA_PROP], "score": [p[3] for p in PKA_PROP]})
    return gt, pr


@pytest.mark.parametrize("max_avg", [None, 2, 100])
def test_oracle_known_answer(max_avg):
    gt, pr = proposal_known_answer_frames()
    recall, avg, ppv = ref.average_recall_vs_avg_nr_proposals(gt, pr, max_avg, PKA_THR)
    points, auc = PKA[max_avg]
    for (t, j), want in points.items():
        assert recall[t, j] == want, (t, j, recall[t, j], want)
    assert abs(ref.auc(avg, ppv) - auc) < 1e-4
    assert np.array_equal(avg, recall.mean(axis=0))
    if max_avg is None:
        # ratio 1: keep a = 4, b = 2, total 6, AN_j = 0.04 (j + 1); at j = 74 video b's cut is int(2 * pcn[74]) with the
        # product exactly 2.0 - the point flips if the device recomputes pcn instead of using the host's values
        pcn = np.arange(1, 101) / 100.0 * (4.0 * 2 / 6)
        assert 2 * pcn[74] == 2.0 and np.allclose(ppv, 0.04 * np.arange(1, 101))
        assert recall[0, 73] == 2 / 3 and recall[0, 74] == 1.0
    if max_avg == 2:
        assert recall[:, :].max() == 2 / 3           # b keeps one proposal (tIoU 0.4) and is never matched
    if max_avg == 100:
        assert np.allclose(ppv, np.arange(1, 101))


def _args(**kw):
    a = native.EvalProposalArgs()
    thr = (ctypes.c_double * 2)(0.5, 0.7)
    frac = (ctypes.c_double * 100)(*(np.arange(1, 101) / 100.0))
    dummy = 4096                          # any 256-aligned address: nothing may be dereferenced on the device side
    a.n_video, a.n_prop, a.n_gt = 2, 10, 3
    a.prop_off = a.prop_seg = a.prop_score = a.keep = a.gt_off = a.gt_seg = a.matches = a.status = dummy
    a.thresholds, a.n_thr, a.an_frac = thr, 2, frac
    a.workspace, a.workspace_bytes = dummy, native.lib().avdf_eval_proposal_workspace_bytes(2)
    for k, v in kw.items():
        setattr(a, k, v)
    return a, (thr, frac)


def _frac(values):
    return (ctypes.c_double * 100)(*values)


BAD_FRAC = {"nan": [float("nan")] + [1.0] * 99, "negative": [-0.01] + [1.0] * 99, "decreasing": [0.5] * 50 + [0.4] * 50,
            "huge": [1e13] * 100}


@pytest.mark.parametrize("bad", [dict(n_thr=17), dict(n_thr=0), dict(n_video=-1), dict(n_prop=-1), dict(n_gt=-1),
                                 dict(prop_off=None), dict(gt_off=None), dict(keep=None), dict(prop_seg=None),
                                 dict(gt_seg=None), dict(matches=None), dict(status=None), dict(workspace=None),
                                 dict(workspace_bytes=16), dict(workspace=4096 + 8), dict(prop_seg=4096 + 8),
                                 dict(gt_seg=4096 + 8), dict(thresholds=None), dict(an_frac=None),
                                 *[dict(an_frac=k) for k in BAD_FRAC]])
def test_proposal_entry_rejects_bad_arguments_before_cuda(bad):
    L = native.lib()
    if isinstance(bad.get("an_frac"), str):
        bad = dict(an_frac=_frac(BAD_FRAC[bad["an_frac"]]))
    a, keep = _args(**bad)
    assert L.avdf_eval_proposal(ctypes.byref(a), None) == -1
    assert b"invalid argument" in L.avdf_last_error()
    assert L.avdf_eval_proposal(None, None) == -1
    a, keep = _args(thresholds=(ctypes.c_double * 2)(0.5, float("nan")))
    assert L.avdf_eval_proposal(ctypes.byref(a), None) == -1          # NaN threshold
    assert L.avdf_eval_proposal_workspace_bytes(-1) == 0


def test_division_by_zero_cases_raise_value_error():
    gt, pr = proposal_known_answer_frames()
    with pytest.raises(ValueError, match="ground truth"):
        average_recall_vs_avg_nr_proposals(gt.iloc[:0], pr, tiou_thresholds=PKA_THR)
    with pytest.raises(ValueError, match="no proposals"):
        average_recall_vs_avg_nr_proposals(gt, pr.iloc[:0], tiou_thresholds=PKA_THR)
    with pytest.raises(ValueError, match="keeps no proposal"):     # ratio 0.5 * 2 / 8: int(4 / 8) = int(2 / 8) = 0
        average_recall_vs_avg_nr_proposals(gt, pr, max_avg_nr_proposals=0.5, tiou_thresholds=PKA_THR)
    with pytest.raises(ValueError, match="keeps no proposal"):     # only the video without GT has proposals
        average_recall_vs_avg_nr_proposals(gt, pr[pr["video-id"] == "c"], tiou_thresholds=PKA_THR)
    with pytest.raises(ValueError, match="NaN"):
        bad = pr.copy()
        bad.loc[0, "score"] = float("nan")
        average_recall_vs_avg_nr_proposals(gt, bad, tiou_thresholds=PKA_THR)


def _write_files(tmp_path):
    gt = {"version": "1.3", "taxonomy": [], "database": {
        "a": {"subset": "validation", "annotations": [{"segment": [0.0, 10.0], "label": "Fake"},
                                                      {"segment": [20.0, 30.0], "label": "Fake"}]},
        "b": {"subset": "validation", "annotations": [{"segment": [5.0, 6.0], "label": "Fake"}]},
        "d": {"subset": "training", "annotations": [{"segment": [1.0, 2.0], "label": "Fake"}]}}}
    results = {"version": "1.3", "external_data": {}, "results": {}}
    for v, s, e, sc in PKA_PROP:
        results["results"].setdefault(v, []).append({"segment": [float(s), float(e)], "score": sc})
    g, p = tmp_path / "gt.json", tmp_path / "proposals.json"
    g.write_text(json.dumps(gt)); p.write_text(json.dumps(results))
    return str(g), str(p)


def test_files_load_like_the_frames(tmp_path):
    g, p = _write_files(tmp_path)
    prop = ANETproposal(g, p, tiou_thresholds=PKA_THR)
    gt, _ = proposal_known_answer_frames()
    pd.testing.assert_frame_equal(prop.ground_truth, gt)          # subset "validation", string labels ignored
    assert prop.blocked_videos == [] and prop.proposal["results"]["c"][1]["score"] == 0.1
    with pytest.raises(IOError):
        ANETproposal(g, p, ground_truth_fields=["database", "missing"])
    with pytest.raises(IOError):
        ANETproposal(g, None)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_evaluate_without_gpu_raises(tmp_path):
    g, p = _write_files(tmp_path)
    prop = ANETproposal(g, p, tiou_thresholds=PKA_THR)
    with pytest.raises(native.AvdfError):
        prop.evaluate()
    from audio_visual_deepfake_detection_b200.libs.utils.Evaluation import eval_proposal
    (tmp_path / "data_left_0.json").write_text(json.dumps([{"video_id": "a", "scores": [0.9], "segments": [[0.0, 10.0]]}]))
    with pytest.raises(native.AvdfError):
        eval_proposal.main(["--gt", g, str(tmp_path)])
