"""CPU checks of the detection evaluator: the pandas oracle (oracle/anet_ref.py) reproduces a hand-derived answer, the two
ground-truth loaders agree, the C entry point rejects bad arguments before touching CUDA, and evaluate() has no CPU
fallback."""
import ctypes
import json

import numpy as np
import pandas as pd
import pytest
import torch

import anet_ref
from audio_visual_deepfake_detection_b200 import native
from audio_visual_deepfake_detection_b200.libs.utils import metrics

# one class; thresholds 0.5 / 0.75 / 0.9
KA_THR = np.array([0.5, 0.75, 0.9])
KA_GT = [("a", 0.0, 10.0), ("a", 20.0, 30.0), ("b", 5.0, 6.0)]
KA_PRED = [("a", 0, 10, .9), ("a", 1, 11, .8), ("a", 20, 28, .7), ("a", 40, 50, .3), ("b", 5, 6, .85), ("b", 4, 6.5, .6),
           ("c", 0, 5, .95)]
KA_AP = [29 / 45, 29 / 45, 4 / 9]
KA_R1 = [2 / 3, 2 / 3, 2 / 3]
KA_R5 = [1.0, 1.0, 2 / 3]
KA_TP05_INPUT = [1, 0, 1, 0, 1, 0, 0]     # TP at 0.5 of the rows above (score order: c F, a T, b T, a F, a T, b F, a F)


def known_answer_frames():
    gt = pd.DataFrame({"video-id": [g[0] for g in KA_GT], "t-start": [g[1] for g in KA_GT], "t-end": [g[2] for g in KA_GT],
                       "label": [0] * len(KA_GT)})
    pr = pd.DataFrame({"video-id": [p[0] for p in KA_PRED], "t-start": [float(p[1]) for p in KA_PRED],
                       "t-end": [float(p[2]) for p in KA_PRED], "label": [0] * len(KA_PRED), "score": [p[3] for p in KA_PRED]})
    return gt, pr


def test_oracle_known_answer():
    gt, pr = known_answer_frames()
    ap, recall, tps, rows = anet_ref.evaluate(gt, pr, KA_THR, (1, 5))
    assert np.allclose(ap[:, 0], KA_AP, rtol=0, atol=1e-15)
    assert np.allclose(recall[:, 0, 0], KA_R1, rtol=0, atol=1e-15) and np.allclose(recall[:, 1, 0], KA_R5, rtol=0, atol=1e-15)
    assert tps[0][0].astype(int).tolist() == KA_TP05_INPUT
    # the closed form the kernels use: AP = (1 / npos) sum over TP rows of max_{j >= i} prec_j
    order = anet_ref.score_order(pr["score"].values)
    for t in range(len(KA_THR)):
        tp = tps[0][t][order]
        prec = np.cumsum(tp) / np.arange(1, len(tp) + 1)
        env = np.maximum.accumulate(prec[::-1])[::-1]
        assert abs((env * tp).sum() / len(gt) - KA_AP[t]) < 1e-15


def _write_gt_files(tmp_path):
    anet = {"database": {
        "v1": {"subset": "test", "annotations": [{"segment": [1.0, 2.5], "label": 0}, {"segment": [4.0, 9.0], "label": 0}]},
        "v2": {"subset": "test", "annotations": []},
        "v3": {"subset": "Test", "annotations": [{"segment": [0.5, 0.75], "label": 0}]},
        "v4": {"subset": "train", "annotations": [{"segment": [3.0, 4.0], "label": 0}]}}}
    meta = [{"file": "v1", "split": "test", "fake_segments": [[1.0, 2.5], [4.0, 9.0]]},
            {"file": "v2", "split": "test", "fake_segments": []},
            {"file": "v3", "split": "test", "fake_segments": [[0.5, 0.75]]},
            {"file": "v4", "split": "train", "fake_segments": [[3.0, 4.0]]}]
    a, m = tmp_path / "anet.json", tmp_path / "meta.json"
    a.write_text(json.dumps(anet)); m.write_text(json.dumps(meta))
    return str(a), str(m)


def test_gt_loaders_agree_and_split_filters(tmp_path):
    a, m = _write_gt_files(tmp_path)
    for split, n in ((None, 4), ("test", 3), ("train", 1)):
        ta = metrics.load_gt_seg_from_json(a, split=split)
        tm = metrics.load_gt_seg_from_metadata(m, split=split)
        assert len(ta) == n
        pd.testing.assert_frame_equal(ta, tm)
        tg = metrics.load_gt(m, split=split)          # format told apart by the JSON's top level
        pd.testing.assert_frame_equal(tg, tm)
    t = metrics.load_gt_seg_from_json(a, split="test")
    assert t["video-id"].tolist() == ["v1", "v1", "v3"] and t["t-end"].tolist() == [2.5, 9.0, 0.75]
    assert (t["label"] == 0).all()


def _args(**kw):
    a = native.EvalArgs()
    thr = (ctypes.c_double * 2)(0.5, 0.7)
    ks = (ctypes.c_int32 * 2)(1, 5)
    dummy = 4096                          # any 256-aligned address: nothing may be dereferenced on the device side
    a.n_pred, a.n_video, a.n_gt = 10, 2, 3
    a.pred_off = a.pred_seg = a.pred_score = a.gt_off = a.gt_seg = a.ap = a.recall_hits = a.status = dummy
    a.thresholds, a.n_thr, a.top_k, a.n_topk = thr, 2, ks, 2
    a.workspace, a.workspace_bytes = dummy, native.lib().avdf_eval_workspace_bytes(10, 2)
    for k, v in kw.items():
        setattr(a, k, v)
    return a, (thr, ks)


@pytest.mark.parametrize("bad", [dict(n_thr=17), dict(n_thr=0), dict(n_topk=5), dict(n_gt=0), dict(n_pred=-1),
                                 dict(pred_off=None), dict(status=None), dict(ap=None), dict(workspace_bytes=16),
                                 dict(workspace=4096 + 8), dict(pred_seg=4096 + 8), dict(tp_mask=4096 + 2)])
def test_eval_entry_rejects_bad_arguments_before_cuda(bad):
    L = native.lib()
    a, keep = _args(**bad)
    assert L.avdf_eval_detection(ctypes.byref(a), None) == -1
    assert b"invalid argument" in L.avdf_last_error()
    assert L.avdf_eval_detection(None, None) == -1
    t = (ctypes.c_int32 * 1)(0)
    a, keep = _args()
    a.top_k = t
    assert L.avdf_eval_detection(ctypes.byref(a), None) == -1        # top_k value 0
    thr = (ctypes.c_double * 2)(0.5, float("nan"))
    a, keep = _args()
    a.thresholds = thr
    assert L.avdf_eval_detection(ctypes.byref(a), None) == -1        # NaN threshold
    assert L.avdf_eval_workspace_bytes(-1, 2) == 0


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_evaluate_without_gpu_raises(tmp_path):
    a, _ = _write_gt_files(tmp_path)
    det = metrics.ANETdetection(a, split="test", tiou_thresholds=KA_THR)
    with pytest.raises(native.AvdfError):
        det.evaluate({"video-id": ["v1"], "t-start": [1.0], "t-end": [2.0], "label": [0], "score": [0.5]})
    with pytest.raises(native.AvdfError):
        metrics.main(["--gt", a, str(tmp_path)])
