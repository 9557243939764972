"""Post-processing sweeps on the GPU (libs/utils/sweep.py, avdf_postprocess_sweep):

  * end to end: every setting of a 14-setting grid returns, bit for bit, what forward_streams returns from a model built
    with that test_cfg and the same weights (counts, scores, segments, video_cls) - two archs, mixed and fp32, dense and
    sparse synthetic weights, batch 32 plus a short last batch;
  * kernel level: the sweep's rows equal avdf_postprocess run once per setting on the same dense buffers (the pyramid
    mask built from the valid lengths), for settings that differ only in decode parameters or only in NMS parameters,
    raw-stream videos and feats items longer than max_seq_len; a permuted settings table gives every setting its row;
  * evaluation: each setting's mAP / Recall@kx equal ANETdetection.evaluate on that setting's records (AP <= 1e-12,
    recall bit-equal) and AR@AN equals ANETproposal."""
import numpy as np
import pandas as pd
import pytest
import torch

import parity_common
from make_golden import MODEL_CASES
from audio_visual_deepfake_detection_b200 import ops
from audio_visual_deepfake_detection_b200.libs.core import load_config_for
from audio_visual_deepfake_detection_b200.libs.modeling import make_meta_arch
from audio_visual_deepfake_detection_b200.libs.modeling.engine import DenseStore
from audio_visual_deepfake_detection_b200.libs.utils import synthetic as syn
from audio_visual_deepfake_detection_b200.libs.utils import sweep
from audio_visual_deepfake_detection_b200.libs.utils.Evaluation.eval_proposal import ANETproposal
from audio_visual_deepfake_detection_b200.libs.utils.metrics import ANETdetection

pytestmark = pytest.mark.gpu
N_VIDEOS = 37          # one batch of 32 and a short last batch of 5

# hard and soft, voting 0 / 0.9, iou 0.1 / 0.5, min_score 0.001 / 0.2, sigma 0.5 / 0.75, max_seg_num 1 / 100,
# two values each of pre_nms_thresh / pre_nms_topk / duration_thresh
SETTINGS = [
    {"nms_method": "soft", "iou_threshold": 0.1, "min_score": 0.2, "nms_sigma": 0.75, "voting_thresh": 0.9},
    {"nms_method": "hard", "iou_threshold": 0.1, "min_score": 0.2, "voting_thresh": 0.9},
    {"nms_method": "soft", "iou_threshold": 0.5, "min_score": 0.001, "nms_sigma": 0.5, "voting_thresh": 0.0},
    {"nms_method": "hard", "iou_threshold": 0.5, "min_score": 0.001, "voting_thresh": 0.0},
    {"nms_method": "soft", "max_seg_num": 1},
    {"nms_method": "hard", "max_seg_num": 1, "voting_thresh": 0.0},
    {"nms_method": "soft", "max_seg_num": 100, "nms_sigma": 0.5},
    {"nms_method": "soft", "pre_nms_thresh": 0.3},
    {"nms_method": "hard", "pre_nms_thresh": 0.3},
    {"nms_method": "soft", "pre_nms_topk": 50},
    {"nms_method": "hard", "pre_nms_topk": 50, "iou_threshold": 0.5},
    {"nms_method": "soft", "duration_thresh": 2.0},
    {"nms_method": "hard", "duration_thresh": 2.0, "voting_thresh": 0.0},
    {"nms_method": "soft", "multiclass_nms": True},
]


def _model(case, precision, weights, test_cfg=None):
    model_name, overrides, _, wseed = MODEL_CASES[case]
    ov = dict(overrides)
    for k, v in (test_cfg or {}).items():
        ov["test_cfg." + k] = v
    cfg = load_config_for(model_name, ov)
    sd = syn.synthetic_state_dict(cfg["model"], model_name, seed=wseed, cls_bias=parity_common.WEIGHTS[weights])
    model = make_meta_arch(cfg["model_name"], **cfg["model"], precision=precision, max_batch=32)
    model.load_state_dict(sd)
    return model.to("cuda").eval()


def _same(a, b):
    assert a["video_id"] == b["video_id"]
    for k in ("segments", "scores", "video_cls"):
        x, y = a[k].numpy(), b[k].numpy()
        assert x.shape == y.shape and np.array_equal(x.view(np.uint32), y.view(np.uint32)), (a["video_id"], k)


@pytest.mark.parametrize("weights", ["dense", "sparse"])
@pytest.mark.parametrize("precision", ["mixed", "fp32"])
@pytest.mark.parametrize("case", ["audio_only", "exp12"])
def test_sweep_equals_a_model_per_setting(case, precision, weights):
    raw = parity_common.make_videos(N_VIDEOS, MODEL_CASES[case][2], seed0=7100)
    model = _model(case, precision, weights)
    store = DenseStore()
    plain = [r for i in range(0, N_VIDEOS, 32) for r in model.forward_streams(raw[i:i + 32], dense=store)]
    again = [r for i in range(0, N_VIDEOS, 32) for r in model.forward_streams(raw[i:i + 32])]
    for a, b in zip(plain, again):          # keeping the dense outputs changes nothing
        _same(a, b)
    base = {k: getattr(model, "test_" + k) for k in sweep.SETTING_KEYS}
    full = [sweep.full_setting(base, s) for s in SETTINGS]
    rows = sweep.sweep_rows(store, full)
    for i, s in enumerate(full):
        ref_model = _model(case, precision, weights, s)
        ref = [r for j in range(0, N_VIDEOS, 32) for r in ref_model.forward_streams(raw[j:j + 32])]
        got = sweep.rows_to_records(store.ids, rows[i])
        assert len(got) == len(ref) == N_VIDEOS
        for a, b in zip(got, ref):
            _same(a, b)
        del ref_model


def _reference_rows(chunk, eng, s, K):
    """avdf_postprocess with setting s on a chunk's dense buffers, as record rows [n, 3 + 3K]."""
    n, L = chunk["n"], chunk["L"]
    dev = chunk["logits"].device
    mask = eng.masks(chunk["valid"][:n].tolist(), L)["pyr"]
    P = chunk["logits"].shape[1]
    k = int(s["max_seg_num"])
    cs = torch.empty((n, P, 2), device=dev); cc = torch.empty((n, P), device=dev); cn = torch.empty(n, dtype=torch.int32, device=dev)
    osg = torch.empty((n, k, 2), device=dev); osc = torch.empty((n, k), device=dev); ocn = torch.empty(n, dtype=torch.int32, device=dev)
    ring = torch.zeros((n, 3 + 3 * k), device=dev)
    counter = torch.zeros(1, dtype=torch.int32, device=dev)
    pos = torch.from_numpy(chunk["pos"][:n]).to(dev)
    ops.postprocess(n, logits=chunk["logits"][:n], offsets=chunk["offsets"][:n], mask=mask, level_len=chunk["level_len"],
                    level_stride=chunk["level_stride"], pre_nms_thresh=s["pre_nms_thresh"], pre_nms_topk=s["pre_nms_topk"],
                    duration_thresh=s["duration_thresh"], cand_segs=cs, cand_scores=cc, cand_count=cn,
                    iou_threshold=s["iou_threshold"], min_score=s["min_score"], sigma=s["nms_sigma"],
                    voting_thresh=0.0 if s["multiclass_nms"] else s["voting_thresh"], max_seg_num=k,
                    use_soft_nms=s["nms_method"] == "soft", vid_meta=[chunk["meta"][i, :n] for i in range(4)],
                    out_segs=osg, out_scores=osc, out_count=ocn, records=(ring, counter, pos, chunk["vcls"][:n]))
    ring = ring.cpu()
    ring = ring[torch.argsort(ring[:, 0])]
    out = torch.zeros((n, 3 + 3 * K))
    out[:, :3] = ring[:, :3]
    out[:, 3:3 + k] = ring[:, 3:3 + k]
    out[:, 3 + K:3 + K + 2 * k] = ring[:, 3 + k:]
    return out


def test_sweep_kernel_equals_postprocess_per_setting():
    model = _model("exp12", "mixed", "dense")
    eng = model.engine()
    raw = parity_common.make_videos(40, True, seed0=7300)
    store = DenseStore(chunk=24)                 # several chunks, the last one short
    for i in range(0, 40, 32):
        model.forward_streams(raw[i:i + 32], dense=store)
    # feats items longer than max_seq_len: a padded pyramid of its own (960 rows at level 0), masked tails
    rng = np.random.RandomState(3)
    feats = [{"video_id": "long%d" % j, "feats": torch.from_numpy(rng.randn(eng.c_in, t).astype(np.float32)), "fps": 25.0,
              "duration": t / 25.0, "feat_stride": 1.0, "feat_num_frames": 1.0} for j, t in enumerate((900, 870, 400))]
    model(feats[:2], dense=store)
    model(feats[2:], dense=store)
    assert {c["L"] for c in store.chunks} == {768, 960}
    base = {k: getattr(model, "test_" + k) for k in sweep.SETTING_KEYS}
    decode_only = [{"pre_nms_thresh": t, "pre_nms_topk": k, "duration_thresh": d}
                   for t in (0.001, 0.25) for k in (2000, 64) for d in (0.001, 1.5)]
    nms_only = [{"nms_method": m, "iou_threshold": i, "min_score": ms, "voting_thresh": v}
                for m in ("hard", "soft") for i, ms, v in ((0.1, 0.2, 0.9), (0.5, 0.001, 0.0), (0.3, 0.05, 0.5))]
    full = [sweep.full_setting(base, s) for s in decode_only + nms_only + [{"max_seg_num": 3}, {"nms_sigma": 0.3}]]
    rows = sweep.sweep_rows(store, full)
    K = rows.shape[2] // 3 - 1
    perm = list(reversed(range(len(full))))
    rows_p = sweep.sweep_rows(store, [full[i] for i in perm])
    for i in range(len(full)):
        assert torch.equal(rows[i].view(torch.int32), rows_p[perm.index(i)].view(torch.int32)), i
    got = rows.cpu()
    for i, s in enumerate(full):
        for c in store.chunks:
            ref = _reference_rows(c, eng, s, K)
            mine = got[i, torch.from_numpy(c["pos"][:c["n"]].astype(np.int64))]
            assert torch.equal(mine.view(torch.int32), ref.view(torch.int32)), (i, s, c["L"])


def _synthetic_gt(ids, seed):
    rng = np.random.RandomState(seed)
    vids, t0, t1 = [], [], []
    for v in list(ids) + ["gt_only_a", "gt_only_b"]:
        for _ in range(2 if v.startswith("gt_only") else rng.randint(0, 4)):
            s = rng.uniform(0, 8)
            vids.append(v); t0.append(s); t1.append(s + rng.uniform(0.05, 2.0))
    return pd.DataFrame({"video-id": vids, "t-start": np.asarray(t0), "t-end": np.asarray(t1), "label": np.zeros(len(vids), np.int64)})


def test_sweep_evaluation_equals_the_evaluators():
    model = _model("audio_only", "mixed", "dense")
    raw = parity_common.make_videos(70, False, seed0=7500)
    gt = _synthetic_gt([r["video_id"] for r in raw], 11)
    tiou = np.linspace(0.1, 0.5, 5)
    res = sweep.sweep_postprocess(model, raw, SETTINGS, gt, tiou_thresholds=tiou, proposals=True, max_bytes=1 << 20)
    assert len(res.results) == len(SETTINGS)
    for i, r in enumerate(res.results):
        records = res.records(i)
        det = ANETdetection(gt, tiou_thresholds=tiou, top_k=(1, 5))
        mAP, avg, mRecall = det.evaluate(records, verbose=False)
        assert np.abs(np.asarray(r["mAP"]) - mAP).max() <= 1e-12, (i, r["mAP"], mAP)
        assert np.array_equal(np.asarray(r["mRecall"]), mRecall), i
        prop = ANETproposal(gt, records, tiou_thresholds=tiou, max_avg_nr_proposals=100.0)
        prop.evaluate()
        for an, v in r["AR@AN"].items():
            j = int(round(an * 100.0 / prop.proposals_per_video[-1])) - 1
            assert v == float(prop.avg_recall[j]), (i, an)
