"""GPU checks of the detection evaluator (csrc/eval.cu, libs/utils/metrics.py) against the pandas oracle
(oracle/anet_ref.py) and against a torch composition of the AP formula at scale."""
import json

import numpy as np
import pandas as pd
import pytest
import torch

import anet_ref
from audio_visual_deepfake_detection_b200 import native, ops
from audio_visual_deepfake_detection_b200.libs.utils import metrics
from test_eval_oracle import KA_AP, KA_R1, KA_R5, KA_THR, KA_TP05_INPUT, known_answer_frames

pytestmark = pytest.mark.gpu


def test_known_answer():
    gt, pr = known_answer_frames()
    det = metrics.ANETdetection(gt, tiou_thresholds=KA_THR)
    ap, recall, tp = det.evaluate_classes(pr, want_tp=True)
    assert np.abs(ap[:, 0] - KA_AP).max() < 1e-12
    assert np.abs(recall[:, 0, 0] - KA_R1).max() < 1e-12 and np.abs(recall[:, 1, 0] - KA_R5).max() < 1e-12
    assert [int(m) & 1 for m in tp] == KA_TP05_INPUT
    mAP, avg, mRecall = det.evaluate(pr, verbose=False)
    assert np.abs(mAP - KA_AP).max() < 1e-12 and abs(avg - np.mean(KA_AP)) < 1e-12 and mRecall.shape == (3, 2)


def random_set(seed, n_video=1000, classes=(0,), score_kind="fp64", grouped=False):
    """GT of 1-3 segments on ~60 % of the videos (real videos have none), 0-12 predictions per video jittered around the
    GT or placed at random; prediction labels include one value that is no GT label (kept as is by the mapping)."""
    rng = np.random.RandomState(seed)
    gt_rows, pr_rows = [], []
    pred_labels = list(classes) + ([1] if len(classes) > 1 and 1 not in classes else [])
    for v in range(n_video):
        vid = "vid%05d" % v
        dur = rng.uniform(5, 60)
        segs = []
        if rng.rand() < 0.6:
            for _ in range(rng.randint(1, 4)):
                s = rng.uniform(0, dur - 1); e = min(dur, s + rng.uniform(0.2, 8))
                lab = classes[rng.randint(len(classes))]
                segs.append((s, e, lab)); gt_rows.append((vid, s, e, lab))
        for _ in range(rng.randint(0, 13)):
            if segs and rng.rand() < 0.7:
                s, e, lab = segs[rng.randint(len(segs))]
                j = rng.normal(0, 0.15 * (e - s), 2)
                ps, pe = s + j[0], max(s + j[0] + 0.05, e + j[1])
                lab = lab if rng.rand() < 0.8 else pred_labels[rng.randint(len(pred_labels))]
            else:
                ps = rng.uniform(0, dur - 1); pe = ps + rng.uniform(0.1, 6); lab = pred_labels[rng.randint(len(pred_labels))]
            sc = rng.rand()
            if score_kind == "grid":
                sc = np.round(sc * 20) / 20                      # many ties
            elif score_kind == "fp32":
                sc = float(np.float32(sc))
            pr_rows.append((vid, float(ps), float(pe), lab, float(sc)))
    gt = pd.DataFrame(gt_rows, columns=["video-id", "t-start", "t-end", "label"])
    pr = pd.DataFrame(pr_rows, columns=["video-id", "t-start", "t-end", "label", "score"])
    if not grouped:
        pr = pr.sample(frac=1.0, random_state=seed).reset_index(drop=True)
    return gt, pr


@pytest.mark.parametrize("classes,score_kind,grouped", [((0,), "grid", False), ((0,), "fp32", True), ((0,), "fp64", False),
                                                        ((3, 7, 11), "grid", False), ((3, 7, 11), "fp64", True)])
def test_against_oracle(classes, score_kind, grouped):
    gt, pr = random_set(7 + len(classes), classes=classes, score_kind=score_kind, grouped=grouped)
    thr = np.linspace(0.5, 0.95, 10)
    ap_ref, rec_ref, tps_ref, rows = anet_ref.evaluate(gt, pr, thr, (1, 5))
    det = metrics.ANETdetection(gt, tiou_thresholds=thr)
    ap, rec, tp = det.evaluate_classes(pr, want_tp=True)
    assert np.abs(ap - ap_ref).max() < 1e-12
    assert np.array_equal(rec, rec_ref)
    for c, sel in rows.items():
        want = (tps_ref[c].astype(np.uint16) << np.arange(len(thr), dtype=np.uint16)[:, None]).sum(0).astype(np.uint16)
        assert np.array_equal(tp[sel], want), c
    if grouped and len(classes) == 1:                  # the same rows as result records
        recs = [{"video_id": v, "scores": g["score"].tolist(), "segments": g[["t-start", "t-end"]].values.tolist()}
                for v, g in pr.groupby("video-id", sort=False)]
        ap2, rec2, _ = det.evaluate_classes(recs)
        assert np.array_equal(ap2, ap) and np.array_equal(rec2, rec)


def _big_csr(n_video, per_video, seed, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    n = n_video * per_video
    n_gt_v = torch.randint(1, 4, (n_video,), generator=g, device=dev, dtype=torch.int32)
    gt_off = torch.zeros(n_video + 1, dtype=torch.int32, device=dev)
    gt_off[1:] = torch.cumsum(n_gt_v, 0)
    G = int(gt_off[-1])
    gs = torch.rand(G, generator=g, device=dev, dtype=torch.float64) * 50
    gt_seg = torch.stack([gs, gs + 0.5 + 5 * torch.rand(G, generator=g, device=dev, dtype=torch.float64)], 1).contiguous()
    vid = torch.arange(n_video, device=dev).repeat_interleave(per_video)
    pick = gt_off[:-1].long()[vid] + (torch.randint(0, 1 << 20, (n,), generator=g, device=dev) % n_gt_v.long()[vid])
    base = gt_seg[pick]
    jit = torch.randn(n, 2, generator=g, device=dev, dtype=torch.float64) * (base[:, 1:] - base[:, :1]) * 0.2
    ps = base[:, 0] + jit[:, 0]
    pred_seg = torch.stack([ps, torch.maximum(ps + 0.01, base[:, 1] + jit[:, 1])], 1).contiguous()
    score = torch.round(torch.rand(n, generator=g, device=dev, dtype=torch.float64) * 1000) / 1000     # ties across videos
    # descending inside every video except every tenth one (those take the shared-memory sort)
    key = vid.double() * 2 - score
    order = torch.argsort(key, stable=True)
    srt = torch.where((vid % 10 == 0), torch.arange(n, device=dev), order)
    score = score[srt].contiguous()
    pred_off = torch.arange(0, n + 1, per_video, device=dev, dtype=torch.int64)
    return pred_off, pred_seg, score, gt_off, gt_seg


def test_large_against_torch_composition_and_deterministic():
    dev = torch.device("cuda")
    pred_off, pred_seg, score, gt_off, gt_seg = _big_csr(100_000, 100, 3, dev)
    thr = np.linspace(0.5, 0.95, 10)
    tp = torch.empty(score.numel(), dtype=torch.uint16, device=dev)
    ap, hits, _ = ops.eval_detection(pred_off, pred_seg, score, gt_off, gt_seg, thr, (1, 5), tp_mask=tp)
    tp2 = torch.empty_like(tp)
    ap2, hits2, _ = ops.eval_detection(pred_off, pred_seg, score, gt_off, gt_seg, thr, (1, 5), tp_mask=tp2)
    assert torch.equal(ap, ap2) and torch.equal(hits, hits2) and torch.equal(tp.view(torch.int16), tp2.view(torch.int16))
    _, idx = torch.sort(score, descending=True, stable=True)
    m = tp.view(torch.int16).int()[idx] & 0xffff
    npos = gt_seg.shape[0]
    pos = torch.arange(1, score.numel() + 1, device=dev, dtype=torch.float64)
    for t in range(len(thr)):
        b = ((m >> t) & 1).double()
        prec = torch.cumsum(b, 0) / pos
        env = torch.flip(torch.cummax(torch.flip(prec, [0]), 0).values, [0])
        want = float((env * b).sum() / npos)
        assert abs(float(ap[t]) - want) < 1e-9, (t, float(ap[t]), want)
    assert 0 < float(ap[0]) < 1 and int(hits[0, 1]) <= npos and (hits[:, 0] <= hits[:, 1]).all()


def test_device_limits_raise_and_write_nothing():
    dev = torch.device("cuda")
    n = 8193
    pred_off = torch.tensor([0, n], dtype=torch.int64, device=dev)
    seg = torch.zeros(n, 2, dtype=torch.float64, device=dev); seg[:, 1] = 1
    score = torch.rand(n, dtype=torch.float64, device=dev)
    gt_off = torch.tensor([0, 1], dtype=torch.int32, device=dev)
    gt = torch.tensor([[0.0, 1.0]], dtype=torch.float64, device=dev)
    with pytest.raises(native.AvdfError, match="8192"):
        ops.eval_detection(pred_off, seg, score, gt_off, gt, [0.5], (1,))
    tp = torch.full((n,), 7, dtype=torch.int16, device=dev).view(torch.uint16)
    ap, hits, st = ops.eval_detection(pred_off, seg, score, gt_off, gt, [0.5], (1,), tp_mask=tp, check_status=False)
    assert int(st) == native.EVAL_PRED_LIMIT and (tp.view(torch.int16) == 7).all()
    gt_off = torch.tensor([0, 65], dtype=torch.int32, device=dev)
    gt = torch.zeros(65, 2, dtype=torch.float64, device=dev); gt[:, 1] = 1
    with pytest.raises(native.AvdfError, match="64"):
        ops.eval_detection(torch.tensor([0, 2], dtype=torch.int64, device=dev), seg[:2].contiguous(), score[:2].contiguous(),
                           gt_off, gt, [0.5], (1,))


def test_valid_one_epoch_and_cli_match_evaluate(tmp_path, capsys):
    import interp_ref
    from audio_visual_deepfake_detection_b200.libs.core import load_config_for
    from audio_visual_deepfake_detection_b200.libs.modeling import EXP12, make_meta_arch
    from audio_visual_deepfake_detection_b200.libs.utils import inference_one_epoch, synthetic as syn, valid_one_epoch
    cfg = load_config_for(EXP12)
    sd = syn.synthetic_state_dict(cfg["model"], EXP12, seed=0)
    model = make_meta_arch(cfg["model_name"], **cfg["model"], max_batch=8)
    model.load_state_dict(sd)
    model.to("cuda").eval()
    rng = np.random.RandomState(5)
    durs = rng.uniform(4, 20, 64)
    items = [interp_ref.dataset_item(syn.synthetic_streams(float(d), 3000 + i), float(d), "v%02d" % i) for i, d in enumerate(durs)]
    loader = [items[i:i + 8] for i in range(0, 64, 8)]
    db = {}
    for i, d in enumerate(durs):
        ann = []
        if i % 3:
            s = rng.uniform(0, d - 2)
            ann.append({"segment": [s, s + rng.uniform(0.5, 2)], "label": 0})
        db["v%02d" % i] = {"subset": "test", "annotations": ann}
    gt_file = tmp_path / "gt.json"
    gt_file.write_text(json.dumps({"database": db}))
    thr = np.linspace(0.1, 0.5, 5)          # loose thresholds: synthetic weights localise nothing in particular

    class Capture(metrics.ANETdetection):
        def evaluate(self, preds, verbose=True):
            self.seen = preds
            return super().evaluate(preds, verbose)
    det = Capture(str(gt_file), split="test", tiou_thresholds=thr)
    avg = valid_one_epoch(loader, model, 0, evaluator=det, print_freq=4)
    assert len(det.seen["score"]) > 0
    mAP, avg2, mRecall = metrics.ANETdetection(str(gt_file), split="test", tiou_thresholds=thr).evaluate(det.seen, verbose=False)
    assert avg == avg2
    inference_one_epoch(loader, model, 0, output_folder=str(tmp_path / "out"))
    capsys.readouterr()
    cli_mAP, cli_avg, cli_rec = metrics.main(["--gt", str(gt_file), "--split", "test", str(tmp_path / "out"), "--tiou", *map(str, thr)])
    line = capsys.readouterr().out.strip().splitlines()[-1]
    res = json.loads(line)
    assert np.array_equal(cli_mAP, mAP) and np.array_equal(cli_rec, mRecall) and res["average_mAP"] == float(avg2)
    assert res["videos"] == 64
