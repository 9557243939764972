"""GPU checks of the proposal evaluator (csrc/eval.cu avdf_eval_proposal, libs/utils/Evaluation/eval_proposal.py) against
the pandas oracle (oracle/anet_proposal_ref.py) and, at AV-Deepfake1M scale, against a vectorised torch composition."""
import json

import numpy as np
import pandas as pd
import pytest
import torch

import anet_proposal_ref as ref
from audio_visual_deepfake_detection_b200 import native, ops
from audio_visual_deepfake_detection_b200.libs.utils import ANETproposal, average_recall_vs_avg_nr_proposals
from audio_visual_deepfake_detection_b200.libs.utils.Evaluation import eval_proposal
from test_proposal_oracle import PKA, PKA_THR, proposal_known_answer_frames

pytestmark = pytest.mark.gpu

THR = np.linspace(0.5, 0.95, 10)


def _records(pr):
    return [{"video_id": v, "scores": g["score"].tolist(), "segments": g[["t-start", "t-end"]].values.tolist()}
            for v, g in pr.groupby("video-id", sort=False)]


def _assert_equal_to_oracle(gt, pr_df, got, max_avg, thr):
    rec_ref, avg_ref, ppv_ref = ref.average_recall_vs_avg_nr_proposals(gt, pr_df, max_avg, thr)
    rec, avg, ppv = got
    assert np.array_equal(rec, rec_ref)
    assert np.array_equal(avg, avg_ref) and np.array_equal(ppv, ppv_ref)
    assert eval_proposal.area_under_curve(avg, ppv) == ref.auc(avg_ref, ppv_ref)
    return rec


@pytest.mark.parametrize("max_avg", [None, 2, 100])
def test_known_answer(max_avg):
    gt, pr = proposal_known_answer_frames()
    got = average_recall_vs_avg_nr_proposals(gt, pr, max_avg, PKA_THR)
    rec = _assert_equal_to_oracle(gt, pr, got, max_avg, PKA_THR)
    points, auc = PKA[max_avg]
    for (t, j), want in points.items():
        assert rec[t, j] == want
    assert abs(eval_proposal.area_under_curve(got[1], got[2]) - auc) < 1e-4
    prop = ANETproposal(gt, pr, tiou_thresholds=PKA_THR, max_avg_nr_proposals=max_avg)
    prop.evaluate()
    assert np.array_equal(prop.recall, rec) and np.array_equal(prop.avg_recall, got[1])
    assert np.array_equal(prop.proposals_per_video, got[2])


def proposal_set(seed, n_video=1000, score_kind="fp64", grouped=True):
    """GT of 1-3 segments on ~60 % of the videos; 0-12 proposals per video jittered around a GT segment or placed at random
    (so GT videos without proposals and videos without GT that have proposals both occur); videos 7, 257, 507, 757 have
    40 GT rows and 300 proposals. grouped: rows grouped by video, score-descending inside each (as result records are);
    else shuffled."""
    rng = np.random.RandomState(seed)
    gt_rows, pr_rows = [], []
    for v in range(n_video):
        vid = "vid%05d" % v
        dur = rng.uniform(5, 60)
        big = v % 250 == 7
        segs = []
        if big or rng.rand() < 0.6:
            for _ in range(40 if big else rng.randint(1, 4)):
                s = rng.uniform(0, dur - 1); e = min(dur, s + rng.uniform(0.2, 8))
                segs.append((s, e)); gt_rows.append((vid, s, e))
        rows = []
        for _ in range(300 if big else rng.randint(0, 13)):
            if segs and rng.rand() < 0.7:
                s, e = segs[rng.randint(len(segs))]
                j = rng.normal(0, 0.15 * (e - s), 2)
                ps, pe = s + j[0], max(s + j[0] + 0.05, e + j[1])
            else:
                ps = rng.uniform(0, dur - 1); pe = ps + rng.uniform(0.1, 6)
            sc = rng.rand()
            if score_kind == "grid":
                sc = np.round(sc * 10) / 10                       # many ties
            rows.append((vid, float(ps), float(pe), float(sc)))
        if grouped:
            rows = [rows[i] for i in np.lexsort((np.arange(len(rows)), [-r[3] for r in rows]))]
        pr_rows += rows
    gt = pd.DataFrame(gt_rows, columns=["video-id", "t-start", "t-end"])
    pr = pd.DataFrame(pr_rows, columns=["video-id", "t-start", "t-end", "score"])
    if not grouped:
        pr = pr.sample(frac=1.0, random_state=seed).reset_index(drop=True)
    return gt, pr


@pytest.mark.parametrize("seed,score_kind,grouped,max_avg,thr", [
    (21, "grid", False, None, THR), (22, "grid", True, 100, THR), (23, "fp64", False, 1.0, THR),
    (24, "grid", False, 3.0, THR), (25, "fp64", True, None, np.linspace(0.05, 1.0, 16))])
def test_against_oracle(seed, score_kind, grouped, max_avg, thr):
    gt, pr = proposal_set(seed, score_kind=score_kind, grouped=grouped)
    gt_v = set(gt["video-id"])
    n_p = pr.groupby("video-id").size()
    assert any(v not in n_p.index for v in gt_v) and any(v not in gt_v for v in n_p.index)
    if max_avg == 1.0:                         # the budget cuts: both 0 < keep < n_p and keep == 0 < n_p occur
        n = n_p[[v for v in n_p.index if v in gt_v]].values
        k = (n * (max_avg * len(gt_v) / len(pr))).astype(np.int64)
        assert ((k > 0) & (k < n)).any() and ((k == 0) & (n > 0)).any()
    got = average_recall_vs_avg_nr_proposals(gt, pr, max_avg, thr)
    rec = _assert_equal_to_oracle(gt, pr, got, max_avg, thr)
    assert 0 < rec[0, -1] <= 1
    if grouped:                                # the same rows as result records
        got2 = average_recall_vs_avg_nr_proposals(gt, _records(pr), max_avg, thr)
        assert all(np.array_equal(a, b) for a, b in zip(got, got2))


def _one_video(n_p, n_gt, keep):
    dev = torch.device("cuda")
    prop_off = torch.tensor([0, n_p], dtype=torch.int64, device=dev)
    seg = torch.zeros(n_p, 2, dtype=torch.float64, device=dev); seg[:, 1] = 1
    score = torch.rand(n_p, dtype=torch.float64, device=dev)
    gt_off = torch.tensor([0, n_gt], dtype=torch.int32, device=dev)
    gt = torch.zeros(n_gt, 2, dtype=torch.float64, device=dev); gt[:, 1] = 1
    return prop_off, seg, score, torch.tensor([keep], dtype=torch.int32, device=dev), gt_off, gt


@pytest.mark.parametrize("n_p,n_gt,keep,bit,msg", [(8193, 1, 8193, native.EVAL_PRED_LIMIT, "8192"),
                                                   (4, 65, 4, native.EVAL_GT_LIMIT, "64"),
                                                   (4, 2, 5, native.EVAL_BAD_KEEP, "keep"),
                                                   (4, 2, -1, native.EVAL_BAD_KEEP, "keep")])
def test_device_limits_raise_and_write_nothing(n_p, n_gt, keep, bit, msg):
    args = _one_video(n_p, n_gt, keep)
    frac = np.arange(1, 101) / 100.0
    with pytest.raises(native.AvdfError, match=msg):
        ops.eval_proposal(*args, THR, frac)
    sentinel = torch.full((len(THR), 100), -7, dtype=torch.int64, device="cuda")
    m, st = ops.eval_proposal(*args, THR, frac, matches=sentinel, check_status=False)
    assert int(st) == bit and (sentinel == -7).all()


def test_bad_offsets_raise():
    prop_off, seg, score, keep, gt_off, gt = _one_video(4, 2, 4)
    with pytest.raises(native.AvdfError, match="offsets"):
        ops.eval_proposal(prop_off, seg, score, keep, torch.tensor([1, 2], dtype=torch.int32, device="cuda"), gt, THR,
                          np.arange(1, 101) / 100.0)


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
    jit = torch.randn(n, 2, generator=g, device=dev, dtype=torch.float64) * (base[:, 1:] - base[:, :1]) * 0.3
    ps = base[:, 0] + jit[:, 0]
    prop_seg = torch.stack([ps, torch.maximum(ps + 0.01, base[:, 1] + jit[:, 1])], 1).contiguous()
    score = torch.round(torch.rand(n, generator=g, device=dev, dtype=torch.float64) * 1000) / 1000     # ties
    # descending inside every video except every tenth one (those take the shared-memory sort)
    order = torch.argsort(vid.double() * 2 - score, stable=True)
    srt = torch.where(vid % 10 == 0, torch.arange(n, device=dev), order)
    score, prop_seg = score[srt].contiguous(), prop_seg[srt].contiguous()
    keep = torch.randint(0, per_video + 1, (n_video,), generator=g, device=dev, dtype=torch.int32)
    prop_off = torch.arange(0, n + 1, per_video, device=dev, dtype=torch.int64)
    return prop_off, prop_seg, score, keep, gt_off, gt_seg


def test_large_against_torch_composition_and_deterministic():
    dev = torch.device("cuda")
    V, P = 343_233, 100
    prop_off, prop_seg, score, keep, gt_off, gt_seg = _big_csr(V, P, 5, dev)
    total = int(keep.sum())
    pcn = np.arange(1, 101) / 100.0 * (60 * float(V) / total)
    m1, _ = ops.eval_proposal(prop_off, prop_seg, score, keep, gt_off, gt_seg, THR, pcn)
    m2, _ = ops.eval_proposal(prop_off, prop_seg, score, keep, gt_off, gt_seg, THR, pcn)
    assert torch.equal(m1, m2)
    # walk order: score descending inside each video, ties by position
    vid = torch.arange(V, device=dev).repeat_interleave(P)
    walk = prop_seg[torch.argsort(vid.double() * 2 - score, stable=True)].view(V, P, 2)
    gv = torch.arange(V, device=dev).repeat_interleave((gt_off[1:] - gt_off[:-1]).long())
    cut = torch.minimum((keep.double()[:, None] * torch.from_numpy(pcn).to(dev)[None]).long(), keep.long()[:, None])
    want = torch.zeros(len(THR), 100, dtype=torch.int64, device=dev)
    for c0 in range(0, gv.numel(), 200_000):            # GT rows in chunks: [rows, P] tIoU matrices
        g = gv[c0:c0 + 200_000]
        p = walk[g]
        gs, ge = gt_seg[c0:c0 + 200_000, 0:1], gt_seg[c0:c0 + 200_000, 1:2]
        inter = torch.clamp(torch.minimum(p[..., 1], ge) - torch.maximum(p[..., 0], gs), min=0)
        tiou = inter / ((ge - gs) + (p[..., 1] - p[..., 0]) - inter)
        walked = torch.arange(P, device=dev)[None] < keep.long()[g][:, None]
        for t, th in enumerate(THR):
            hit = (tiou >= th) & walked
            first = torch.where(hit.any(1), hit.int().argmax(1), torch.full_like(g, P + 1))
            want[t] += (first[:, None] < cut[g]).sum(0)
    assert torch.equal(m1, want)
    assert 0 < int(m1[0, -1]) <= gv.numel() and (m1[:, 1:] >= m1[:, :-1]).all()


def test_cli_matches_evaluate(tmp_path, capsys):
    gt, pr = proposal_set(3, n_video=400, score_kind="grid", grouped=True)
    db = {}
    for v, s, e in gt.itertuples(index=False):
        db.setdefault(v, {"subset": "test", "annotations": []})["annotations"].append({"segment": [s, e], "label": "Fake"})
    db["other"] = {"subset": "train", "annotations": [{"segment": [1.0, 2.0], "label": "Fake"}]}
    gt_file = tmp_path / "gt.json"
    gt_file.write_text(json.dumps({"database": db}))
    recs = _records(pr)
    out = tmp_path / "out"
    out.mkdir()
    (out / "data_left_0.json").write_text(json.dumps(recs[:150]))
    (out / "data_left_1.json").write_text(json.dumps(recs[150:]))
    prop = ANETproposal(str(gt_file), recs, ground_truth_fields=["database"], subset="test", max_avg_nr_proposals=100)
    prop.evaluate()
    capsys.readouterr()
    rec, avg, ppv, auc = eval_proposal.main(["--gt", str(gt_file), "--split", "test", str(out)])
    res = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert np.array_equal(rec, prop.recall) and np.array_equal(avg, prop.avg_recall)
    assert np.array_equal(ppv, prop.proposals_per_video)
    assert auc == eval_proposal.area_under_curve(prop.avg_recall, prop.proposals_per_video) == res["auc"]
    for an in (1, 5, 10, 20, 50, 100):
        assert res["AR@%d" % an] == float(prop.avg_recall[an - 1])
    assert res["videos"] == len(recs) and res["proposals"] == len(pr)
    _assert_equal_to_oracle(gt, pr, (rec, avg, ppv), 100, THR)
