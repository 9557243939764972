"""Proposal-evaluation benchmark (csrc/eval.cu avdf_eval_proposal): the AV-Deepfake1M-sized synthetic test set of
scripts/eval_bench.py (the same `synth`: 343,233 videos x 100 proposals, GT on --gt-share of the videos).

    python scripts/proposal_bench.py [--videos 343233] [--per-video 100] [--max-avg-nr-proposals 100] [--out FILE]

Reports, in one JSON line:
  * device time of one evaluation from device-resident CSR arrays of the GT videos (CUDA events; warm-up, then --repeats
    calls: median, min);
  * time from host arrays: H2D copy of those CSR arrays + evaluation + the match counts back (host clock around a
    synchronised call);
  * the pandas oracle (oracle/anet_proposal_ref.py) on the first 1,000 videos only, with its size - not extrapolated - and
    the GPU result on the same subset (through average_recall_vs_avg_nr_proposals) compared with it;
  * the GPU name and power limit, read in the same run.
As in the reference, the budget counts the proposals of the videos without GT, so --max-avg-nr-proposals 100 keeps
int(100 * ratio) of each GT video's 100 proposals, ratio = 100 * (GT videos) / (all proposals).
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "scripts")]

from audio_visual_deepfake_detection_b200 import ops  # noqa: E402
from eval_bench import gpu_info, synth  # noqa: E402

THR = np.linspace(0.5, 0.95, 10)


def gt_video_csr(host, max_avg):
    """eval_bench.synth's CSR over all videos -> the CSR of the GT videos, keep and pcn (the reference's arithmetic)."""
    pred_off, seg, score, gt_off, gt_seg = host
    n_gt_v = np.diff(gt_off)
    has = n_gt_v > 0
    n_p = np.diff(pred_off)
    rows = np.repeat(has, n_p)
    prop_off = np.zeros(int(has.sum()) + 1, dtype=np.int64)
    prop_off[1:] = np.cumsum(n_p[has])
    g_off = np.zeros(int(has.sum()) + 1, dtype=np.int32)
    g_off[1:] = np.cumsum(n_gt_v[has])
    n_video, n_all = int(has.sum()), int(score.size)
    ratio = max_avg * float(n_video) / n_all
    keep = np.minimum((n_p[has] * ratio).astype(np.int64), n_p[has])
    total = int(keep.sum())
    pcn = np.arange(1, 101) / 100.0 * (max_avg * float(n_video) / total)
    arrs = (prop_off, np.ascontiguousarray(seg[rows]), np.ascontiguousarray(score[rows]), keep.astype(np.int32), g_off,
            gt_seg)
    return arrs, pcn, total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--videos", type=int, default=343233)
    ap.add_argument("--per-video", type=int, default=100)
    ap.add_argument("--gt-share", type=float, default=0.5)
    ap.add_argument("--max-avg-nr-proposals", type=float, default=100.0)
    ap.add_argument("--repeats", type=int, default=20)
    ap.add_argument("--oracle-videos", type=int, default=1000)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("proposal_bench needs a GPU (no CPU fallback)")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    host = synth(args.videos, args.per_video, args.gt_share, args.seed)
    arrs, pcn, total = gt_video_csr(host, args.max_avg_nr_proposals)
    d = [torch.from_numpy(x).to(dev) for x in arrs]
    ws = torch.empty(ops.nv.lib().avdf_eval_proposal_workspace_bytes(arrs[0].size - 1), dtype=torch.uint8, device=dev)

    def run(a):
        return ops.eval_proposal(*a, THR, pcn, workspace=ws, check_status=False)

    for _ in range(3):
        out = run(d)
    assert int(out[1].item()) == 0
    times = []
    for _ in range(args.repeats):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); run(d); e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    m_a = run(d)[0].cpu().numpy()
    deterministic = bool(np.array_equal(m_a, run(d)[0].cpu().numpy()))
    pinned = [torch.from_numpy(x).pin_memory() for x in arrs]
    host_times = []
    for _ in range(max(3, args.repeats // 4)):
        torch.cuda.synchronize()
        h0 = time.perf_counter()
        dd = [p.to(dev, non_blocking=True) for p in pinned]
        run(dd)[0].cpu()
        host_times.append((time.perf_counter() - h0) * 1e3)
    n_gt = int(arrs[4][-1])
    avg_recall = (m_a / float(n_gt)).mean(axis=0)
    ppv = pcn * (float(total) / (arrs[0].size - 1))

    # oracle on the first videos only (their proposals include those of the videos without GT)
    import anet_proposal_ref as ref
    import pandas as pd
    from audio_visual_deepfake_detection_b200.libs.utils import average_recall_vs_avg_nr_proposals
    nv = args.oracle_videos
    pred_off, seg, score, gt_off, gt_seg = host
    P, G = int(pred_off[nv]), int(gt_off[nv])
    gt_df = pd.DataFrame({"video-id": np.repeat(np.arange(nv), np.diff(gt_off[:nv + 1])), "t-start": gt_seg[:G, 0],
                          "t-end": gt_seg[:G, 1]})
    pr_df = pd.DataFrame({"video-id": np.repeat(np.arange(nv), np.diff(pred_off[:nv + 1])), "t-start": seg[:P, 0],
                          "t-end": seg[:P, 1], "score": score[:P]})
    o0 = time.perf_counter()
    rec_ref, avg_ref, ppv_ref = ref.average_recall_vs_avg_nr_proposals(gt_df, pr_df, args.max_avg_nr_proposals, THR)
    t_oracle = time.perf_counter() - o0
    rec_s, avg_s, ppv_s = average_recall_vs_avg_nr_proposals(gt_df, pr_df, args.max_avg_nr_proposals, THR)
    name, smi = gpu_info()
    trapz = getattr(np, "trapezoid", None) or np.trapz
    res = {"bench": "eval_proposal", "gpu": name, "nvidia_smi": smi, "videos": args.videos, "proposals": int(host[2].size),
           "gt_videos": int(arrs[0].size - 1), "gt_rows": n_gt, "gt_share_synthetic": args.gt_share,
           "max_avg_nr_proposals": args.max_avg_nr_proposals, "proposals_walked": total, "thresholds": len(THR),
           "device_ms_median": float(np.median(times)), "device_ms_min": float(np.min(times)), "repeats": args.repeats,
           "from_host_arrays_ms_median": float(np.median(host_times)), "deterministic": deterministic,
           "AR@1": float(avg_recall[0]), "AR@100": float(avg_recall[-1]),
           "auc": 100.0 * float(trapz(avg_recall, ppv)) / ppv[-1],
           "oracle_videos": nv, "oracle_proposals": P, "oracle_s": t_oracle,
           "oracle_vs_gpu_recall_equal": bool(np.array_equal(rec_s, rec_ref)),
           "oracle_vs_gpu_avg_recall_equal": bool(np.array_equal(avg_s, avg_ref) and np.array_equal(ppv_s, ppv_ref))}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
