"""Detection-evaluation benchmark (csrc/eval.cu): an AV-Deepfake1M-sized synthetic test set, one class.

    python scripts/eval_bench.py [--videos 343233] [--per-video 100] [--repeats 20] [--out FILE]

Synthetic data (seeded): 343,233 videos x 100 predictions; ground truth of 1-3 segments on a share of the videos (--gt-share,
default 0.5 - a synthetic choice, not AV-Deepfake1M's real share); predictions jittered around a GT segment of their video
(at random on videos without GT); fp32-derived scores, descending inside each video as result records are.
Reports, in one JSON line:
  * device time of one evaluation from device-resident CSR arrays (CUDA events; warm-up, then --repeats calls: median, min);
  * time from host arrays: H2D copy of the CSR arrays + evaluation + results back (host clock around a synchronised call);
  * the pandas oracle (oracle/anet_ref.py) on the first 1,000 videos only, with its size - not extrapolated - and the GPU
    result on the same subset compared with it;
  * the GPU name and power limit, read in the same run;
  * the bytes the kernels move (counted from the launch sequence: see `traffic`) over the median time, as a fraction of
    7.7 TB/s HBM bandwidth. The working set is larger than L2 only in part, so this is a fraction of a floor estimate.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle")]

from audio_visual_deepfake_detection_b200 import ops  # noqa: E402

THR = np.linspace(0.5, 0.95, 10)
TOPK = (1, 5)
HBM_BYTES_PER_S = 7.7e12


def synth(n_video, per_video, gt_share, seed):
    rng = np.random.default_rng(seed)
    dur = rng.uniform(5, 60, n_video)
    n_gt_v = np.where(rng.random(n_video) < gt_share, rng.integers(1, 4, n_video), 0)
    gt_off = np.zeros(n_video + 1, dtype=np.int64)
    gt_off[1:] = np.cumsum(n_gt_v)
    G = int(gt_off[-1])
    gv = np.repeat(np.arange(n_video), n_gt_v)
    gs = rng.random(G) * (dur[gv] - 1)
    gt_seg = np.stack([gs, np.minimum(dur[gv], gs + rng.uniform(0.2, 8, G))], 1)
    n = n_video * per_video
    pv = np.repeat(np.arange(n_video), per_video)
    has = n_gt_v[pv] > 0
    pick = gt_off[pv] + (rng.integers(0, 1 << 30, n) % np.maximum(n_gt_v[pv], 1))
    base = np.where(has[:, None], gt_seg[np.minimum(pick, max(G - 1, 0))], 0.0)
    ln = base[:, 1] - base[:, 0]
    rs = rng.random(n) * (dur[pv] - 1)
    ps = np.where(has, base[:, 0] + rng.normal(0, 1, n) * 0.15 * ln, rs)
    pe = np.where(has, np.maximum(ps + 0.05, base[:, 1] + rng.normal(0, 1, n) * 0.15 * ln), rs + rng.uniform(0.1, 6, n))
    score = rng.random(n).astype(np.float32).astype(np.float64)
    order = np.lexsort((-score, pv))                    # descending inside each video
    score, ps, pe = score[order], ps[order], pe[order]
    pred_off = np.arange(0, n + 1, per_video, dtype=np.int64)
    return pred_off, np.stack([ps, pe], 1), score, gt_off.astype(np.int32), np.ascontiguousarray(gt_seg)


def traffic(n, score):
    """Bytes the launch sequence moves for n predictions (reads + writes of every kernel, per call)."""
    k = score.view(np.uint64).copy()
    k = np.where(k >> 63, ~k, k | np.uint64(1 << 63))
    active = sum(1 for d in range(8) if np.unique((k >> np.uint64(8 * d)) & np.uint64(255)).size > 1)
    per = 16 + 8 + 2          # match: segments, scores (order check), tp mask
    per += 8                  # histogram of all digits
    for a in range(active):   # upsweep key read, scatter key + payload read, payload (+ key unless last) write
        per += 8 + 10 + 2 + (8 if a + 1 < active else 0)
    per += 3 * 2              # AP scan: three passes over the sorted masks
    return per * n, active


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as exc:       # noqa: BLE001
        q = "nvidia-smi unavailable: %s" % exc
    return name, q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--videos", type=int, default=343233)
    ap.add_argument("--per-video", type=int, default=100)
    ap.add_argument("--gt-share", type=float, default=0.5)
    ap.add_argument("--repeats", type=int, default=20)
    ap.add_argument("--oracle-videos", type=int, default=1000)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("eval_bench needs a GPU (no CPU fallback)")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    t0 = time.perf_counter()
    host = synth(args.videos, args.per_video, args.gt_share, args.seed)
    t_synth = time.perf_counter() - t0
    n = host[2].size
    d = [torch.from_numpy(x).to(dev) for x in host]
    ws = torch.empty(ops.nv.lib().avdf_eval_workspace_bytes(n, args.videos), dtype=torch.uint8, device=dev)

    def run(arrs):
        return ops.eval_detection(*arrs, THR, TOPK, workspace=ws, check_status=False)

    for _ in range(3):
        out = run(d)
    assert int(out[2].item()) == 0
    times = []
    for _ in range(args.repeats):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); run(d); e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    ap_dev, hits, _ = run(d)
    ap_a, hits_a = ap_dev.cpu().numpy(), hits.cpu().numpy()
    ap_b, hits_b, _ = run(d)
    deterministic = bool(np.array_equal(ap_a, ap_b.cpu().numpy()) and np.array_equal(hits_a, hits_b.cpu().numpy()))
    # from host arrays: pinned copies of the CSR, H2D + evaluation + results back
    pinned = [torch.from_numpy(x).pin_memory() for x in host]
    host_times = []
    for _ in range(max(3, args.repeats // 4)):
        torch.cuda.synchronize()
        h0 = time.perf_counter()
        dd = [p.to(dev, non_blocking=True) for p in pinned]
        a_, h_, _ = run(dd)
        a_.cpu(); h_.cpu()
        host_times.append((time.perf_counter() - h0) * 1e3)
    # oracle on the first videos only
    import anet_ref
    import pandas as pd
    nv = args.oracle_videos
    pred_off, seg, score, gt_off, gt_seg = host
    P, G = int(pred_off[nv]), int(gt_off[nv])
    gt_df = pd.DataFrame({"video-id": np.repeat(np.arange(nv), np.diff(gt_off[:nv + 1])), "t-start": gt_seg[:G, 0],
                          "t-end": gt_seg[:G, 1], "label": 0})
    pr_df = pd.DataFrame({"video-id": np.repeat(np.arange(nv), np.diff(pred_off[:nv + 1])), "t-start": seg[:P, 0],
                          "t-end": seg[:P, 1], "label": 0, "score": score[:P]})
    o0 = time.perf_counter()
    ap_ref, rec_ref, _, _ = anet_ref.evaluate(gt_df, pr_df, THR, TOPK)
    t_oracle = time.perf_counter() - o0
    sub = [torch.from_numpy(np.ascontiguousarray(x)).to(dev) for x in (pred_off[:nv + 1], seg[:P], score[:P], gt_off[:nv + 1], gt_seg[:G])]
    ap_s, hits_s, _ = ops.eval_detection(*sub, THR, TOPK)
    sub_ap_err = float(np.abs(ap_s.cpu().numpy() - ap_ref[:, 0]).max())
    sub_rec_equal = bool(np.array_equal(hits_s.cpu().numpy() / G, rec_ref[:, :, 0]))
    nbytes, active = traffic(n, score)
    med = float(np.median(times))
    name, smi = gpu_info()
    res = {"bench": "eval_detection", "gpu": name, "nvidia_smi": smi, "videos": args.videos, "predictions": int(n),
           "gt_rows": int(host[3][-1]), "gt_share_synthetic": args.gt_share, "thresholds": len(THR), "top_k": list(TOPK),
           "device_ms_median": med, "device_ms_min": float(np.min(times)), "repeats": args.repeats,
           "from_host_arrays_ms_median": float(np.median(host_times)), "radix_passes": active,
           "bytes_moved_est": int(nbytes), "hbm_floor_ms_est": nbytes / HBM_BYTES_PER_S * 1e3,
           "fraction_of_hbm_floor": nbytes / HBM_BYTES_PER_S * 1e3 / med, "deterministic": deterministic,
           "mAP": [float(x) for x in ap_a], "recall_at_1x": [float(x) for x in hits_a[:, 0] / host[3][-1]],
           "oracle_videos": nv, "oracle_predictions": P, "oracle_s": t_oracle, "oracle_vs_gpu_ap_max_abs_err": sub_ap_err,
           "oracle_vs_gpu_recall_equal": sub_rec_equal, "synth_s": t_synth}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
