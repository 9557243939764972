"""Sliding-window benchmark (model.forward_streams(..., window, hop)): the audio-only exp12 workload of bench.py (BYOL-A
2048 + Emotion2Vec 768, synthetic weights, batch 32) on synthetic recordings of --minutes minutes, window --window s,
hop --hop s.

    python scripts/window_bench.py [--recordings 8] [--minutes 10] [--window 10] [--hop 5] [--repeats 3] [--out FILE]

Reports, in one JSON line:
  * media-seconds per second of wall time (host clock around whole synchronised calls, after a warm-up call that
    captures the graphs) and windows/s;
  * media-seconds per second of device time: device time = the summed durations of every kernel and copy of one call in
    a torch.profiler trace (a separate, traced call); the merge's share = its three launches (window_gather_kernel,
    the postprocess_kernel that follows it, window_finalize_kernel) over that sum;
  * host -> device bytes per media-second as sent (each recording once), next to what packing every window as a
    video of its own would send (the rows of all windows);
  * the GPU name and power limit, read in the same run.
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "scripts")]

from audio_visual_deepfake_detection_b200.libs.core import load_config_for  # noqa: E402
from audio_visual_deepfake_detection_b200.libs.modeling import EXP12, make_meta_arch  # noqa: E402
from audio_visual_deepfake_detection_b200.libs.modeling.windows import window_plan  # noqa: E402
from audio_visual_deepfake_detection_b200.libs.utils import synthetic as syn  # noqa: E402
from eval_bench import gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--recordings", type=int, default=8)
    ap.add_argument("--minutes", type=float, default=10.0)
    ap.add_argument("--window", type=float, default=10.0)
    ap.add_argument("--hop", type=float, default=5.0)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "window_bench.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("window_bench needs a GPU")
    cfg = load_config_for(EXP12, {"dataset.video_input_dim": 0})
    model = make_meta_arch(cfg["model_name"], **cfg["model"], max_batch=32)
    model.load_state_dict(syn.synthetic_state_dict(cfg["model"], EXP12, seed=0))
    model.to("cuda").eval()
    D = args.minutes * 60.0
    recs = [{"video_id": "long%d" % i, "duration": D, "streams": syn.synthetic_streams(D, 5000 + i, video_dim=0)}
            for i in range(args.recordings)]
    media = D * len(recs)
    n_win, dup_bytes, sent_bytes = 0, 0, 0
    for r in recs:
        arrs = [r["streams"].get(n) for n in ("video", "byola", "emo")]
        plan = window_plan(D, [None if a is None else a.shape[0] for a in arrs], args.window, args.hop)
        n_win += len(plan)
        sent_bytes += sum(a.nbytes for a in arrs if a is not None)
        dup_bytes += sum(m * a.shape[1] * a.itemsize for _, rng in plan for a, (_, m) in zip(arrs, rng) if a is not None)

    def call():
        return model.forward_streams(recs, window=args.window, hop=args.hop)
    call()                                                          # graphs captured, staging sized
    runner = model.runner()
    h0 = runner.h2d_bytes
    walls = []
    for _ in range(args.repeats):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = call()
        walls.append(time.perf_counter() - t0)
    h2d = (runner.h2d_bytes - h0) / args.repeats
    n_segs = sum(int(o["scores"].numel()) for o in out)

    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        call()
        torch.cuda.synchronize()
    evs = sorted([e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA], key=lambda e: e.time_range.start)
    dev_us, merge_us, after_gather = 0.0, 0.0, False
    for e in evs:
        d = e.time_range.end - e.time_range.start
        dev_us += d
        if "window_gather_kernel" in e.name or "window_finalize_kernel" in e.name:
            merge_us += d
            after_gather = "window_gather_kernel" in e.name
        elif after_gather and "postprocess_kernel" in e.name:
            merge_us += d
            after_gather = False
    name, smi = gpu_info()
    wall = float(np.median(walls))
    res = {
        "workload": "audio-only exp12 (BYOL-A 2048 + Emotion2Vec 768), synthetic weights, max_batch 32",
        "recordings": len(recs), "recording_seconds": D, "window_s": args.window, "hop_s": args.hop, "windows": n_win,
        "segments_out": n_segs,
        "wall_s_median": wall, "wall_s_all": walls,
        "media_s_per_wall_s": media / wall, "windows_per_wall_s": n_win / wall,
        "device_ms_traced": dev_us / 1e3, "media_s_per_device_s": media / (dev_us / 1e6),
        "windows_per_device_s": n_win / (dev_us / 1e6),
        "merge_ms_traced": merge_us / 1e3, "merge_share_of_device_time": merge_us / dev_us,
        "h2d_bytes_per_media_s": h2d / media,
        "h2d_bytes_per_media_s_if_windows_packed_separately": dup_bytes / media,
        "stream_bytes_per_media_s": sent_bytes / media,
        "gpu": name, "nvidia_smi_name_power_limit_max_sm_clock": smi,
        "notes": "device time = summed kernel + copy durations of one traced call (torch.profiler); wall time = host clock "
                 "around untraced synchronised calls after a warm-up call",
    }
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
