"""Sliding windows through launch-plan sessions (avdf_session_run_windows) next to the Python windowed path
(model.forward_streams(..., window, hop)), on window_bench.py's workload: audio-only exp12 (BYOL-A 2048 + Emotion2Vec 768,
synthetic weights, max_batch 32), --recordings synthetic recordings of --minutes minutes, window --window s, hop --hop s,
a plan exported with every batch size and enough --max-seconds of staging for one session's recordings.

    python scripts/plan_window_bench.py [--recordings 8] [--minutes 10] [--window 10] [--hop 5] [--repeats 3] [--out FILE]

Reports, in one JSON line, windows/s and media-seconds/s (host clock around synchronised calls, median of --repeats,
after a warm-up call that captures the graphs) for:
  * forward_streams(window=...): host packing + one host -> device copy per stream + the windows + merge + results to host;
  * one plan session: avdf_session_run_windows with the recordings already in the session's staging (the copy into the
    staging is the caller's, timed separately as `plan_staging_s`);
  * 2 and 4 sessions of the plan, each with its own recordings in its own staging, launched on separate streams.
Outputs are compared bit for bit: the session against forward_streams on the same recordings, the concurrent sessions
against their own sequential runs. The GPU name and power limit are read in the same run.
"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "scripts")]

from audio_visual_deepfake_detection_b200.libs.core import load_config_for  # noqa: E402
from audio_visual_deepfake_detection_b200.libs.modeling import EXP12, make_meta_arch  # noqa: E402
from audio_visual_deepfake_detection_b200.libs.modeling import plan as pl  # noqa: E402
from audio_visual_deepfake_detection_b200.libs.modeling.windows import window_plan  # noqa: E402
from audio_visual_deepfake_detection_b200.libs.utils import synthetic as syn  # noqa: E402
from eval_bench import gpu_info  # noqa: E402


def same(a, b):
    return len(a) == len(b) and all(
        x["video_id"] == y["video_id"] and x["segments"].shape == y["segments"].shape and
        all(torch.equal(x[k], y[k]) for k in ("segments", "scores", "video_cls")) for x, y in zip(a, b))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--recordings", type=int, default=8)
    ap.add_argument("--minutes", type=float, default=10.0)
    ap.add_argument("--window", type=float, default=10.0)
    ap.add_argument("--hop", type=float, default=5.0)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--sessions", type=int, nargs="+", default=[2, 4])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "plan_window_bench.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("plan_window_bench needs a GPU")
    cfg = load_config_for(EXP12, {"dataset.video_input_dim": 0})
    model = make_meta_arch(cfg["model_name"], **cfg["model"], max_batch=32)
    model.load_state_dict(syn.synthetic_state_dict(cfg["model"], EXP12, seed=0))
    model.to("cuda").eval()
    D, W, H = args.minutes * 60.0, args.window, args.hop
    n_sets = max([1] + args.sessions)
    sets = [[{"video_id": "long%d_%d" % (j, i), "duration": D, "streams": syn.synthetic_streams(D, 5000 + 100 * j + i, video_dim=0)}
             for i in range(args.recordings)] for j in range(n_sets)]
    recs = sets[0]
    per_rec = len(window_plan(D, [None] + [recs[0]["streams"][n].shape[0] for n in ("byola", "emo")], W, H))
    n_win = per_rec * len(recs)
    media = D * len(recs)

    def timed(fn):
        fn()                                                                      # warm-up: graphs captured
        walls = []
        for _ in range(args.repeats):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            walls.append(time.perf_counter() - t0)
        return float(np.median(walls)), walls

    res = {"workload": "audio-only exp12 (BYOL-A 2048 + Emotion2Vec 768), synthetic weights, max_batch 32",
           "recordings_per_session": len(recs), "recording_seconds": D, "window_s": W, "hop_s": H, "windows_per_session": n_win}
    want = model.forward_streams(recs, window=W, hop=H)
    wall, walls = timed(lambda: model.forward_streams(recs, window=W, hop=H))
    res["forward_streams"] = {"wall_s_median": wall, "wall_s_all": walls, "windows_per_s": n_win / wall,
                              "media_s_per_s": media / wall}

    tmp = tempfile.mkdtemp(prefix="plan_window_bench_")
    max_seconds = D * len(recs) / model.max_batch + 1.0                          # one session's recordings fit the staging
    path = model.export_plan(os.path.join(tmp, "exp12_audio.plan"), max_seconds=max_seconds)
    plan = pl.Plan(path)
    try:
        K = plan.info.max_seg_num
        sessions = []
        for j in range(n_sets):
            s = plan.session()
            s.attach_windows(n_win, per_rec)
            sessions.append(s)
        rows = [[[c["streams"][n].shape[0] if n in c["streams"] else 0 for n in pl.STREAM_NAMES] for c in st] for st in sets]
        durs = [[c["duration"] for c in st] for st in sets]
        outs = [(torch.empty((len(st), K, 2), device="cuda"), torch.empty((len(st), K), device="cuda"),
                 torch.empty((len(st),), dtype=torch.int32, device="cuda"), torch.empty((len(st),), device="cuda")) for st in sets]

        def results(j):
            segs, scores, counts, vcls = (t.cpu() for t in outs[j])
            return [{"video_id": c["video_id"], "segments": segs[r, :int(counts[r])], "scores": scores[r, :int(counts[r])],
                     "video_cls": vcls[r:r + 1]} for r, c in enumerate(sets[j])]

        t0 = time.perf_counter()
        for j in range(n_sets):
            with torch.cuda.stream(sessions[j].stream):
                pl._stage_streams(sets[j], sessions[j].streams)
        torch.cuda.synchronize()
        res["plan_staging_s"] = (time.perf_counter() - t0) / n_sets
        res["plan_max_seconds"] = max_seconds
        ok = same(sessions[0].run_windows(recs, W, H), want)
        with torch.cuda.stream(sessions[0].stream):
            pl._stage_streams(sets[0], sessions[0].streams)
        torch.cuda.synchronize()
        seq = []
        for j in range(n_sets):                                                   # sequential reference of every set
            sessions[j].launch_windows(durs[j], rows[j], W, H, outs[j])
            torch.cuda.synchronize()
            seq.append(results(j))

        def run(n):
            for j in range(n):
                sessions[j].launch_windows(durs[j], rows[j], W, H, outs[j])
        for n in [1] + args.sessions:
            wall, walls = timed(lambda: run(n))
            ok_n = all(same(results(j), seq[j]) for j in range(n))
            res["plan_sessions_%d" % n] = {"wall_s_median": wall, "wall_s_all": walls, "windows_per_s": n * n_win / wall,
                                           "media_s_per_s": n * media / wall, "bit_identical_to_sequential": ok_n}
            ok = ok and ok_n
        res["plan_bit_identical_to_forward_streams"] = same(seq[0], want)
        res["bit_identical"] = bool(ok and res["plan_bit_identical_to_forward_streams"])
    finally:
        plan.close()
        for f in os.listdir(tmp):
            os.remove(os.path.join(tmp, f))
        os.rmdir(tmp)
    name, smi = gpu_info()
    res.update({"gpu": name, "nvidia_smi_name_power_limit_max_sm_clock": smi,
                "notes": "wall time = host clock around synchronised calls after a warm-up call, median of the repeats; "
                         "plan sessions time avdf_session_run_windows with inputs already staged; forward_streams includes "
                         "its own host packing and host -> device copy"})
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")
    if not res["bit_identical"]:
        raise SystemExit("plan_window_bench: outputs differ")


if __name__ == "__main__":
    main()
