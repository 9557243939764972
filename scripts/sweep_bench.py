"""Post-processing sweep (libs/utils/sweep.py) against the ways a setting is scored without it.

    python scripts/sweep_bench.py [--videos 32768] [--weights sparse] [--full-passes 2] [--json profiles/sweep_bench.json]

Workload: audio-only exp12 model with synthetic weights (`sparse`: cls prior -7, a handful of segments per video like a
trained detector; `dense`: the golden fixtures' stress weights), `--videos` synthetic AV-Deepfake1M-length videos (a pool
of 256 distinct raw-stream sets reused under distinct ids), batch 32, precision mixed, a synthetic ground truth (0-3
segments per video), and a 48-setting grid: nms_method {hard, soft} x iou_threshold {0.1, 0.3, 0.5} x min_score
{0.001, 0.2} x voting_thresh {0, 0.9} x pre_nms_thresh {0.001, 0.05} (two decode groups). Reports:
  - the forward pass over all videos with and without dense capture (host clock around synchronised runs);
  - sweep-kernel device time for all 48 settings (CUDA events, median of 3, warm), per setting and per (video, setting);
  - (a) the same rows from 48 launches of avdf_postprocess: per decode group one decode-mode launch, then candidate-mode
    launches from its candidate list (CUDA events, median of 3), and whether its results equal the sweep's;
  - evaluation device time per setting (CUDA events around ANETdetection.evaluate_rows, median over the settings);
  - total wall time of sweep_postprocess over the kept outputs (kernel + evaluation of every setting);
  - (b) full forward_streams passes for the first `--full-passes` settings, wall time each;
  - the card name and power limit, read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    sys.path.insert(0, p)

import numpy as np  # noqa: E402
import pandas as pd  # noqa: E402
import torch  # noqa: E402

from audio_visual_deepfake_detection_b200 import ops  # noqa: E402
from audio_visual_deepfake_detection_b200.libs.core import load_config_for  # noqa: E402
from audio_visual_deepfake_detection_b200.libs.modeling import EXP12, make_meta_arch  # noqa: E402
from audio_visual_deepfake_detection_b200.libs.modeling.engine import DenseStore  # noqa: E402
from audio_visual_deepfake_detection_b200.libs.utils import synthetic as syn  # noqa: E402
from audio_visual_deepfake_detection_b200.libs.utils import sweep  # noqa: E402
from audio_visual_deepfake_detection_b200.libs.utils.metrics import ANETdetection, RowsLayout  # noqa: E402

GRID = [("nms_method", ["hard", "soft"]), ("iou_threshold", [0.1, 0.3, 0.5]), ("min_score", [0.001, 0.2]),
        ("voting_thresh", [0.0, 0.9]), ("pre_nms_thresh", [0.001, 0.05])]
WEIGHTS = {"dense": -3.0, "sparse": -7.0}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as exc:       # noqa: BLE001
        q = "nvidia-smi unavailable: %s" % exc
    return torch.cuda.get_device_name(0), q


def events(fn, reps=3):
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    return statistics.median(ts)


def wall(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t, out


def loop_postprocess(store, eng, full, K):
    """Rows of every setting from avdf_postprocess: one decode-mode launch per decode group, candidate mode after it."""
    rows = torch.zeros((len(full), len(store), 3 + 3 * K), dtype=torch.float32, device="cuda")
    groups = {}
    for i, s in enumerate(full):
        groups.setdefault((s["pre_nms_thresh"], s["pre_nms_topk"], s["duration_thresh"]), []).append(i)
    for c in store.chunks:
        n, P = c["n"], c["logits"].shape[1]
        mask = eng.masks(c["valid"][:n].tolist(), c["L"])["pyr"]
        pos = torch.from_numpy(c["pos"][:n]).cuda()
        cs = torch.empty((n, P, 2), device="cuda"); cc = torch.empty((n, P), device="cuda")
        cn = torch.empty(n, dtype=torch.int32, device="cuda")
        meta = [c["meta"][i, :n] for i in range(4)]
        for members in groups.values():
            for j, i in enumerate(members):
                s = full[i]
                k = int(s["max_seg_num"])
                osg = torch.empty((n, k, 2), device="cuda"); osc = torch.empty((n, k), device="cuda")
                ocn = torch.empty(n, dtype=torch.int32, device="cuda")
                dec = dict(logits=c["logits"][:n], offsets=c["offsets"][:n], mask=mask) if j == 0 else {}
                ops.postprocess(n, **dec, level_len=c["level_len"], level_stride=c["level_stride"],
                                pre_nms_thresh=s["pre_nms_thresh"], pre_nms_topk=s["pre_nms_topk"],
                                duration_thresh=s["duration_thresh"], cand_segs=cs, cand_scores=cc, cand_count=cn,
                                iou_threshold=s["iou_threshold"], min_score=s["min_score"], sigma=s["nms_sigma"],
                                voting_thresh=0.0 if s["multiclass_nms"] else s["voting_thresh"], max_seg_num=k,
                                use_soft_nms=s["nms_method"] == "soft", vid_meta=meta, out_segs=osg, out_scores=osc,
                                out_count=ocn)
                r = rows[i].index_select(0, pos.long())
                r[:, 1] = ocn.float()
                r[:, 3:3 + k] = osc
                r[:, 3 + K:3 + K + 2 * k] = osg.reshape(n, -1)
                rows[i].index_copy_(0, pos.long(), r)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--videos", type=int, default=32768)
    ap.add_argument("--weights", default="sparse", choices=sorted(WEIGHTS))
    ap.add_argument("--full-passes", type=int, default=2)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    name, smi = gpu_info()
    cfg = load_config_for(EXP12, {"dataset.video_input_dim": 0})
    sd = syn.synthetic_state_dict(cfg["model"], EXP12, seed=3, cls_bias=WEIGHTS[args.weights])

    def build(test_cfg=None):
        c = load_config_for(EXP12, dict({"dataset.video_input_dim": 0}, **{"test_cfg." + k: v for k, v in (test_cfg or {}).items()}))
        m = make_meta_arch(c["model_name"], **c["model"], precision="mixed", max_batch=32)
        m.load_state_dict(sd)
        return m.to("cuda").eval()

    model = build()
    durs = syn.sample_durations(256, seed=1)
    pool = [syn.synthetic_streams(float(d), 9000 + i, video_dim=0) for i, d in enumerate(durs)]
    raw = [{"video_id": "v%06d" % i, "duration": float(durs[i % 256]), "streams": pool[i % 256]} for i in range(args.videos)]
    batches = [raw[i:i + 32] for i in range(0, len(raw), 32)]
    for _ in model.stream(batches[:8]):            # warm: graphs captured, staging sized
        pass
    t_plain, _ = wall(lambda: [r for b in model.stream(batches) for r in b])
    store = DenseStore()
    t_dense, _ = wall(lambda: [r for b in model.stream(batches, dense=store) for r in b])
    rng = np.random.RandomState(0)
    gv, g0, g1 = [], [], []
    for v in store.ids:
        for _ in range(rng.randint(0, 4)):
            s = rng.uniform(0, 8)
            gv.append(v); g0.append(s); g1.append(s + rng.uniform(0.1, 3.0))
    gt = pd.DataFrame({"video-id": gv, "t-start": np.asarray(g0), "t-end": np.asarray(g1), "label": np.zeros(len(gv), np.int64)})
    base = {k: getattr(model, "test_" + k) for k in sweep.SETTING_KEYS}
    full = [sweep.full_setting(base, s) for s in sweep.grid(GRID)]
    S, N = len(full), len(store)
    K = max(int(s["max_seg_num"]) for s in full)
    rows = sweep.sweep_rows(store, full)            # warm
    t_sweep = events(lambda: sweep.sweep_rows(store, full))
    eng = model.engine()
    rows_a = loop_postprocess(store, eng, full, K)  # warm
    t_loop = events(lambda: loop_postprocess(store, eng, full, K))
    # avdf_postprocess leaves out_* beyond each video's count unwritten: compare counts and the live entries
    live = torch.arange(K, device="cuda")[None, None, :] < rows[:, :, 1:2]
    live_seg = live.repeat_interleave(2, dim=2)
    same = bool(torch.equal(rows_a[:, :, 1], rows[:, :, 1]) and
                torch.equal(rows_a[:, :, 3:3 + K][live].view(torch.int32), rows[:, :, 3:3 + K][live].view(torch.int32)) and
                torch.equal(rows_a[:, :, 3 + K:][live_seg].view(torch.int32), rows[:, :, 3 + K:][live_seg].view(torch.int32)))
    del rows_a
    det = ANETdetection(gt, tiou_thresholds=np.linspace(0.5, 0.95, 10))
    layout = RowsLayout(det.ground_truth, store.ids)
    t_eval = [events(lambda: det.evaluate_rows(rows[s], K, layout), reps=1) for s in range(S)]
    del rows
    t_total, res = wall(lambda: sweep.sweep_postprocess(model, store, sweep.grid(GRID), gt))
    t_full = []
    for s in full[:args.full_passes]:
        m = build({k: s[k] for k in sweep.SETTING_KEYS})
        for _ in m.stream(batches[:8]):
            pass
        t, _ = wall(lambda: [r for b in m.stream(batches) for r in b])
        t_full.append(t)
        del m
    out = {
        "gpu": name, "nvidia_smi_name_power_limit_max_sm_clock": smi, "weights": args.weights, "videos": N,
        "settings": S, "decode_groups": 2, "dense_store_bytes": store.nbytes(),
        "forward_s": {"plain": t_plain, "with_dense_capture": t_dense},
        "sweep_kernel_ms": {"all_settings": t_sweep, "per_setting": t_sweep / S, "per_video_setting_us": 1e3 * t_sweep / (S * N)},
        "loop_postprocess_ms": {"all_settings": t_loop, "per_setting": t_loop / S, "equal_rows": same,
                                "sweep_speedup": t_loop / t_sweep},
        "eval_ms_per_setting": {"median": statistics.median(t_eval), "max": max(t_eval)},
        "sweep_postprocess_wall_s": t_total,
        "full_forward_pass_s_per_setting": t_full,
        "best_setting": max(res.results, key=lambda r: r["average_mAP"])["setting"],
    }
    print(json.dumps(out, indent=1))
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
