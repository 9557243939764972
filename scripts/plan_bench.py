"""Launch-plan replay (avdf_session_run, csrc/plan.cu) against the Python path's captured graphs, in the same run.

    python scripts/plan_bench.py [--out profiles/plan_bench.json] [--seconds 1.5]

Workload: the audio-only exp12 model (BYOL-A + emotion2vec streams, mixed precision, synthetic weights), batches of 32
seeded AV-Deepfake1M-length recordings resident on the device (no host -> device copy in the timed region). Each lane is
one buffer set on its own stream - a PlanSession for the plan, an engine lane with its GraphedPass for Python - and every
launch replays one CUDA graph of the whole pass. Timed with CUDA events around at least --seconds of launches per
configuration; 1 and 8 lanes, plan and Python alternated, two rounds. Also reported: host time per launch call (what the
caller's thread spends to enqueue one batch). Writes the card name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from audio_visual_deepfake_detection_b200.libs.core import load_config_for          # noqa: E402
from audio_visual_deepfake_detection_b200.libs.modeling import EXP12, make_meta_arch  # noqa: E402
from audio_visual_deepfake_detection_b200.libs.modeling import plan as pl           # noqa: E402
from audio_visual_deepfake_detection_b200.libs.utils import synthetic as syn       # noqa: E402

B = 32


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
        name, limit = [v.strip() for v in q.split(",")]
    except Exception as exc:           # the name from torch, the power limit unknown
        return {"name": torch.cuda.get_device_name(), "power_limit": "unavailable (%s)" % exc}
    return {"name": name, "power_limit": limit}


def timed(lanes, seconds):
    """lanes: [(launch(), stream)] -> (batches, device seconds, host us per launch call), round-robin over the lanes."""
    def go(n):
        start = torch.cuda.Event(enable_timing=True)
        end = torch.cuda.Event(enable_timing=True)
        start.record()
        for _, st in lanes:
            st.wait_event(start)
        host = 0.0
        for i in range(n):
            fn, st = lanes[i % len(lanes)]
            with torch.cuda.stream(st):
                t0 = time.perf_counter()
                fn()
                host += time.perf_counter() - t0
        cur = torch.cuda.current_stream()
        for _, st in lanes:
            cur.wait_stream(st)
        end.record()
        end.synchronize()
        return start.elapsed_time(end) / 1e3, host / n * 1e6

    t, _ = go(8 * len(lanes))                # warm
    n = 8 * len(lanes)
    while True:
        t, host = go(n)
        if t >= seconds:
            return n, t, host
        n = int(n * max(1.5, 1.1 * seconds / max(t, 1e-3)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "plan_bench.json"))
    ap.add_argument("--seconds", type=float, default=1.5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("plan_bench needs a CUDA device")
    cfg = load_config_for(EXP12, {"dataset.video_input_dim": 0})
    model = make_meta_arch(cfg["model_name"], **cfg["model"], precision="mixed", max_batch=B)
    model.load_state_dict(syn.synthetic_state_dict(cfg["model"], EXP12, seed=3, cls_bias=-7.0))
    model = model.to("cuda").eval()
    items = pl._synthetic_items((0, 2048, 768), B, 4321)
    tmp = tempfile.mkdtemp()
    path = model.export_plan(os.path.join(tmp, "audio_only.plan"), batch_sizes=(B,))
    plan = pl.Plan(path)
    dev = torch.device("cuda", torch.cuda.current_device())

    sessions = [plan.session() for _ in range(8)]
    rows = None
    for s in sessions:
        rows = s.stage(items)
    torch.cuda.synchronize()

    graphs = []                       # Python path: one engine lane + captured pass per lane, inputs resident
    info = plan.info
    for lane in range(8):
        streams = [torch.zeros((info.stream_rows[s], info.channels[s]), device=dev) if info.channels[s] else None for s in range(3)]
        offs = torch.zeros((3, B + 1), dtype=torch.int32, device=dev)
        meta = torch.zeros(4 * B, device=dev)
        pl._stage_items(items, streams, offs, meta, info.t_out)
        staged = {"ids": [c["video_id"] for c in items], "B": B, "meta": meta.view(4, B), "streams": streams,
                  "offs": [offs[s, :B + 1] if info.channels[s] else None for s in range(3)]}
        graphs.append(model.capture(staged, lane=lane))
    torch.cuda.synchronize()

    streams = [torch.cuda.Stream() for _ in range(8)]
    plan_lanes = [(lambda s=s, st=st: s.launch(B, rows, st), st) for s, st in zip(sessions, streams)]
    py_lanes = [(g.replay, st) for g, st in zip(graphs, streams)]
    # the same bits from both paths before anything is timed
    plan_lanes[0][0]()
    torch.cuda.synchronize()
    res = graphs[0].replay()
    torch.cuda.synchronize()
    s0 = sessions[0]
    same = torch.equal(s0.counts, res["counts"]) and torch.equal(s0.vcls, res["vcls"]) and all(    # rows past counts are unwritten
        torch.equal(s0.segs[b, :n], res["segs"][b, :n]) and torch.equal(s0.scores[b, :n], res["scores"][b, :n])
        for b, n in enumerate(res["counts"].tolist()))
    rows_out = []
    for rnd in range(2):
        for n_lanes in (1, 8):
            for name, lanes in (("plan", plan_lanes), ("python", py_lanes)):
                n, t, host = timed(lanes[:n_lanes], a.seconds)
                rows_out.append({"round": rnd, "path": name, "lanes": n_lanes, "batches": n, "seconds": round(t, 4),
                                 "videos_per_s": round(n * B / t, 1), "host_us_per_launch": round(host, 2)})
                print(json.dumps(rows_out[-1]), flush=True)
    out = {"workload": "audio-only exp12 (byola 2048 + emo 768), mixed precision, synthetic weights, batch %d, "
                       "inputs resident on the device, one CUDA graph replay per batch" % B,
           "card": card(), "torch": torch.__version__, "plan_bytes": os.path.getsize(path),
           "plan_matches_python_bit_for_bit": bool(same), "results": rows_out}
    for s in sessions:
        s.close()
    plan.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out["card"]), "plan == python:", same)


if __name__ == "__main__":
    main()
