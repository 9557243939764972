#!/usr/bin/env python
"""Benchmark of the localization-inference hot path (BASELINE.json: videos/s, fwd + decode + soft-NMS).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload audio|av12|av13] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One step = 32 batches of 32 synthetic AV-Deepfake1M-shaped videos (1024 videos) on every rank, each batch one pass of
the path: interp+concat of the raw per-stream features (K1) -> video-level branch + embedding + 18 ConvTransformer
blocks + FPN + heads -> decode -> soft-NMS + voting + seconds conversion -> one result record per video. Videos are
sharded over ranks (weak scaling: 1024 videos per rank per step, no data-path collective); the fixed-size result records
are all-gathered once at the end of the timed region (the path's only exchange).

  value     videos/s with the raw features already resident in HBM (CUDA events, max over ranks)
  e2e       videos/s through the public API (model.forward_streams on HOST numpy buffers): pinned H2D of every
            step's features and D2H of every step's results inside the timed region
  roofline  tensor-core GEMM kernel (conv_gemm_tc_kernel), tensor bound: algorithmic FLOPs of all its launches / their
            summed CUDA-event durations, measured in an instrumented pass right after the timed region
  cpu_baseline / --impl reference: the oracle (CPU restatement of the reference, oracle/) on the host cores (all
            cores and one thread), bounded sample of the same workload; its outputs also check the CUDA path's
            final segment sets (`parity`)
  extra     (single GPU) av12 / av13 workloads and the 1k-100k NMS sweep (BASELINE.json configs[2], [3]).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (meta-arch key, cfg overrides, use video stream, description)
    "audio": ("exp12", {"dataset.video_input_dim": 0}, False,
              "audio-only (BYOL-A 2048 + Emotion2Vec 768) exp12-arch localization, synthetic AV-Deepfake1M-length sequences, batch 32"),
    "av12": ("exp12", {}, True, "audio-visual fused exp12-arch localization (3072 ch), batch 32"),
    "av13": ("exp13", {}, True, "audio-visual fused exp13-arch localization (SegmentandCls branch), batch 32"),
    # SURVEY 8(f).3: the exp5-style arch (live reconstruction branch), visual stream + emotion2vec (1024 ch) like its yaml
    "av5": ("exp5", {}, "video+emo", "audio-visual exp5-style localization with the live reconstruction branch (1024 ch), batch 32"),
}
BATCH = 32
TRAFFIC_FILE = "r2_o_step_traffic.json"    # per-kernel DRAM bytes of one pass (ncu pass, see profiles/README.md)
PIPE_FILE = "r2_n_tensor_pipe.json"          # sm__pipe_tensor_cycles_active per kernel from the committed ncu --set full page
N_POOL = 8              # distinct resident input batches rotated through the timed region (8 x ~75 MB > 126 MB L2)


def flops_per_video(cfg_model, exp13, recon=False):
    """Algorithmic FLOPs per video (SURVEY.md 8d: embedding once, dead Expansion dropped)."""
    cin = cfg_model["video_input_dim"] + cfg_model["audio_input_dim"]
    C, T = cfg_model["embd_dim"], cfg_model["max_seq_len"]
    embed = 2 * T * C * 3 * cin + 2 * T * C * 3 * C
    blocks = 1.573e6 * 7632 * (T / 768.0)
    fpn = 0.201e9
    heads = 2.385e9
    if exp13:
        dims = [cin, 1024, 512, 256, 128, 64]
        vc = sum(2 * T * dims[i + 1] * 3 * dims[i] for i in range(5))
    else:
        dims = [cin, C, 2 * C, 4 * C, 8 * C, C]
        vc = sum(2 * (T >> (i + 1)) * dims[i + 1] * 3 * dims[i] for i in range(5))
    if recon:       # exp5-style: the Expansion (ConvTranspose1d k3: 3 taps per input position, blocks.py:1568-1590) + a second embedding pass
        up = [C, 2048, 1024, 512, 256, cin]
        vc += sum(2 * (T >> (5 - i)) * up[i] * 3 * up[i + 1] for i in range(5)) + embed
    return embed + blocks + fpn + heads + vc


def build_cfg(workload):
    from audio_visual_deepfake_detection_b200.libs.core import load_config_for
    from audio_visual_deepfake_detection_b200.libs.modeling import EXP5, EXP12, EXP13
    key, overrides, use_video, desc = WORKLOADS[workload]
    name = {"exp12": EXP12, "exp13": EXP13, "exp5": EXP5}[key]
    # the metric is quoted with soft-NMS (BASELINE.json); the shipped yaml resolves to hard
    cfg = load_config_for(name, dict(overrides, **{"test_cfg.nms_method": "soft"}))
    return cfg, name, use_video, desc


def make_raw_batches(n_batches, use_video, seed0):
    from audio_visual_deepfake_detection_b200.libs.utils import synthetic as syn
    durs = syn.sample_durations(n_batches * BATCH, seed=seed0)
    out = []
    for i in range(n_batches):
        out.append([{"video_id": "v%06d" % (seed0 * 100000 + i * BATCH + j), "duration": float(durs[i * BATCH + j]),
                     "streams": syn.synthetic_streams(float(durs[i * BATCH + j]), seed0 * 100000 + i * BATCH + j,
                                                      video_dim=256 if use_video else 0,
                                                      byola_dim=0 if use_video == "video+emo" else 2048)} for j in range(BATCH)])
    return out


def pin_batches(batches):
    """The same batches with every stream array living in page-locked host memory: one pinned block per batch, collated
    stream-major by the product's loader-side helper (libs/modeling/streaming.py collate_pinned)."""
    from audio_visual_deepfake_detection_b200.libs.modeling.streaming import collate_pinned
    return [collate_pinned(chunk) for chunk in batches]


# --------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    QUERY = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def wait_ready(self, timeout=3.0):
        """Block until nvidia-smi has printed its first sample (it needs ~0.1-0.3 s to start)."""
        t0 = time.time()
        while self.proc is not None and not self.rows and time.time() - t0 < timeout:
            time.sleep(0.01)

    def mark(self):
        self.first = len(self.rows)

    def count(self):
        return len(self.rows) - getattr(self, "first", 0)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.rows = self.rows[getattr(self, "first", 0):]
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------- CPU reference arm
def cpu_reference(workload, n_videos, threads, keep_outputs=False, cls_bias=-3.0):
    """Times the oracle (oracle/model_ref.py + oracle/nms_ref.c: the CPU restatement of the reference path,
    pinned to the reference's outputs by tests/test_oracle_golden.py) on `n_videos` videos of the workload:
    numpy interp+concat, fp32 forward, decode, soft-NMS, one video per call like the reference
    (av_fd_no_recon.py:456). Returns (videos/s, seconds[, raw videos, oracle outputs])."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import interp_ref, model_ref, nms_ref
    from audio_visual_deepfake_detection_b200.libs.utils import synthetic as syn
    torch.set_num_threads(threads)
    cfg, name, use_video, _ = build_cfg(workload)
    sd = syn.synthetic_state_dict(cfg["model"], name, seed=0, cls_bias=cls_bias)
    om = model_ref.OracleModel(cfg["model"], sd, name)
    raw = make_raw_batches(1, use_video, seed0=7)[0][:n_videos]
    nms_ref.lib()
    om([interp_ref.dataset_item(raw[0]["streams"], raw[0]["duration"], raw[0]["video_id"])], nms_ref.batched_nms)   # warm-up
    outs = []
    t0 = time.perf_counter()
    for r in raw:
        item = interp_ref.dataset_item(r["streams"], r["duration"], r["video_id"])
        o = om([item], nms_ref.batched_nms)
        if keep_outputs:
            outs.append(o[0])
    dt = time.perf_counter() - t0
    if keep_outputs:
        return n_videos / dt, dt, raw, outs
    return n_videos / dt, dt


def parity_vs_oracle(model, raw, ref_outs):
    """The checker half of the cpu_baseline leg: the oracle's final sets for its timed sample against the CUDA path's sets for
    the same videos (after the 0.2 score filter: same membership, start/end within 1e-3 s; oracle/parity.py)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import parity
    got = model.forward_streams(raw)
    st = {"videos": len(raw), "identical_sets": 0, "membership_diff": 0, "boundary_over_1ms_only": 0, "members_ref": 0,
          "members_over_1ms": 0, "max_boundary_dev_s": 0.0}
    for g, r in zip(got, ref_outs):
        c = parity.compare_sets(g["segments"].numpy(), g["scores"].numpy(), r["segments"].numpy(), r["scores"].numpy())
        st["members_ref"] += c["n_ref"]; st["members_over_1ms"] += c["n_dt_over"]
        st["max_boundary_dev_s"] = max(st["max_boundary_dev_s"], c["max_dt"])
        if c["same_membership"] and c["n_dt_over"] == 0:
            st["identical_sets"] += 1
        elif c["same_membership"]:
            st["boundary_over_1ms_only"] += 1
        else:
            st["membership_diff"] += 1
    return st


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    n = args.ref_videos
    cfg, name, use_video, desc = build_cfg(args.workload)
    vals = []
    for _ in range(args.warmup if args.warmup < 1 else 1):
        cpu_reference(args.workload, 2, threads)
    for _ in range(args.steps):
        vals.append(cpu_reference(args.workload, n, threads)[0])
    v = float(np.mean(vals))
    line = {"impl": "reference", "metric": "videos/sec localization inference (fwd+decode+soft-NMS)", "value": v, "unit": "videos/s",
            "n_gpus": args.gpus, "steps": len(vals), "warmup": args.warmup, "ms_per_step": 1000.0 * n / v,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": desc, "videos_per_step": n, "nms": "soft", "note": "CPU, B=1 per call like the reference"},
            "cpu_baseline": {"value": v, "unit": "videos/s", "cores": threads, "kind": "port",
                             "sample": "%d videos per step, oracle/model_ref.py + oracle/nms_ref.c, torch CPU fp32" % n},
            "e2e": {"value": v, "unit": "videos/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# --------------------------------------------------------------------------------------------- NMS sweep
def nms_sweep(dev):
    """BASELINE.json configs[3]: hard and soft NMS over N = 1k ... 100k candidate segments of one video (SURVEY 8d:
    centres U(0,768), lengths U(0.01,40), scores U(0,1)): GPU time of avdf_nms_hard / avdf_nms_soft (CUDA events, warm,
    full pick lists like nms_1d_cpu) next to the CPU time of the oracle's C port of nms_cpu.cpp on the host."""
    import torch
    from audio_visual_deepfake_detection_b200 import ops
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import nms_ref
    out = {}
    for n in (1000, 1512, 10000, 100000):
        rng = np.random.RandomState(7000 + n)
        c = rng.uniform(0, 768, n).astype(np.float32); ln = rng.uniform(0.01, 40, n).astype(np.float32)
        segs = np.stack([c - ln / 2, c + ln / 2], 1).astype(np.float32); sc = rng.uniform(0, 1, n).astype(np.float32)
        keep = sc > 0.2
        hs, hp = np.ascontiguousarray(segs[keep]), np.ascontiguousarray(sc[keep])      # NMSop pre-filter (nms.py:15-19)
        d_hs, d_hp = torch.from_numpy(hs).to(dev), torch.from_numpy(hp).to(dev)
        d_s, d_p = torch.from_numpy(segs).to(dev), torch.from_numpy(sc).to(dev)
        dets = torch.zeros((n, 3), device=dev)
        res = {}
        for kind in ("hard", "soft"):
            fn = (lambda: ops.nms_hard(d_hs, d_hp, 0.1)) if kind == "hard" else (lambda: ops.nms_soft(d_s, d_p, dets, 0.1, 0.75, 0.2, 2))
            got = fn()
            torch.cuda.synchronize()
            reps = 3 if n >= 100000 else 10
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record(); torch.cuda.synchronize()
            gpu_us = 1000.0 * e0.elapsed_time(e1) / reps
            t0 = time.perf_counter()
            if kind == "hard":
                want = nms_ref.nms(hs, hp, 0.1)
            else:
                want, _ = nms_ref.softnms(segs, sc, 0.1, 0.75, 0.2, 2)
            cpu_ms = 1000.0 * (time.perf_counter() - t0)
            res[kind] = {"gpu_us": gpu_us, "cpu_ms": cpu_ms, "picks": int(len(want)),
                         "bit_equal": bool(np.array_equal(got.cpu().numpy(), want))}
            if n <= 1512:
                # the product's shape: ONE launch of the fused postprocess kernel over a batch of videos, one CTA per video
                # (NMS + voting + the final sort, max_seg_num 100 like the shipped test_cfg) - 148 copies of this list
                B = 148
                cs = d_s[None].repeat(B, 1, 1).contiguous(); cc = d_p[None].repeat(B, 1).contiguous()
                cn = torch.full((B,), n, dtype=torch.int32, device=dev)
                osg = torch.zeros((B, 100, 2), device=dev); osc = torch.zeros((B, 100), device=dev)
                ocn = torch.zeros(B, dtype=torch.int32, device=dev)
                bf = lambda: ops.postprocess(B, cand_segs=cs, cand_scores=cc, cand_count=cn, iou_threshold=0.1, min_score=0.2, sigma=0.75,   # noqa: E731
                                             voting_thresh=0.9, max_seg_num=100, use_soft_nms=(kind == "soft"), out_segs=osg,
                                             out_scores=osc, out_count=ocn)
                bf(); torch.cuda.synchronize()
                e0.record()
                for _ in range(10):
                    bf()
                e1.record(); torch.cuda.synchronize()
                res[kind]["batched_148_videos_us_per_video"] = 1000.0 * e0.elapsed_time(e1) / 10 / B
        out[str(n)] = res
    out["note"] = ("gpu_us: one list per launch, full pick list like nms_1d_cpu (N <= 6144: one CTA in shared memory; larger: a cluster of "
                   "16 CTAs, the working arrays distributed over their shared memory); batched_148_videos_us_per_video: the fused "
                   "postprocess kernel, one CTA per video, 100 picks + voting; cpu_ms: oracle/nms_ref.c (port of nms_cpu.cpp), one core")
    return out


def byola_extractor_bench(dev):
    """SURVEY 8(f).4: the BYOL-A extractor in front of the path (wav -> [T, 2048] features), 32 clips of AV-Deepfake1M
    lengths per batch: device-resident (wav in HBM, CUDA events), end to end from host arrays (pinned staging + copy inside
    `extract`), the per-kernel times of one batch, the CPU oracle (torch CPU fp32, one clip per call like the reference
    script) on a bounded sample, and the parity of the sampled clips."""
    import torch
    from audio_visual_deepfake_detection_b200 import ops
    from audio_visual_deepfake_detection_b200.libs.features import AudioNTT2020Task6, BatchPlan, LogMelSpectrogram
    from audio_visual_deepfake_detection_b200.libs.utils import synthetic as syn
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import byola_ref
    sd = syn.synthetic_byola_state_dict(0)
    m = AudioNTT2020Task6(n_mels=64, d=2048, precision="mixed").load_state_dict(sd).to(dev).eval()
    durs = syn.sample_durations(8 * 32, seed=4321)
    batches = [[syn.synthetic_wav(int(16000 * d), 9000 + 32 * b + i) for i, d in enumerate(durs[32 * b:32 * b + 32])] for b in range(8)]
    mel = LogMelSpectrogram(dev)
    plans = [BatchPlan([w.shape[0] for w in bt], dev) for bt in batches]
    d_wavs = [torch.from_numpy(np.concatenate(bt)).to(dev) for bt in batches]

    def resident():
        for w, pl in zip(d_wavs, plans):
            m.forward_packed(mel.packed(w, pl), pl)
    for _ in range(2):
        resident()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 5
    e0.record()
    for _ in range(reps):
        resident()
    e1.record(); torch.cuda.synchronize()
    res_ms = e0.elapsed_time(e1) / reps / len(batches)
    for bt in batches:                     # warm-up of the host path (pinned staging buffer at its final size)
        m.extract(bt)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(2):
        for bt in batches:
            outs = m.extract(bt)
    torch.cuda.synchronize()
    e2e_ms = 1000.0 * (time.perf_counter() - t0) / 2 / len(batches)
    # per-kernel times of one batch
    ops.Profile.on = True; ops.Profile.records = []
    m.forward_packed(mel.packed(d_wavs[0], plans[0]), plans[0])
    torch.cuda.synchronize()
    ops.Profile.on = False
    kern = {}
    for name, work, a, b in ops.Profile.records:
        if "k" in (work or {}):
            name = "%s[k=%d,n=%d]" % (name, work["k"], work["n"])
        k = kern.setdefault(name, {"us": 0.0, "launches": 0, "gflop": 0.0, "mb": 0.0})
        k["us"] += 1000.0 * a.elapsed_time(b); k["launches"] += 1
        k["gflop"] += (work or {}).get("flops", 0.0) / 1e9; k["mb"] += (work or {}).get("bytes", 0.0) / 1e6
    ops.Profile.records = []
    for k in kern.values():
        k["tflops"] = k["gflop"] / k["us"] * 1e3 if k["gflop"] else None
        k["gbs"] = k["mb"] / k["us"] * 1e3 if k["us"] else None
    # CPU oracle + parity on a bounded sample (one clip per call, all host threads)
    n_cpu = 6
    t0 = time.perf_counter()
    want = [byola_ref.extract(w, sd) for w in batches[0][:n_cpu]]
    cpu_s = time.perf_counter() - t0
    got = m.extract(batches[0])
    err = max(float(np.abs(g.cpu().numpy() - w).max() / np.abs(w).max()) for g, w in zip(got, want))
    secs = float(np.sum(durs)) / len(batches)
    return {"workload": "BYOL-A AudioNTT2020Task6 (d = 2048) on 16 kHz audio, 32 clips per batch, AV-Deepfake1M durations (mean %.1f s)" % (secs / 32),
            "value": 32.0 / res_ms * 1e3, "unit": "clips/s", "ms_per_batch": res_ms, "audio_seconds_per_second": secs / res_ms * 1e3,
            "e2e": {"value": 32.0 / e2e_ms * 1e3, "unit": "clips/s", "note": "host float arrays in, device features out (pageable -> pinned -> H2D inside extract)"},
            "kernels": kern, "precision": "mixed (fp16 operands, fp32 accumulate; log-mel and conv1 in fp32)",
            "cpu_baseline": {"value": n_cpu / cpu_s, "unit": "clips/s", "cores": os.cpu_count(), "kind": "port",
                             "sample": "%d clips, oracle/byola_ref.py (numpy FFT + torch CPU fp32), one clip per call" % n_cpu},
            "parity": {"max_rel_err_vs_oracle": err, "bar": 1e-2, "clips": n_cpu}}


# --------------------------------------------------------------------------------------------- our arm
BATCHES_PER_STEP = 32        # one step = 4 passes over the 8-batch pool = 1024 videos per GPU


def measure_workload(args, workload, steps, rank, world, local, dist, full):
    """Resident value + e2e of one workload. full: also the pageable-input e2e leg, the per-kernel pass, clocks."""
    import torch
    from audio_visual_deepfake_detection_b200 import native, ops
    from audio_visual_deepfake_detection_b200.libs.modeling import make_meta_arch
    from audio_visual_deepfake_detection_b200.libs.utils import synthetic as syn

    dev = torch.device("cuda", local)
    cfg, name, use_video, desc = build_cfg(workload)
    model = make_meta_arch(cfg["model_name"], **cfg["model"], precision=args.precision, max_batch=BATCH)
    model.load_state_dict(syn.synthetic_state_dict(cfg["model"], name, seed=0))
    model.to(dev).eval()
    K = int(cfg["test_cfg"]["max_seg_num"])
    rec_w = 3 + 3 * K                           # [video index, count, video_cls, scores[K], segs[K,2]] as fp32

    raw = make_raw_batches(N_POOL, use_video, seed0=11 + rank)
    packed = [model.pack_streams(b) for b in raw]
    staged = [model.stage(p) for p in packed]
    n_batches = steps * BATCHES_PER_STEP
    # result records: written by the postprocess kernel itself into a device ring (one row per video), all-gathered once
    ring = torch.zeros((n_batches * BATCH, rec_w), dtype=torch.float32, device=dev)
    counter = torch.zeros(1, dtype=torch.int32, device=dev)
    for i, s_ in enumerate(staged):
        s_["records"] = (ring, counter)
        s_["vidx"] = torch.arange(BATCH, dtype=torch.int32, device=dev) + (rank * N_POOL + i) * BATCH
    torch.cuda.synchronize()
    h2d = int(np.mean([model.h2d_bytes(p) for p in packed]))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def gather():
        if world > 1:
            out = torch.empty((world * ring.shape[0], rec_w), dtype=torch.float32, device=dev)
            dist.all_gather_into_tensor(out, ring)
            return out
        return ring

    # ---------------- device-resident throughput ----------------
    # n_lanes batches are in flight at once, each on its own stream and buffer set: while one batch is in the
    # small pyramid levels (6..48 CTAs on 148 SMs) the other fills the idle SMs
    n_lanes = max(1, args.lanes)
    if args.no_graph:
        class _Eager:
            def __init__(self, st, lane): self.st, self.lane = st, lane
            def replay(self): return model.run_staged(self.st, self.lane)
        passes = [_Eager(s_, i % n_lanes) for i, s_ in enumerate(staged)]
    else:
        # one CUDA graph per resident input batch; batch i runs on lane (buffer set) i % n_lanes
        passes = [model.capture(s_, lane=i % n_lanes) for i, s_ in enumerate(staged)]
    lanes = [torch.cuda.Stream() for _ in range(n_lanes)]

    def run_batches(n):
        main = torch.cuda.current_stream()
        for s_ in lanes:
            s_.wait_stream(main)
        for i in range(n):
            with torch.cuda.stream(lanes[i % n_lanes]):
                passes[i % N_POOL].replay()
        for s_ in lanes:
            main.wait_stream(s_)

    sampler = ClockSampler(local) if (rank == 0 and full) else None
    run_batches(max(args.warmup * N_POOL, 2 * N_POOL))
    gather()
    if sampler:
        sampler.wait_ready()
    counter.zero_()
    barrier()
    if sampler:
        sampler.mark()                  # clocks are sampled (20 ms period) from here on, i.e. under the timed load
    native.LAUNCHES["n"] = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run_batches(n_batches)
    allrec = gather()
    e1.record()
    barrier()
    launches = native.LAUNCHES["n"]
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    clocks = sampler.stop() if sampler else None
    value = world * n_batches * BATCH / (ms / 1000.0)
    assert int(counter.item()) == n_batches * BATCH and allrec.shape[0] == world * n_batches * BATCH
    assert bool((ring[:, 1] >= 0).all()) and float(ring[:, 1].max()) <= K
    last_step = None
    if full and args.dump_outputs:
        # every step replays the same pool of batches, so the last step computed one result per pool video of every rank.
        # The lanes append records in whatever order they finish and a step's last records can land after the next
        # step's first ones: keep one row per video index over all timed rows (rows sorted by index, then contents).
        rows = allrec.cpu().numpy()
        rows = rows[np.lexsort(rows.T[::-1])]
        last_step = rows[np.unique(rows[:, 0], return_index=True)[1]]

    # ---------------- end to end through the public API (host buffers) ----------------
    # model.stream(batches): host numpy arrays in, host tensors out; every step packs its videos into pinned
    # memory, copies them H2D, replays the pass and reads the results back D2H - all inside the timed region.
    # Two measurements of the same call: (1) the inputs sit in PINNED host memory (the state the contract's e2e starts
    # from - a loader that reads the .npy files into a page-locked pool): the copy engine reads them in place;
    # (2) the inputs are ordinary pageable numpy arrays: one host-side gather into pinned staging per batch first.
    for s_ in staged:
        s_.pop("records", None)
    runner = model.runner()
    runner.use_graph = not args.no_graph

    def e2e_leg(pool):
        for _ in model.stream(pool[i % N_POOL] for i in range(max(args.warmup * N_POOL, 2 * len(runner.slots)))):   # every slot captures its graph here
            pass
        barrier()
        runner.h2d_bytes = runner.d2h_bytes = 0
        t0 = time.perf_counter()
        n_out = 0
        for out in model.stream(pool[i % N_POOL] for i in range(n_batches)):
            n_out += len(out)
        torch.cuda.synchronize()
        dt = torch.tensor([time.perf_counter() - t0], device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        return world * n_out / float(dt.item()), runner.h2d_bytes // steps, runner.d2h_bytes // steps
    e2e_pageable = e2e_leg(raw)[0] if full else None
    e2e_value, h2d_step, d2h_step = e2e_leg(pin_batches(raw))
    # (3) the opt-in 16-bit feature-shard format (streaming.bf16_shard: the raw streams stored as bf16): half the bytes over PCIe
    e2e_shard = None
    if full:
        from audio_visual_deepfake_detection_b200.libs.modeling.streaming import bf16_shard
        shard = [[{**c, "streams": {k: bf16_shard(a) for k, a in c["streams"].items()}} for c in chunk] for chunk in raw]
        v_, h_, _ = e2e_leg(pin_batches(shard))
        e2e_shard = {"value": v_, "h2d_bytes_per_step": h_}
    # (4) what the box can deliver: every rank copies one of its pinned batches host -> device back to back for ~1 s, all
    # ranks at once, nothing else on the GPUs (scripts/h2d_ceiling.py is the stand-alone version with per-span copies)
    ceiling = None
    if full:
        pk = packed[0]
        srcs = [t for t in pk["streams"] if t is not None]
        dsts = [torch.empty_like(t, device=dev) for t in srcs]
        nb = sum(t.numel() * t.element_size() for t in srcs)
        cst = torch.cuda.Stream()
        barrier()
        with torch.cuda.stream(cst):
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record(cst)
            t0_, k_ = time.perf_counter(), 0
            while time.perf_counter() - t0_ < 1.0:
                for s_t, d_t in zip(srcs, dsts):
                    d_t.copy_(s_t, non_blocking=True)
                k_ += 1
                if k_ % 8 == 0:
                    cst.synchronize()
            c1.record(cst)
            cst.synchronize()
        gbs = torch.tensor([k_ * nb / (c0.elapsed_time(c1) * 1e-3) / 1e9], device=dev)
        allg = [torch.zeros_like(gbs) for _ in range(world)] if world > 1 else [gbs]
        if world > 1:
            dist.all_gather(allg, gbs)
        per_rank = [round(float(g.item()), 1) for g in allg]
        bpv = nb / BATCH
        ceiling = {"per_rank_gbs": per_rank, "aggregate_gbs": round(sum(per_rank), 1), "bytes_per_video_fp32": bpv,
                   "videos_per_s_fed_fp32": round(sum(per_rank) * 1e9 / bpv), "videos_per_s_fed_if_every_rank_waits_for_the_slowest": round(min(per_rank) * world * 1e9 / bpv),
                   "note": "pinned host -> device copies only, all ranks at once, ~1 s: the host-memory / PCIe path of this box; e2e.value (fp32 "
                           "features) cannot exceed it, bf16 shards halve the bytes"}
        del dsts
    res = {"value": value, "ms": ms, "launches": launches, "clocks": clocks, "e2e": e2e_value, "e2e_pageable": e2e_pageable,
           "e2e_shard": e2e_shard, "h2d_ceiling": ceiling,
           "h2d": h2d_step, "d2h": d2h_step, "desc": desc, "cfg": cfg, "name": name, "n_lanes": n_lanes, "h2d_batch": h2d,
           "last_step": last_step, "K": K}
    if not full:
        return res, None

    # ---------------- per-kernel timing (instrumented pass, not part of the numbers above) ----------------
    res["kernels"], res["roof"], res["step_roof_ms"] = {}, None, None
    if rank == 0:
        ops.Profile.on, ops.Profile.records = True, []
        psteps = 4
        for i in range(psteps):
            # stall the stream (~20 ms) so the host can enqueue the whole pass: the events then bracket GPU
            # execution only, not Python launch latency
            torch.cuda._sleep(40_000_000)
            model.run_staged(staged[i % N_POOL])
        torch.cuda.synchronize()
        ops.Profile.on = False
        agg = {}
        for nm, work, a, b in ops.Profile.records:
            d = agg.setdefault(nm, {"ms": 0.0, "n": 0, "flops": 0.0, "bytes": 0.0})
            d["ms"] += a.elapsed_time(b); d["n"] += 1
            d["flops"] += work.get("flops", 0.0); d["bytes"] += work.get("bytes", 0.0)
        if args.dump_launches:
            rows = [{"call": nm, "us": 1000.0 * a.elapsed_time(b), **{k: v for k, v in work.items()}} for nm, work, a, b in ops.Profile.records]
            json.dump(rows[-(len(rows) // psteps):], open(args.dump_launches, "w"), indent=0)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
        peak_gbs = peaks.get("hbm_gbs", 6650.0)
        pipe = {}
        try:        # tensor-pipe utilisation per kernel from the committed ncu page (profiles/), not measured live
            pipe = json.load(open(os.path.join(ROOT, "profiles", PIPE_FILE)))["kernels"]
        except Exception:
            pass
        # per-launch roofline time = max(FLOP / tensor peak, algorithmic bytes / HBM peak); summed per kernel and per pass
        for nm, work, a, b in ops.Profile.records:
            agg[nm]["roof_ms"] = agg[nm].get("roof_ms", 0.0) + 1e3 * max(work.get("flops", 0.0) / (peak_tf * 1e12), work.get("bytes", 0.0) / (peak_gbs * 1e9))
        tot = sum(d["ms"] for d in agg.values())
        kernels = res["kernels"]
        for nm, d in agg.items():
            kernels[nm] = {"ms_per_batch": d["ms"] / psteps, "launches_per_batch": d["n"] / psteps, "share": d["ms"] / tot,
                           "tflops": (d["flops"] / (d["ms"] * 1e-3) / 1e12) if d["flops"] else None,
                           "gbs": (d["bytes"] / (d["ms"] * 1e-3) / 1e9) if d["bytes"] else None,
                           "roofline_frac": (d.get("roof_ms", 0.0) / d["ms"]) if d.get("roof_ms") else None}
            if kernels[nm]["tflops"]:
                kernels[nm]["tensor_frac"] = kernels[nm]["tflops"] / peak_tf
            if nm in pipe:
                kernels[nm]["tensor_pipe_pct_ncu"] = pipe[nm]
        for nm, kv in kernels.items():                 # HBM-roofline fraction of the memory-bound kernels (algorithmic bytes)
            if kv["gbs"] and not kv["tflops"]:
                kv["hbm_frac"] = kv["gbs"] / peak_gbs
        # the same fraction on each kernel's LARGEST launch (the level-0 / T = 768 one): the small pyramid levels (12 MB and
        # less per launch) are bound by launch latency, not by a roofline, and pull the all-launch figure down
        big = {}
        for nm, work, a, b in ops.Profile.records:
            key = max(work.get("flops", 0.0) / (peak_tf * 1e12), work.get("bytes", 0.0) / (peak_gbs * 1e9))
            if key > 0:
                cur = big.setdefault(nm, {"roof_s": key, "ms": []})
                if key > cur["roof_s"] * 1.001:
                    cur["roof_s"], cur["ms"] = key, []
                if key > cur["roof_s"] * 0.999:
                    cur["ms"].append(a.elapsed_time(b))
        for nm, v in big.items():
            if nm in kernels and v["ms"]:
                med = sorted(v["ms"])[len(v["ms"]) // 2]
                kernels[nm]["largest_launch"] = {"us": 1000.0 * med, "roofline_frac": v["roof_s"] * 1e3 / med}
        traffic = None
        try:        # DRAM bytes per launch of the GEMM kernel from the committed ncu pass (profiles/), not measured live
            tj = json.load(open(os.path.join(ROOT, "profiles", TRAFFIC_FILE)))["kernels"]["tc::conv_gemm_tc_kernel"]
            traffic = (tj["dram_read_bytes_per_step"] + tj["dram_write_bytes_per_step"]) / tj["launches_per_step"]
        except Exception:
            pass
        g = agg.get("avdf_conv_gemm")
        if g and args.precision != "fp32":
            # dominant kernel = conv_gemm_tc_kernel (largest share of the pass). SURVEY 8(d): the path is a dense contraction
            # workload, i.e. TENSOR bound: achieved = sum of algorithmic FLOP of its launches / sum of their CUDA-event
            # durations, against the sustained bf16 peak. The HBM view of the same launches is kept as secondary keys.
            secs = g["ms"] * 1e-3
            t_tensor = g["flops"] / (peak_tf * 1e12)
            t_hbm = g["bytes"] / (peak_gbs * 1e9)
            res["roof"] = {"bound": "tensor", "kernel": "conv_gemm_tc_kernel", "achieved": g["flops"] / secs / 1e12, "peak": peak_tf,
                           "unit": "TFLOP/s", "frac": t_tensor / secs, "traffic": traffic,
                           "traffic_note": "mean DRAM read+write bytes per launch, ncu pass profiles/%s (audio workload)" % TRAFFIC_FILE,
                           "algorithmic_gflop_per_launch": g["flops"] / g["n"] / 1e9, "algorithmic_bytes_per_launch": g["bytes"] / g["n"],
                           "hbm_gbs": g["bytes"] / secs / 1e9, "hbm_frac": t_hbm / secs,
                           "tensor_pipe_pct_ncu": pipe.get("avdf_conv_gemm"),
                           "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained / hbm_gbs (of measured)" if peaks else "fallback 1.4 PFLOP/s / 6650 GB/s (of fallback)",
                           "launches_per_batch": g["n"] / psteps, "avg_launch_us": 1000.0 * g["ms"] / g["n"]}
        res["step_roof_ms"] = sum(d.get("roof_ms", 0.0) for d in agg.values()) / psteps
        res["peak_tf"] = peak_tf
    return res, model


def run_ours(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL logs (e.g. its version banner when NCCL_DEBUG is set in the image) go to stderr: stdout carries one JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    r, model = measure_workload(args, args.workload, args.steps, rank, world, local, dist, full=True)
    cfg, name = r["cfg"], r["name"]
    n_batches = args.steps * BATCHES_PER_STEP
    gflop = flops_per_video(cfg["model"], name.endswith("THE"), name.endswith("NoNorm")) / 1e9

    line = None
    if rank == 0:
        if args.dump_outputs:
            dump_records(args.dump_outputs, r["last_step"], r["K"])
        ms_step = r["ms"] / args.steps
        line = {"metric": "videos/sec localization inference (fwd+decode+soft-NMS)", "value": r["value"], "unit": "videos/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": {"mixed": "bf16", "fp32": "f32"}[args.precision], "data": "synthetic",
                "config": {"workload": r["desc"], "step": "one step = %d batches of %d videos per GPU (%d passes over the pool of %d resident batches) = %d videos per GPU"
                                                          % (BATCHES_PER_STEP, BATCH, BATCHES_PER_STEP // N_POOL, N_POOL, BATCHES_PER_STEP * BATCH),
                           "videos_per_step_per_gpu": BATCHES_PER_STEP * BATCH, "batch": BATCH, "t": cfg["model"]["max_seq_len"], "nms": "soft",
                           "precision": args.precision + (" (bf16 raw-feature operands, fp16 bounded activations, fp32 accumulate/stream)" if args.precision == "mixed" else ""),
                           "l2": "inputs rotate over %d distinct resident batches (%.0f MB total > 126 MB L2)" % (N_POOL, N_POOL * r["h2d_batch"] / 1e6),
                           "lanes": r["n_lanes"], "launch": "eager (one Python call per kernel)" if args.no_graph else "CUDA graph per resident batch (one cudaGraphLaunch per batch)",
                           "records": "written by the postprocess kernel into a device ring (one fixed-size row per video)",
                           "parallelism": "videos sharded over %d rank(s); one all-gather of result records per run" % world,
                           "gflop_per_video": gflop},
                "e2e": {"value": r["e2e"], "unit": "videos/s", "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"],
                        "inputs": "host numpy arrays in pinned memory (one block per batch, collated stream-major: collate_pinned), copied H2D where they are (model.stream)",
                        "pageable_inputs_value": r["e2e_pageable"],
                        "pageable_inputs_note": "same call on pageable numpy arrays: one host gather (avdf_host_pack) into pinned "
                                                "staging per batch first; bounded by the host cores all ranks share",
                        "h2d_ceiling": r["h2d_ceiling"],
                        "bf16_shards": r["e2e_shard"],
                        "bf16_shards_note": "same call on the opt-in 16-bit feature-shard format (raw streams stored as bf16, pinned, collated): "
                                            "half the PCIe bytes; tests/test_gpu_model.py::test_bf16_feature_shards_and_collated_pinned_batches"},
                "gpu_launches": r["launches"], "clocks": r["clocks"], "roofline": r["roof"],
                "step_roofline": {"tensor_frac": (r["value"] / world) * gflop * 1e9 / (r["peak_tf"] * 1e12),
                                  "min_ms_per_batch": r["step_roof_ms"], "achieved_ms_per_batch": r["ms"] / n_batches,
                                  "frac": r["step_roof_ms"] / (r["ms"] / n_batches),
                                  "note": "tensor_frac: whole-pass algorithmic FLOP/s per GPU over the sustained bf16 peak; frac: sum over the pass's "
                                          "launches of max(FLOP / tensor peak, algorithmic bytes / HBM peak) against the timed pass"},
                "kernels": r["kernels"]}
        if world == 1 and not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            v1, dt1 = cpu_reference(args.workload, max(2, args.ref_videos // 4), 1)
            v, dt_cpu, raw_ref, ref_outs = cpu_reference(args.workload, args.ref_videos, threads, keep_outputs=True)
            line["cpu_baseline"] = {"value": v, "unit": "videos/s", "cores": threads, "kind": "port",
                                    "sample": "%d videos (%.1f s), oracle/model_ref.py + oracle/nms_ref.c, torch CPU fp32, B=1 per call" % (args.ref_videos, dt_cpu),
                                    "one_thread": {"value": v1, "cores": 1, "sample": "%d videos (%.1f s)" % (max(2, args.ref_videos // 4), dt1)}}
            # the oracle's outputs for its timed sample double as the checker of the CUDA path's final sets
            par = {"bar": "final sets after the 0.2 score filter: same membership, start/end within 1e-3 s (BASELINE.json north_star)",
                   "benchmark_weights (cls prior -3: ~1000 of 1512 points above 0.2, every threshold is crowded)": parity_vs_oracle(model, raw_ref, ref_outs)}
            try:
                from audio_visual_deepfake_detection_b200.libs.modeling import make_meta_arch
                from audio_visual_deepfake_detection_b200.libs.utils import synthetic as syn
                sp = make_meta_arch(cfg["model_name"], **cfg["model"], precision=args.precision, max_batch=BATCH)
                sp.load_state_dict(syn.synthetic_state_dict(cfg["model"], name, seed=0, cls_bias=-7.0))
                sp.to(dev).eval()
                _, _, raw_sp, ref_sp = cpu_reference(args.workload, args.ref_videos, threads, keep_outputs=True, cls_bias=-7.0)
                par["sparse_weights (cls prior -7: a handful of segments per video, like a trained detector)"] = parity_vs_oracle(sp, raw_sp, ref_sp)
                del sp
            except Exception as exc:     # the parity object is a report, never a reason to lose the bench line
                par["sparse_weights_error"] = repr(exc)
            par["test"] = "tests/test_gpu_parity_sets.py asserts this over 256 videos x 3 configs x 2 weight sets x hard/soft with the threshold-margin analysis of oracle/parity.py"
            line["parity"] = par
        if world == 1 and not args.no_extra:
            del model
            torch.cuda.empty_cache()
            extra = {}
            for wl in ("av12", "av13", "av5"):
                if wl == args.workload:
                    continue
                rr, _ = measure_workload(args, wl, max(2, args.steps // 4), rank, world, local, dist, full=False)
                extra[wl] = {"workload": rr["desc"], "value": rr["value"], "unit": "videos/s", "e2e": rr["e2e"], "steps": max(2, args.steps // 4),
                             "gflop_per_video": flops_per_video(rr["cfg"]["model"], rr["name"].endswith("THE"), rr["name"].endswith("NoNorm")) / 1e9}
                torch.cuda.empty_cache()
            extra["nms_sweep"] = nms_sweep(dev)
            try:
                extra["byola_extractor"] = byola_extractor_bench(dev)
            except Exception as exc:     # an extra never costs the bench line
                extra["byola_extractor_error"] = repr(exc)
            line["extra"] = extra
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def dump_records(out_dir, rows, K):
    """The timed pass's per-video results (what model.forward_streams returns per video, padded to K segments) as
    out_dir/<name>.npy: video_index, n_segments, video_cls [N]; scores [N, K]; segments [N, K, 2] (seconds)."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"video_index": rows[:, 0], "n_segments": rows[:, 1], "video_cls": rows[:, 2],
              "scores": rows[:, 3:3 + K], "segments": rows[:, 3 + K:3 + 3 * K].reshape(-1, K, 2)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


_REAL_STDOUT = None


def capture_stdout():
    """Everything libraries print to fd 1 (e.g. NCCL's version banner) is re-routed to stderr; the one JSON line goes
    to the original stdout through emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="audio", choices=list(WORKLOADS))
    ap.add_argument("--precision", default="mixed", choices=["mixed", "fp32"])
    ap.add_argument("--ref-videos", type=int, default=24)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the av12 / av13 / av5 / NMS-sweep extras of the single-GPU line")
    ap.add_argument("--lanes", type=int, default=8, help="batches in flight at once (each on its own stream and buffer set)")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from Python instead of replaying CUDA graphs")
    ap.add_argument("--dump-launches", default=None, help="write the per-launch CUDA-event timings of one step to this json")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the per-video results of the last timed step as DIR/<name>.npy (same inputs on every run)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "ours" and args.gpus > 1 and world == 1:
        # convenience: relaunch under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus), "--master-addr",
               "127.0.0.1", "--master-port", "29533", os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    capture_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        if args.warmup < 3:
            args.warmup = 3
        run_ours(args)


if __name__ == "__main__":
    main()
