"""Sliding windows on launch plans (avdf_session_attach_windows / avdf_session_run_windows, csrc/plan.cu) on the GPU:
bit-identical to `model.forward_streams(items, window=W, hop=H)` on the same seeded recordings - every MODEL_CASES arch,
mixed / hard and fp32 / soft, bf16 shards, (W, H) = (10, 5) and (30, 12.5), 40 s to 10 min recordings mixed with ones
shorter than W, more recordings than max_batch, a plan with every batch size and one with only 32 (padded last batch) -
from a Python-free C caller too; graphs replay on new inputs; sessions on two streams are independent; windowed and
plain runs interleave on one session; refusals launch nothing."""
import ctypes
import os
import struct
import subprocess

import numpy as np
import pytest
import torch

from make_golden import MODEL_CASES
from test_plan_windows import write_plan
from audio_visual_deepfake_detection_b200 import native as nv
from audio_visual_deepfake_detection_b200.libs.core import load_config_for
from audio_visual_deepfake_detection_b200.libs.modeling import make_meta_arch
from audio_visual_deepfake_detection_b200.libs.modeling import plan as pl
from audio_visual_deepfake_detection_b200.libs.modeling.streaming import bf16_shard
from audio_visual_deepfake_detection_b200.libs.utils import synthetic as syn

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BATCHES = (1, 5, 32)
WH = ((10.0, 5.0), (30.0, 12.5))
LONG = (600.0, 7.42, 45.0, 3.9, 130.0, 40.0, 25.0)     # seconds: long recordings mixed with ones shorter than W


def make_model(case, precision="mixed", nms="hard"):
    model_name, overrides, _, wseed = MODEL_CASES[case]
    cfg = load_config_for(model_name, dict(overrides, **{"test_cfg.nms_method": nms}))
    model = make_meta_arch(cfg["model_name"], **cfg["model"], precision=precision, max_batch=32)
    model.load_state_dict(syn.synthetic_state_dict(cfg["model"], model_name, seed=wseed))
    return model.to("cuda").eval()


def dims(case):
    use_video = MODEL_CASES[case][2]
    return (256 if use_video else 0, 0 if use_video == "video+emo" else 2048, 768)


def recordings(case, durations, seed, shards=False):
    d = dims(case)
    items = [{"video_id": "w%d_%d" % (seed, i), "duration": float(D),
              "streams": syn.synthetic_streams(float(D), seed + i, video_dim=d[0], byola_dim=d[1], emo_dim=d[2])}
             for i, D in enumerate(durations)]
    if shards:
        items = [dict(c, streams={k: bf16_shard(a) for k, a in c["streams"].items()}) for c in items]
    return items


def assert_same(got, want, what):
    assert len(got) == len(want), what
    for g, w in zip(got, want):
        assert g["video_id"] == w["video_id"]
        assert g["segments"].shape == w["segments"].shape, "%s: %s segment count" % (what, w["video_id"])
        for k in ("segments", "scores", "video_cls"):
            assert torch.equal(g[k], w[k]), "%s: %s %s differs" % (what, w["video_id"], k)


CASES = [(c, "mixed", "hard", False) for c in MODEL_CASES] + [(c, "fp32", "soft", False) for c in MODEL_CASES]
CASES += [("exp12", "mixed", "soft", True)]


@pytest.mark.parametrize("case,precision,nms,shards", CASES,
                         ids=["%s-%s-%s%s" % (c, p, n, "-bf16shards" if s else "") for c, p, n, s in CASES])
def test_run_windows_is_bit_identical_to_forward_streams(case, precision, nms, shards, tmp_path):
    model = make_model(case, precision, nms)
    plan = pl.Plan(model.export_plan(str(tmp_path / "m.plan"), batch_sizes=BATCHES, shards=shards))
    try:
        sess = plan.session()
        sess.attach_windows(512, 128)
        items = recordings(case, LONG, 300, shards)
        for W, H in WH:
            got = sess.run_windows(items, W, H)
            assert_same(got, model.forward_streams(items, window=W, hop=H), "%s W=%g H=%g" % (case, W, H))
        assert sum(int(r["scores"].numel()) for r in got) > 0
    finally:
        plan.close()


@pytest.fixture(scope="module")
def exp12(tmp_path_factory):
    model = make_model("exp12", "mixed", "soft")
    d = tmp_path_factory.mktemp("wplan")
    every = pl.Plan(model.export_plan(str(d / "every.plan")))                       # batch sizes 1 .. 32
    only32 = pl.Plan(model.export_plan(str(d / "only32.plan"), batch_sizes=(32,)))
    yield model, every, only32, str(d / "every.plan")
    every.close()
    only32.close()


def test_every_batch_size_and_padded_batches(exp12):
    model, every, only32, _ = exp12
    items = recordings("exp12", LONG, 400)
    for plan in (every, only32):
        sess = plan.session()
        sess.attach_windows(512, 128)
        for W, H in WH:
            assert_same(sess.run_windows(items, W, H), model.forward_streams(items, window=W, hop=H),
                        "batch mask %#x W=%g" % (plan.info.batch_mask, W))


def test_more_recordings_than_max_batch(exp12):
    model, every, only32, _ = exp12
    items = recordings("exp12", list(syn.sample_durations(38, 5)) + [95.0, 61.0], 500)
    for plan in (every, only32):
        sess = plan.session()
        sess.attach_windows(256, 32)
        assert_same(sess.run_windows(items, 10.0), model.forward_streams(items, window=10.0, hop=5.0),
                    "40 recordings, batch mask %#x" % plan.info.batch_mask)


def test_replays_read_new_inputs_in_place(exp12):
    model, every, _, _ = exp12
    sess = every.session()
    sess.attach_windows(512, 128)
    a, b = recordings("exp12", LONG, 600), recordings("exp12", (77.0, 12.0, 300.0), 700)
    first = sess.run_windows(a, 10.0, 5.0)                  # eager passes, captures, replays
    second = sess.run_windows(b, 10.0, 5.0)                 # replays on new staging contents and a new table
    third = sess.run_windows(a, 10.0, 5.0)
    assert_same(third, first, "replay vs first call")
    assert_same(second, model.forward_streams(b, window=10.0, hop=5.0), "replay on new inputs")
    assert_same(first, model.forward_streams(a, window=10.0, hop=5.0), "first call")


def _outs(R, K):
    return (torch.full((R, K, 2), -3.0, device="cuda"), torch.full((R, K), -3.0, device="cuda"),
            torch.full((R,), -3, dtype=torch.int32, device="cuda"), torch.full((R,), -3.0, device="cuda"))


def _results(items, outs):
    torch.cuda.synchronize()
    segs, scores, counts, vcls = (t.cpu() for t in outs)
    return [{"video_id": c["video_id"], "segments": segs[r, :int(counts[r])], "scores": scores[r, :int(counts[r])],
             "video_cls": vcls[r:r + 1]} for r, c in enumerate(items)]


def test_two_sessions_on_two_streams_match_sequential_runs(exp12):
    _, every, _, _ = exp12
    K = every.info.max_seg_num
    s1, s2 = every.session(), every.session()
    s1.attach_windows(512, 128)
    s2.attach_windows(512, 128)
    a, b = recordings("exp12", LONG, 800), recordings("exp12", (240.0, 5.0, 33.0, 71.5), 900)
    want_a, want_b = s1.run_windows(a, 10.0, 5.0), s2.run_windows(b, 10.0, 5.0)
    ra = [[c["streams"][n].shape[0] if n in c["streams"] else 0 for n in pl.STREAM_NAMES] for c in a]
    rb = [[c["streams"][n].shape[0] if n in c["streams"] else 0 for n in pl.STREAM_NAMES] for c in b]
    with torch.cuda.stream(s1.stream):
        pl._stage_streams(a, s1.streams)
    with torch.cuda.stream(s2.stream):
        pl._stage_streams(b, s2.streams)
    torch.cuda.synchronize()
    oa, ob = _outs(len(a), K), _outs(len(b), K)
    st1, st2 = torch.cuda.Stream(), torch.cuda.Stream()
    for _ in range(3):                                      # both in flight at once
        s1.launch_windows([c["duration"] for c in a], ra, 10.0, 5.0, oa, st1)
        s2.launch_windows([c["duration"] for c in b], rb, 10.0, 5.0, ob, st2)
    torch.cuda.synchronize()
    assert_same(_results(a, oa), want_a, "session 1")
    assert_same(_results(b, ob), want_b, "session 2")


def test_interleaved_plain_and_windowed_runs(exp12):
    model, every, _, _ = exp12
    sess = every.session()
    sess.attach_windows(512, 128)
    short, long = pl._synthetic_items(dims("exp12"), 5, 1100), recordings("exp12", (150.0, 9.0), 1200)
    want_short, want_long = model.forward_streams(short), model.forward_streams(long, window=30.0, hop=12.5)
    for _ in range(2):
        assert_same(sess.run(short), want_short, "plain run")
        assert_same(sess.run_windows(long, 30.0, 12.5), want_long, "windowed run")


def test_refusals_launch_nothing(exp12):
    _, every, _, _ = exp12
    info, L = every.info, every.L
    K = info.max_seg_num
    bare = every.session()
    sess = every.session()
    sess.attach_windows(64, 20)
    items = recordings("exp12", (100.0, 20.0), 1300)
    with torch.cuda.stream(sess.stream):
        pl._stage_streams(items, sess.streams)
    torch.cuda.synchronize()
    rows = [[c["streams"][n].shape[0] for n in pl.STREAM_NAMES] for c in items]
    durs = [c["duration"] for c in items]
    outs = _outs(2, K)
    big = rows[0][:1] + [int(info.stream_rows[1])] + rows[0][2:]
    bad = [(bare, durs, rows, 10.0, 5.0, "has no window block"),
           (sess, [], [], 10.0, 5.0, "n_rec is 0"),
           (sess, durs, rows, 0.0, 0.0, "window must be > 0"),
           (sess, durs, rows, 10.0, 12.0, "hop must satisfy"),
           (sess, [1000.0, 20.0], [[rows[0][0], 3, rows[0][2]], rows[1]], 10.0, 5.0, "holds no row of stream 1"),
           (sess, durs, [[0] + rows[0][1:], rows[1]], 10.0, 5.0, "stream 0 is present in the plan but has 0 rows"),
           (sess, durs, [big, rows[1]], 10.0, 5.0, "stream 1: %d rows, the staging holds" % (big[1] + rows[1][1])),
           (sess, durs, rows, 10.0, 1.0, "recording 0 has 91 windows, the window block holds 20 per recording"),
           (sess, [100.0] * 4, rows * 2, 10.0, 5.0, "76 windows, the window block holds 64")]
    for s, d, r, W, H, msg in bad:
        with pytest.raises(nv.AvdfError, match=msg):
            s.launch_windows(d, r, W, H, outs)
    a = nv.WindowRunArgs()
    dur = (ctypes.c_double * 2)(*durs)
    rw = (ctypes.c_int64 * 6)(*[v for r in rows for v in r])
    a.n_rec, a.duration, a.rows, a.window, a.hop = 2, dur, rw, 10.0, 5.0
    a.out_segs, a.out_scores, a.out_count, a.out_cls = (t.data_ptr() for t in outs)
    assert L.avdf_session_run_windows(sess.h, ctypes.byref(a), None) == -1
    assert b"legacy default stream" in L.avdf_last_error()
    torch.cuda.synchronize()
    for t in outs:
        assert bool((t == -3).all())


def test_attach_refuses_a_plan_that_cannot_run_windows(tmp_path):
    sms, ccma, ccmi = ctypes.c_int32(), ctypes.c_int32(), ctypes.c_int32()
    nv.check(nv.lib().avdf_device_info(ctypes.byref(sms), ctypes.byref(ccma), ctypes.byref(ccmi)))
    from test_plan_windows import ln_rows
    path = write_plan(tmp_path, device=(ccma.value, ccmi.value, sms.value), first=lambda B: ln_rows((4, 4, 4)))
    plan = pl.Plan(str(path))
    try:
        sess = plan.session()
        block = torch.empty(1 << 20, dtype=torch.uint8, device="cuda")
        rc = plan.L.avdf_session_attach_windows(sess.h, block.data_ptr(), block.numel(), 16, 4)
        assert rc == -3
        assert plan.L.avdf_last_error().decode() == ("avdf_session_attach_windows: the launch list for batch 1 does not "
                                                     "start with avdf_interp_concat_in (it starts with avdf_ln_rows)")
        with pytest.raises(nv.AvdfError, match=r"avdf_session_window_bytes: the launch list for batch 1 does not start "
                                               r"with avdf_interp_concat_in"):
            sess.attach_windows(16, 4)            # PlanSession sizes the block first: the same check refuses
        assert sess.win_block is None
    finally:
        plan.close()


def test_c_driver_without_python_matches_forward_streams(exp12, tmp_path):
    model, _, _, path = exp12
    exe = tmp_path / "plan_window_driver"
    csrc = os.path.join(ROOT, "audio_visual_deepfake_detection_b200", "csrc")
    subprocess.run(["/usr/local/cuda/bin/nvcc" if os.path.exists("/usr/local/cuda/bin/nvcc") else "nvcc", "-O2", "-Wno-deprecated-gpu-targets",
                    "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "plan_window_driver.c"), "-o", str(exe),
                    "-L", csrc, "-lavdf_sm100", "-Xlinker", "-rpath", "-Xlinker", csrc], check=True)
    items = recordings("exp12", LONG, 1400)
    R, W, H = len(items), 30.0, 12.5
    blob = [struct.pack("<i2d", R, W, H)]
    for c in items:
        blob.append(struct.pack("<d3q", c["duration"], *[c["streams"][n].shape[0] for n in pl.STREAM_NAMES]))
    for n in pl.STREAM_NAMES:
        blob += [np.ascontiguousarray(c["streams"][n], np.float32).tobytes() for c in items]
    (tmp_path / "in.bin").write_bytes(b"".join(blob))
    env = {k: v for k, v in os.environ.items() if not k.startswith("PYTHON")}
    r = subprocess.run([str(exe), path, str(tmp_path / "in.bin"), str(tmp_path / "out.bin")], env=env,
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    raw = (tmp_path / "out.bin").read_bytes()
    r_, K = struct.unpack("<2i", raw[:8])
    assert r_ == R
    o = 8
    segs = np.frombuffer(raw, np.float32, R * K * 2, o).reshape(R, K, 2); o += R * K * 8
    scores = np.frombuffer(raw, np.float32, R * K, o).reshape(R, K); o += R * K * 4
    counts = np.frombuffer(raw, np.int32, R, o); o += R * 4
    vcls = np.frombuffer(raw, np.float32, R, o)
    got = [{"video_id": c["video_id"], "segments": torch.from_numpy(segs[b, :counts[b]].copy()),
            "scores": torch.from_numpy(scores[b, :counts[b]].copy()), "video_cls": torch.from_numpy(vcls[b:b + 1].copy())}
           for b, c in enumerate(items)]
    assert_same(got, model.forward_streams(items, window=W, hop=H), "C driver")
