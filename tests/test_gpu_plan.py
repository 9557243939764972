"""Launch plans on the GPU (libs/modeling/plan.py, csrc/plan.cu): the pass replayed by avdf_session_run is bit-identical
to `model.forward_streams` on the same seeded recordings - every MODEL_CASES arch, mixed and fp32, hard and soft NMS,
batch sizes 1 / 5 / 32, fp32 streams and bf16 feature shards - from a Python-free C caller too; the captured graph reads
its inputs in place; sessions are independent; recording does not depend on input values; the exporter and the runtime
refuse what they cannot run and launch nothing when they refuse."""
import os
import struct
import subprocess

import numpy as np
import pytest
import torch

from make_golden import MODEL_CASES
from audio_visual_deepfake_detection_b200 import native as nv
from audio_visual_deepfake_detection_b200 import ops
from audio_visual_deepfake_detection_b200.libs.core import load_config_for
from audio_visual_deepfake_detection_b200.libs.modeling import make_meta_arch
from audio_visual_deepfake_detection_b200.libs.modeling import plan as pl
from audio_visual_deepfake_detection_b200.libs.modeling.streaming import bf16_shard
from audio_visual_deepfake_detection_b200.libs.utils import synthetic as syn

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BATCHES = (1, 5, 32)


def make_model(case, precision="mixed", nms="hard"):
    model_name, overrides, _, wseed = MODEL_CASES[case]
    cfg = load_config_for(model_name, dict(overrides, **{"test_cfg.nms_method": nms}))
    model = make_meta_arch(cfg["model_name"], **cfg["model"], precision=precision, max_batch=32)
    model.load_state_dict(syn.synthetic_state_dict(cfg["model"], model_name, seed=wseed))
    return model.to("cuda").eval()


def make_items(case, n, seed, shards=False):
    use_video = MODEL_CASES[case][2]
    dims = (256 if use_video else 0, 0 if use_video == "video+emo" else 2048, 768)
    items = pl._synthetic_items(dims, n, seed)
    if shards:
        items = [dict(c, streams={k: bf16_shard(a) for k, a in c["streams"].items()}) for c in items]
    return items


def assert_same(got, want, what):
    assert len(got) == len(want), what
    for g, w in zip(got, want):
        assert g["video_id"] == w["video_id"]
        for k in ("segments", "scores", "video_cls"):
            assert g[k].shape == w[k].shape and torch.equal(g[k], w[k]), "%s: %s %s differs" % (what, w["video_id"], k)


CASES = [(c, "mixed", "hard", False) for c in MODEL_CASES] + [(c, "fp32", "soft", False) for c in MODEL_CASES]
CASES += [("exp12", "mixed", "soft", True)]


@pytest.mark.parametrize("case,precision,nms,shards", CASES,
                         ids=["%s-%s-%s%s" % (c, p, n, "-bf16shards" if s else "") for c, p, n, s in CASES])
def test_session_run_is_bit_identical_to_forward_streams(case, precision, nms, shards, tmp_path):
    model = make_model(case, precision, nms)
    path = model.export_plan(str(tmp_path / "m.plan"), batch_sizes=BATCHES, shards=shards)
    plan = pl.Plan(path)
    try:
        assert plan.info.batch_mask == sum(1 << (b - 1) for b in BATCHES)
        assert ("precision=%s" % precision) in plan.info.description.decode()
        sess = plan.session()
        for i, B in enumerate(BATCHES):
            items = make_items(case, B, 1000 + 100 * i, shards)
            assert_same(sess.run(items), model.forward_streams(items), "%s B=%d" % (case, B))
    finally:
        plan.close()


@pytest.fixture(scope="module")
def exp12(tmp_path_factory):
    model = make_model("exp12")
    path = model.export_plan(str(tmp_path_factory.mktemp("plan") / "exp12.plan"), batch_sizes=BATCHES)
    plan = pl.Plan(path)
    yield model, plan, path
    plan.close()


def test_first_run_and_replays_agree_and_read_inputs_in_place(exp12):
    model, plan, _ = exp12
    sess = plan.session()
    a, b = make_items("exp12", 32, 7), make_items("exp12", 32, 8)
    first = sess.run(a)                       # eager pass, capture, replay
    second = sess.run(b)                      # replay on new input contents
    third = sess.run(a)
    assert_same(third, first, "replay vs first run")
    assert_same(second, model.forward_streams(b), "replay on new inputs")
    assert any(not torch.equal(x["video_cls"], y["video_cls"]) for x, y in zip(first, second))


def test_two_sessions_on_two_streams_match_sequential_runs(exp12):
    _, plan, _ = exp12
    s1, s2 = plan.session(), plan.session()
    a, b = make_items("exp12", 32, 21), make_items("exp12", 5, 22)
    want_a, want_b = s1.run(a), s2.run(b)      # one after the other (also captures both graphs)
    s1.segs.zero_(); s2.segs.zero_()
    torch.cuda.synchronize()
    ra, rb = s1.stage(a), s2.stage(b)
    torch.cuda.synchronize()
    st1, st2 = torch.cuda.Stream(), torch.cuda.Stream()
    for _ in range(3):                         # both in flight at once
        s1.launch(32, ra, st1)
        s2.launch(5, rb, st2)
    torch.cuda.synchronize()
    assert_same(s1.results([c["video_id"] for c in a]), want_a, "session 1")
    assert_same(s2.results([c["video_id"] for c in b]), want_b, "session 2")


def test_recording_does_not_depend_on_input_values():
    model = make_model("audio_only")
    one = pl.encode_plan(*pl.record_plan(model, batch_sizes=(2, 3), items=make_items("audio_only", 3, 1)))
    two = pl.encode_plan(*pl.record_plan(model, batch_sizes=(2, 3), items=make_items("audio_only", 3, 2)))
    assert one == two


def test_export_refusals(tmp_path, monkeypatch):
    model = make_model("audio_only")
    feats = [{"video_id": "x", "feats": torch.zeros(2816, 768), "fps": 25.0, "duration": 4.0, "feat_stride": 1.0,
              "feat_num_frames": 1.0}]
    with pytest.raises(nv.AvdfError, match="'feats' items"):
        model.export_plan(str(tmp_path / "a.plan"), batch_sizes=(1,), items=feats)
    model.test_nms_method = "none"
    with pytest.raises(nv.AvdfError, match="nms_method 'none'"):
        model.export_plan(str(tmp_path / "b.plan"), batch_sizes=(1,))
    model.test_nms_method = "hard"
    orig = ops.conv_gemm

    def foreign_bias(*args, **kw):            # one launch reads a tensor the engine does not own
        if kw.get("bias") is not None and kw.get("taps") == 3 and kw.get("stride") == 2:
            kw["bias"] = kw["bias"].clone()
        return orig(*args, **kw)

    monkeypatch.setattr(ops, "conv_gemm", foreign_bias)
    with pytest.raises(nv.AvdfError, match=r"avdf_conv_gemm field bias: device pointer 0x[0-9a-f]+ is outside"):
        model.export_plan(str(tmp_path / "c.plan"), batch_sizes=(1,))
    assert not any(p.name.startswith("c.plan") for p in tmp_path.iterdir())


def test_session_run_refusals_launch_nothing(exp12):
    _, plan, _ = exp12
    sess = plan.session()
    sess.segs.fill_(-3.0)
    torch.cuda.synchronize()
    rows = list(plan.info.stream_rows)
    bad = [(2, rows, "no launch list for batch size 2"),
           (5, [rows[0] + 1, rows[1], rows[2]], "stream 0: %d rows" % (rows[0] + 1)),
           (33, rows, "no launch list for batch size 33")]
    for B, r, msg in bad:
        with pytest.raises(nv.AvdfError, match=msg):
            sess.launch(B, r)
    torch.cuda.synchronize()
    assert bool((sess.segs == -3.0).all())


def test_c_driver_without_python_matches_forward_streams(exp12, tmp_path):
    model, _, path = exp12
    exe = tmp_path / "plan_driver"
    csrc = os.path.join(ROOT, "audio_visual_deepfake_detection_b200", "csrc")
    subprocess.run(["/usr/local/cuda/bin/nvcc" if os.path.exists("/usr/local/cuda/bin/nvcc") else "nvcc", "-O2", "-Wno-deprecated-gpu-targets",
                    "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "plan_driver.c"), "-o", str(exe),
                    "-L", csrc, "-lavdf_sm100", "-Xlinker", "-rpath", "-Xlinker", csrc], check=True)
    items = make_items("exp12", 5, 31)
    B = len(items)
    blob = [struct.pack("<i", B)]
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
    b_, K = struct.unpack("<2i", raw[:8])
    assert b_ == B
    o = 8
    segs = np.frombuffer(raw, np.float32, B * K * 2, o).reshape(B, K, 2); o += B * K * 8
    scores = np.frombuffer(raw, np.float32, B * K, o).reshape(B, K); o += B * K * 4
    counts = np.frombuffer(raw, np.int32, B, o); o += B * 4
    vcls = np.frombuffer(raw, np.float32, B, o)
    got = [{"video_id": c["video_id"], "segments": torch.from_numpy(segs[b, :counts[b]].copy()),
            "scores": torch.from_numpy(scores[b, :counts[b]].copy()), "video_cls": torch.from_numpy(vcls[b:b + 1].copy())}
           for b, c in enumerate(items)]
    assert_same(got, model.forward_streams(items), "C driver")
