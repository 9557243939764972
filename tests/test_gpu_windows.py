"""Sliding-window inference over long recordings (libs/modeling/windows.py, csrc/window.cu, avdf_interp_concat_ranges):
the range resampling against the CSR kernel, and the windowed API against the composition oracle (host-sliced windows
through today's forward_streams, merged by oracle/window_ref.py with the reference's batched_nms), bit for bit."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import window_ref
from audio_visual_deepfake_detection_b200 import ops
from audio_visual_deepfake_detection_b200.libs.core import load_config_for
from audio_visual_deepfake_detection_b200.libs.datasets import make_inference_dataset
from audio_visual_deepfake_detection_b200.libs.modeling import EXP12, make_meta_arch
from audio_visual_deepfake_detection_b200.libs.modeling.streaming import bf16_shard
from audio_visual_deepfake_detection_b200.native import AvdfError
from audio_visual_deepfake_detection_b200.libs.utils import synthetic as syn

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
AUDIO = {"dataset.video_input_dim": 0}


@pytest.fixture(scope="module")
def model():
    cfg = load_config_for(EXP12, AUDIO)
    m = make_meta_arch(cfg["model_name"], **cfg["model"], max_batch=8)
    m.load_state_dict(syn.synthetic_state_dict(cfg["model"], EXP12, seed=3))
    m.to("cuda").eval()
    saved = m.test_key()
    yield m
    for k, v in zip(m._TEST_ATTRS, saved):
        setattr(m, "test_" + k, v)


def rec(dur, seed, video=False):
    return {"video_id": "r%d" % seed, "duration": dur, "streams": syn.synthetic_streams(dur, seed, video_dim=256 if video else 0)}


def same(a, b):
    assert a["segments"].shape == b["segments"].shape, (a["segments"].shape, b["segments"].shape)
    assert torch.equal(a["segments"].reshape(-1, 2), b["segments"].reshape(-1, 2))
    assert torch.equal(a["scores"], b["scores"])
    assert torch.equal(a["video_cls"].reshape(-1), b["video_cls"].reshape(-1))


# ---------------------------------------------------------------- range resampling
@pytest.mark.parametrize("shard", [False, True])
@pytest.mark.parametrize("out_dt", [torch.float32, torch.bfloat16, torch.float16])
def test_interp_ranges_equal_csr_on_sliced_copies(shard, out_dt):
    dev = torch.device("cuda")
    recs = [syn.synthetic_streams(d, 700 + i) for i, d in enumerate((61.3, 15.0, 40.0))]
    names = ("video", "byola", "emo")
    # (recording, start row, rows) per stream: overlapping windows, windows ending at the stream end, count == 768
    wins = []
    for r, st in enumerate(recs):
        T = [st[n].shape[0] for n in names]
        wins += [(r, [0] * 3, [t // 3 for t in T]), (r, [t // 6 for t in T], [t // 3 for t in T]),
                 (r, [t - t // 4 for t in T], [t // 4 for t in T])]
    T0 = [recs[0][n].shape[0] for n in names]
    wins.append((0, [0, 0, T0[2] - 768], [T0[0] // 2, T0[1] // 2, 768]))
    conv = (lambda a: bf16_shard(a)) if shard else (lambda a: a)
    tdt = torch.bfloat16 if shard else torch.float32

    def tens(a):
        t = torch.from_numpy(np.ascontiguousarray(a))
        return (t.view(torch.bfloat16) if shard else t).to(dev)
    base = np.cumsum([[0] * 3] + [[st[n].shape[0] for n in names] for st in recs], axis=0)
    srcs = [tens(np.concatenate([conv(st[n]) for st in recs])) for n in names]
    start = torch.tensor([[int(base[r][s]) + a[s] for r, a, _ in wins] for s in range(3)], dtype=torch.int32, device=dev)
    count = torch.tensor([[m[s] for _, _, m in wins] for s in range(3)], dtype=torch.int32, device=dev)
    C = sum(x.shape[1] for x in srcs)
    got = torch.empty((len(wins), 768, C), dtype=out_dt, device=dev)
    ops.interp_concat_ranges(srcs, start, count, 768, got)
    # the same windows as host-sliced contiguous copies through the CSR kernel
    cps = [[conv(recs[r][n][a[s]:a[s] + m[s]]) for r, a, m in wins] for s, n in enumerate(names)]
    csr = [tens(np.concatenate(c)) for c in cps]
    offs = [torch.tensor(np.concatenate([[0], np.cumsum([x.shape[0] for x in c])]), dtype=torch.int32, device=dev) for c in cps]
    want = torch.empty_like(got)
    ops.interp_concat(csr, offs, 768, want)
    assert srcs[0].dtype == tdt
    assert torch.equal(got.view(torch.int16) if out_dt != torch.float32 else got.view(torch.int32),
                       want.view(torch.int16) if out_dt != torch.float32 else want.view(torch.int32))


# ---------------------------------------------------------------- the windowed API
def test_recordings_within_the_window_are_unchanged(model):
    recs = [rec(d, 10 + i) for i, d in enumerate((4.03, 9.04, 26.37, 7.42, 30.0, 5.5, 12.0, 8.0, 6.6, 29.9))]
    want = model.forward_streams(recs)
    got = model.forward_streams(recs, window=30.0)
    for a, b in zip(got, want):
        assert a["video_id"] == b["video_id"]
        same(a, b)


CONFIGS = [("hard", 0.0, False), ("hard", 0.9, False), ("soft", 0.0, False), ("soft", 0.75, False), ("soft", 0.9, True)]


@pytest.mark.parametrize("wh", [(10.0, 5.0), (30.0, 12.5)])
@pytest.mark.parametrize("method,voting,multiclass", CONFIGS)
def test_composition_oracle(model, wh, method, voting, multiclass):
    W, H = wh
    model.test_nms_method, model.test_voting_thresh, model.test_multiclass_nms = method, voting, multiclass
    recs = [rec(40.0, 1), rec(600.0, 2), rec(7.42, 3), rec(137.7, 4)]
    got = model.forward_streams(recs, window=W, hop=H)
    want = window_ref.run(model, recs, W, H)
    for a, b in zip(got, want):
        same(a, b)
    assert sum(int(a["scores"].numel()) for a in got) > 0


def test_grouping_does_not_change_results(model):
    model.test_nms_method, model.test_voting_thresh, model.test_multiclass_nms = "soft", 0.75, False
    long = rec(95.0, 21)
    shorts = [rec(d, 30 + i) for i, d in enumerate((4.03, 6.0, 9.5))]
    alone = model.forward_streams([long], window=10.0)[0]
    mixed = model.forward_streams([shorts[0], long, shorts[1], shorts[2]], window=10.0)
    same(mixed[1], alone)
    for s, m in zip(shorts, (mixed[0], mixed[2], mixed[3])):
        same(m, model.forward_streams([s])[0])
    runner = model.runner()
    saved = runner.GROUP_BYTES
    try:
        runner.GROUP_BYTES = 1                  # one recording per group: other batch boundaries, other staging
        split = model.forward_streams([shorts[0], long, shorts[1]], window=10.0)
        runner.use_graph = False
        eager = model.forward_streams([long], window=10.0)[0]
    finally:
        runner.GROUP_BYTES, runner.use_graph = saved, True
    same(split[1], alone)
    same(eager, alone)
    streamed = [r for out in model.stream(iter([[shorts[0]], [long, shorts[1]]]), window=10.0) for r in out]
    same(streamed[1], alone)


def test_bf16_shards_and_audio_visual_streams():
    cfg = load_config_for(EXP12)
    m = make_meta_arch(cfg["model_name"], **cfg["model"], max_batch=4)
    m.load_state_dict(syn.synthetic_state_dict(cfg["model"], EXP12, seed=0))
    m.to("cuda").eval()
    recs = [rec(47.0, 50, video=True), rec(8.0, 51, video=True)]
    same(m.forward_streams(recs, window=12.0, hop=5.0)[0], window_ref.run(m, recs[:1], 12.0, 5.0)[0])
    sh = [{**r, "streams": {k: bf16_shard(a) for k, a in r["streams"].items()}} for r in recs]
    for a, b in zip(m.forward_streams(sh, window=12.0, hop=5.0), window_ref.run(m, sh, 12.0, 5.0)):
        same(a, b)


def test_errors(model):
    r = [rec(40.0, 60)]
    for W, H in ((0.0, None), (10.0, 0.0), (10.0, 11.0), (-5.0, 1.0)):
        with pytest.raises(ValueError):
            model.forward_streams(r, window=W, hop=H)
    with pytest.raises(ValueError):                 # a window with no row of the stream
        model.forward_streams([{"video_id": "x", "duration": 1000.0,
                                "streams": {"byola": np.zeros((3, 2048), np.float32), "emo": np.zeros((50000, 768), np.float32)}}],
                              window=10.0)
    with pytest.raises(AvdfError):
        model.forward_streams([{"video_id": "x", "duration": 40.0, "feats": torch.zeros(2816, 768)}], window=10.0)
    saved = model.test_nms_method
    model.test_nms_method = "none"
    try:
        with pytest.raises(AvdfError):
            model.forward_streams(r, window=10.0)
    finally:
        model.test_nms_method = saved


# ---------------------------------------------------------------- drivers
def write_corpus(root, durs):
    folders = {k: os.path.join(root, k) for k in ("video", "byola", "emo", "lists")}
    for f in folders.values():
        os.makedirs(f, exist_ok=True)
    lines = []
    for i, d in enumerate(durs):
        st = syn.synthetic_streams(d, 80 + i)
        vid = f"id{i:03d}/clip.mp4"
        for k in ("video", "byola", "emo"):
            path = os.path.join(folders[k], vid.replace(".mp4", ".npy"))
            os.makedirs(os.path.dirname(path), exist_ok=True)
            np.save(path, st[k])
        lines.append(f"{vid},{d}")
    with open(os.path.join(folders["lists"], "deepfake_test_sub3.txt"), "w") as f:
        f.write("\n".join(lines) + "\n")
    return folders


def corpus_setup(tmp_path, durs):
    import yaml
    folders = write_corpus(str(tmp_path / "data"), durs)
    cfg = yaml.load(open(os.path.join(ROOT, "configs", "deepfake_exp12_test.yaml")), Loader=yaml.FullLoader)
    cfg["dataset"].update(video_feat_folder=folders["video"], audio_byola_feat_folder=folders["byola"],
                          audio_emo_feat_folder=folders["emo"], test_folder=folders["lists"])
    cfg["loader"] = {"batch_size": 1, "num_workers": 0}
    cfg_path = str(tmp_path / "cfg.yaml")
    yaml.dump(cfg, open(cfg_path, "w"))
    full = load_config_for(EXP12)
    sd = syn.synthetic_state_dict(full["model"], EXP12, seed=0)
    ds = make_inference_dataset("deepfake_video_audioEmoBYOLA_inference", False, ["test"], 3, crop_ratio=None,
                                default_fps=None, downsample_rate=0, video_feat_folder=folders["video"], audio_feat_folder=None,
                                audio_byola_feat_folder=folders["byola"], audio_emo_feat_folder=folders["emo"],
                                audio_file_ext=".npy", num_classes=1, input_dim=0, video_input_dim=256, audio_input_dim=2816,
                                feat_stride=1, num_frames=1, test_folder=folders["lists"], trunc_thresh=0.5, max_seq_len=768,
                                force_upsampling=True)
    return cfg_path, full, sd, ds


def api_records(model, ds, window, hop=None):
    from audio_visual_deepfake_detection_b200.libs.utils.infer_utils import result_item
    items = [ds[i] for i in range(len(ds))]
    return [result_item(it["video_id"], r) for it, r in zip(items, model.forward_streams(items, window=window, hop=hop))]


def test_inference_sharded_window_equals_api(tmp_path):
    from audio_visual_deepfake_detection_b200.libs.utils import inference_sharded
    cfg_path, full, sd, ds = corpus_setup(tmp_path, [62.0, 4.03, 7.42, 35.5, 9.04])
    model = make_meta_arch(full["model_name"], **full["model"], max_batch=4)
    model.load_state_dict(sd)
    model.to("cuda").eval()
    got = inference_sharded(ds, model, str(tmp_path / "out"), batch_size=2, window=10.0)
    assert got == api_records(model, ds, 10.0)
    assert json.load(open(tmp_path / "out" / "data_left.json")) == got


def test_inference_cli_window(tmp_path):
    cfg_path, full, sd, ds = corpus_setup(tmp_path, [75.0, 6.2])
    ckpt = str(tmp_path / "run" / "epoch_010.pth.tar")
    os.makedirs(os.path.dirname(ckpt))
    torch.save({"epoch": 10, "state_dict_ema": {"module." + k: v for k, v in sd.items()}}, ckpt)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "inference.py"), cfg_path, "3", ckpt, "-b", "4", "--window", "20"],
                       capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    model = make_meta_arch(full["model_name"], **full["model"], max_batch=4)
    model.load_state_dict(sd)
    model.to("cuda").eval()
    want = api_records(model, ds, 20.0, 10.0)
    assert json.load(open(tmp_path / "run" / "3" / "data_left.json")) == want
    assert len(want) == 2


def test_two_rank_window_inference_equals_one_rank(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cfg_path, full, sd, ds = corpus_setup(tmp_path, [62.0, 4.03, 7.42, 35.5, 9.04])
    outs = []
    for tag, launcher in (("one", [sys.executable]),
                          ("two", [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                                   "--master-addr", "127.0.0.1", "--master-port", "29613"])):
        ckpt = str(tmp_path / tag / "epoch_010.pth.tar")
        os.makedirs(os.path.dirname(ckpt))
        torch.save({"epoch": 10, "state_dict_ema": {"module." + k: v for k, v in sd.items()}}, ckpt)
        r = subprocess.run(launcher + [os.path.join(ROOT, "inference.py"), cfg_path, "3", ckpt, "-b", "4", "--window", "10"],
                           capture_output=True, text=True, cwd=ROOT, timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        outs.append(json.load(open(tmp_path / tag / "3" / "data_left.json")))
    assert outs[0] == outs[1]
