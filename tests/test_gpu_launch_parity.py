"""Every kernel launch of real forward passes, checked one by one against the float64 references of
oracle/launch_ref.py (tests/launch_check.py: a fixture wraps the `ops` entry points the engine calls; each launch gets
the overlap, replay, error and zeros checks at once). A failure names the op, the engine call site and block, the shapes /
dtypes and the worst element with both values.
Passes: every MODEL_CASES entry in fp32 and mixed at batch 3 and in mixed at batch 32 (the benchmark's batch: the only
passes that take the launch configurations that depend on the SM count), and exp12 mixed at batch 32 with each of the
engine's A/B switches AVDF_FUSE_TAIL, AVDF_FUSE_LN2, AVDF_FUSED_MLP turned off. Each pass ends in the fused postprocess
(decode, NMS - soft in the mixed batch-3 passes, hard otherwise - voting, seconds), checked the same way."""
import collections
import time

import pytest
import torch

import launch_check
import launch_ref
from make_golden import MODEL_CASES, VIDEO_CASES, make_item
from audio_visual_deepfake_detection_b200.libs.core import load_config_for
from audio_visual_deepfake_detection_b200.libs.modeling import make_meta_arch
from audio_visual_deepfake_detection_b200.libs.utils import synthetic as syn

pytestmark = pytest.mark.gpu

STATS = collections.defaultdict(lambda: [0, 0.0])          # op -> [launches, worst error / bar] over the whole module


@pytest.fixture
def recorder(monkeypatch):
    """Wraps every `ops` entry point that has a float64 reference; each call is checked as soon as it returns."""
    return launch_check.install(monkeypatch, launch_ref.REFERENCES, launch_check.ENGINE_FILE)


_ITEMS = {}


def _items(use_video, batch):
    """batch items cycling through VIDEO_CASES' durations and the interp / ragged modes (ragged masks)."""
    if use_video not in _ITEMS:
        _ITEMS[use_video] = [make_item(d, s, m, use_video) for d, s, m in VIDEO_CASES]
    base = _ITEMS[use_video]
    return [base[i % len(base)] for i in range(batch)]


PASSES = [(case, prec, b, None) for case in MODEL_CASES for prec, b in (("fp32", 3), ("mixed", 3), ("mixed", 32))]
PASSES += [("exp12", "mixed", 32, env) for env in ("AVDF_FUSE_TAIL", "AVDF_FUSE_LN2", "AVDF_FUSED_MLP")]


@pytest.mark.parametrize("case,precision,batch,switch_off", PASSES,
                         ids=["%s-%s-b%d%s" % (c, p, b, "" if e is None else "-%s=0" % e) for c, p, b, e in PASSES])
def test_every_launch_of_a_forward_pass(case, precision, batch, switch_off, recorder, monkeypatch):
    if switch_off is not None:
        monkeypatch.setenv(switch_off, "0")          # read when the engine is built
    model_name, overrides, use_video, wseed = MODEL_CASES[case]
    cfg = load_config_for(model_name, dict(overrides))
    model = make_meta_arch(cfg["model_name"], **cfg["model"], precision=precision, max_batch=batch)
    model.load_state_dict(syn.synthetic_state_dict(cfg["model"], model_name, seed=wseed))
    model = model.to("cuda").eval()
    if precision == "mixed" and batch == 3:
        model.test_nms_method = "soft"               # the configs ship hard NMS; these passes check the soft path
    t0 = time.time()
    launch_ref.reset_postprocess_stats()
    model(_items(use_video, batch))                  # forward pass + decode / NMS / voting / seconds (postprocess)
    torch.cuda.synchronize()
    n = sum(recorder.count.values())
    assert n > 0 and recorder.count["pack_feats"] == batch and recorder.count["postprocess"] == 1
    for op in ("conv_gemm", "attention", "ln_dwconv_ln"):
        assert recorder.count[op] > 0, op
    ps = launch_ref.POSTPROCESS_STATS
    assert ps["videos"] == batch
    print("\nlaunch parity %s: %d launches checked in %.1f s; %s; worst error / bar: %s; postprocess (%s NMS): %d decode "
          "points near the cut exempt, %d of them kept or dropped unlike float64; voting error / bound %.3g" % (
              "-".join(str(v) for v in (case, precision, batch, switch_off) if v is not None), n, time.time() - t0,
              dict(recorder.count), {k: round(v, 3) for k, v in sorted(recorder.worst.items())}, model.test_nms_method,
              ps["near_cut"], ps["near_cut_moved"], recorder.worst_path.get(("postprocess", "out_segs"), 0.0)))
    for k, v in recorder.count.items():
        STATS[k][0] += v
        STATS[k][1] = max(STATS[k][1], recorder.worst.get(k, 0.0))


def teardown_module(module):
    launch_check.report("launch parity", STATS)
