"""CPU-side checks of the post-processing sweep (libs/utils/sweep.py, avdf_postprocess_sweep): grid parsing and the
Cartesian product order, every setting the sweep refuses, and argument errors of the C entry point returned as -1
before any CUDA call (so these run without a GPU)."""
import ctypes
import math

import pytest

from audio_visual_deepfake_detection_b200 import native
from audio_visual_deepfake_detection_b200.libs.utils import sweep

BASE = {"nms_method": "soft", "iou_threshold": 0.1, "min_score": 0.2, "nms_sigma": 0.75, "voting_thresh": 0.9,
        "pre_nms_thresh": 0.001, "pre_nms_topk": 2000, "duration_thresh": 0.001, "max_seg_num": 100, "multiclass_nms": False}


def test_parse_set_types():
    assert sweep.parse_set("nms_method=hard,soft") == ("nms_method", ["hard", "soft"])
    assert sweep.parse_set("iou_threshold=0.1, 0.5") == ("iou_threshold", [0.1, 0.5])
    k, v = sweep.parse_set("max_seg_num=1,100")
    assert v == [1, 100] and all(isinstance(x, int) for x in v)
    assert sweep.parse_set("multiclass_nms=true,false") == ("multiclass_nms", [True, False])
    for bad in ("iou_threshold", "bogus=1", "iou_threshold=", "multiclass_nms=maybe", "max_seg_num=1.5"):
        with pytest.raises(ValueError):
            sweep.parse_set(bad)


def test_grid_is_the_cartesian_product_last_key_fastest():
    g = sweep.grid([("nms_method", ["hard", "soft"]), ("iou_threshold", [0.1, 0.3, 0.5])])
    assert g == [{"nms_method": m, "iou_threshold": t} for m in ("hard", "soft") for t in (0.1, 0.3, 0.5)]
    assert sweep.grid([]) == [{}]
    with pytest.raises(ValueError):
        sweep.grid([("min_score", [0.1]), ("min_score", [0.2])])


def test_full_setting_fills_from_test_cfg():
    s = sweep.full_setting(BASE, {"nms_method": "hard", "max_seg_num": 1})
    assert s == dict(BASE, nms_method="hard", max_seg_num=1)
    c = sweep.c_setting(dict(s, multiclass_nms=True))
    assert c.use_soft_nms == 0 and c.voting_thresh == 0.0 and c.max_seg_num == 1 and c.pre_nms_topk == 2000


@pytest.mark.parametrize("setting", [
    {"nms_method": "none"},
    {"max_seg_num": 0},
    {"max_seg_num": native.MAX_SEGS + 1},
    {"nms_method": "soft", "nms_sigma": 0.0},
    {"nms_method": "soft", "nms_sigma": -1.0},
    {"iou_threshold": math.nan},
    {"min_score": math.inf},
    {"voting_thresh": -math.inf},
    {"pre_nms_thresh": math.nan},
    {"duration_thresh": math.inf},
])
def test_refused_settings(setting):
    with pytest.raises(native.AvdfError):
        sweep.full_setting(BASE, setting)


def test_refused_multiclass_with_several_classes_and_unknown_keys():
    with pytest.raises(native.AvdfError):
        sweep.full_setting(BASE, {"multiclass_nms": True}, num_classes=2)
    sweep.full_setting(BASE, {"multiclass_nms": True}, num_classes=1)
    with pytest.raises(ValueError):
        sweep.full_setting(BASE, {"nms_thresh": 0.5})


def test_empty_grid_is_refused():
    with pytest.raises(native.AvdfError):
        sweep.sweep_rows(None, [])


def _args(n_settings=1, **kw):
    table = (native.SweepSetting * max(1, n_settings))(*[sweep.c_setting(BASE)] * max(1, n_settings))
    a = native.PostprocessSweepArgs()
    a.batch, a.n_levels = 2, 2
    a.level_len[0], a.level_len[1] = 8, 4
    a.level_stride[0], a.level_stride[1] = 1.0, 2.0
    fake = 0x1000                      # never dereferenced: every call below fails validation first
    a.logits = a.offsets = a.valid_len = a.out_rows = a.workspace = fake
    a.workspace_bytes = 1 << 30
    a.n_settings, a.settings = n_settings, table
    a.rows_per_setting, a.row_k = 2, 100
    for k, v in kw.items():
        setattr(a, k, v)
    return a, table


def _set(table, **kw):
    for k, v in kw.items():
        setattr(table[0], k, v)


def test_sweep_bad_arguments_return_minus_one():
    L = native.lib()
    assert L.avdf_postprocess_sweep(None, None) == -1
    assert L.avdf_postprocess_sweep_workspace_bytes(0, 12) == 0
    assert L.avdf_postprocess_sweep_workspace_bytes(2, 12) > 0
    cases = [dict(n_settings=0), dict(n_settings=65), dict(row_k=0), dict(row_k=native.MAX_SEGS + 1), dict(n_levels=0),
             dict(batch=-1), dict(rows_per_setting=1), dict(out_rows=None), dict(workspace_bytes=0), dict(valid_len=None)]
    for kw in cases:
        n = kw.pop("n_settings", 1)
        a, table = _args(n_settings=max(n, 0) if n <= 64 else 64, **kw)
        a.n_settings = n
        assert L.avdf_postprocess_sweep(ctypes.byref(a), None) == -1, kw
        assert b"invalid argument" in L.avdf_last_error()
    for bad in (dict(use_soft_nms=2), dict(use_soft_nms=-1), dict(max_seg_num=0), dict(max_seg_num=101),
                dict(use_soft_nms=1, sigma=0.0), dict(iou_threshold=math.nan), dict(min_score=math.inf),
                dict(pre_nms_thresh=math.nan), dict(duration_thresh=-math.inf), dict(voting_thresh=math.nan),
                dict(pre_nms_topk=-1)):
        a, table = _args()
        _set(table, **bad)
        assert L.avdf_postprocess_sweep(ctypes.byref(a), None) == -1, bad
    a, table = _args()
    a.level_len[1] = 0
    assert L.avdf_postprocess_sweep(ctypes.byref(a), None) == -1
    a, table = _args()
    a.level_stride[0] = math.nan
    assert L.avdf_postprocess_sweep(ctypes.byref(a), None) == -1
