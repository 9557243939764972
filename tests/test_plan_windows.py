"""CPU-side checks of sliding windows on launch plans (csrc/plan.cu, include/avdf.h "sliding windows on a session"):
avdf_plan_window_layout is the C++ port of windows.window_plan + video_meta / window_meta and matches it bit for bit on
seeded cases; every bad input is refused with its own message; avdf_session_window_bytes is the documented sum and
refuses a plan whose launch lists cannot run windows. Hand-built plans, as in test_plan.py: no GPU needed."""
import ctypes
import math
import os

import numpy as np
import pytest

from audio_visual_deepfake_detection_b200 import native as nv
from audio_visual_deepfake_detection_b200.libs.modeling import plan as pl
from audio_visual_deepfake_detection_b200.libs.modeling.streaming import video_meta
from audio_visual_deepfake_detection_b200.libs.modeling.windows import window_meta, window_plan
from audio_visual_deepfake_detection_b200.libs.utils import synthetic as syn

MB, K, L = 4, 5, 768
PP = nv.PostprocessArgs


def allocs(channels):
    out = []
    for s, role in enumerate((pl.ROLE_VIDEO, pl.ROLE_BYOLA, pl.ROLE_EMO)):
        if channels[s]:
            out.append((pl.KIND_INPUT, role, 10 * channels[s] * 4, 0))
    out += [(pl.KIND_INPUT, pl.ROLE_OFFSETS, 3 * (MB + 1) * 4, 0), (pl.KIND_INPUT, pl.ROLE_META, 4 * MB * 4, 0),
            (pl.KIND_OUTPUT, pl.ROLE_SEGS, MB * K * 8, 0), (pl.KIND_OUTPUT, pl.ROLE_SCORES, MB * K * 4, 0),
            (pl.KIND_OUTPUT, pl.ROLE_COUNTS, MB * 4, 0), (pl.KIND_OUTPUT, pl.ROLE_VCLS, MB * 4, 0),
            (pl.KIND_SCRATCH, pl.ROLE_NONE, 1 << 16, 0)]
    return out


def ids(channels):
    """allocation id of every io role (absent streams have none) and of the scratch buffer"""
    n_in = sum(1 for c in channels if c)
    io = {}
    k = 0
    for s, role in enumerate((pl.ROLE_VIDEO, pl.ROLE_BYOLA, pl.ROLE_EMO)):
        if channels[s]:
            io[role] = k
            k += 1
    for j, role in enumerate((pl.ROLE_OFFSETS, pl.ROLE_META, pl.ROLE_SEGS, pl.ROLE_SCORES, pl.ROLE_COUNTS, pl.ROLE_VCLS)):
        io[role] = n_in + j
    return io, n_in + 6


def interp(channels, B, batch_arg=None, offsets=True):
    io, scratch = ids(channels)
    streams = [(pl.TAG_PTR, (io[r], 0) if channels[s] else (None, 0))
               for s, r in enumerate((pl.ROLE_VIDEO, pl.ROLE_BYOLA, pl.ROLE_EMO))]
    offs = [(pl.TAG_PTR, ((io[pl.ROLE_OFFSETS] if offsets else scratch), 4 * s * (MB + 1)) if channels[s] else (None, 0))
            for s in range(3)]
    return ("avdf_interp_concat_in", streams + [(pl.TAG_I32, nv.DTYPE_F32)] + offs +
            [(pl.TAG_I32, B if batch_arg is None else batch_arg)] + [(pl.TAG_I32, c) for c in channels] +
            [(pl.TAG_I32, L), (pl.TAG_PTR, (scratch, 0)), (pl.TAG_I32, nv.DTYPE_F32), (pl.TAG_STREAM, None)])


def postprocess(channels, B, soft=1, method=2, records=False):
    io, scratch = ids(channels)
    a = PP()
    a.batch, a.max_seg_num, a.use_soft_nms, a.soft_method = B, K, soft, method
    a.iou_threshold, a.min_score, a.sigma, a.voting_thresh = 0.1, 0.001, 0.75, 0.0
    raw = bytes(ctypes.string_at(ctypes.addressof(a), ctypes.sizeof(a)))
    relocs = [(PP.out_segs.offset, io[pl.ROLE_SEGS], 0), (PP.out_scores.offset, io[pl.ROLE_SCORES], 0),
              (PP.out_count.offset, io[pl.ROLE_COUNTS], 0), (PP.cand_segs.offset, scratch, 1024)]
    if records:
        relocs.append((PP.rec_ring.offset, scratch, 4096))
    return ("avdf_postprocess", [(pl.TAG_STRUCT, (raw, relocs)), (pl.TAG_STREAM, None)])


def ln_rows(channels):
    _, scratch = ids(channels)
    return ("avdf_ln_rows", [(pl.TAG_PTR, (scratch, 0)), (pl.TAG_PTR, (scratch, 64)), (pl.TAG_PTR, (scratch, 128)),
                             (pl.TAG_PTR, (scratch, 2048)), (pl.TAG_I32, nv.DTYPE_F32), (pl.TAG_I64, 4), (pl.TAG_I32, 4),
                             (pl.TAG_STREAM, None)])


def make_lists(channels, batches=(1, 3, MB), **bad):
    out = {}
    for B in batches:
        first = bad["first"](B) if "first" in bad else interp(channels, B)
        post = [postprocess(channels, B, **bad.get("post", {}))] * bad.get("n_post", 1)
        out[B] = [first, ln_rows(channels)] + post
    return out


def write_plan(tmp_path, channels=(4, 4, 4), name="p.avdfplan", device=(10, 0, 148), **bad):
    header = dict(cc_major=device[0], cc_minor=device[1], sm_count=device[2], max_batch=MB, max_seg_num=K, t_out=L,
                  in_dtype=nv.DTYPE_F32, channels=list(channels), stream_rows=[10 if c else 0 for c in channels],
                  description="windows")
    data = pl.encode_plan(header, allocs(channels), bytes(256), make_lists(channels, **bad))
    path = tmp_path / name
    path.write_bytes(data)
    return path


def open_plan(tmp_path, channels=(4, 4, 4), name="p.avdfplan", **bad):
    path = write_plan(tmp_path, channels, name, **bad)
    h = ctypes.c_void_p()
    lib = nv.lib()
    assert lib.avdf_plan_open(os.fsencode(str(path)), ctypes.byref(h)) == 0, lib.avdf_last_error()
    return h


@pytest.fixture
def plans(tmp_path):
    lib = nv.lib()
    hs = {"av": open_plan(tmp_path, (4, 4, 4), "av.plan"), "audio": open_plan(tmp_path, (0, 4, 4), "audio.plan")}
    yield hs
    for h in hs.values():
        lib.avdf_plan_close(h)


def layout(h, D, rows, W, H):
    """avdf_plan_window_layout -> (n, start [n,3], count [n,3], meta [n,4], win_start [n]) or (rc, message)"""
    lib = nv.lib()
    r = (ctypes.c_int64 * 3)(*rows)
    n = lib.avdf_plan_window_layout(h, D, r, W, H, 0, None, None, None, None)
    if n < 0:
        return n, lib.avdf_last_error().decode()
    st, ct = np.zeros((n, 3), np.int32), np.zeros((n, 3), np.int32)
    me, ws = np.zeros((n, 4), np.float32), np.zeros(n, np.float32)
    p32, pf = ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_float)
    got = lib.avdf_plan_window_layout(h, D, r, W, H, n, st.ctypes.data_as(p32), ct.ctypes.data_as(p32),
                                      me.ctypes.data_as(pf), ws.ctypes.data_as(pf))
    assert got == n
    return n, st, ct, me, ws


def reference(D, rows, W, H, channels):
    lens = [int(rows[s]) if channels[s] else None for s in range(3)]
    wp = window_plan(D, lens, W, H)
    first = 0 if channels[0] else 1
    st = np.array([[a for a, _ in rng] for _, rng in wp], np.int32)
    ct = np.array([[m for _, m in rng] for _, rng in wp], np.int32)
    if len(wp) == 1:
        me = np.array([video_meta({"duration": D}, lens[first], L)], np.float32)
    else:
        me = np.array([window_meta(rng[first][1], W, L) for _, rng in wp], np.float32)
    ws = np.array([np.float32(s) for s, _ in wp], np.float32)
    return len(wp), st, ct, me, ws


def cases(seed, n):
    """(D, rows, W, H): durations 4 s .. 2 h, rows at the synthetic stream rates and off them, H == W and tiny hops,
    D == W and one ulp above it, near-integer products s * T / D"""
    rng = np.random.RandomState(seed)
    out = []
    for i in range(n):
        kind = i % 8
        W = float(rng.choice([2.0, 4.0, 10.0, 12.5, 30.0, 60.0, 7.3, 300.0]))
        H = float(rng.choice([W, W / 2, W / 3, 0.4 * W, 5.0 if W > 5 else W, 0.1 if W >= 1 else W]))
        D = float(math.exp(rng.uniform(math.log(4.0), math.log(7200.0))))
        if D / H > 2000:                                    # keep the Python reference fast: <= 2000 windows
            D = W + H * rng.uniform(0, 2000)
        if kind == 0:
            rows = list(syn.stream_lengths(D))
        elif kind == 1:
            rows = [int(rng.randint(1, 200000)) for _ in range(3)]
        elif kind == 2:                                     # D == W, and one ulp above
            D = W if rng.rand() < 0.5 else float(np.nextafter(W, np.inf))
            rows = list(syn.stream_lengths(D))
        elif kind == 3:                                     # tiny hop, few windows
            H = float(rng.choice([1e-3, 1e-6, 0.0137]))
            D = W + H * rng.uniform(0, 300)
            rows = list(syn.stream_lengths(D))
        elif kind == 4:                                     # T / D at an exact rate: s * T / D lands on or next to integers
            rate = float(rng.choice([25.0, 50.0, 12.497, 30.0, 0.1]))
            T = int(rng.randint(max(2, int(W * rate) + 2), 200000))
            D = T / rate
            rows = [T, max(2, int(D * 12.497)), max(2, int(D * 50) - 1)]
            H = float(rng.choice([0.1, 0.3, 1.0 / 3.0, 0.7, W]))
            H = min(H, W)
            if D / H > 2000:
                D, rows = W + H * 500, list(syn.stream_lengths(W + H * 500))
        elif kind == 5:                                     # k * H clamped to D - W: D - W not a multiple of H
            D = W + H * (int(rng.randint(1, 300)) + float(rng.uniform(0.001, 0.999)))
            rows = list(syn.stream_lengths(D))
        elif kind == 6:                                     # D shorter than W
            D = float(rng.uniform(0.05, 1.0)) * W
            rows = [int(rng.randint(1, 5000)) for _ in range(3)]
        else:                                               # few rows: m = floor(W * T / D) near 1
            T = int(max(1, math.ceil(D / W)) + rng.randint(0, 3))
            rows = [T, T + int(rng.randint(0, 3)), T]
        out.append((D, rows, W, H))
    return out


@pytest.mark.parametrize("which", ["av", "audio"])
def test_layout_matches_window_plan_bit_for_bit(plans, which):
    channels = (4, 4, 4) if which == "av" else (0, 4, 4)
    h = plans[which]
    checked = refused = windows = 0
    for D, rows, W, H in cases(7 if which == "av" else 8, 5200):
        rows = [r if channels[s] else 0 for s, r in enumerate(rows)]
        try:
            want = reference(D, rows, W, H, channels)
        except ValueError:
            rc, msg = layout(h, D, rows, W, H)
            assert rc == -1 and "holds no row" in msg, (D, rows, W, H, msg)
            refused += 1
            continue
        got = layout(h, D, rows, W, H)
        assert got[0] == want[0], (D, rows, W, H)
        for g, w, what in zip(got[1:], want[1:], ("start", "count", "meta", "win_start")):
            assert g.dtype == w.dtype and np.array_equal(g, w), (what, D, rows, W, H)
            assert np.array_equal(g.view(np.uint32 if g.dtype == np.float32 else np.int32),
                                  w.view(np.uint32 if w.dtype == np.float32 else np.int32)), (what, D, rows, W, H)
        checked += 1
        windows += want[0]
    assert checked + refused == 5200 and checked >= 5000 and windows > 500000


def test_layout_capacity_and_no_arrays(plans):
    h, lib = plans["av"], nv.lib()
    r = (ctypes.c_int64 * 3)(15000, 7498, 29999)
    n = lib.avdf_plan_window_layout(h, 600.0, r, 10.0, 5.0, 0, None, None, None, None)
    assert n == math.ceil(590 / 5) + 1
    st = np.full((n, 3), -7, np.int32)
    p32, pf = ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_float)
    dummy = np.zeros((n, 4), np.float32)
    assert lib.avdf_plan_window_layout(h, 600.0, r, 10.0, 5.0, n - 1, st.ctypes.data_as(p32), st.ctypes.data_as(p32),
                                       dummy.ctypes.data_as(pf), dummy.ctypes.data_as(pf)) == n
    assert (st == -7).all()                                  # cap < n: nothing written


@pytest.mark.parametrize("D,rows,W,H,message", [
    (40.0, [1000, 500, 2000], 0.0, 0.0, "window must be > 0 seconds"),
    (40.0, [1000, 500, 2000], -5.0, 1.0, "window must be > 0 seconds"),
    (40.0, [1000, 500, 2000], float("nan"), 1.0, "window must be > 0 seconds"),
    (40.0, [1000, 500, 2000], 10.0, 0.0, "hop must satisfy 0 < hop <= window"),
    (40.0, [1000, 500, 2000], 10.0, 11.0, "hop must satisfy 0 < hop <= window"),
    (40.0, [1000, 500, 2000], 10.0, float("nan"), "hop must satisfy 0 < hop <= window"),
    (0.0, [1000, 500, 2000], 10.0, 5.0, "duration must be a positive finite number"),
    (float("inf"), [1000, 500, 2000], 10.0, 5.0, "duration must be a positive finite number"),
    (float("nan"), [1000, 500, 2000], 10.0, 5.0, "duration must be a positive finite number"),
    (40.0, [1000, 0, 2000], 10.0, 5.0, "stream 1 is present in the plan but has 0 rows"),
    (1000.0, [1000, 3, 50000], 10.0, 5.0, "holds no row of stream 1 (3 rows)"),
])
def test_layout_refusals(plans, D, rows, W, H, message):
    rc, msg = layout(plans["av"], D, rows, W, H)
    assert rc == -1 and message in msg, msg


def test_layout_refuses_rows_of_an_absent_stream(plans):
    rc, msg = layout(plans["audio"], 40.0, [1000, 500, 2000], 10.0, 5.0)
    assert rc == -1 and "stream 0 is absent from the plan but has 1000 rows" in msg, msg


def align(n):
    return (n + 255) // 256 * 256


@pytest.mark.parametrize("mw,per", [(1, 1), (37, 5), (1000, 120), (64, 64)])
def test_window_bytes_is_the_documented_sum(plans, mw, per):
    lib = nv.lib()
    want = (align(4 * (12 * mw + 10 * MB)) + align(24 * MB) + align(8 * K * mw) + align(4 * K * mw) + align(4 * mw)
            + align(4 * mw) + lib.avdf_window_merge_workspace_bytes(mw, K * per))
    assert lib.avdf_session_window_bytes(plans["av"], mw, per) == want


def test_window_bytes_refuses_bad_limits(plans):
    lib = nv.lib()
    for mw, per in ((0, 1), (10, 0), (10, 11), ((1 << 24) + 1, 1)):
        assert lib.avdf_session_window_bytes(plans["av"], mw, per) == 0
        assert b"max_windows_per_recording" in lib.avdf_last_error()


@pytest.mark.parametrize("bad,message", [
    (dict(first=lambda B: ln_rows((4, 4, 4))), "the launch list for batch 1 does not start with avdf_interp_concat_in"),
    (dict(first=lambda B: interp((4, 4, 4), B, offsets=False)), "stream 0 offsets are not the io offsets"),
    (dict(first=lambda B: interp((4, 4, 4), B, batch_arg=MB)), "batch 1: the resampling runs 4 recordings"),
    (dict(n_post=2), "batch 1: more than one avdf_postprocess"),
    (dict(n_post=0), "batch 1: no avdf_postprocess"),
    (dict(post=dict(records=True)), "avdf_postprocess keeps result records"),
    (dict(post=dict(soft=-1)), "use_soft_nms -1"),
    (dict(post=dict(soft=1, method=1)), "use_soft_nms 1 (method 1)"),
])
def test_window_bytes_refuses_plans_that_cannot_run_windows(tmp_path, bad, message):
    lib = nv.lib()
    h = open_plan(tmp_path, **bad)
    try:
        assert lib.avdf_session_window_bytes(h, 16, 4) == 0
        msg = lib.avdf_last_error().decode()
        assert msg.startswith("avdf_session_window_bytes: ") and message in msg, msg
    finally:
        lib.avdf_plan_close(h)


def test_hard_nms_plan_is_accepted(tmp_path):
    lib = nv.lib()
    h = open_plan(tmp_path, post=dict(soft=0, method=0))
    try:
        assert lib.avdf_session_window_bytes(h, 16, 4) > 0
    finally:
        lib.avdf_plan_close(h)


def test_run_and_attach_refuse_null_without_a_gpu():
    lib = nv.lib()
    a = nv.WindowRunArgs()
    assert lib.avdf_session_run_windows(None, ctypes.byref(a), None) == -1
    assert b"session / args is NULL" in lib.avdf_last_error()
    assert lib.avdf_session_attach_windows(None, None, 0, 1, 1) == -1
