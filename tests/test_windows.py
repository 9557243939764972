"""Window plan of the sliding-window path (libs/modeling/windows.py), checked against its stated rules on the host."""
import math

import numpy as np
import pytest

from audio_visual_deepfake_detection_b200.libs.modeling.streaming import video_meta
from audio_visual_deepfake_detection_b200.libs.modeling.windows import check_window, window_meta, window_plan
from audio_visual_deepfake_detection_b200.libs.utils import synthetic as syn


def lens_of(D):
    return list(syn.stream_lengths(D))


def check_rules(D, lens, W, H):
    plan = window_plan(D, lens, W, H)
    if D <= W:
        assert plan == [(0.0, [(0, T) for T in lens])]
        return plan
    n = math.ceil((D - W) / H) + 1
    assert len(plan) == n
    for k, (s, rng) in enumerate(plan):
        assert s == min(k * H, D - W)
        for T, (a, m) in zip(lens, rng):
            assert a == math.floor(s * T / D) and m == math.floor(W * T / D)
            assert m >= 1 and 0 <= a and a + m <= T
    assert plan[-1][0] + W == D                                   # the last window ends at D
    assert plan[0][0] == 0.0
    for (s0, _), (s1, _) in zip(plan, plan[1:]):                  # every instant of [0, D] lies in some window
        assert s0 < s1 <= s0 + W
        assert s1 - s0 <= H
    return plan


def test_recording_no_longer_than_the_window_is_one_window():
    for D in (4.03, 9.99, 10.0):
        plan = check_rules(D, lens_of(D), 10.0, 5.0)
        assert len(plan) == 1


def test_just_above_the_window():
    D = 10.01
    plan = check_rules(D, lens_of(D), 10.0, 5.0)
    assert len(plan) == 2 and plan[1][0] == pytest.approx(0.01)


@pytest.mark.parametrize("D,W,H", [(40.0, 10.0, 5.0), (47.3, 10.0, 5.0), (600.0, 10.0, 5.0), (601.7, 30.0, 12.5),
                                   (123.4, 30.0, 30.0), (75.0, 30.0, 7.0)])
def test_plan_rules(D, W, H):
    plan = check_rules(D, lens_of(D), W, H)
    if (D - W) % H:                                               # non-divisible: the last hop is shorter
        assert plan[-1][0] - plan[-2][0] < H


def test_absent_stream_and_default_hop():
    D = 100.0
    t_v, t_b, t_e = lens_of(D)
    plan = window_plan(D, [None, t_b, t_e], 20.0)
    assert len(plan) == math.ceil((D - 20.0) / 10.0) + 1
    assert all(rng[0] == (0, 0) for _, rng in plan)
    assert check_window(20.0, None) == (20.0, 10.0)


def test_segment_no_longer_than_w_minus_h_lies_in_a_window():
    D, W, H = 97.0, 10.0, 4.0
    starts = [s for s, _ in window_plan(D, lens_of(D), W, H)]
    rng = np.random.RandomState(0)
    for _ in range(2000):
        length = rng.uniform(0, W - H)
        t0 = rng.uniform(0, D - length)
        assert any(s <= t0 and t0 + length <= s + W for s in starts)


def test_window_meta_is_video_meta_of_a_w_second_item():
    m, W, L = 250, 10.0, 768
    assert window_meta(m, W, L) == video_meta({"duration": W}, m, L)
    assert window_meta(m, W, L, 16, 32) == video_meta({"duration": W}, m, L, 16, 32)
    # item-level fps / feat_stride describe the whole recording and are not used
    assert window_meta(m, W, L)[2] == np.float32(m / W)


@pytest.mark.parametrize("W,H", [(0.0, None), (-1.0, 0.5), (10.0, 0.0), (10.0, -2.0), (10.0, 10.5)])
def test_bad_window_or_hop(W, H):
    with pytest.raises(ValueError):
        window_plan(100.0, lens_of(100.0), W, H)


def test_window_without_a_row_of_some_stream():
    # 2 rows over 1000 s: a 10 s window holds floor(10 * 2 / 1000) = 0 of them
    with pytest.raises(ValueError):
        window_plan(1000.0, [None, 2, 50000], 10.0, 5.0)
