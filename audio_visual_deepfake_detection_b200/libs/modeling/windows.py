"""Sliding-window plan for recordings longer than the model's training clips.

Every path into the model resamples a whole recording to max_seq_len (768) steps. AV-Deepfake1M clips are 4-33 s, so a
step is 5-43 ms; a 10-minute recording would get 781 ms steps, a time scale the model never saw. With a window `W` and
hop `H` (seconds, 0 < H <= W) a recording of duration D is cut into windows of W seconds, each of which runs through
the ordinary pass as a video of its own, and the window outputs are merged per recording (csrc/window.cu).

Geometry (host, float64):
  D <= W   one window: the recording itself (all rows, its own fps / feat_stride); its result is today's result.
  D >  W   n = ceil((D - W) / H) + 1 windows; window k starts at s_k = min(k * H, D - W), so the last ends at D.
           Stream s (T_s rows) of window k is rows [a, a + m), a = floor(s_k * T_s / D), m = floor(W * T_s / D);
           m < 1 for any stream raises ValueError.
Consecutive windows overlap by W - H seconds, so any segment no longer than W - H lies inside some window. H = W / 2 is
the suggested default. W and H are user parameters: no trained weights or long recordings are in this repository, so
no choice of them has been validated for detection quality.
"""
import math

import numpy as np

from .streaming import video_meta


def check_window(window, hop):
    """(W, H) as floats; H defaults to W / 2. Raises ValueError unless 0 < H <= W."""
    W = float(window)
    H = W / 2.0 if hop is None else float(hop)
    if not W > 0:
        raise ValueError("window must be > 0 seconds, got %r" % (window,))
    if not (0 < H <= W):
        raise ValueError("hop must satisfy 0 < hop <= window, got hop %r, window %r" % (hop, window))
    return W, H


def window_plan(duration, lengths, window, hop=None):
    """Windows of one recording: a list of (s_k seconds, [(a, m) per stream]) with `lengths` the rows T_s of each
    stream (None for an absent stream: (0, 0) in its place). A recording no longer than the window gives
    [(0.0, [(0, T_s), ...])]."""
    W, H = check_window(window, hop)
    D = float(duration)
    if D <= W:
        return [(0.0, [(0, 0) if T is None else (0, int(T)) for T in lengths])]
    n = int(math.ceil((D - W) / H)) + 1
    m = [None if T is None else int(math.floor(W * T / D)) for T in lengths]
    if any(x is not None and x < 1 for x in m):
        raise ValueError("a %.3f s window of a %.3f s recording holds no row of a stream with %s rows" % (W, D, list(lengths)))
    plan = []
    for k in range(n):
        s = min(k * H, D - W)
        plan.append((s, [(0, 0) if T is None else (int(math.floor(s * T / D)), mk) for T, mk in zip(lengths, m)]))
    return plan


def window_meta(m_first, window, L, feat_stride=1, num_frames=1):
    """(feat_stride, 0.5 * feat_num_frames, fps, duration) fp32 of a window with m_first rows of its first stream: what
    video_meta derives for an item of duration W without item-level fps / feat_stride / feat_num_frames (those
    describe the whole recording), from the dataset-level feat_stride / num_frames."""
    return video_meta({"duration": float(window)}, m_first, L, feat_stride, num_frames)


def stream_lengths(item, names):
    """Row count of each named stream of a raw-stream item (None where absent)."""
    return [np.shape(item["streams"][n])[0] if n in item["streams"] else None for n in names]
