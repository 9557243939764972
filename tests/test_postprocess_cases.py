"""Self-checks of the adversarial post-processing inputs (tests/postprocess_cases.py), on the CPU: each generator is
deterministic, float32, and really reaches the edge it is named for - checked with the float32 restatement of the
kernels' arithmetic and, where it decides, with the C oracle (oracle/nms_ref.c)."""
import numpy as np
import pytest

import nms_ref
import postprocess_cases as pc

F32 = np.float32


@pytest.mark.parametrize("family", list(pc.FAMILIES))
@pytest.mark.parametrize("n", [1, 33, 6145])
def test_families_are_deterministic_float32(family, n):
    a, b = pc.FAMILIES[family](n, 5), pc.FAMILIES[family](n, 5)
    assert a[0].dtype == F32 and a[1].dtype == F32 and a[0].shape == (n, 2) and a[1].shape == (n,)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    assert np.isfinite(a[0]).all() and ((a[1] >= 0) & (a[1] <= 1)).all()


def test_tie_families_tie():
    s = pc.grid_ties(4000, 1)[1]
    assert (s == F32(1)).mean() > 0.25 and len(np.unique(s)) <= 17
    s = pc.min_score_ties(4000, 1)[1]
    assert (s == F32(0.2)).mean() > 0.3
    segs = pc.identical_segments(4000, 1)[0]
    assert len(np.unique(segs, axis=0)) <= 500


def test_degenerate_geometry():
    segs, _ = pc.nested_touching(2000, 2)
    unit = segs[(segs[:, 1] - segs[:, 0]) == 1]
    i, j = np.nonzero(unit[:, 1][:, None] == unit[:, 0][None, :])
    assert len(i) > 10 and (pc.ovr_eps(unit[i, 0], unit[i, 1], unit[j, 0], unit[j, 1]) == 0).all()
    segs, _ = pc.zero_length(2000, 2)
    assert (segs[:, 0] == segs[:, 1]).mean() > 0.2


@pytest.mark.parametrize("thr", [0.1, 0.3, 0.75])
def test_exact_iou_pairs_hit_the_threshold(thr):
    at, below = pc.exact_iou_pairs(thr, 11)
    assert len(at) >= 8 and len(below) >= 8
    assert (pc.ovr_eps(*at.T) == F32(thr)).all()
    assert (pc.ovr_eps(*below.T) == np.nextafter(F32(thr), F32(0))).all()
    # the oracle's '>=': the lower-scored partner at the threshold is suppressed, the one just below is kept
    segs, sc = pc.exact_iou(200, 11, thr)
    kept = set(nms_ref.nms(segs, sc, thr).tolist())
    assert all(2 * i + 1 not in kept for i in range(len(at)))
    assert all(2 * (len(at) + i) + 1 in kept for i in range(len(below)))


def test_linear_decay_lands_on_min_score():
    segs, sc = pc.linear_decay_to_min(40, 3)
    assert len(sc) >= 60
    o = pc.ovr_eps(segs[0::2, 0], segs[0::2, 1], segs[1::2, 0], segs[1::2, 1])
    assert (o >= F32(0.1)).all() and ((sc[1::2] * (F32(1) - o)) == F32(0.2)).all()
    inds, dets = nms_ref.softnms(segs, sc, 0.1, 0.75, 0.2, 1)
    assert len(inds) == len(sc) and (dets[:, 2] == F32(0.2)).sum() >= len(sc) // 2   # decayed onto min_score, kept


def _first_step_failures(segs, sc, thr=0.1):
    """Positions failing in the first soft-NMS step (method 0) after the reference's swap of the pick to position 0."""
    mp = int(np.argmax(sc))                  # first maximum in position order
    order = np.arange(len(sc))
    order[[0, mp]] = order[[mp, 0]]
    o = pc.ovr_eps(segs[mp, 0], segs[mp, 1], segs[order[1:], 0], segs[order[1:], 1])
    return np.nonzero(o >= F32(thr))[0] + 1


def test_soft_nms_step_edges():
    n = 3000
    segs, sc = pc.suppress_all(n, 4)
    assert len(_first_step_failures(segs, sc)) == n - 1                # F = nsegs - 1
    inds, _ = nms_ref.softnms(segs, sc, 0.1, 0.75, 0.2, 0)
    assert len(inds) == 1
    segs, sc = pc.disjoint(n, 4)
    assert len(_first_step_failures(segs, sc)) == 0 and (sc >= F32(0.25)).all()
    assert len(nms_ref.softnms(segs, sc, 0.1, 0.75, 0.2, 2)[0]) == n   # F == 0 at every step
    segs, sc = pc.chunk_straddle(n, 4)
    fail = _first_step_failures(segs, sc)
    chunk = -(-(n - 1) // pc.NMS_THREADS)
    assert chunk >= 2
    r = (fail - 1) % chunk
    assert (r == 0).any() and (r == chunk - 1).any()                  # failures on both ends of a thread's chunk
    new_n = n - len(fail)
    assert (fail < new_n).any() and (fail >= new_n).any()             # holes below the new end, failures above it


def test_cluster_slices_and_paths():
    assert pc.cluster_slice(6145) == 416 and 15 * 416 >= 6145          # the last CTA owns no position
    assert pc.cluster_slice(180224) == pc.NMS_CL_SLICE_MAX
    assert [pc.nms_path(n) for n in (6144, 6145, 180224, 180225)] == ["smem", "cluster", "cluster", "global"]
    assert pc.nms_path(6145, cluster=False) == "global"


def test_decode_case_edges():
    lens, topk = [2048, 1000, 333, 17, 1], 300
    logits, offsets, mask = pc.decode_case(21, lens, topk)
    assert logits.dtype == F32 and offsets.dtype == F32 and mask.dtype == np.uint8 and logits.shape == (5, sum(lens))
    assert (logits[0, :lens[0]] >= 17).sum() > topk                     # the cut falls inside the saturated group
    v, c = np.unique(logits[1, :lens[0]], return_counts=True)
    assert len(v) <= 7 and (c > 1).all()
    assert mask[2].sum() == 0
    off = np.cumsum([0] + lens)
    exact = 0
    for l, n in enumerate(lens):
        s = F32(2 ** l)
        tt = np.arange(n).astype(F32) * s
        of = offsets[3, off[l]:off[l + 1]]
        d = (tt + of[:, 1] * s) - (tt - of[:, 0] * s)
        exact += int((d == F32(0.001)).sum())
    assert exact >= len(lens)            # right - left exactly duration_thresh (at least point 0 of every level)
    grid = np.concatenate([logits[4], logits[3]])
    assert (grid * 16 == np.round(grid * 16)).all()                    # distinct logits on the 1/16 grid
