"""Post-processing at its edges (csrc/nms.cu): the adversarial inputs of tests/postprocess_cases.py through every NMS
code path, checked against the C oracle (oracle/nms_ref.c, bit-exact), the stable-sort decode of
model_ref.OracleModel, and the float64 voting reference with its derived bound (launch_ref.voting_ref).

NMS paths of avdf_nms_hard / avdf_nms_soft: 'smem' (n <= 6144), 'cluster' (16 CTAs, n <= 16 x 11264 = 180224), 'global'
(one CTA from the workspace: longer lists, or any list > 6144 with the cluster switched off). avdf_postprocess takes
'smem' or 'global' per video, from that video's n. Every list > 6144 runs twice, the second time with the cluster off."""
import collections
import ctypes
import time

import numpy as np
import pytest
import torch

import launch_ref
import model_ref
import nms_ref
import postprocess_cases as pc
from audio_visual_deepfake_detection_b200 import native as nv
from audio_visual_deepfake_detection_b200 import ops
from audio_visual_deepfake_detection_b200.libs.utils import nms as front

pytestmark = pytest.mark.gpu
DEV = "cuda"
THR, SIGMA, MIN_SCORE = 0.1, 0.75, 0.2
PATHS = collections.defaultdict(set)           # path -> list sizes that reached it
VOTING = [0.0]                                 # worst voting error / bound
T0 = [time.time()]


def dev(a):
    return torch.as_tensor(np.ascontiguousarray(a)).to(DEV)


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


@pytest.fixture
def cluster():
    """Switches the 16-CTA cluster path on or off (a process-global setting); restores the previous value."""
    fn = nv.lib().avdf_debug_nms_cluster
    fn.restype, fn.argtypes = ctypes.c_int, [ctypes.c_int]
    prev = fn(1)
    try:
        yield lambda on: fn(int(on))
    finally:
        fn(prev)


def _modes(n):
    return (True, False) if n > pc.NMS_SMEM_CAP else (True,)


def check_standalone(segs, sc, method, max_num=0, thr=THR, on=True, what=""):
    """One avdf_nms_hard (method None) / avdf_nms_soft call against the C oracle: indices, dets and count bit-exact."""
    n = len(sc)
    PATHS[pc.nms_path(n, on)].add(n)
    if method is None:
        got = ops.nms_hard(dev(segs), dev(sc), thr, max_num).cpu().numpy()
        want = nms_ref.nms(segs, sc, thr)
        want = want[:max_num] if max_num > 0 else want
        assert np.array_equal(got, want), "%s hard n=%d max_num=%d: %d picks vs %d" % (what, n, max_num, len(got), len(want))
        return len(want)
    dets = torch.full((max(n, 1), 3), float("nan"), device=DEV)
    got = ops.nms_soft(dev(segs), dev(sc), dets, thr, SIGMA, MIN_SCORE, method, max_num).cpu().numpy()
    want_i, want_d = nms_ref.softnms(segs, sc, thr, SIGMA, MIN_SCORE, method, max_num=max_num)
    assert np.array_equal(got, want_i), "%s soft m%d n=%d max_num=%d: %d picks vs %d" % (what, method, n, max_num, len(got), len(want_i))
    assert np.array_equal(bits(dets[:len(got)].cpu().numpy()), bits(want_d)), "%s soft m%d n=%d: dets differ" % (what, method, n)
    return len(want_i)


# --------------------------------------------------------------------------------------------- standalone NMS
SIZES = [1, 2, 31, 32, 33, 511, 512, 513, 6143, 6144, 6145, 16 * 416 + 1, 180224, 180225]


@pytest.mark.parametrize("n", SIZES)
def test_standalone_nms_at_path_boundaries(n, cluster):
    """Tied grid scores at every size around the block / shared-memory / cluster limits (6145: S = 416, CTA 15 owns no
    position), hard and soft methods 0/1/2; lists past 20000 stop soft NMS after 300 picks (the oracle's prefix)."""
    segs, sc = pc.grid_ties(n, 100 + n)
    cap = 300 if n > 20000 else 0
    for on in _modes(n):
        cluster(on)
        check_standalone(segs, sc, None, on=on, what="grid_ties")
        for m in (0, 1, 2):
            check_standalone(segs, sc, m, cap, on=on, what="grid_ties")


@pytest.mark.parametrize("n", [33, 513, 6145, 9000])
def test_standalone_max_num_edges(n, cluster):
    """max_num = 1, k - 1, k, k + 1 where k is the uncapped pick count."""
    segs, sc = pc.identical_segments(n, 200 + n)
    for on in _modes(n):
        cluster(on)
        for method in (None, 0, 2):
            k = check_standalone(segs, sc, method, on=on)
            for mx in sorted({1, max(k - 1, 1), k, k + 1}):
                check_standalone(segs, sc, method, mx, on=on, what="max_num")


FAM_SIZES = (2000, 6144, 6145, 12289)


@pytest.mark.parametrize("family", list(pc.FAMILIES))
def test_standalone_nms_families(family, cluster):
    """Every generator family on both sides of the shared-memory limit, hard and soft methods 0/1/2 (soft past 6144
    stops after 400 picks)."""
    gen = pc.FAMILIES[family]
    for n in FAM_SIZES:
        segs, sc = gen(n, 300 + n)
        for on in _modes(n):
            cluster(on)
            check_standalone(segs, sc, None, on=on, what=family)
            for m in (0, 1, 2):
                check_standalone(segs, sc, m, 400 if n > pc.NMS_SMEM_CAP else 0, on=on, what=family)


def test_standalone_exact_threshold_iou(cluster):
    """IoU exactly at the threshold suppresses ('>='), one ulp below does not: thresholds 0.1, 0.3, 0.75, every path."""
    for thr in (0.1, 0.3, 0.75):
        for n in (200, 7000):
            segs, sc = pc.exact_iou(n, 11, thr)
            at, below = pc.exact_iou_pairs(thr, 11)
            want = set(nms_ref.nms(segs, sc, thr).tolist())
            assert not any(2 * i + 1 in want for i in range(len(at)))                     # the partner at the threshold goes
            assert all(2 * (len(at) + i) + 1 in want for i in range(len(below)))          # the one just below stays
            for on in _modes(n):
                cluster(on)
                check_standalone(segs, sc, None, thr=thr, on=on, what="exact_iou")
                for m in (0, 1):
                    check_standalone(segs, sc, m, thr=thr, on=on, what="exact_iou")


# --------------------------------------------------------------------------------------------- postprocess, candidate mode
def _pp_candidates(cases, K, soft, voting, method=2):
    B = len(cases)
    cap = max(max(len(s) for _, s in cases), 1)
    cs = torch.zeros((B, cap, 2), device=DEV)
    cc = torch.zeros((B, cap), device=DEV)
    cn = torch.tensor([len(s) for _, s in cases], dtype=torch.int32, device=DEV)
    for b, (segs, sc) in enumerate(cases):
        if len(sc):
            cs[b, :len(sc)] = dev(segs); cc[b, :len(sc)] = dev(sc)

    def run():
        o = (torch.full((B, K, 2), float("nan"), device=DEV), torch.full((B, K), float("nan"), device=DEV),
             torch.full((B,), -7, dtype=torch.int32, device=DEV), torch.full((B, K), -7, dtype=torch.int32, device=DEV))
        ops.postprocess(B, cand_segs=cs, cand_scores=cc, cand_count=cn, iou_threshold=THR, min_score=MIN_SCORE, sigma=SIGMA,
                        voting_thresh=voting, max_seg_num=K, use_soft_nms=soft, soft_method=method, out_segs=o[0],
                        out_scores=o[1], out_count=o[2], out_index=o[3])
        return [t.cpu() for t in o]
    first, again = run(), run()
    for a, b in zip(first, again):                 # a replay into fresh NaN-filled outputs is bit-identical
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))
    return first


def _check_candidates(cases, out, K, soft, voting, method=2):
    osg, osc, ocn, oix = (t.numpy() for t in out)
    for b, (segs, sc) in enumerate(cases):
        PATHS["postprocess " + ("smem" if len(sc) <= pc.NMS_SMEM_CAP else "global")].add(len(sc))
        idx, ps, pseg = launch_ref.nms_picks(segs, sc, THR, MIN_SCORE, SIGMA, K, soft, method)
        order = np.argsort(-ps, kind="stable")
        idx, ps, pseg = idx[order], ps[order], pseg[order]
        k = len(idx)
        what = "video %d (n=%d, K=%d, %s, voting %s)" % (b, len(sc), K, "soft" if soft else "hard", voting)
        assert ocn[b] == k, "%s: %d outputs, oracle %d" % (what, ocn[b], k)
        assert np.array_equal(bits(osc[b, :k]), bits(ps)), what
        assert np.array_equal(oix[b, :k], idx), what + ": out_index"
        assert np.isnan(osg[b, k:]).all() and np.isnan(osc[b, k:]).all() and (oix[b, k:] == -7).all(), what + ": wrote past k"
        if voting > 0 and k:
            val, bnd = launch_ref.voting_ref(pseg, segs, sc, voting)
            got = osg[b, :k].astype(np.float64)
            nan = np.isnan(val)
            assert np.array_equal(np.isnan(got), nan), what + ": NaN pattern of voting"
            if (~nan).any():
                r = float((np.abs(got - val)[~nan] / bnd[~nan]).max())
                VOTING[0] = max(VOTING[0], r)
                assert r <= 1.0, "%s: voting error / bound %.3g" % (what, r)
        else:
            assert np.array_equal(bits(osg[b, :k]), bits(pseg)), what


@pytest.mark.parametrize("soft", [False, True])
@pytest.mark.parametrize("voting", [0.0, 0.75])
def test_postprocess_candidates_mixed_paths(soft, voting):
    """One launch whose videos take shared memory (n <= 6144) and the global workspace (n > 6144) inside a 12289-wide
    buffer; ties, zero-length segments (voting NaN), exact-threshold pairs, min_score ties, an empty video; K = 1,
    the pick count of video 0, and 1024."""
    cases = [pc.grid_ties(300, 1), pc.zero_length(6144, 2), pc.min_score_ties(6145, 3), pc.exact_iou(9000, 4),
             pc.identical_segments(12289, 5), (np.zeros((0, 2), np.float32), np.zeros(0, np.float32))]
    k0 = len(launch_ref.nms_picks(*cases[0], THR, MIN_SCORE, SIGMA, 1024, soft, 2)[0])
    for K in (1, k0, 1024):
        _check_candidates(cases, _pp_candidates(cases, K, soft, voting), K, soft, voting)


@pytest.mark.parametrize("family", ["suppress_all", "disjoint", "chunk_straddle", "decay_to_min", "nested_touching"])
def test_postprocess_candidates_soft_decay_edges(family):
    """Soft-NMS bookkeeping inside postprocess (methods 0, 1, 2) on the decay-edge families, both per-video paths."""
    gen = pc.FAMILIES[family]
    cases = [gen(3000, 7), gen(7001, 8)]
    for method in (0, 1, 2):
        _check_candidates(cases, _pp_candidates(cases, 1024, True, 0.0, method), 1024, True, 0.0, method)


# --------------------------------------------------------------------------------------------- postprocess, decode mode
LENS = [2048, 1000, 333, 17, 1]
TOPK = 300


def _oracle_decode(logits, offsets, mask, lens, topk):
    class Stub(model_ref.OracleModel):
        def __init__(self):
            self.test_cfg = {"pre_nms_thresh": 0.001, "pre_nms_topk": topk, "duration_thresh": 0.001}
            self.fpn_strides = [2 ** l for l in range(len(lens))]; self.num_classes = 1
    off = np.cumsum([0] + lens)
    sl = lambda a, l: torch.from_numpy(np.ascontiguousarray(a[off[l]:off[l + 1]]))
    segs, scores, _ = Stub().decode([sl(logits, l).unsqueeze(-1) for l in range(len(lens))],
                                    [sl(offsets, l) for l in range(len(lens))],
                                    [sl(mask, l).bool() for l in range(len(lens))])
    return segs.numpy(), scores.numpy()


@pytest.mark.parametrize("method", ["hard", "soft", "none"])
def test_postprocess_decode_ties_and_cuts(method):
    """Decode of saturated (exactly 1.0f) and duplicated logits with the pre_nms_topk cut inside a tied group (the
    lowest point indices survive), an all-masked video, segments exactly duration_thresh long (dropped), level lengths
    2048 (DEC_MAX_T), 1000, 333, 17 and 1: candidates equal the stable-sort oracle (segments and order bit for bit,
    scores within the sigmoid's bound), then NMS on them equals the C oracle."""
    logits, offsets, mask = pc.decode_case(21, LENS, TOPK)
    B, P = logits.shape
    cs = torch.full((B, P, 2), float("nan"), device=DEV); cc = torch.full((B, P), float("nan"), device=DEV)
    cn = torch.full((B,), -7, dtype=torch.int32, device=DEV)
    K = P if method == "none" else 100
    osg = torch.full((B, K, 2), float("nan"), device=DEV); osc = torch.full((B, K), float("nan"), device=DEV)
    ocn = torch.zeros(B, dtype=torch.int32, device=DEV)
    ops.postprocess(B, logits=dev(logits), offsets=dev(offsets), mask=dev(mask), level_len=LENS,
                    level_stride=pc.decode_level_strides(LENS), pre_nms_thresh=0.001, pre_nms_topk=TOPK, duration_thresh=0.001,
                    cand_segs=cs, cand_scores=cc, cand_count=cn, iou_threshold=THR, min_score=MIN_SCORE, sigma=SIGMA,
                    voting_thresh=0.0, max_seg_num=100,
                    use_soft_nms=None if method == "none" else method == "soft", out_segs=osg, out_scores=osc, out_count=ocn)
    cs, cc, cn, osg, osc, ocn = (t.cpu().numpy() for t in (cs, cc, cn, osg, osc, ocn))
    for b in range(B):
        segs, scores = _oracle_decode(logits[b], offsets[b], mask[b], LENS, TOPK)
        n = int(cn[b])
        assert n == len(scores), (b, n, len(scores))
        assert np.array_equal(bits(cs[b, :n]), bits(segs)), "video %d: decoded segments / order differ from the oracle" % b
        p64 = 1.0 / (1.0 + np.exp(-logits[b].astype(np.float64)))
        assert bool((np.abs(cc[b, :n] - scores.astype(np.float64)) <= 2 * launch_ref.SIGMOID_REL * scores).all()), b
        assert bool((cc[b, :n] <= 1.0).all()) and p64.size
        if b == 0:                                     # the cut inside the saturated group keeps the lowest indices
            sat = np.nonzero(logits[0, :LENS[0]] >= 17)[0]
            tt = sat[:TOPK].astype(np.float32)
            want = np.stack([tt - offsets[0, sat[:TOPK], 0], tt + offsets[0, sat[:TOPK], 1]], 1)
            ok = (want[:, 1] - want[:, 0]) > np.float32(0.001)
            assert len(sat) > TOPK and (scores[:int(ok.sum())] == 1.0).all()
            assert np.array_equal(segs[:int(ok.sum())], want[ok])
        if b == 2:
            assert n == 0
        if method == "none":
            assert ocn[b] == n and np.array_equal(bits(osg[b, :n]), bits(cs[b, :n])) and np.array_equal(bits(osc[b, :n]), bits(cc[b, :n]))
            continue
        idx, ps, pseg = launch_ref.nms_picks(cs[b, :n], cc[b, :n], THR, MIN_SCORE, SIGMA, 100, method == "soft", 2)
        order = np.argsort(-ps, kind="stable")
        k = len(idx)
        assert ocn[b] == k and np.array_equal(bits(osc[b, :k]), bits(ps[order])) and np.array_equal(bits(osg[b, :k]), bits(pseg[order]))
    PATHS["decode"].update(LENS)


# --------------------------------------------------------------------------------------------- batched_nms front-end
def _many_picks(n=3000, seed=9):
    """Disjoint segments: every candidate is a pick (> 1024 picks), three labels."""
    r = np.random.RandomState(seed)
    k = r.permutation(n).astype(np.float32) * 2
    segs = np.stack([k, k + 1], 1).astype(np.float32)
    sc = (r.randint(4, 17, n) / 16.0).astype(np.float32)
    return torch.from_numpy(segs), torch.from_numpy(sc), torch.from_numpy(r.randint(0, 3, n).astype(np.int64))


@pytest.mark.parametrize("multiclass", [False, True])
@pytest.mark.parametrize("soft", [False, True])
def test_batched_nms_max_seg_num_matches_the_reference(multiclass, soft):
    """libs.utils.nms.batched_nms against nms_ref.batched_nms for max_seg_num 0, -1, 1024, 2000 on lists with more
    than 1024 picks: the same results where the kernel's 1024-pick limit allows them, AvdfError naming the limit where
    it does not - never a silent cut."""
    for n in (900, 1025, 3000):
        segs, sc, cls = _many_picks(n)
        for m in (0, -1, 1024, 2000):
            want = nms_ref.batched_nms(segs, sc, cls, THR, MIN_SCORE, m, use_soft_nms=soft, multiclass=multiclass,
                                       sigma=SIGMA, voting_thresh=0.0)
            per_class = [int((cls == c).sum()) for c in range(3)] if multiclass else [n]
            need = len(want[1]) if not multiclass else max(len(range(p)[:m if m > 0 else None]) for p in per_class)
            if m != 0 and need > 1024:
                with pytest.raises(nv.AvdfError, match="1024"):
                    front.batched_nms(segs, sc, cls, THR, MIN_SCORE, m, use_soft_nms=soft, multiclass=multiclass, sigma=SIGMA,
                                      voting_thresh=0.0)
                continue
            got = front.batched_nms(segs, sc, cls, THR, MIN_SCORE, m, use_soft_nms=soft, multiclass=multiclass, sigma=SIGMA,
                                    voting_thresh=0.0)
            what = "n=%d max_seg_num=%d" % (n, m)
            assert len(got[1]) == len(want[1]), "%s: %d results, reference %d" % (what, len(got[1]), len(want[1]))
            assert torch.equal(got[1], want[1]) and torch.equal(got[0].reshape(-1, 2), want[0].reshape(-1, 2)), what
            assert torch.equal(got[2], want[2]), what


def teardown_module(module):
    print("\nNMS paths reached, by list size:")
    for k in sorted(PATHS):
        print("  %-20s %s" % (k, sorted(PATHS[k])))
    print("voting: worst error / bound %.3g; module time %.1f s" % (VOTING[0], time.time() - T0[0]))
