"""Deterministic adversarial inputs for the post-processing kernels (csrc/nms.cu): tied scores, degenerate geometry,
IoU exactly at the threshold, soft-NMS decay edges, and decode inputs with exact probability ties. numpy only, so the
generators and their self-checks (tests/test_postprocess_cases.py) run without a GPU.

Candidate generators take (n, seed, **params) and return (segs [n, 2], scores [n]) float32. The float32 arithmetic of
the kernels is restated here with numpy float32 operations, which are IEEE single operations with round-to-nearest
like the kernel's __fadd_rn / __fsub_rn / __fdiv_rn:
    ar = (x2 - x1) + 1e-6f,  ovr = inter / ((ar_i + ar_j) - inter),  inter = max(0, min(x2_i, x2_j) - max(x1_i, x1_j)).
Decode ties come only from saturated logits (>= 17, where both the device sigmoid and torch's give exactly 1.0f) or from
the same logit value at several points: the device expf may differ from the host's by 2 ulp, so distinct logits are
drawn from a 1/16 grid whose probabilities lie hundreds of ulp apart.
"""
import numpy as np

F32 = np.float32
EPS = F32(1e-6)
NMS_SMEM_CAP = 6144            # csrc/nms.cu: lists up to this size run from shared memory
NMS_CL, NMS_CL_SLICE_MAX = 16, 11264
NMS_THREADS = 512


def cluster_slice(n):
    """Positions per CTA of the 16-CTA cluster path for a list of n (csrc/nms.cu launch_standalone)."""
    return ((n + NMS_CL - 1) // NMS_CL + 31) // 32 * 32


def nms_path(n, cluster=True):
    """The code path avdf_nms_hard / avdf_nms_soft take for a list of n: 'smem', 'cluster' or 'global'."""
    if n <= NMS_SMEM_CAP:
        return "smem"
    return "cluster" if cluster and n <= NMS_CL * NMS_CL_SLICE_MAX else "global"


def ovr_eps(x1i, x2i, x1j, x2j):
    """The kernels' IoU with epsilon'd areas, elementwise in float32."""
    x1i, x2i, x1j, x2j = (np.asarray(v, F32) for v in (x1i, x2i, x1j, x2j))
    ari, arj = (x2i - x1i) + EPS, (x2j - x1j) + EPS
    inter = np.fmax(F32(0), np.fmin(x2i, x2j) - np.fmax(x1i, x1j))
    with np.errstate(divide="ignore", invalid="ignore"):
        return inter / ((ari + arj) - inter)


def _rng(seed):
    return np.random.RandomState(seed)


def _sweep_segs(rng, n, span=768.0, max_len=40.0):
    c = rng.uniform(0, span, n).astype(F32)
    ln = rng.uniform(0.01, max_len, n).astype(F32)
    return np.stack([c - ln / 2, c + ln / 2], 1).astype(F32)


def _grid_scores(rng, n, p_one=0.3):
    """Scores k / 16, k = 0..16, with a share p_one exactly 1.0."""
    s = (rng.randint(0, 17, n) / 16.0).astype(F32)
    s[rng.uniform(size=n) < p_one] = F32(1.0)
    return s


# --------------------------------------------------------------------------------------------- tied scores
def grid_ties(n, seed):
    """Sweep-like segments, scores on a k/16 grid with many exactly 1.0: every pick is a tie break."""
    r = _rng(seed)
    return _sweep_segs(r, n), _grid_scores(r, n)


def min_score_ties(n, seed, min_score=0.2):
    """Groups of scores exactly float32(min_score) (hard NMS drops them: strict '>'; soft NMS keeps them: a failure is
    strict '<'), the rest on the k/16 grid."""
    r = _rng(seed)
    s = _grid_scores(r, n, p_one=0.1)
    s[r.uniform(size=n) < 0.4] = F32(min_score)
    return _sweep_segs(r, n), s


# --------------------------------------------------------------------------------------------- degenerate geometry
def identical_segments(n, seed):
    """About n / 8 distinct segments, each repeated at scattered indices, with grid scores (identical boxes tie)."""
    r = _rng(seed)
    base = _sweep_segs(r, max(1, n // 8))
    return base[r.randint(0, len(base), n)].copy(), _grid_scores(r, n)


def nested_touching(n, seed):
    """Segments nested around shared centres plus chains of touching unit cells [k, k + 1] (intersection exactly 0)."""
    r = _rng(seed)
    half = n // 2
    centres = (r.randint(0, 96, half) * 8).astype(F32)
    radius = (r.randint(1, 33, half) / 4.0).astype(F32)
    nested = np.stack([centres - radius, centres + radius], 1)
    k = r.randint(0, 800, n - half).astype(F32)
    touching = np.stack([k, k + F32(1)], 1)
    segs = np.concatenate([nested, touching]).astype(F32)
    perm = r.permutation(n)
    return segs[perm].copy(), _grid_scores(r, n)


def zero_length(n, seed):
    """A quarter of the segments have x1 == x2 (the candidate path only: decode drops them). Voting with a zero-length
    pick divides 0 by 0."""
    r = _rng(seed)
    segs = _sweep_segs(r, n)
    z = r.uniform(size=n) < 0.25
    segs[z, 1] = segs[z, 0]
    return segs, _grid_scores(r, n)


# --------------------------------------------------------------------------------------------- IoU exactly at the threshold
def exact_iou_pairs(iou_threshold, seed):
    """Segment pairs (i, j) whose float32 ovr_eps is exactly float32(iou_threshold), and pairs whose ovr_eps is the
    next float32 below it. Returns (at [m, 4], below [m', 4]), rows x1_i, x2_i, x1_j, x2_j.
    A pair is found by scanning float32 neighbours of the real-valued solution. The epsilon'd areas make an exact
    quotient rare unless the coordinates' ulp is no coarser than the lengths', so pair k sits at its own scale
    4^m: i = [c, c + l_i] with |c| ~ 4^m and lengths in [4^m / 2, 4^m); pairs of different scales never overlap."""
    r = _rng(seed)
    thr = F32(iou_threshold)
    down = np.nextafter(thr, F32(0))
    t = float(thr)
    at, below = [], []
    k = np.arange(-24, 25).astype(F32)
    for m in range(-2, 9):
        for sign in (1, -1):
            scale = 4.0 ** m
            c = F32(scale if sign > 0 else -3 * scale)            # the pair lies in [scale, 3 scale) or [-3 scale, -scale)
            want, dst = (thr, at) if len(at) <= len(below) else (down, below)
            for _ in range(400):
                li, lj = F32(scale * r.randint(32, 64) / 64), F32(scale * r.randint(32, 64) / 64)
                # j = [c + d, c + d + lj] overlaps the right end of i = [c, c + li]: inter = li - d, union = lj + d
                d = (float(li) - t * float(lj)) / (1.0 + t)
                if not (0.0 < d < float(li) and d + float(lj) > float(li)):
                    continue
                x0 = F32(float(c) + d)
                x2 = F32(x0 + lj)
                x1j = np.repeat((x0 + k * np.spacing(x0)).astype(F32), len(k))      # every (x1_j, x2_j) of ulp steps
                x2j = np.tile((x2 + k * np.spacing(x2)).astype(F32), len(k))
                hit = np.nonzero(ovr_eps(c, c + li, x1j, x2j) == want)[0]
                if len(hit):
                    dst.append((c, F32(c + li), x1j[hit[0]], x2j[hit[0]]))
                    break
    return np.array(at, F32).reshape(-1, 4), np.array(below, F32).reshape(-1, 4)


def exact_iou(n, seed, iou_threshold=0.1):
    """Pairs whose IoU is exactly the threshold (the lower-scored one must be suppressed: '>='), pairs one ulp below
    it (both kept), each pair apart from the others; the rest is grid-score filler far beyond them."""
    r = _rng(seed)
    at, below = exact_iou_pairs(iou_threshold, seed)
    pairs = np.concatenate([at, below]).reshape(-1, 2)
    sc = np.tile(np.array([0.9, 0.6], F32), len(pairs) // 2)
    fill = max(0, n - len(sc))
    fs = _sweep_segs(r, fill) + F32(300000)            # beyond the largest pair scale
    segs = np.concatenate([pairs, fs]).astype(F32)[:n]
    return segs.copy(), np.concatenate([sc, _grid_scores(r, fill)]).astype(F32)[:n].copy()


# --------------------------------------------------------------------------------------------- soft-NMS decay edges
def linear_decay_to_min(count, seed, iou_threshold=0.1, min_score=0.2):
    """Pairs (pick, other) for soft-NMS method 1 where the other's decayed score fl(s * fl(1 - ovr)) is exactly
    float32(min_score) (it survives: a failure is strict '<'), each pair apart from the others. Returns
    (segs [2m, 2], scores [2m])."""
    r = _rng(seed)
    ms = F32(min_score)
    segs, scores = [], []
    tries = 0
    while len(scores) < 2 * count and tries < 100 * count + 100:
        tries += 1
        c = F32(100 * (len(scores) // 2) + r.randint(0, 10))      # pair k in [100 k, 100 k + 60)
        li = F32(r.randint(4, 40) / 2.0)
        d = F32(r.uniform(0.0, 0.5) * li)
        i, j = (c, F32(c + li)), (F32(c + d), F32(c + d + li))
        o = ovr_eps(*i, *j)
        if not o >= F32(iou_threshold):
            continue
        w = F32(1) - o
        s0 = F32(ms / w)
        cand = (s0 + np.arange(-8, 9).astype(F32) * np.spacing(s0)).astype(F32)
        hit = cand[(cand * w == ms) & (cand < F32(1))]
        if len(hit) == 0:
            continue
        segs += [i, j]
        scores += [F32(1.0), hit[0]]
    return np.array(segs, F32).reshape(-1, 2), np.array(scores, F32)


def decay_to_min(n, seed, iou_threshold=0.1, min_score=0.2):
    """Method-1 pairs decayed exactly onto min_score, each in its own region, plus grid-score filler further out."""
    r = _rng(seed)
    segs, scores = linear_decay_to_min(max(0, min(n // 4, 48)), seed, iou_threshold, min_score)
    segs, scores = segs[:n], scores[:n]
    fill = n - len(scores)
    fs = _sweep_segs(r, fill) + F32(20000)
    return np.concatenate([segs, fs]).astype(F32), np.concatenate([scores, _grid_scores(r, fill)]).astype(F32)


def suppress_all(n, seed):
    """Near-identical segments: the first pick overlaps every other one with IoU ~ 1, so with method 0 (and hard NMS)
    everything after it fails at once (F = nsegs - 1). The pick sits at a random index, not at position 0."""
    r = _rng(seed)
    x1 = (F32(100) + (r.randint(0, 4, n) / 64.0)).astype(F32)
    segs = np.stack([x1, x1 + F32(50)], 1).astype(F32)
    s = (r.randint(1, 12, n) / 16.0).astype(F32)
    s[r.randint(0, n)] = F32(1.0)
    return segs, s


def disjoint(n, seed):
    """Disjoint unit segments with scores above min_score: no decay, no failure (the F == 0 step), ties on the grid."""
    r = _rng(seed)
    k = r.permutation(n).astype(F32) * F32(2)
    return np.stack([k, k + F32(1)], 1).astype(F32), (r.randint(4, 17, n) / 16.0).astype(F32)


def chunk_straddle(n, seed):
    """Index 0 is the first pick ([0, 100], score 1.0); about half of the others overlap it (IoU >= 0.5, they fail under
    method 0) and the rest lie beyond it. Failures then fall on every residue of step 4's per-thread chunks of
    ceil((n - 1) / 512) positions, on both chunk ends, and below and above the new end."""
    r = _rng(seed)
    fail = r.uniform(size=n) < 0.5
    fail[0] = False
    a = r.randint(0, 8, n).astype(F32)
    segs = np.where(fail[:, None], np.stack([a, a + F32(96)], 1),
                    np.stack([F32(200) + a * 40, F32(200) + a * 40 + F32(30)], 1)).astype(F32)
    segs[0] = (F32(0), F32(100))
    s = (r.randint(4, 16, n) / 16.0).astype(F32)
    s[0] = F32(1.0)
    return segs, s


FAMILIES = {f.__name__: f for f in (grid_ties, min_score_ties, identical_segments, nested_touching, zero_length, exact_iou,
                                    decay_to_min, suppress_all, disjoint, chunk_straddle)}


# --------------------------------------------------------------------------------------------- decode inputs
def duration_edge_offsets(stride, duration_thresh, points, seed):
    """For each point index t of `points`, offsets (o0, o1) >= 0 with right - left exactly float32(duration_thresh)
    under the kernel's float32 formula (tt = t * s, left = tt - o0 * s, right = tt + o1 * s), or None where the scan
    finds none. The kernel keeps right - left > duration_thresh: these points must be dropped."""
    s, dt = F32(stride), F32(duration_thresh)
    out = []
    for t in points:
        tt = F32(t) * s
        base = F32(dt / s)
        o1 = (base + np.arange(-64, 65).astype(F32) * np.spacing(base)).astype(F32)
        o1 = o1[o1 >= 0]
        right, left = tt + o1 * s, tt - F32(0) * s
        hit = o1[(right - left) == dt]
        out.append(None if len(hit) == 0 else (F32(0), hit[0]))
    return out


def decode_case(seed, level_len, pre_nms_topk, pre_nms_thresh=0.001, duration_thresh=0.001):
    """Five videos over levels `level_len` (strides 2^l), as (logits [5, P], offsets [5, P, 2], mask [5, P] uint8):
      0  saturated: a third of the points have logits >= 17 (probability exactly 1.0f) - in the longest level more
         of them than pre_nms_topk, so the cut falls inside the tied group
      1  duplicated: every logit is one of 7 grid values, so each level is a few groups of exact ties, cut by topk
      2  all points masked
      3  duration edges: every 3rd point has right - left exactly duration_thresh, its neighbour one ulp above
      4  distinct grid logits with a ragged mask tail
    Distinct logits come from a 1/16 grid in [-9, 9]: their probabilities are far apart in ulps, and far from
    pre_nms_thresh, so a 2-ulp expf difference changes no order and no threshold decision."""
    r = _rng(seed)
    P = sum(level_len)
    B = 5
    grid = lambda *shape: (r.randint(-144, 145, shape) / 16.0).astype(F32)
    logits = grid(B, P)
    offsets = (r.randint(0, 64, (B, P, 2)) / 8.0).astype(F32)
    mask = np.ones((B, P), np.uint8)
    sat = r.uniform(size=P) < 0.34
    off = np.cumsum([0] + list(level_len))
    big = int(np.argmax(level_len))
    l0 = off[big]
    need = min(level_len[big], pre_nms_topk + 40)
    sat[l0:l0 + need] = True
    logits[0, sat] = (17 + r.randint(0, 8, int(sat.sum()))).astype(F32)
    vals = np.array([-7.5, -2.0, 0.5, 1.25, 3.0, 6.0, 20.0], F32)
    logits[1] = vals[r.randint(0, len(vals), P)]
    mask[2] = 0
    for l, n in enumerate(level_len):
        pts = list(range(0, n, 3))
        offs = duration_edge_offsets(2.0 ** l, duration_thresh, pts, seed + l)
        for t, o in zip(pts, offs):
            if o is None:
                continue
            offsets[3, off[l] + t] = o
            if t + 1 < n:
                offsets[3, off[l] + t + 1] = (o[0], np.nextafter(o[1], F32(np.inf)))
    logits[3] = np.abs(logits[3]) + F32(1)          # well above pre_nms_thresh: only the duration cut decides
    for l, n in enumerate(level_len):
        cut = (n * 3) // 4
        mask[4, off[l] + cut:off[l + 1]] = 0
    return logits, offsets, mask


def decode_level_strides(level_len):
    return [float(2 ** l) for l in range(len(level_len))]
