"""Tensor-level wrappers of the C-ABI entry points (include/avdf.h).

Each function takes CUDA torch tensors (device memory + current stream are all
torch provides), checks shapes/dtypes, and calls straight into
libavdf_sm100.so through `native`. No arithmetic happens in Python.
Layout: activations are token-major [B, T, C]; conv weights are packed
[c_out, taps * c_in] with the tap index outermost inside a row.
"""
import ctypes
from ctypes import c_float, c_int32, c_void_p

import torch

from . import native as nv
from .native import DTYPE_BF16, DTYPE_F16, DTYPE_F32, ACT_NONE, ACT_RELU, ACT_GELU  # noqa: F401


def _dt(t):
    if t.dtype == torch.float32:
        return DTYPE_F32
    if t.dtype == torch.bfloat16:
        return DTYPE_BF16
    if t.dtype == torch.float16:
        return DTYPE_F16
    raise TypeError("unsupported dtype %s" % t.dtype)


# Device of the tensors of the call being marshalled. The library launches on the CURRENT device and takes the stream it is
# given, so every entry point runs with the tensors' device current and on that device's current stream - a model on
# 'cuda:3' (what the reference yaml ships) must not launch on GPU 0.
_dev = [None]


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream(_dev[0]).cuda_stream)


def _chk(t, dtype=None, name="tensor"):
    if t is None:
        return
    if not t.is_cuda:
        raise nv.AvdfError("%s must be a CUDA tensor (no CPU fallback)" % name)
    _dev[0] = t.device
    if not t.is_contiguous():
        raise nv.AvdfError("%s must be contiguous" % name)
    if dtype is not None and t.dtype != dtype:
        raise TypeError("%s must be %s, got %s" % (name, dtype, t.dtype))


class Profile:
    """Optional per-launch CUDA-event timing (bench.py's roofline leg). Off by default: zero overhead."""
    on = False
    records = []          # (entry point, work dict, start event, end event)


def _call(name, fn, args, launches=1, work=None):
    dev = _dev[0]
    if dev is not None and dev.index is not None and dev.index != torch.cuda.current_device():
        with torch.cuda.device(dev):
            return _call_on_current(name, fn, args, launches, work)
    return _call_on_current(name, fn, args, launches, work)


def _call_on_current(name, fn, args, launches, work):
    if Profile.on:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = fn(*args)
        e1.record()
        Profile.records.append((name, work or {}, e0, e1))
    else:
        rc = fn(*args)
    nv.check(rc, name)
    nv.count(launches)


def _nbytes(*ts):
    return sum(t.numel() * t.element_size() for t in ts if t is not None)


def _levels(level_len):
    arr = (c_int32 * len(level_len))(*[int(v) for v in level_len])
    return arr


# ---------------------------------------------------------------------------- K1
def interp_concat(streams, offsets, t_out, out):
    """streams: (video|None, byola|None, emo|None) packed [sum_T, C_s], all fp32 or all bf16 (16-bit feature shards);
    offsets: matching int32 [B+1] row prefix tensors; out [B, t_out, C_total]."""
    L = nv.lib()
    ptrs, offs, cs = [], [], []
    batch = None
    in_dt = next(s.dtype for s in streams if s is not None)
    if in_dt not in (torch.float32, torch.bfloat16):
        raise TypeError("streams must be fp32 or bf16")
    for s, o in zip(streams, offsets):
        if s is None:
            ptrs.append(None); offs.append(None); cs.append(0)
            continue
        _chk(s, in_dt, "stream"); _chk(o, torch.int32, "offsets")
        ptrs.append(nv.ptr(s)); offs.append(nv.ptr(o)); cs.append(s.shape[1])
        batch = o.numel() - 1
    _chk(out, None, "out")
    assert out.shape == (batch, t_out, sum(cs)), (out.shape, batch, t_out, cs)
    _call("avdf_interp_concat", L.avdf_interp_concat_in, (ptrs[0], ptrs[1], ptrs[2], DTYPE_F32 if in_dt == torch.float32 else DTYPE_BF16,
                                  offs[0], offs[1], offs[2], batch, cs[0], cs[1], cs[2],
                                  t_out, nv.ptr(out), _dt(out), _stream(),), launches=1, work={"bytes": _nbytes(*[t for t in streams if t is not None]) + _nbytes(out)})
    return out


def interp_concat_ranges(streams, start, count, t_out, out):
    """Row-range form of interp_concat: video b of stream s is rows [start[s, b], start[s, b] + count[s, b]) of
    streams[s]; start / count: int32 [3, B] device tensors (rows of absent streams are ignored). Overlapping ranges
    read the same source rows: the windows of one recording share its one device copy."""
    L = nv.lib()
    cs = [0 if s is None else s.shape[1] for s in streams]
    in_dt = next(s.dtype for s in streams if s is not None)
    if in_dt not in (torch.float32, torch.bfloat16):
        raise TypeError("streams must be fp32 or bf16")
    for s in streams:
        if s is not None:
            _chk(s, in_dt, "stream")
    _chk(start, torch.int32, "start"); _chk(count, torch.int32, "count"); _chk(out, None, "out")
    batch = start.shape[1]
    assert start.shape == (3, batch) and count.shape == (3, batch), (start.shape, count.shape)
    assert out.shape == (batch, t_out, sum(cs)), (out.shape, batch, t_out, cs)
    _call("avdf_interp_concat_ranges", L.avdf_interp_concat_ranges,
          (nv.ptr(streams[0]), nv.ptr(streams[1]), nv.ptr(streams[2]), DTYPE_F32 if in_dt == torch.float32 else DTYPE_BF16,
           nv.ptr(start), nv.ptr(count), batch, cs[0], cs[1], cs[2], t_out, nv.ptr(out), _dt(out), _stream(),),
          launches=1, work=None)
    return out


def pack_feats(feats_ct, out):
    """feats_ct [C, T] fp32 (device) -> out [L, C] token-major, zero-padded rows T..L."""
    L = nv.lib()
    _chk(feats_ct, torch.float32, "feats"); _chk(out, None, "out")
    C, T = feats_ct.shape
    assert out.shape[1] == C and out.shape[0] >= T
    _call("avdf_pack_feats", L.avdf_pack_feats, (nv.ptr(feats_ct), C, T, out.shape[0], nv.ptr(out), _dt(out), _stream(),), launches=1, work=None)


# ---------------------------------------------------------------------------- NMS
def nms_hard(segs, scores, iou_threshold, max_num=0):
    """nms_1d_cpu.nms on device tensors -> kept indices (int64, device)."""
    L = nv.lib()
    _chk(segs, torch.float32, "segs"); _chk(scores, torch.float32, "scores")
    n = scores.numel()
    out_idx = torch.empty(max(n, 1), dtype=torch.int64, device=scores.device)
    out_count = torch.zeros(1, dtype=torch.int32, device=scores.device)
    wsb = L.avdf_nms_workspace_bytes(n)
    ws = torch.empty(max(wsb, 1), dtype=torch.uint8, device=scores.device)
    _call("avdf_nms_hard", L.avdf_nms_hard, (nv.ptr(segs), nv.ptr(scores), n, float(iou_threshold), int(max_num), nv.ptr(out_idx),
                             nv.ptr(out_count), nv.ptr(ws), wsb, _stream(),), launches=1, work=None)
    return out_idx[: int(out_count.item())]


def nms_soft(segs, scores, dets, iou_threshold, sigma, min_score, method, max_num=0):
    """nms_1d_cpu.softnms on device tensors: writes dets[:K] in place, returns indices."""
    L = nv.lib()
    _chk(segs, torch.float32, "segs"); _chk(scores, torch.float32, "scores"); _chk(dets, torch.float32, "dets")
    n = scores.numel()
    out_idx = torch.empty(max(n, 1), dtype=torch.int64, device=scores.device)
    out_count = torch.zeros(1, dtype=torch.int32, device=scores.device)
    wsb = L.avdf_nms_workspace_bytes(n)
    ws = torch.empty(max(wsb, 1), dtype=torch.uint8, device=scores.device)
    _call("avdf_nms_soft", L.avdf_nms_soft, (nv.ptr(segs), nv.ptr(scores), n, nv.ptr(dets), float(iou_threshold), float(sigma),
                             float(min_score), int(method), int(max_num), nv.ptr(out_idx), nv.ptr(out_count),
                             nv.ptr(ws), wsb, _stream(),), launches=1, work=None)
    return out_idx[: int(out_count.item())]


def postprocess(batch, *, logits=None, offsets=None, mask=None, level_len=(), level_stride=(), pre_nms_thresh=0.001,
                pre_nms_topk=2000, duration_thresh=0.001, cand_segs, cand_scores, cand_count, iou_threshold, min_score,
                sigma, voting_thresh, max_seg_num, use_soft_nms, soft_method=2, vid_meta=None, out_segs, out_scores,
                out_count, workspace=None, records=None, out_index=None):
    """Fused decode + batched_nms (class-agnostic) + seconds conversion; one CTA per video. use_soft_nms: True / False,
    or None for nms_method 'none' (the decoded candidates, out_* sized cand_cap). records: optional
    (ring [cap, 3 + 3K] f32, counter [1] i32, vid_index [B] i32 | None, vid_cls [B] f32 | None)."""
    L = nv.lib()
    a = nv.PostprocessArgs()
    a.batch = batch
    if logits is not None:
        _chk(logits, torch.float32, "logits"); _chk(offsets, torch.float32, "offsets"); _chk(mask, torch.uint8, "mask")
        a.logits, a.offsets, a.mask = logits.data_ptr(), offsets.data_ptr(), mask.data_ptr()
        a.n_levels = len(level_len)
        for i, (n, s) in enumerate(zip(level_len, level_stride)):
            a.level_len[i] = int(n); a.level_stride[i] = float(s)
    a.pre_nms_thresh, a.pre_nms_topk, a.duration_thresh = float(pre_nms_thresh), int(pre_nms_topk), float(duration_thresh)
    _chk(cand_segs, torch.float32, "cand_segs"); _chk(cand_scores, torch.float32, "cand_scores"); _chk(cand_count, torch.int32, "cand_count")
    a.cand_segs, a.cand_scores, a.cand_count = cand_segs.data_ptr(), cand_scores.data_ptr(), cand_count.data_ptr()
    a.cand_cap = cand_scores.shape[1]
    a.iou_threshold, a.min_score, a.sigma, a.voting_thresh = float(iou_threshold), float(min_score), float(sigma), float(voting_thresh)
    a.max_seg_num, a.use_soft_nms, a.soft_method = int(max_seg_num), (-1 if use_soft_nms is None else int(bool(use_soft_nms))), int(soft_method)
    if records is not None:
        ring, counter, vidx, vcls = records
        _chk(ring, torch.float32, "rec_ring"); _chk(counter, torch.int32, "rec_counter"); _chk(vidx, torch.int32, "vid_index"); _chk(vcls, torch.float32, "vid_cls")
        if ring.shape[1] != 3 + 3 * int(max_seg_num):
            raise ValueError("record rows must hold 3 + 3 * max_seg_num floats")
        a.rec_ring, a.rec_counter, a.rec_cap = ring.data_ptr(), counter.data_ptr(), ring.shape[0]
        a.vid_index = vidx.data_ptr() if vidx is not None else None
        a.vid_cls = vcls.data_ptr() if vcls is not None else None
    if vid_meta is not None:
        for t in vid_meta:
            _chk(t, torch.float32, "vid_meta")
        a.vid_feat_stride, a.vid_half_nframes, a.vid_fps, a.vid_duration = [t.data_ptr() for t in vid_meta]
    _chk(out_segs, torch.float32, "out_segs"); _chk(out_scores, torch.float32, "out_scores"); _chk(out_count, torch.int32, "out_count")
    a.out_segs, a.out_scores, a.out_count = out_segs.data_ptr(), out_scores.data_ptr(), out_count.data_ptr()
    _chk(out_index, torch.int32, "out_index")
    a.out_index = out_index.data_ptr() if out_index is not None else None
    need = L.avdf_postprocess_workspace_bytes(batch, a.cand_cap)
    if need:
        if workspace is None or workspace.numel() * workspace.element_size() < need:
            workspace = torch.empty(need, dtype=torch.uint8, device=out_segs.device)
        a.workspace, a.workspace_bytes = workspace.data_ptr(), need
    _call("avdf_postprocess", L.avdf_postprocess, (ctypes.byref(a), _stream(),), launches=1, work=None)


def window_merge(rec_win, win_start, win_segs, win_scores, win_count, win_cls, *, cand_cap, iou_threshold, min_score, sigma,
                 voting_thresh, use_soft_nms, out_segs, out_scores, out_count, out_cls, workspace=None, records=None):
    """Cross-window merge (csrc/window.cu): rec_win int32 [R+1] windows per recording (CSR), win_start fp32 [W] seconds,
    window outputs win_segs [W, K, 2] / win_scores [W, K] / win_count [W] / win_cls [W] -> out_* [R, ...].
    records: optional (ring [cap, 3 + 3K] f32, counter [1] i32, vid_index [R] i32)."""
    L = nv.lib()
    a = nv.WindowMergeArgs()
    R = rec_win.numel() - 1
    K = win_scores.shape[1]
    for t, dt, name in ((rec_win, torch.int32, "rec_win"), (win_start, torch.float32, "win_start"), (win_segs, torch.float32, "win_segs"),
                        (win_scores, torch.float32, "win_scores"), (win_count, torch.int32, "win_count"), (win_cls, torch.float32, "win_cls"),
                        (out_segs, torch.float32, "out_segs"), (out_scores, torch.float32, "out_scores"),
                        (out_count, torch.int32, "out_count"), (out_cls, torch.float32, "out_cls")):
        _chk(t, dt, name)
    a.n_rec, a.rec_win, a.win_start = R, rec_win.data_ptr(), win_start.data_ptr()
    a.win_segs, a.win_scores, a.win_count, a.win_cls = win_segs.data_ptr(), win_scores.data_ptr(), win_count.data_ptr(), win_cls.data_ptr()
    a.cand_cap = int(cand_cap)
    a.iou_threshold, a.min_score, a.sigma, a.voting_thresh = float(iou_threshold), float(min_score), float(sigma), float(voting_thresh)
    a.max_seg_num, a.use_soft_nms = K, int(bool(use_soft_nms))
    a.out_segs, a.out_scores, a.out_count, a.out_cls = out_segs.data_ptr(), out_scores.data_ptr(), out_count.data_ptr(), out_cls.data_ptr()
    if records is not None:
        ring, counter, vidx = records
        _chk(ring, torch.float32, "rec_ring"); _chk(counter, torch.int32, "rec_counter"); _chk(vidx, torch.int32, "vid_index")
        if ring.shape[1] != 3 + 3 * K:
            raise ValueError("record rows must hold 3 + 3 * max_seg_num floats")
        a.rec_ring, a.rec_counter, a.rec_cap = ring.data_ptr(), counter.data_ptr(), ring.shape[0]
        a.vid_index = vidx.data_ptr() if vidx is not None else None
    need = L.avdf_window_merge_workspace_bytes(R, a.cand_cap)
    if need and (workspace is None or workspace.numel() * workspace.element_size() < need):
        workspace = torch.empty(need, dtype=torch.uint8, device=out_segs.device)
    if need:
        a.workspace, a.workspace_bytes = workspace.data_ptr(), need
    _call("avdf_window_merge", L.avdf_window_merge, (ctypes.byref(a), _stream(),), launches=3, work=None)


def postprocess_workspace_bytes(batch, cand_cap):
    return nv.lib().avdf_postprocess_workspace_bytes(batch, cand_cap)


def postprocess_sweep(logits, offsets, valid_len, *, level_len, level_stride, settings, out_rows, vid_meta=None, vid_cls=None,
                      vid_index=None, workspace=None):
    """Post-processing of the same dense outputs under up to 64 settings in one launch (include/avdf.h
    avdf_postprocess_sweep). logits [B, P] / offsets [B, P, 2] fp32, valid_len int32 [B]; settings: sequence of
    nv.SweepSetting; out_rows fp32 [S, R, 3 + 3K] (video b of setting s -> out_rows[s, vid_index[b] or b]).
    vid_meta: optional 4 fp32 [B] tensors (feat_stride, half frames, fps, duration). Returns the workspace used."""
    L = nv.lib()
    _chk(logits, torch.float32, "logits"); _chk(offsets, torch.float32, "offsets"); _chk(valid_len, torch.int32, "valid_len")
    _chk(out_rows, torch.float32, "out_rows"); _chk(vid_cls, torch.float32, "vid_cls"); _chk(vid_index, torch.int32, "vid_index")
    B, P = logits.shape
    S = len(settings)
    assert offsets.shape == (B, P, 2) and valid_len.numel() == B and out_rows.dim() == 3 and out_rows.shape[0] == S
    a = nv.PostprocessSweepArgs()
    a.batch, a.logits, a.offsets, a.valid_len = B, logits.data_ptr(), offsets.data_ptr(), valid_len.data_ptr()
    a.n_levels = len(level_len)
    for i, (n, s) in enumerate(zip(level_len, level_stride)):
        a.level_len[i] = int(n); a.level_stride[i] = float(s)
    if vid_meta is not None:
        for t in vid_meta:
            _chk(t, torch.float32, "vid_meta")
        a.vid_feat_stride, a.vid_half_nframes, a.vid_fps, a.vid_duration = [t.data_ptr() for t in vid_meta]
    a.vid_cls = vid_cls.data_ptr() if vid_cls is not None else None
    a.vid_index = vid_index.data_ptr() if vid_index is not None else None
    table = (nv.SweepSetting * max(1, S))(*settings)
    a.n_settings, a.settings = S, table
    a.out_rows, a.rows_per_setting, a.row_k = out_rows.data_ptr(), out_rows.shape[1], (out_rows.shape[2] - 3) // 3
    need = L.avdf_postprocess_sweep_workspace_bytes(B, P)
    if need and (workspace is None or workspace.numel() * workspace.element_size() < need):
        workspace = torch.empty(need, dtype=torch.uint8, device=logits.device)
    if need:
        a.workspace, a.workspace_bytes = workspace.data_ptr(), need
    _call("avdf_postprocess_sweep", L.avdf_postprocess_sweep, (ctypes.byref(a), _stream(),), launches=1, work=None)
    return workspace


# ---------------------------------------------------------------------------- conv GEMM
def conv_gemm(a, w, *, taps, stride=1, batch, c_in, n_out, segs, a_rows, o_rows, bias=None, row_mask=None, ln=None,
              act=ACT_NONE, pe=None, residual=None, gamma=None, out_f32=None, out_h=None, workspace=None,
              ln_after_residual=False, tap_mode=0, dots=None, tap_rows=None):
    """segs: list of (t_out, a_row, o_row[, w_row]) per segment. a: [batch, a_rows, c_in]; w: [n_w_rows, taps*c_in]
    (same dtype as a: fp32 -> CUDA-core parity path, bf16 / fp16 -> tcgen05 path). Outputs [batch, o_rows, n_out]:
    out_f32 and/or out_h (a bf16 or fp16 copy)."""
    L = nv.lib()
    _chk(a, None, "a"); _chk(w, a.dtype, "w")
    g = nv.ConvGemmArgs()
    g.batch, g.n_out, g.c_in, g.taps, g.stride, g.n_seg = batch, n_out, c_in, taps, stride, len(segs)
    for i, sg in enumerate(segs):
        g.seg_t_out[i], g.seg_a_row[i], g.seg_o_row[i] = int(sg[0]), int(sg[1]), int(sg[2])
        g.seg_w_row[i] = int(sg[3]) if len(sg) > 3 else 0
    g.n_w_rows = w.shape[0]
    g.a_rows_per_video, g.o_rows_per_video = int(a_rows), int(o_rows)
    g.a, g.w, g.dtype = a.data_ptr(), w.data_ptr(), _dt(a)
    for name, t in (("bias", bias), ("pe", pe), ("residual", residual), ("gamma", gamma)):
        _chk(t, torch.float32, name)
    _chk(row_mask, torch.uint8, "row_mask")
    g.bias = bias.data_ptr() if bias is not None else None
    g.row_mask = row_mask.data_ptr() if row_mask is not None else None
    if ln is not None:
        _chk(ln[0], torch.float32, "ln_w"); _chk(ln[1], torch.float32, "ln_b")
        g.ln_w, g.ln_b = ln[0].data_ptr(), ln[1].data_ptr()
    g.act = act
    g.ln_after_residual, g.tap_mode = int(bool(ln_after_residual)), int(tap_mode)
    if dots is not None:                 # (dot_w [n, n_out] fp32, dot_out [batch, o_rows, n] fp32): row dot products of the result
        _chk(dots[0], torch.float32, "dot_w"); _chk(dots[1], torch.float32, "dot_out")
        assert dots[0].shape[1] == n_out and dots[1].shape[-1] == dots[0].shape[0]
        g.dot_w, g.dot_n, g.dot_out = dots[0].data_ptr(), dots[0].shape[0], dots[1].data_ptr()
    if tap_rows is not None:             # explicit row offset per tap (a 3x3 Conv2d over a flattened, padded grid)
        assert len(tap_rows) == taps
        tr = (c_int32 * taps)(*[int(v) for v in tap_rows])
        g.tap_rows = tr
    g.pe = pe.data_ptr() if pe is not None else None
    g.residual = residual.data_ptr() if residual is not None else None
    g.gamma = gamma.data_ptr() if gamma is not None else None
    _chk(out_f32, torch.float32, "out_f32"); _chk(out_h, None, "out_h")
    g.out_f32 = out_f32.data_ptr() if out_f32 is not None else None
    if out_h is not None:
        if out_h.dtype not in (torch.bfloat16, torch.float16):
            raise TypeError("out_h must be bf16 or fp16")
        g.out_h, g.out_h_dtype = out_h.data_ptr(), _dt(out_h)
    need = L.avdf_conv_gemm_workspace_bytes(ctypes.byref(g))
    if need:
        if workspace is None or workspace.numel() * workspace.element_size() < need:
            workspace = torch.empty(need, dtype=torch.uint8, device=a.device)
        g.workspace, g.workspace_bytes = workspace.data_ptr(), workspace.numel() * workspace.element_size()
    _call("avdf_conv_gemm", L.avdf_conv_gemm, (ctypes.byref(g), _stream(),), launches=2 if g.dtype == DTYPE_F32 else 1, work={"flops": 2.0 * batch * sum(sg[0] for sg in segs) * n_out * taps * c_in, "m": batch * sum(sg[0] for sg in segs), "n": n_out, "k": taps * c_in,
                "bytes": _nbytes(a, w, out_f32, out_h, residual)})


# ---------------------------------------------------------------------------- block kernels
def mlp_fused(x, w1, b1, w2, b2, *, row_mask, residual, gamma, out, out_h=None, out_h_level=None, proj=None):
    """out = residual*mask + gamma * ((GELU(x w1^T + b1) w2^T + b2) * mask); x [..., 256] fp16|bf16, w1 [1024, 256],
    w2 [256, 1024] of the same dtype, residual / out fp32 [..., 256]. One launch; the hidden activations stay on chip.
    proj = (att, w_o, b_o, gamma_attn, (ln2_w, ln2_b), skip, y | None): the block tail - the attention projection and LN2 in
    the same launch, the residual stream y kept in the accumulator: w2 / b2 must come pre-scaled by the MLP's scale and
    gamma must be None; x may be None (its dtype is att's), residual is ignored."""
    L = nv.lib()
    if proj is not None:
        x = proj[0] if x is None else x
        residual = proj[5]                 # (placeholder for the checks below: the kernel ignores it)
    _chk(x, None, "x"); _chk(w1, x.dtype, "w1"); _chk(w2, x.dtype, "w2")
    _chk(b1, torch.float32, "b1"); _chk(b2, torch.float32, "b2"); _chk(gamma, torch.float32, "gamma")
    _chk(row_mask, torch.uint8, "row_mask"); _chk(residual, torch.float32, "residual"); _chk(out, torch.float32, "out")
    C, H = x.shape[-1], w1.shape[0]
    rows = x.numel() // C
    assert w1.shape == (H, C) and w2.shape == (C, H) and out.numel() == rows * C and residual.numel() == rows * C
    a = nv.MlpFusedArgs()
    a.rows, a.channels, a.hidden, a.dtype = rows, C, H, _dt(x)
    a.x, a.w1, a.w2 = x.data_ptr(), w1.data_ptr(), w2.data_ptr()
    a.b1 = b1.data_ptr() if b1 is not None else None
    a.b2 = b2.data_ptr() if b2 is not None else None
    a.row_mask = row_mask.data_ptr() if row_mask is not None else None
    a.gamma = gamma.data_ptr() if gamma is not None else None
    a.residual, a.out = residual.data_ptr(), out.data_ptr()
    _chk(out_h, x.dtype, "out_h")
    a.out_h = out_h.data_ptr() if out_h is not None else None
    if out_h_level is not None:          # (t, pitch, row0): out_h is a [batch, pitch, C] pyramid buffer, this level at row0
        a.out_h_t, a.out_h_pitch, a.out_h_row0 = [int(v) for v in out_h_level]
    flops, nbytes = 4.0 * rows * C * H, rows * C * (x.element_size() + 8) + 2 * C * H * x.element_size()
    if proj is not None:
        att, w_o, b_o, ga, ln2, skip, y = proj
        _chk(att, x.dtype, "att"); _chk(w_o, x.dtype, "w_o"); _chk(b_o, torch.float32, "b_o"); _chk(ga, torch.float32, "gamma_attn")
        _chk(ln2[0], torch.float32, "ln2_w"); _chk(ln2[1], torch.float32, "ln2_b"); _chk(skip, torch.float32, "skip"); _chk(y, torch.float32, "y")
        assert att.numel() == rows * C and skip.numel() == rows * C and (y is None or y.numel() == rows * C) and w_o.shape == (C, C)
        assert gamma is None, "block tail: fold the MLP's scale into w2 / b2"
        a.att, a.w_o, a.skip = att.data_ptr(), w_o.data_ptr(), skip.data_ptr()
        a.y = y.data_ptr() if y is not None else None
        a.b_o = b_o.data_ptr() if b_o is not None else None
        a.gamma_attn = ga.data_ptr() if ga is not None else None
        a.ln2_w, a.ln2_b = ln2[0].data_ptr(), ln2[1].data_ptr()
        flops += 2.0 * rows * C * C
        nbytes += C * C * x.element_size() - rows * C * x.element_size()   # att in instead of x in (+ skip in counted as the residual), + Wo
    _call("avdf_mlp_fused", L.avdf_mlp_fused, (ctypes.byref(a), _stream(),), launches=1,
          work={"flops": flops, "bytes": nbytes, "m": rows, "n": C, "k": H})
    return out


def ln_dwconv_ln(src, *, batch, t_src, t_virt, shift, stride, mask_out, ln_in, dw, ln_out, outs, skip_out=None, out_rows=0,
                 out_row_offsets=None, tile_rows=0):
    """ln_in / ln_out: lists of (w, b); dw: list of [C,3]; outs: list of output tensors. Dense: each
    [batch, t_virt/stride, C]. Interleaved: every entry is the SAME base tensor [batch, out_rows, C] and
    out_row_offsets[i] is the first row of stream i inside a video's block."""
    L = nv.lib()
    _chk(src, torch.float32, "src"); _chk(mask_out, torch.uint8, "mask_out"); _chk(skip_out, torch.float32, "skip_out")
    n = len(outs)
    a = nv.LnDwconvLnArgs()
    a.batch, a.channels, a.t_src, a.t_virt, a.shift, a.stride, a.n_streams = batch, src.shape[-1], t_src, t_virt, shift, stride, n
    a.src = src.data_ptr()
    a.mask_out = mask_out.data_ptr() if mask_out is not None else None
    for i in range(n):
        for t in (ln_in[i][0], ln_in[i][1], dw[i], ln_out[i][0], ln_out[i][1]):
            _chk(t, torch.float32, "param")
        _chk(outs[i], outs[0].dtype, "out")
        a.ln_in_w[i], a.ln_in_b[i] = ln_in[i][0].data_ptr(), ln_in[i][1].data_ptr()
        a.dw_w[i] = dw[i].data_ptr()
        a.ln_out_w[i], a.ln_out_b[i] = ln_out[i][0].data_ptr(), ln_out[i][1].data_ptr()
        a.out[i] = outs[i].data_ptr() + (out_row_offsets[i] * src.shape[-1] * outs[i].element_size() if out_row_offsets else 0)
    a.out_dtype = _dt(outs[0])
    a.out_rows_per_video = int(out_rows)
    a.skip_out = skip_out.data_ptr() if skip_out is not None else None
    a.tile_rows = int(tile_rows)
    C, t_out = src.shape[-1], t_virt // stride
    nbytes = batch * min(t_src, t_virt) * C * 4 + n * batch * t_out * C * outs[0].element_size() + (batch * t_out * C * 4 if skip_out is not None else 0)
    _call("avdf_ln_dwconv_ln", L.avdf_ln_dwconv_ln, (ctypes.byref(a), _stream(),), launches=1, work={"bytes": nbytes})


def attention(q, k, v, kv_mask, out, *, batch, t, n_head, window, qkv=None):
    """q, k, v: [batch, t, C] each, or `qkv` = one [batch, 3t, C] tensor holding a video's q rows, k rows, v rows."""
    L = nv.lib()
    rpv = 0
    if qkv is not None:
        _chk(qkv, None, "qkv")
        C, es = qkv.shape[-1], qkv.element_size()
        base = qkv.data_ptr()
        qp, kp, vp = (c_void_p(base + i * t * C * es) for i in range(3))
        q, rpv = qkv, 3 * t
    else:
        _chk(q, None, "q"); _chk(k, q.dtype, "k"); _chk(v, q.dtype, "v")
        qp, kp, vp = nv.ptr(q), nv.ptr(k), nv.ptr(v)
    _chk(out, None, "out"); _chk(kv_mask, torch.uint8, "kv_mask")
    _call("avdf_attention", L.avdf_attention, (qp, kp, vp, nv.ptr(kv_mask), nv.ptr(out), _dt(q), _dt(out), batch, t, rpv,
                              q.shape[-1], n_head, window, _stream(),), launches=1, work={"bytes": (_nbytes(qkv) if qkv is not None else _nbytes(q, k, v)) + _nbytes(out)})


def ln_rows(x, w, b, out, rows):
    L = nv.lib()
    _chk(x, torch.float32, "x"); _chk(w, torch.float32, "w"); _chk(b, torch.float32, "b"); _chk(out, None, "out")
    _call("avdf_ln_rows", L.avdf_ln_rows, (nv.ptr(x), nv.ptr(w), nv.ptr(b), nv.ptr(out), _dt(out), rows, x.shape[-1], _stream(),), launches=1, work={"bytes": rows * x.shape[-1] * (4 + out.element_size())})


def instnorm_lrelu(x, out, *, batch, t, channels, slope=0.2):
    L = nv.lib()
    _chk(x, torch.float32, "x"); _chk(out, None, "out")
    _call("avdf_instnorm_lrelu", L.avdf_instnorm_lrelu, (nv.ptr(x), nv.ptr(out), _dt(out), batch, t, channels, float(slope), _stream(),), launches=1, work={"bytes": batch * t * channels * (4 + out.element_size())})


def fpn_fuse(lat, mask, dw_w, ln_w, ln_b, out, *, batch, level_len):
    L = nv.lib()
    _chk(lat, torch.float32, "lat"); _chk(mask, torch.uint8, "mask"); _chk(dw_w, torch.float32, "dw_w"); _chk(out, None, "out")
    _call("avdf_fpn_fuse", L.avdf_fpn_fuse, (nv.ptr(lat), nv.ptr(mask), nv.ptr(dw_w), nv.ptr(ln_w), nv.ptr(ln_b), nv.ptr(out), _dt(out), batch,
                             lat.shape[-1], len(level_len), _levels(level_len), _stream(),), launches=1, work={"bytes": _nbytes(lat, out)})


def head_final(cls_feat, reg_feat, mask, cls_w, cls_b, reg_w, reg_b, level_scale, logits, offsets, *, batch, level_len):
    L = nv.lib()
    _chk(cls_feat, None, "cls_feat"); _chk(reg_feat, cls_feat.dtype, "reg_feat"); _chk(mask, torch.uint8, "mask")
    for t in (cls_w, cls_b, reg_w, reg_b, logits, offsets):
        _chk(t, torch.float32, "head tensor")
    sc = (c_float * len(level_scale))(*[float(s) for s in level_scale])
    _call("avdf_head_final", L.avdf_head_final, (nv.ptr(cls_feat), nv.ptr(reg_feat), _dt(cls_feat), nv.ptr(mask), nv.ptr(cls_w), nv.ptr(cls_b),
                               nv.ptr(reg_w), nv.ptr(reg_b), sc, nv.ptr(logits), nv.ptr(offsets), batch, cls_feat.shape[-1],
                               len(level_len), _levels(level_len), _stream(),), launches=1, work=None)


def head_combine(cls_dots, reg_dots, mask, cls_b, reg_b, level_scale, logits, offsets, *, batch, level_len):
    """logits / offsets from the per-tap partial sums the last tower layers emit (conv_gemm dots=...)."""
    L = nv.lib()
    for t in (cls_dots, reg_dots, cls_b, reg_b, logits, offsets):
        _chk(t, torch.float32, "head tensor")
    _chk(mask, torch.uint8, "mask")
    assert cls_dots.shape[-1] == 3 and reg_dots.shape[-1] == 6
    sc = (c_float * len(level_scale))(*[float(s) for s in level_scale])
    _call("avdf_head_combine", L.avdf_head_combine, (nv.ptr(cls_dots), nv.ptr(reg_dots), nv.ptr(mask), nv.ptr(cls_b), nv.ptr(reg_b), sc,
                               nv.ptr(logits), nv.ptr(offsets), batch, len(level_len), _levels(level_len), _stream(),), launches=1, work=None)


def vcls_exp12(z, conv0_w, lin1_w, ln_w, ln_b, lin2_w, lin2_b, out, *, batch, t):
    L = nv.lib()
    _chk(z, None, "z")
    for x in (conv0_w, lin1_w, ln_w, ln_b, lin2_w, lin2_b, out):
        _chk(x, torch.float32, "vcls tensor")
    _call("avdf_vcls_exp12", L.avdf_vcls_exp12, (nv.ptr(z), _dt(z), nv.ptr(conv0_w), nv.ptr(lin1_w), nv.ptr(ln_w), nv.ptr(ln_b), nv.ptr(lin2_w),
                               nv.ptr(lin2_b), nv.ptr(out), batch, t, z.shape[-1], _stream(),), launches=1, work=None)


def vcls_exp13(z, conv0_w, seg_w, seg_b, cls_w, cls_b, out, *, batch, t):
    L = nv.lib()
    _chk(z, None, "z")
    for x in (conv0_w, seg_w, seg_b, cls_w, cls_b, out):
        _chk(x, torch.float32, "vcls tensor")
    _call("avdf_vcls_exp13", L.avdf_vcls_exp13, (nv.ptr(z), _dt(z), nv.ptr(conv0_w), nv.ptr(seg_w), nv.ptr(seg_b), nv.ptr(cls_w), nv.ptr(cls_b),
                               nv.ptr(out), batch, t, z.shape[-1], _stream(),), launches=1, work=None)


# ---------------------------------------------------------------------------- BYOL-A extractor (SURVEY 8(f).4)
def logmel(wav, clip_sample_off, clip_frame_off, clip_pair_off, total_pairs, window, twiddle, mel, lms, *, mean, std):
    """wav: the clips back to back (fp32); lms [total_frames, 64] receives the normalised log-mel rows.
    mel = (lo int32 [64], cnt int32 [64], w fp32 [64, stride]): the mel triangles in sparse form."""
    L = nv.lib()
    mel_lo, mel_cnt, mel_w = mel
    for t, n in ((wav, "wav"), (window, "window"), (twiddle, "twiddle"), (mel_w, "mel_w"), (lms, "lms")):
        _chk(t, torch.float32, n)
    _chk(clip_sample_off, torch.int64, "clip_sample_off")
    for t in (clip_frame_off, clip_pair_off, mel_lo, mel_cnt):
        _chk(t, torch.int32, "index array")
    assert window.numel() == 1024 and twiddle.numel() == 2048 and mel_lo.numel() == 64 and mel_cnt.numel() == 64 and mel_w.shape[0] == 64
    n_clips, frames = clip_frame_off.numel() - 1, lms.shape[0]
    _call("avdf_logmel", L.avdf_logmel, (nv.ptr(wav), nv.ptr(clip_sample_off), nv.ptr(clip_frame_off), nv.ptr(clip_pair_off), n_clips, frames,
                                         int(total_pairs), nv.ptr(window), nv.ptr(twiddle), nv.ptr(mel_lo), nv.ptr(mel_cnt), nv.ptr(mel_w),
                                         int(mel_w.shape[1]), float(mean), float(std), nv.ptr(lms), _stream(),),
          launches=1, work={"bytes": _nbytes(wav, lms), "flops": frames * (5.0 * 1024 * 10 / 2 + 2.0 * 970)})


def byola_conv1_pool(lms, clip_frame_off, w, b, clip_of_step, t_of_step, out, mask_out=None):
    L = nv.lib()
    _chk(lms, torch.float32, "lms"); _chk(w, torch.float32, "w"); _chk(b, torch.float32, "b"); _chk(out, None, "out")
    for t in (clip_frame_off, clip_of_step, t_of_step):
        _chk(t, torch.int32, "index array")
    _chk(mask_out, torch.uint8, "mask_out")
    n_steps = clip_of_step.numel()
    assert out.numel() == n_steps * 34 * 64 and w.numel() == 64 * 9
    _call("avdf_byola_conv1_pool", L.avdf_byola_conv1_pool, (nv.ptr(lms), nv.ptr(clip_frame_off), nv.ptr(w), nv.ptr(b), nv.ptr(clip_of_step),
          nv.ptr(t_of_step), n_steps, nv.ptr(out), _dt(out), nv.ptr(mask_out) if mask_out is not None else None, _stream(),),
          launches=1, work={"bytes": _nbytes(lms, out)})


def byola_pool(x, clip_step_in, clip_of_step, t_of_step, out, *, mel_in, pad_out, mask_out=None):
    L = nv.lib()
    _chk(x, None, "x"); _chk(out, x.dtype, "out"); _chk(mask_out, torch.uint8, "mask_out")
    for t in (clip_step_in, clip_of_step, t_of_step):
        _chk(t, torch.int32, "index array")
    n_steps = clip_of_step.numel()
    assert out.numel() == n_steps * (mel_in // 2 + 2 * pad_out) * 64
    _call("avdf_byola_pool", L.avdf_byola_pool, (nv.ptr(x), _dt(x), mel_in, nv.ptr(clip_step_in), nv.ptr(clip_of_step), nv.ptr(t_of_step), n_steps,
          int(pad_out), nv.ptr(out), nv.ptr(mask_out) if mask_out is not None else None, _stream(),), launches=1, work={"bytes": _nbytes(x, out)})


# ---------------------------------------------------------------------------- detection evaluation (one class)
def eval_detection(pred_off, pred_seg, pred_score, gt_off, gt_seg, thresholds, top_k, *, tp_mask=None, pred_rank=None,
                   workspace=None, check_status=True):
    """ActivityNet AP per tIoU threshold + Recall@kx hit counts of one class, videos in CSR form (include/avdf.h
    avdf_eval_detection): pred_off int64 [V+1], pred_seg fp64 [N, 2], pred_score fp64 [N], gt_off int32 [V+1],
    gt_seg fp64 [G, 2] (G >= 1); thresholds / top_k host sequences. tp_mask: optional uint16 [N] output. pred_rank:
    optional int32 [N] permutation that orders equal scores instead of the CSR position.
    Returns (ap fp64 [n_thr], hits int64 [n_thr, n_topk], status int32 [1]) on the device. check_status reads the status
    word (a synchronisation) and raises AvdfError when a per-video limit was exceeded (no results were written)."""
    L = nv.lib()
    _chk(pred_off, torch.int64, "pred_off"); _chk(pred_seg, torch.float64, "pred_seg"); _chk(pred_score, torch.float64, "pred_score")
    _chk(gt_off, torch.int32, "gt_off"); _chk(gt_seg, torch.float64, "gt_seg"); _chk(tp_mask, torch.uint16, "tp_mask")
    _chk(pred_rank, torch.int32, "pred_rank")
    n, n_video, n_gt = pred_score.numel(), pred_off.numel() - 1, gt_seg.shape[0]
    assert pred_seg.shape == (n, 2) and gt_seg.shape == (n_gt, 2) and gt_off.numel() == n_video + 1
    assert tp_mask is None or tp_mask.numel() == n
    dev = pred_off.device
    thr = [float(t) for t in thresholds]
    ks = [int(k) for k in top_k]
    ap = torch.empty(len(thr), dtype=torch.float64, device=dev)
    hits = torch.empty((len(thr), len(ks)), dtype=torch.int64, device=dev)
    status = torch.empty(1, dtype=torch.int32, device=dev)
    need = L.avdf_eval_workspace_bytes(n, n_video)
    if workspace is None or workspace.numel() * workspace.element_size() < need:
        workspace = torch.empty(need, dtype=torch.uint8, device=dev)
    a = nv.EvalArgs()
    a.n_pred, a.n_video, a.n_gt = n, n_video, n_gt
    a.pred_off, a.pred_seg, a.pred_score = pred_off.data_ptr(), pred_seg.data_ptr() if n else None, pred_score.data_ptr() if n else None
    a.gt_off, a.gt_seg = gt_off.data_ptr(), gt_seg.data_ptr()
    thr_arr, k_arr = (ctypes.c_double * max(1, len(thr)))(*thr), (c_int32 * max(1, len(ks)))(*ks)
    a.thresholds, a.n_thr, a.top_k, a.n_topk = thr_arr, len(thr), k_arr, len(ks)
    a.ap, a.recall_hits, a.status = ap.data_ptr(), hits.data_ptr(), status.data_ptr()
    a.tp_mask = tp_mask.data_ptr() if tp_mask is not None and n else None
    a.pred_rank = pred_rank.data_ptr() if pred_rank is not None and n else None
    a.workspace, a.workspace_bytes = workspace.data_ptr(), workspace.numel() * workspace.element_size()
    _call("avdf_eval_detection", L.avdf_eval_detection, (ctypes.byref(a), _stream(),), launches=1,
          work={"bytes": n * (16 + 8) + n_gt * 16})
    if check_status:
        st = int(status.item())
        if st:
            why = [w for b, w in ((nv.EVAL_PRED_LIMIT, "a video has more than 8192 predictions"),
                                  (nv.EVAL_GT_LIMIT, "a video has more than 64 ground-truth rows"),
                                  (nv.EVAL_BAD_OFFSETS, "malformed CSR offsets")) if st & b]
            raise nv.AvdfError("avdf_eval_detection: %s (status %d); no results were written" % ("; ".join(why), st))
    return ap, hits, status


def eval_proposal(prop_off, prop_seg, prop_score, keep, gt_off, gt_seg, thresholds, an_frac, *, matches=None, workspace=None,
                  check_status=True):
    """ActivityNet proposal matches per tIoU threshold and point of the AR-AN curve, videos in CSR form (include/avdf.h
    avdf_eval_proposal): prop_off int64 [V+1], prop_seg fp64 [N, 2], prop_score fp64 [N], keep int32 [V] (proposals walked
    per video), gt_off int32 [V+1], gt_seg fp64 [G, 2]; thresholds and an_frac (100 values) host sequences. matches: optional
    int64 [n_thr, 100] output. Returns (matches, status int32 [1]) on the device; check_status reads the status word (a
    synchronisation) and raises AvdfError when a per-video check failed (matches was not written)."""
    L = nv.lib()
    _chk(prop_off, torch.int64, "prop_off"); _chk(prop_seg, torch.float64, "prop_seg"); _chk(prop_score, torch.float64, "prop_score")
    _chk(keep, torch.int32, "keep"); _chk(gt_off, torch.int32, "gt_off"); _chk(gt_seg, torch.float64, "gt_seg")
    _chk(matches, torch.int64, "matches")
    n, n_video, n_gt = prop_score.numel(), prop_off.numel() - 1, gt_seg.shape[0]
    assert prop_seg.shape == (n, 2) and gt_seg.shape == (n_gt, 2) and gt_off.numel() == n_video + 1 and keep.numel() == n_video
    dev = prop_off.device
    thr = [float(t) for t in thresholds]
    frac = [float(f) for f in an_frac]
    assert len(frac) == 100, "an_frac must hold the 100 points of the AR-AN curve"
    if matches is None:
        matches = torch.empty((len(thr), 100), dtype=torch.int64, device=dev)
    assert matches.numel() == len(thr) * 100
    status = torch.empty(1, dtype=torch.int32, device=dev)
    need = L.avdf_eval_proposal_workspace_bytes(n_video)
    if workspace is None or workspace.numel() * workspace.element_size() < need:
        workspace = torch.empty(need, dtype=torch.uint8, device=dev)
    a = nv.EvalProposalArgs()
    a.n_video, a.n_prop, a.n_gt = n_video, n, n_gt
    a.prop_off, a.keep, a.gt_off = prop_off.data_ptr(), keep.data_ptr(), gt_off.data_ptr()
    a.prop_seg, a.prop_score = (prop_seg.data_ptr(), prop_score.data_ptr()) if n else (None, None)
    a.gt_seg = gt_seg.data_ptr() if n_gt else None
    thr_arr, frac_arr = (ctypes.c_double * max(1, len(thr)))(*thr), (ctypes.c_double * 100)(*frac)
    a.thresholds, a.n_thr, a.an_frac = thr_arr, len(thr), frac_arr
    a.matches, a.status = matches.data_ptr(), status.data_ptr()
    a.workspace, a.workspace_bytes = workspace.data_ptr(), workspace.numel() * workspace.element_size()
    _call("avdf_eval_proposal", L.avdf_eval_proposal, (ctypes.byref(a), _stream(),), launches=1,
          work={"bytes": n * (16 + 8) + n_gt * 16})
    if check_status:
        st = int(status.item())
        if st:
            why = [w for b, w in ((nv.EVAL_PRED_LIMIT, "a video has more than 8192 proposals"),
                                  (nv.EVAL_GT_LIMIT, "a video has more than 64 ground-truth rows"),
                                  (nv.EVAL_BAD_OFFSETS, "malformed CSR offsets"),
                                  (nv.EVAL_BAD_KEEP, "keep is outside 0 .. proposals of its video")) if st & b]
            raise nv.AvdfError("avdf_eval_proposal: %s (status %d); no results were written" % ("; ".join(why), st))
    return matches, status


# ---------------------------------------------------------------------------- result files (JSON text)
def format_results(mode, records, K, order, ids, id_off, id_bytes_max, pos_begin, n_rows, out, out_bytes, *, min_score=0.2,
                   workspace=None):
    """JSON text of output positions [pos_begin, pos_begin + n_rows) into the uint8 buffer `out`, its byte count into
    int64 out_bytes [1] (include/avdf.h avdf_format_results; -1 when a row was invalid). records fp32 [R, 3 + 3K],
    order int32 [P], ids uint8 blob, id_off int64 [P + 1] (device); mode nv.FORMAT_RECORDS or nv.FORMAT_PREDICTIONS.
    Returns the workspace used (pass it back to reuse it)."""
    L = nv.lib()
    _chk(records, torch.float32, "records"); _chk(order, torch.int32, "order"); _chk(ids, torch.uint8, "ids")
    _chk(id_off, torch.int64, "id_off"); _chk(out, torch.uint8, "out"); _chk(out_bytes, torch.int64, "out_bytes")
    assert records.dim() == 2 and records.shape[1] == 3 + 3 * K and id_off.numel() == order.numel() + 1
    need = L.avdf_format_results_workspace_bytes(n_rows)
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty(need, dtype=torch.uint8, device=records.device)
    a = nv.FormatArgs()
    a.mode, a.K, a.records, a.n_records = mode, K, records.data_ptr(), records.shape[0]
    a.order, a.n_pos, a.ids, a.id_off, a.id_bytes_max = order.data_ptr(), order.numel(), ids.data_ptr(), id_off.data_ptr(), id_bytes_max
    a.pos_begin, a.n_rows, a.min_score = pos_begin, n_rows, float(min_score)
    a.out, a.out_capacity, a.out_bytes = out.data_ptr(), out.numel(), out_bytes.data_ptr()
    a.workspace, a.workspace_bytes = workspace.data_ptr(), workspace.numel()
    _call("avdf_format_results", L.avdf_format_results, (ctypes.byref(a), _stream(),), launches=3,
          work={"bytes": n_rows * records.shape[1] * 4})
    return workspace
