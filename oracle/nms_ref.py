"""ctypes front-end of oracle/nms_ref.c + a restatement of
libs/utils/nms.py:8-64,103-190 (NMSop / SoftNMSop / batched_nms dispatch).

TEST INFRASTRUCTURE — see oracle/model_ref.py's header for who may import it.
"""
import ctypes
import os
import subprocess

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "nms_ref.c")
_OUT = os.path.join(_HERE, "_build", "libnms_ref.so")
_lib = None


def build(force=False):
    if force or not os.path.isfile(_OUT) or os.path.getmtime(_OUT) < os.path.getmtime(_SRC):
        os.makedirs(os.path.dirname(_OUT), exist_ok=True)
        subprocess.run(["gcc", "-O2", "-ffp-contract=off", "-shared", "-fPIC", _SRC, "-o", _OUT, "-lm"], check=True)
    return _OUT


def lib():
    global _lib
    if _lib is None:
        L = ctypes.CDLL(build())
        f32p, i64p = ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_int64)
        L.ref_nms_1d.restype = ctypes.c_int64
        L.ref_nms_1d.argtypes = [f32p, f32p, ctypes.c_int64, ctypes.c_float, i64p]
        L.ref_softnms_1d.restype = ctypes.c_int64
        L.ref_softnms_1d.argtypes = [f32p, f32p, f32p, ctypes.c_int64, ctypes.c_float, ctypes.c_float,
                                     ctypes.c_float, ctypes.c_int, i64p]
        L.ref_softnms_1d_capped.restype = ctypes.c_int64
        L.ref_softnms_1d_capped.argtypes = [f32p, f32p, f32p, ctypes.c_int64, ctypes.c_float, ctypes.c_float,
                                            ctypes.c_float, ctypes.c_int, ctypes.c_int64, i64p]
        L.ref_seg_voting.restype = None
        L.ref_seg_voting.argtypes = [f32p, ctypes.c_int64, f32p, f32p, ctypes.c_int64, ctypes.c_float, f32p]
        _lib = L
    return _lib


def _f(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))


def _i(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))


def nms(segs, scores, iou_threshold):
    """nms_1d_cpu.nms equivalent (numpy in / numpy out)."""
    segs = np.ascontiguousarray(segs, np.float32).reshape(-1, 2)
    scores = np.ascontiguousarray(scores, np.float32)
    out = np.empty(max(len(scores), 1), np.int64)
    k = lib().ref_nms_1d(_f(segs), _f(scores), len(scores), float(iou_threshold), _i(out))
    return out[:k].copy()


def softnms(segs, scores, iou_threshold, sigma, min_score, method, max_num=0):
    """nms_1d_cpu.softnms equivalent; returns (inds, dets[:K]). max_num > 0: the first max_num picks only (the prefix
    of the full result)."""
    segs = np.ascontiguousarray(segs, np.float32).reshape(-1, 2)
    scores = np.ascontiguousarray(scores, np.float32)
    n = len(scores)
    dets = np.zeros((max(n, 1), 3), np.float32)
    out = np.empty(max(n, 1), np.int64)
    k = lib().ref_softnms_1d_capped(_f(segs), _f(scores), _f(dets), n, float(iou_threshold), float(sigma),
                                    float(min_score), int(method), int(max_num), _i(out))
    return out[:k].copy(), dets[:k].copy()


def seg_voting(nms_segs, all_segs, all_scores, iou_threshold):
    nms_segs = np.ascontiguousarray(nms_segs, np.float32).reshape(-1, 2)
    all_segs = np.ascontiguousarray(all_segs, np.float32).reshape(-1, 2)
    all_scores = np.ascontiguousarray(all_scores, np.float32)
    out = np.zeros_like(nms_segs)
    lib().ref_seg_voting(_f(nms_segs), len(nms_segs), _f(all_segs), _f(all_scores), len(all_scores),
                         float(iou_threshold), _f(out))
    return out


def _hard(segs, scores, cls, iou_threshold, min_score, max_num):
    """NMSop.forward, nms.py:8-35."""
    if min_score > 0:
        keep = scores > np.float32(min_score)
        segs, scores, cls = segs[keep], scores[keep], cls[keep]
    inds = nms(segs, scores, iou_threshold)
    if max_num > 0:
        inds = inds[:min(max_num, len(inds))]
    return segs[inds], scores[inds], cls[inds]


def _soft(segs, scores, cls, iou_threshold, sigma, min_score, method, max_num):
    """SoftNMSop.forward, nms.py:38-64."""
    inds, dets = softnms(segs, scores, iou_threshold, sigma, min_score, method)
    n = min(len(inds), max_num) if max_num > 0 else len(inds)
    return dets[:n, :2].copy(), dets[:n, 2].copy(), cls[inds][:n]


def batched_nms(segs, scores, cls_idxs, iou_threshold, min_score, max_seg_num,
                use_soft_nms=True, multiclass=True, sigma=0.5, voting_thresh=0.75):
    """batched_nms, nms.py:103-190. torch tensors in / out like the reference."""
    if segs.shape[0] == 0:
        return torch.zeros([0, 2]), torch.zeros([0]), torch.zeros([0], dtype=cls_idxs.dtype)
    s = segs.detach().cpu().numpy().astype(np.float32)
    p = scores.detach().cpu().numpy().astype(np.float32)
    c = cls_idxs.detach().cpu().numpy()
    if multiclass:
        outs = []
        for cid in np.unique(c):
            sel = c == cid
            outs.append(_soft(s[sel], p[sel], c[sel], iou_threshold, sigma, min_score, 2, max_seg_num)
                        if use_soft_nms else _hard(s[sel], p[sel], c[sel], iou_threshold, min_score, max_seg_num))
        ns = np.concatenate([o[0] for o in outs]); nsc = np.concatenate([o[1] for o in outs])
        nc = np.concatenate([o[2] for o in outs])
    else:
        ns, nsc, nc = (_soft(s, p, c, iou_threshold, sigma, min_score, 2, max_seg_num) if use_soft_nms
                       else _hard(s, p, c, iou_threshold, min_score, max_seg_num))
        if voting_thresh > 0 and len(ns) > 0:
            ns = seg_voting(ns, s, p, voting_thresh)
    order = np.argsort(-nsc, kind="stable")[:min(max_seg_num, len(nsc))]
    return (torch.from_numpy(ns[order].reshape(-1, 2).copy()), torch.from_numpy(nsc[order].copy()),
            torch.from_numpy(nc[order].copy()))
