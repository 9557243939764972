"""1-D NMS front-end with the reference's API (libs/utils/nms.py:8-190), running on the
sm_100a kernels of libavdf_sm100 (csrc/nms.cu).

`batched_nms(segs, scores, cls_idxs, iou_threshold, min_score, max_seg_num, use_soft_nms,
multiclass, sigma, voting_thresh)` keeps the reference's signature, defaults, return types
(CPU tensors, empty-input shapes nms.py:118-121) and selection semantics. Inputs may live on
the CPU (like the reference's callers, av_fd_no_recon.py:841-858) or on the GPU; CPU inputs
are staged to the device - the arithmetic always runs in the CUDA kernels, there is no CPU
implementation here.

`nms_1d_cpu` below is a stand-in for the reference's pybind11 module of that name
(libs/utils/csrc/nms_cpu.cpp:172-182): same two functions, same argument order, same
in-place `dets` contract, executed by avdf_nms_hard / avdf_nms_soft.
"""
import torch

from ... import ops
from ...native import AvdfError


def _device():
    if not torch.cuda.is_available():
        raise AvdfError("libs.utils.nms runs on sm_100a kernels only; no CUDA device is visible (no CPU fallback)")
    return torch.device("cuda", torch.cuda.current_device())


class nms_1d_cpu:                      # noqa: N801  (module-like namespace, name kept for drop-in imports)
    @staticmethod
    def nms(segs, scores, iou_threshold):
        """-> LongTensor[K] (CPU): kept indices into the input, descending score (nms_cpu.cpp:19-65)."""
        dev = _device()
        if scores.numel() == 0:
            return torch.empty(0, dtype=torch.long)
        idx = ops.nms_hard(segs.to(dev, torch.float32).contiguous(), scores.to(dev, torch.float32).contiguous(),
                           float(iou_threshold))
        return idx.cpu()

    @staticmethod
    def softnms(segs, scores, dets, iou_threshold, sigma, min_score, method):
        """-> LongTensor[K] (CPU); writes dets[:K] = (x1, x2, decayed score) in place (nms_cpu.cpp:67-169)."""
        dev = _device()
        if scores.numel() == 0:
            return torch.empty(0, dtype=torch.long)
        d = torch.empty((scores.numel(), 3), dtype=torch.float32, device=dev)
        idx = ops.nms_soft(segs.to(dev, torch.float32).contiguous(), scores.to(dev, torch.float32).contiguous(), d,
                           float(iou_threshold), float(sigma), float(min_score), int(method))
        k = idx.numel()
        dets[:k].copy_(d[:k])
        return idx.cpu()


MAX_SEGS = 1024                        # AVDF_MAX_SEGS: the most picks one avdf_postprocess call returns per video


def _wanted(max_seg_num, total):
    """Picks kept by the reference's final cut `idxs[:min(max_seg_num, total)]` (nms.py:184-189) out of `total`, in
    Python slice semantics: 0 keeps none, a negative value drops that many from the end."""
    return len(range(total)[:min(int(max_seg_num), total)])


def _single_class(segs_d, scores_d, iou_threshold, min_score, max_seg_num, use_soft_nms, sigma, voting_thresh, final_cut):
    """One class-agnostic NMS on device candidates [N,2], [N] -> (segs [K,2], scores [K], candidate index [K]) on device,
    in descending score. NMSop / SoftNMSop cap the picks at max_seg_num when it is > 0 (nms.py:24-25, 57-58); with
    final_cut the reference's final slice follows as well. Picks come out of both NMS kinds in non-increasing score,
    so the first K picks are the first K of the sorted list. More than MAX_SEGS picks wanted raises AvdfError."""
    dev = segs_d.device
    n = scores_d.numel()
    cap = int(max_seg_num) if max_seg_num > 0 else None
    K = min(cap, MAX_SEGS) if cap is not None else MAX_SEGS
    cand_count = torch.tensor([n], dtype=torch.int32, device=dev)
    out_segs = torch.empty((1, K, 2), dtype=torch.float32, device=dev)
    out_scores = torch.empty((1, K), dtype=torch.float32, device=dev)
    out_count = torch.zeros(1, dtype=torch.int32, device=dev)
    out_index = torch.zeros((1, K), dtype=torch.int32, device=dev)
    ops.postprocess(1, cand_segs=segs_d.view(1, n, 2), cand_scores=scores_d.view(1, n), cand_count=cand_count,
                    iou_threshold=iou_threshold, min_score=min_score, sigma=sigma, voting_thresh=voting_thresh,
                    max_seg_num=K, use_soft_nms=use_soft_nms, out_segs=out_segs, out_scores=out_scores, out_count=out_count,
                    out_index=out_index)
    k = int(out_count.item())
    total = k
    if k == K and (cap is None or cap > K):
        total = _pick_count(segs_d, scores_d, iou_threshold, min_score, cap, use_soft_nms, sigma)
    want = min(total, cap) if cap is not None else total
    if final_cut:
        want = _wanted(max_seg_num, want)
    if want > k:
        raise AvdfError("batched_nms: %d picks wanted (max_seg_num=%d), more than the %d (AVDF_MAX_SEGS) one "
                        "postprocess call returns per class" % (want, int(max_seg_num), MAX_SEGS))
    return out_segs[0, :want], out_scores[0, :want], out_index[0, :want]


def _pick_count(segs_d, scores_d, iou_threshold, min_score, cap, use_soft_nms, sigma):
    """The number of picks of the whole NMS (at most cap + 1 when capped), by the standalone kernels."""
    limit = 0 if cap is None else cap + 1
    if use_soft_nms:
        dets = torch.empty((scores_d.numel(), 3), dtype=torch.float32, device=scores_d.device)
        return ops.nms_soft(segs_d, scores_d, dets, float(iou_threshold), float(sigma), float(min_score), 2, limit).numel()
    if min_score > 0:                  # NMSop's score filter (nms.py:15-21)
        keep = torch.nonzero(scores_d > float(min_score)).flatten()
        segs_d, scores_d = segs_d[keep].contiguous(), scores_d[keep].contiguous()
    if scores_d.numel() == 0:
        return 0
    return ops.nms_hard(segs_d, scores_d, float(iou_threshold), limit).numel()


def batched_nms(segs, scores, cls_idxs, iou_threshold, min_score, max_seg_num, use_soft_nms=True, multiclass=True,
                sigma=0.5, voting_thresh=0.75):
    num_segs = segs.shape[0]
    if num_segs == 0 or max_seg_num == 0:          # nms.py:118-121; the final cut [:0] keeps nothing (nms.py:186-189)
        return torch.zeros([0, 2]), torch.zeros([0, ]), torch.zeros([0, ], dtype=cls_idxs.dtype)
    dev = _device()
    segs_d = segs.to(dev, torch.float32).contiguous()
    scores_d = scores.to(dev, torch.float32).contiguous()
    if multiclass:
        # per class, no voting (nms.py:123-156); the final cross-class sort + cut follows nms.py:182-189
        cls_cpu = cls_idxs.cpu()
        new_segs, new_scores, new_cls = [], [], []
        for class_id in torch.unique(cls_cpu):
            cur = torch.where(cls_cpu == class_id)[0].to(dev)
            s, p, _ = _single_class(segs_d[cur].contiguous(), scores_d[cur].contiguous(), iou_threshold, min_score,
                                    max_seg_num, use_soft_nms, sigma, 0.0, final_cut=False)
            new_segs.append(s); new_scores.append(p)
            new_cls.append(torch.full((p.numel(),), int(class_id), dtype=cls_idxs.dtype))
        new_segs, new_scores, new_cls = torch.cat(new_segs).cpu(), torch.cat(new_scores).cpu(), torch.cat(new_cls)
        _, idxs = new_scores.sort(descending=True, stable=True)
        idxs = idxs[:min(max_seg_num, new_segs.shape[0])]
        return new_segs[idxs], new_scores[idxs], new_cls[idxs]
    s, p, idx = _single_class(segs_d, scores_d, iou_threshold, min_score, max_seg_num, use_soft_nms, sigma, voting_thresh,
                              final_cut=True)
    # class-agnostic (nms.py:159-180): one NMS over all candidates; every pick keeps the label of its candidate
    return s.cpu(), p.cpu(), cls_idxs.cpu()[idx.cpu().long()]
