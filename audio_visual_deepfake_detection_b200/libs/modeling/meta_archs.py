"""The two meta-archs of the hot path behind the reference's plugin API.

`make_meta_arch("AVLocPointTransformerRecoveryNoNormNorecon", **cfg['model'])`
(exp12, libs/modeling/av_fd_no_recon.py:162-876) and `...NoreconTHE` (exp13,
libs/modeling/av_fd_no_recon2.py:163) return an nn.Module with the reference's
constructor signature, `load_state_dict` contract (reference tensor names,
optional DataParallel `module.` prefix, the dead `interpolator.expansion.*`
tensors accepted) and eval-mode call contract:

    model(video_list) -> [ {video_id, segments [N,2] s, scores [N], labels [N], video_cls [1]} ]

All compute runs in libavdf_sm100 kernels through LocalizationEngine; there is
no CPU path (a model on a machine without CUDA raises at the first call).
New capabilities over the reference: any batch size per call (the reference
asserts len(video_list) == 1, av_fd_no_recon.py:456; videos are independent)
and `forward_streams`, which takes the RAW per-stream features and runs the
dataset-side resampling (libs/datasets/deepfake_video_audio.py:513-547) on the
GPU as the first kernel of the pass.
"""
import gc
from collections import OrderedDict

import numpy as np
import torch
from torch import nn

from ... import ops
from ...native import AvdfError
from .engine import LocalizationEngine
from .models import register_backbone, register_generator, register_meta_arch, register_neck
from .spec import EXP5, EXP12, EXP13, state_dict_spec


def _on_model_device(fn):
    """Run a method with the model's device current: the library launches on the current device and graph capture
    records on it, whatever device the caller's thread happens to have selected (the reference yaml ships
    devices: ['cuda:3'] and inference.py only calls model.to(device))."""
    import functools

    @functools.wraps(fn)
    def wrapped(self, *args, **kwargs):
        dev = self.engine().device
        if dev.index is not None and dev.index != torch.cuda.current_device():
            with torch.cuda.device(dev):
                return fn(self, *args, **kwargs)
        return fn(self, *args, **kwargs)
    return wrapped


class _LocalizationBase(nn.Module):
    MODEL_NAME = None

    def __init__(self, backbone_type, fpn_type, backbone_arch, scale_factor, video_input_dim, audio_input_dim,
                 max_seq_len, max_buffer_len_factor, n_head, n_mha_win_size, embd_kernel_size, embd_dim, embd_with_ln,
                 fpn_dim, fpn_with_ln, fpn_start_level, head_dim, regression_range, head_num_layers, head_kernel_size,
                 head_with_ln, use_abs_pe, use_rel_pe, num_classes, train_cfg, test_cfg, mlp_ratio=None,
                 precision="mixed", max_batch=32):
        super().__init__()
        # same structural assertion as av_fd_no_recon.py:253
        assert backbone_type == "convHRLRFullResSelfAttTransformerRevised"
        self.model_cfg = dict(
            backbone_type=backbone_type, fpn_type=fpn_type, backbone_arch=tuple(backbone_arch), scale_factor=scale_factor,
            video_input_dim=video_input_dim, audio_input_dim=audio_input_dim, max_seq_len=max_seq_len,
            max_buffer_len_factor=max_buffer_len_factor, n_head=n_head, n_mha_win_size=n_mha_win_size,
            embd_kernel_size=embd_kernel_size, embd_dim=embd_dim, embd_with_ln=embd_with_ln, fpn_dim=fpn_dim,
            fpn_with_ln=fpn_with_ln, fpn_start_level=fpn_start_level, head_dim=head_dim, regression_range=regression_range,
            head_num_layers=head_num_layers, head_kernel_size=head_kernel_size, head_with_ln=head_with_ln,
            use_abs_pe=use_abs_pe, use_rel_pe=use_rel_pe, num_classes=num_classes, train_cfg=train_cfg, test_cfg=test_cfg)
        self.precision = precision
        self.max_batch = int(max_batch)
        self.max_seq_len = max_seq_len
        self.num_classes = num_classes
        # test-time config, same attribute names as av_fd_no_recon.py:229-241
        self.test_pre_nms_thresh = test_cfg["pre_nms_thresh"]
        self.test_pre_nms_topk = test_cfg["pre_nms_topk"]
        self.test_iou_threshold = test_cfg["iou_threshold"]
        self.test_min_score = test_cfg["min_score"]
        self.test_max_seg_num = test_cfg["max_seg_num"]
        self.test_nms_method = test_cfg["nms_method"]
        assert self.test_nms_method in ["soft", "hard", "none"]
        self.test_duration_thresh = test_cfg["duration_thresh"]
        self.test_multiclass_nms = test_cfg["multiclass_nms"]
        self.test_nms_sigma = test_cfg["nms_sigma"]
        self.test_voting_thresh = test_cfg["voting_thresh"]
        self._spec = state_dict_spec(self.model_cfg, self.MODEL_NAME)
        self._sd = None               # reference-named tensors (CPU) once loaded
        self._engine = None
        self._device = torch.device("cpu")

    # ------------------------------------------------------------------ nn.Module surface
    def state_dict(self, *args, prefix="", **kwargs):
        if self._sd is None:
            raise AvdfError("no weights loaded: call load_state_dict() first")
        return OrderedDict((prefix + k, v) for k, v in self._sd.items())

    def load_state_dict(self, state_dict, strict=True, **kwargs):
        """Accepts the reference's checkpoints as they are saved: `ckpt['state_dict_ema']` keys carry the
        DataParallel `module.` prefix (inference.py:70-76)."""
        sd = OrderedDict()
        for k, v in state_dict.items():
            k = k[7:] if k.startswith("module.") else k
            sd[k] = v.detach().to("cpu")
        missing = [k for k in self._spec if k not in sd]
        unexpected = [k for k in sd if k not in self._spec]
        bad_shape = [k for k in self._spec if k in sd and tuple(sd[k].shape) != tuple(self._spec[k])]
        if bad_shape:
            k = bad_shape[0]
            raise RuntimeError("size mismatch for %s: checkpoint %s vs model %s" % (k, tuple(sd[k].shape), tuple(self._spec[k])))
        if strict and (missing or unexpected):
            raise RuntimeError("Error(s) in loading state_dict: missing %s unexpected %s" % (missing[:5], unexpected[:5]))
        self._sd = sd
        self._engine = None
        return torch.nn.modules.module._IncompatibleKeys(missing, unexpected)

    def _apply(self, fn, *args, **kwargs):          # .to() / .cuda(): remember the device, weights are packed lazily
        probe = fn(torch.empty(0))
        if probe.device != self._device:
            self._device = probe.device
            self._engine = None
        return self

    @property
    def device(self):
        return self._device

    _TEST_ATTRS = ("pre_nms_thresh", "pre_nms_topk", "iou_threshold", "min_score", "max_seg_num", "duration_thresh",
                   "multiclass_nms", "nms_sigma", "voting_thresh", "nms_method")

    def test_key(self):
        """The test-time configuration as the reference reads it: from the `test_*` attributes at CALL time
        (av_fd_no_recon.py:229-241, 760-876). Captured CUDA graphs are keyed by it."""
        return tuple(getattr(self, "test_" + k) for k in self._TEST_ATTRS)

    def _sync_test_cfg(self, eng):
        for k in self._TEST_ATTRS:
            eng.test_cfg[k] = getattr(self, "test_" + k)

    def engine(self):
        if self._engine is None:
            if self._sd is None:
                raise AvdfError("no weights loaded: call load_state_dict() first")
            dev = self._device
            if dev.type != "cuda":
                if not torch.cuda.is_available():
                    raise AvdfError("this model runs on sm_100a kernels only; no CUDA device is visible (no CPU fallback)")
                dev = torch.device("cuda", torch.cuda.current_device())
                self._device = dev
            cfg = dict(self.model_cfg)
            cfg["test_cfg"] = dict(cfg["test_cfg"], pre_nms_thresh=self.test_pre_nms_thresh, pre_nms_topk=self.test_pre_nms_topk,
                                   iou_threshold=self.test_iou_threshold, min_score=self.test_min_score,
                                   max_seg_num=self.test_max_seg_num, duration_thresh=self.test_duration_thresh,
                                   multiclass_nms=self.test_multiclass_nms, nms_sigma=self.test_nms_sigma,
                                   voting_thresh=self.test_voting_thresh, nms_method=self.test_nms_method)
            self._engine = LocalizationEngine(cfg, self.MODEL_NAME, self._sd, dev, self.precision, self.max_batch)
        return self._engine

    # ------------------------------------------------------------------ forward
    def forward(self, video_list):
        if self.training:
            raise NotImplementedError("training (losses / label assignment) is outside the accelerated inference path")
        if len(video_list) and "feats" not in video_list[0] and "streams" in video_list[0]:
            # items of the inference datasets of this package: raw streams, resampled on the GPU
            return self.forward_streams(video_list)
        out = []
        for i in range(0, len(video_list), self.max_batch):
            out.extend(self._forward_items(video_list[i:i + self.max_batch]))
        return out

    @torch.no_grad()
    @_on_model_device
    def _forward_items(self, items):
        eng = self.engine()
        B = len(items)
        lens = [int(it["feats"].shape[-1]) for it in items]
        L = eng.padded_len(max(lens))                         # av_fd_no_recon.py:458-466
        x = eng.buf("x_in_%d" % L, (B, L, eng.c_in), eng.in_dt)
        for b, it in enumerate(items):                        # preprocessing: pad + batch layout (av_fd_no_recon.py:431-479)
            f = it["feats"]
            if f.shape[0] != eng.c_in:
                raise AvdfError("feats has %d channels, model expects %d" % (f.shape[0], eng.c_in))
            f = f.to(device=eng.device, dtype=torch.float32, non_blocking=True).contiguous()
            ops.pack_feats(f, x[b])
        return self._run(eng, x, lens, items)

    @torch.no_grad()
    @_on_model_device
    def dense_outputs(self, items):
        """Diagnostics / parity tests: the dense head outputs of `items` (<= max_batch videos) as CPU tensors:
        logits [B, P], offsets [B, P, 2], video_cls [B] (levels concatenated in pyramid order)."""
        eng = self.engine()
        B = len(items)
        lens = [int(it["feats"].shape[-1]) for it in items]
        L = eng.padded_len(max(lens))
        x = eng.buf("x_in_%d" % L, (B, L, eng.c_in), eng.in_dt)
        for b, it in enumerate(items):
            ops.pack_feats(it["feats"].to(device=eng.device, dtype=torch.float32).contiguous(), x[b])
        logits, offsets, vcls, _, _ = eng.forward_dense(x, lens)
        return logits.cpu(), offsets.cpu(), vcls.cpu()

    @torch.no_grad()
    def forward_streams(self, batch, window=None, hop=None):
        """batch: list of dicts {video_id, duration, streams: {'video'?: [T_v,256], 'byola': [T_b,2048],
        'emo': [T_e,768]} fp32 numpy/torch, time-major like the `.npy` files}. Runs the dataset's resampling to
        max_seq_len + concat (deepfake_video_audio.py:513-547) on the GPU, then the model; returns the same list
        of dicts as forward(). Host buffers in, host tensors out (pinned staging + CUDA graph inside).

        window / hop (seconds, hop defaults to window / 2): recordings longer than `window` are cut into overlapping
        windows that each run at the model's trained time scale, and their results are merged on the GPU into one
        result per recording (libs/modeling/windows.py). Recordings no longer than `window` give exactly the
        result they give without it."""
        runner = self.runner()
        if window is not None:
            return runner.run_windows(batch, window, hop)
        out = []
        for i in range(0, len(batch), self.max_batch):
            out.extend(runner.run(batch[i:i + self.max_batch]))
        return out

    @torch.no_grad()
    def stream(self, batches, window=None, hop=None):
        """Pipelined variant for serving loops: `for results in model.stream(iterable_of_batches)` overlaps the
        host-side packing of batch i+1 with the copies and GPU work of batch i (two pinned staging slots).
        window / hop: as forward_streams; each batch's recordings are windowed and merged, one result per recording."""
        if window is None:
            yield from self.runner().stream(batches)
            return
        runner = self.runner()
        for chunk in batches:
            yield runner.run_windows(chunk, window, hop)

    def runner(self):
        if getattr(self, "_runner", None) is None or self._runner.eng is not self.engine():
            from .streaming import StreamRunner
            self._runner = StreamRunner(self)
        return self._runner

    # The raw-stream path in four explicit stages, so that a serving loop (and bench.py) can overlap them:
    #   pack_streams  host:  ragged per-video arrays -> one pinned buffer per stream + row offsets + per-video meta
    #   stage         H2D:   async copies on the current stream
    #   run_staged    GPU:   interp_concat -> forward -> decode/NMS; returns DEVICE tensors, no host sync
    #   fetch         D2H:   results -> the reference's list of dicts
    def pack_streams(self, chunk, feat_stride=1, num_frames=1):
        from .streaming import video_meta
        L = self.max_seq_len
        B = len(chunk)
        packed = {"ids": [c["video_id"] for c in chunk], "streams": [], "offs": [], "B": B}
        for n in ("video", "byola", "emo"):
            if n not in chunk[0]["streams"]:
                packed["streams"].append(None); packed["offs"].append(None)
                continue
            from .streaming import _stream_array
            arrs = [_stream_array(c["streams"][n]) for c in chunk]              # fp32, or uint16 = bf16 feature shards
            off = np.zeros(B + 1, np.int32)
            off[1:] = np.cumsum([a.shape[0] for a in arrs])
            shard16 = arrs[0].dtype == np.uint16
            host = torch.empty((int(off[-1]), arrs[0].shape[1]), dtype=torch.bfloat16 if shard16 else torch.float32,
                               pin_memory=torch.cuda.is_available())
            np.concatenate(arrs, axis=0, out=host.view(torch.int16).numpy().view(np.uint16) if shard16 else host.numpy())
            packed["streams"].append(host)
            packed["offs"].append(torch.from_numpy(off))
        meta = np.empty((4, B), np.float32)
        for b, c in enumerate(chunk):
            first = c["streams"]["video"] if "video" in c["streams"] else c["streams"]["byola"]
            meta[:, b] = video_meta(c, first.shape[0], L, feat_stride, num_frames)
        packed["meta"] = torch.from_numpy(meta)
        return packed

    @_on_model_device
    def stage(self, packed):
        dev = self.engine().device
        staged = dict(packed)
        staged["streams"] = [None if t is None else t.to(dev, non_blocking=True) for t in packed["streams"]]
        staged["offs"] = [None if t is None else t.to(dev, non_blocking=True) for t in packed["offs"]]
        staged["meta"] = packed["meta"].to(dev, non_blocking=True)
        return staged

    @staticmethod
    def h2d_bytes(packed):
        n = packed["meta"].numel() * 4
        for t in packed["streams"] + packed["offs"]:
            if t is not None:
                n += t.numel() * t.element_size()
        return n

    @torch.no_grad()
    @_on_model_device
    def run_staged(self, staged, lane=0):
        """lane selects the engine's buffer set: batches that are in flight at the same time (different CUDA
        streams) must use different lanes."""
        eng = self.engine()
        self._sync_test_cfg(eng)
        eng.lane = lane
        B, L = staged["B"], eng.max_seq_len
        x = eng.buf("x_in_%d" % L, (B, L, eng.c_in), eng.in_dt)
        if staged.get("ranges") is not None:      # sliding windows: (start, count) [3, B] rows into the group's staging
            ops.interp_concat_ranges(staged["streams"], *staged["ranges"], L, x)
        else:
            ops.interp_concat(staged["streams"], staged["offs"], L, x)
        logits, offsets, vcls, masks, lens = eng.forward_dense(x, [L] * B)
        rec = staged.get("records")      # (ring, counter): result records for the multi-GPU gather, written by the kernel
        if rec is not None:
            rec = (rec[0], rec[1], staged.get("vidx"))
        osg, osc, ocn = eng.postprocess(logits, offsets, masks, lens, staged["meta"], nms_method=self.test_nms_method,
                                        records=rec, vcls=vcls)
        eng.lane = 0
        return {"ids": staged["ids"], "segs": osg, "scores": osc, "counts": ocn, "vcls": vcls}

    @_on_model_device
    def capture(self, staged, lane=0):
        """Record the whole pass over a staged (device-resident) batch into a CUDA graph: ~190 kernel launches
        become one cudaGraphLaunch, which removes the host launch cost that otherwise bounds the step
        (measured: 25 us of Python + driver time per launch vs 7-40 us of GPU time per kernel). The graph reads
        the staged tensors and writes the engine's static buffers, so `staged` must stay alive and unchanged in
        place; replay() returns the same device-side result dict as run_staged()."""
        from ... import native
        warm = dict(staged)
        warm.pop("records", None)                   # the warm-up pass must not append result records
        self.run_staged(warm, lane)                 # allocates every static buffer / cache outside the capture
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        n0 = native.LAUNCHES["n"]
        # thread_local: other host threads (the streaming runner's packer allocating pinned staging, a data loader)
        # may call the CUDA allocator while this thread records; in the default global mode that invalidates the capture
        eng = self.engine()
        eng._capture_refs = []
        # no cyclic garbage collection while recording: collecting a discarded model frees its captured graphs, a call
        # this thread may not make during a capture (it invalidates the capture)
        gc_on = gc.isenabled()
        gc.collect()
        gc.disable()
        try:
            with torch.cuda.graph(graph, capture_error_mode="thread_local"):
                res = self.run_staged(staged, lane)
            keep = eng._capture_refs
        finally:
            eng._capture_refs = None
            if gc_on:
                gc.enable()
        return GraphedPass(graph, res, native.LAUNCHES["n"] - n0, staged, keep)

    def export_plan(self, path, batch_sizes=None, shards=False, max_seconds=36.0, items=None):
        """Write the launch plan of the raw-stream pass (libs/modeling/plan.py): what libavdf_sm100.so's
        avdf_session_run replays as a CUDA graph, with no Python in the process."""
        from .plan import export_plan
        return export_plan(self, path, batch_sizes=batch_sizes, shards=shards, max_seconds=max_seconds, items=items)

    @staticmethod
    def fetch(res):
        segs, scores, counts, vc = res["segs"].cpu(), res["scores"].cpu(), res["counts"].cpu(), res["vcls"].cpu()
        out = []
        for b, vid in enumerate(res["ids"]):
            n = int(counts[b])
            out.append({"video_id": vid, "segments": segs[b, :n].clone(), "scores": scores[b, :n].clone(),
                        "labels": torch.zeros(n, dtype=torch.long), "video_cls": vc[b:b + 1].clone()})
        return out

    @staticmethod
    def d2h_bytes(res):
        return sum(res[k].numel() * res[k].element_size() for k in ("segs", "scores", "counts", "vcls"))

    def _run(self, eng, x, valid, items):
        B = x.shape[0]
        self._sync_test_cfg(eng)
        logits, offsets, vcls, masks, lens = eng.forward_dense(x, valid)
        meta = np.empty((4, B), np.float32)
        for b, it in enumerate(items):                        # av_fd_no_recon.py:860-865 (python-float scalars -> fp32)
            meta[:, b] = (np.float32(it["feat_stride"]), np.float32(0.5 * it["feat_num_frames"]), np.float32(it["fps"]),
                          np.float32(it["duration"]))
        meta_d = torch.from_numpy(meta).to(eng.device, non_blocking=True)
        osg, osc, ocn = eng.postprocess(logits, offsets, masks, lens, meta_d, nms_method=self.test_nms_method)
        return self.fetch({"ids": [it["video_id"] for it in items], "segs": osg, "scores": osc, "counts": ocn, "vcls": vcls})


class GraphedPass:
    """A captured pass (see _LocalizationBase.capture)."""

    def __init__(self, graph, result, n_launches, staged, keep=None):
        self.graph, self.result, self.n_launches, self.staged = graph, result, n_launches, staged
        self.keep = keep          # mask tables / workspaces the captured launches point at (see engine._capture_refs)

    def replay(self):
        from ... import native
        self.graph.replay()
        native.count(self.n_launches)
        return self.result


@register_meta_arch(EXP12)
class AVPtTransformerRecovery(_LocalizationBase):
    """exp12: video-level branch = DeepInterpolator (Contraction + classifier), av_fd_no_recon.py:318."""
    MODEL_NAME = EXP12


@register_meta_arch(EXP5)
class AVPtTransformerRecoveryRecon(_LocalizationBase):
    """exp5-style: DeepInterpolator with its Expansion live - the reconstruction is embedded and attended to as K by
    backbone.resselfattention (av_fd_meta_arch.py:162, 346-348; blocks.py:1568-1590)."""
    MODEL_NAME = EXP5


@register_meta_arch(EXP13)
class AVPtTransformerRecoveryTHE(_LocalizationBase):
    """exp13: video-level branch = SegmentandCls (Extract + segment head), av_fd_no_recon2.py:318,348."""
    MODEL_NAME = EXP13


# ---- descriptors for the component registries (see models.py's docstring) ------------------------
@register_backbone("convHRLRFullResSelfAttTransformerRevised")
class BackboneDescriptor:
    """Configuration of ConvHRLRFullResSelfAttTransformerBackboneRevised (backbones.py:272-405)."""

    def __init__(self, **kw):
        self.kw = kw
        assert kw.get("n_embd", 256) == 256 and kw.get("n_head", 4) == 4, "kernels are specialised for 256 x 4 heads"


@register_neck("fpn")
class FPNDescriptor:
    """Configuration of FPN1D (necks.py:10-60)."""

    def __init__(self, **kw):
        self.kw = kw


@register_generator("point")
class PointGenerator:
    """loc_generators.py:27-84: per-level constant tables [T_l, 4] = (t, reg_lo, reg_hi, stride). On the
    accelerated path the decode kernel regenerates t = i * stride on the fly; this class reproduces the
    tables for callers that want them."""

    def __init__(self, max_seq_len, fpn_levels, scale_factor, regression_range, use_offset=False):
        assert len(regression_range) == fpn_levels
        self.points = []
        for l in range(fpn_levels):
            stride = scale_factor ** l
            pts = torch.arange(0, max_seq_len, stride, dtype=torch.float32)[:, None]
            if use_offset:
                pts += 0.5 * stride
            rr = torch.as_tensor(regression_range[l], dtype=torch.float32)[None].repeat(pts.shape[0], 1)
            st = torch.full((pts.shape[0], 1), float(stride))
            self.points.append(torch.cat([pts, rr, st], dim=1))

    def __call__(self, feats):
        return [p[: f.shape[-1]] for p, f in zip(self.points, feats)]
