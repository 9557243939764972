"""ctypes binding of libavdf_sm100.so (the C-ABI declared in include/avdf.h).

This is the only door between the Python host code and the sm_100a kernels.
There is NO fallback: if the library is missing `lib()` raises, and every
wrapper raises `AvdfError` with the library's message when a call fails.
PyTorch is used by the callers for device memory and streams only; the
signatures below take raw device pointers.
"""
import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_float, c_int32, c_int64, c_size_t, c_uint8, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("AVDF_LIB_PATH") or os.path.join(HERE, "csrc", "libavdf_sm100.so")      # (override: kernel experiments)

MAX_LEVELS = 8
MAX_SEGS = 1024
DTYPE_F32, DTYPE_BF16, DTYPE_F16 = 0, 1, 2
ACT_NONE, ACT_RELU, ACT_GELU = 0, 1, 2

# every symbol include/avdf.h declares (checked by tests/test_abi.py)
EXPORTS = [
    "avdf_abi_version", "avdf_last_error", "avdf_device_info", "avdf_interp_concat", "avdf_interp_concat_in", "avdf_pack_feats",
    "avdf_nms_workspace_bytes", "avdf_nms_hard", "avdf_nms_soft",
    "avdf_postprocess_workspace_bytes", "avdf_postprocess",
    "avdf_conv_gemm_workspace_bytes", "avdf_conv_gemm", "avdf_mlp_fused", "avdf_ln_dwconv_ln", "avdf_attention",
    "avdf_ln_rows", "avdf_instnorm_lrelu", "avdf_fpn_fuse", "avdf_head_final", "avdf_head_combine",
    "avdf_vcls_exp12", "avdf_vcls_exp13", "avdf_host_pack", "avdf_host_all_pinned", "avdf_h2d_gather",
    "avdf_logmel", "avdf_byola_conv1_pool", "avdf_byola_pool", "avdf_eval_workspace_bytes", "avdf_eval_detection",
    "avdf_eval_proposal_workspace_bytes", "avdf_eval_proposal", "avdf_interp_concat_ranges",
    "avdf_window_merge_workspace_bytes", "avdf_window_merge",
    "avdf_plan_open", "avdf_plan_get_info", "avdf_plan_upload", "avdf_plan_close",
    "avdf_session_create", "avdf_session_get_io", "avdf_session_run", "avdf_session_destroy",
    "avdf_plan_window_layout", "avdf_session_window_bytes", "avdf_session_attach_windows", "avdf_session_run_windows",
    "avdf_format_results_workspace_bytes", "avdf_format_results",
    "avdf_postprocess_sweep_workspace_bytes", "avdf_postprocess_sweep",
]


class AvdfError(RuntimeError):
    pass


class PostprocessArgs(Structure):
    _fields_ = [
        ("batch", c_int32),
        ("logits", c_void_p), ("offsets", c_void_p), ("mask", c_void_p),
        ("n_levels", c_int32),
        ("level_len", c_int32 * MAX_LEVELS), ("level_stride", c_float * MAX_LEVELS),
        ("pre_nms_thresh", c_float), ("pre_nms_topk", c_int32), ("duration_thresh", c_float),
        ("cand_segs", c_void_p), ("cand_scores", c_void_p), ("cand_count", c_void_p), ("cand_cap", c_int32),
        ("iou_threshold", c_float), ("min_score", c_float), ("sigma", c_float), ("voting_thresh", c_float),
        ("max_seg_num", c_int32), ("use_soft_nms", c_int32), ("soft_method", c_int32),
        ("vid_feat_stride", c_void_p), ("vid_half_nframes", c_void_p), ("vid_fps", c_void_p), ("vid_duration", c_void_p),
        ("out_segs", c_void_p), ("out_scores", c_void_p), ("out_count", c_void_p),
        ("workspace", c_void_p), ("workspace_bytes", c_size_t),
        ("rec_ring", c_void_p), ("rec_counter", c_void_p), ("rec_cap", c_int32), ("vid_index", c_void_p), ("vid_cls", c_void_p),
        ("out_index", c_void_p),
    ]


class SweepSetting(Structure):
    _fields_ = [
        ("pre_nms_thresh", c_float), ("pre_nms_topk", c_int32), ("duration_thresh", c_float),
        ("iou_threshold", c_float), ("min_score", c_float), ("sigma", c_float), ("voting_thresh", c_float),
        ("max_seg_num", c_int32), ("use_soft_nms", c_int32),
    ]


class PostprocessSweepArgs(Structure):
    _fields_ = [
        ("batch", c_int32),
        ("logits", c_void_p), ("offsets", c_void_p), ("valid_len", c_void_p),
        ("n_levels", c_int32),
        ("level_len", c_int32 * MAX_LEVELS), ("level_stride", c_float * MAX_LEVELS),
        ("vid_feat_stride", c_void_p), ("vid_half_nframes", c_void_p), ("vid_fps", c_void_p), ("vid_duration", c_void_p),
        ("vid_cls", c_void_p), ("vid_index", c_void_p),
        ("n_settings", c_int32), ("settings", POINTER(SweepSetting)),
        ("out_rows", c_void_p), ("rows_per_setting", c_int64), ("row_k", c_int32),
        ("workspace", c_void_p), ("workspace_bytes", c_size_t),
    ]


class WindowMergeArgs(Structure):
    _fields_ = [
        ("n_rec", c_int32), ("rec_win", c_void_p), ("win_start", c_void_p),
        ("win_segs", c_void_p), ("win_scores", c_void_p), ("win_count", c_void_p), ("win_cls", c_void_p),
        ("cand_cap", c_int32),
        ("iou_threshold", c_float), ("min_score", c_float), ("sigma", c_float), ("voting_thresh", c_float),
        ("max_seg_num", c_int32), ("use_soft_nms", c_int32),
        ("out_segs", c_void_p), ("out_scores", c_void_p), ("out_count", c_void_p), ("out_cls", c_void_p),
        ("workspace", c_void_p), ("workspace_bytes", c_size_t),
        ("rec_ring", c_void_p), ("rec_counter", c_void_p), ("rec_cap", c_int32), ("vid_index", c_void_p),
    ]


class ConvGemmArgs(Structure):
    _fields_ = [
        ("batch", c_int32), ("n_out", c_int32), ("c_in", c_int32), ("taps", c_int32), ("stride", c_int32), ("n_seg", c_int32),
        ("seg_t_out", c_int32 * MAX_LEVELS), ("seg_a_row", c_int32 * MAX_LEVELS), ("seg_o_row", c_int32 * MAX_LEVELS),
        ("seg_w_row", c_int32 * MAX_LEVELS), ("n_w_rows", c_int32),
        ("a_rows_per_video", c_int64), ("o_rows_per_video", c_int64),
        ("a", c_void_p), ("w", c_void_p), ("dtype", c_int32),
        ("bias", c_void_p), ("row_mask", c_void_p), ("ln_w", c_void_p), ("ln_b", c_void_p), ("act", c_int32),
        ("pe", c_void_p), ("residual", c_void_p), ("gamma", c_void_p),
        ("out_f32", c_void_p), ("out_h", c_void_p), ("out_h_dtype", c_int32),
        ("workspace", c_void_p), ("workspace_bytes", c_size_t),
        ("ln_after_residual", c_int32), ("tap_mode", c_int32),
        ("dot_w", c_void_p), ("dot_n", c_int32), ("dot_out", c_void_p),
        ("tap_rows", POINTER(c_int32)),
    ]


class LnDwconvLnArgs(Structure):
    _fields_ = [
        ("batch", c_int32), ("channels", c_int32), ("t_src", c_int32), ("t_virt", c_int32), ("shift", c_int32),
        ("stride", c_int32), ("n_streams", c_int32),
        ("src", c_void_p), ("mask_out", c_void_p),
        ("ln_in_w", c_void_p * 3), ("ln_in_b", c_void_p * 3), ("dw_w", c_void_p * 3),
        ("ln_out_w", c_void_p * 3), ("ln_out_b", c_void_p * 3),
        ("out", c_void_p * 3), ("out_dtype", c_int32), ("out_rows_per_video", c_int32), ("skip_out", c_void_p),
        ("tile_rows", c_int32),
    ]


class MlpFusedArgs(Structure):
    _fields_ = [
        ("rows", c_int32), ("channels", c_int32), ("hidden", c_int32), ("dtype", c_int32),
        ("x", c_void_p), ("w1", c_void_p), ("b1", c_void_p), ("w2", c_void_p), ("b2", c_void_p),
        ("row_mask", c_void_p), ("residual", c_void_p), ("gamma", c_void_p), ("out", c_void_p), ("out_h", c_void_p),
        ("out_h_t", c_int32), ("out_h_pitch", c_int32), ("out_h_row0", c_int32),
        ("att", c_void_p), ("w_o", c_void_p), ("b_o", c_void_p), ("gamma_attn", c_void_p), ("ln2_w", c_void_p), ("ln2_b", c_void_p),
        ("skip", c_void_p), ("y", c_void_p),
    ]


class EvalArgs(Structure):
    _fields_ = [
        ("n_pred", c_int64), ("n_video", c_int32), ("n_gt", c_int32),
        ("pred_off", c_void_p), ("pred_seg", c_void_p), ("pred_score", c_void_p), ("gt_off", c_void_p), ("gt_seg", c_void_p),
        ("thresholds", POINTER(c_double)), ("n_thr", c_int32), ("top_k", POINTER(c_int32)), ("n_topk", c_int32),
        ("ap", c_void_p), ("recall_hits", c_void_p), ("tp_mask", c_void_p), ("pred_rank", c_void_p), ("status", c_void_p),
        ("workspace", c_void_p), ("workspace_bytes", c_size_t),
    ]


class EvalProposalArgs(Structure):
    _fields_ = [
        ("n_video", c_int32), ("n_prop", c_int64), ("n_gt", c_int32),
        ("prop_off", c_void_p), ("prop_seg", c_void_p), ("prop_score", c_void_p), ("keep", c_void_p),
        ("gt_off", c_void_p), ("gt_seg", c_void_p),
        ("thresholds", POINTER(c_double)), ("n_thr", c_int32), ("an_frac", POINTER(c_double)),
        ("matches", c_void_p), ("status", c_void_p),
        ("workspace", c_void_p), ("workspace_bytes", c_size_t),
    ]


class PlanInfo(Structure):
    _fields_ = [
        ("abi_version", c_int32), ("cc_major", c_int32), ("cc_minor", c_int32), ("sm_count", c_int32), ("max_batch", c_int32),
        ("max_seg_num", c_int32), ("t_out", c_int32), ("in_dtype", c_int32),
        ("channels", c_int32 * 3), ("stream_rows", c_int64 * 3), ("batch_mask", ctypes.c_uint64),
        ("const_bytes", c_size_t), ("session_bytes", c_size_t), ("description", ctypes.c_char * 1024),
    ]


class SessionIO(Structure):
    _fields_ = [
        ("streams", c_void_p * 3), ("offsets", c_void_p), ("meta", c_void_p),
        ("segs", c_void_p), ("scores", c_void_p), ("counts", c_void_p), ("video_cls", c_void_p),
    ]


class WindowRunArgs(Structure):
    _fields_ = [
        ("n_rec", c_int32), ("duration", POINTER(c_double)), ("rows", POINTER(c_int64)), ("window", c_double), ("hop", c_double),
        ("out_segs", c_void_p), ("out_scores", c_void_p), ("out_count", c_void_p), ("out_cls", c_void_p),
    ]


class FormatArgs(Structure):
    _fields_ = [
        ("mode", c_int32), ("K", c_int32), ("records", c_void_p), ("n_records", c_int64), ("order", c_void_p), ("n_pos", c_int64),
        ("ids", c_void_p), ("id_off", c_void_p), ("id_bytes_max", c_int32), ("pos_begin", c_int64), ("n_rows", c_int32),
        ("min_score", c_double), ("out", c_void_p), ("out_capacity", c_size_t), ("out_bytes", c_void_p),
        ("workspace", c_void_p), ("workspace_bytes", c_size_t),
    ]


FORMAT_RECORDS, FORMAT_PREDICTIONS = 0, 1

# status bits of avdf_eval_detection / avdf_eval_proposal (AVDF_EVAL_*)
EVAL_PRED_LIMIT, EVAL_GT_LIMIT, EVAL_BAD_OFFSETS, EVAL_BAD_KEEP = 1, 2, 4, 8

_lib = None


def lib():
    """The loaded library; raises if it has not been built (python -m
    audio_visual_deepfake_detection_b200.csrc.build, or __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise AvdfError("libavdf_sm100.so is not built (%s); run `python -m audio_visual_deepfake_detection_b200.csrc.build` "
                        "- there is no CPU fallback" % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    L.avdf_abi_version.restype = c_int32
    L.avdf_last_error.restype = c_char_p
    L.avdf_device_info.argtypes = [POINTER(c_int32)] * 3
    L.avdf_interp_concat.argtypes = [c_void_p] * 6 + [c_int32] * 5 + [c_void_p, c_int32, c_void_p]
    L.avdf_interp_concat_in.argtypes = [c_void_p] * 3 + [c_int32] + [c_void_p] * 3 + [c_int32] * 5 + [c_void_p, c_int32, c_void_p]
    L.avdf_interp_concat_ranges.argtypes = [c_void_p] * 3 + [c_int32] + [c_void_p] * 2 + [c_int32] * 5 + [c_void_p, c_int32, c_void_p]
    L.avdf_window_merge_workspace_bytes.restype = c_size_t
    L.avdf_window_merge_workspace_bytes.argtypes = [c_int32, c_int32]
    L.avdf_window_merge.argtypes = [POINTER(WindowMergeArgs), c_void_p]
    L.avdf_pack_feats.argtypes = [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_int32, c_void_p]
    L.avdf_nms_workspace_bytes.restype = c_size_t
    L.avdf_nms_workspace_bytes.argtypes = [c_int32]
    L.avdf_nms_hard.argtypes = [c_void_p, c_void_p, c_int32, c_float, c_int32, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]
    L.avdf_nms_soft.argtypes = [c_void_p, c_void_p, c_int32, c_void_p, c_float, c_float, c_float, c_int32, c_int32,
                                c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]
    L.avdf_postprocess_workspace_bytes.restype = c_size_t
    L.avdf_postprocess_workspace_bytes.argtypes = [c_int32, c_int32]
    L.avdf_postprocess.argtypes = [POINTER(PostprocessArgs), c_void_p]
    L.avdf_postprocess_sweep_workspace_bytes.restype = c_size_t
    L.avdf_postprocess_sweep_workspace_bytes.argtypes = [c_int32, c_int32]
    L.avdf_postprocess_sweep.argtypes = [POINTER(PostprocessSweepArgs), c_void_p]
    L.avdf_conv_gemm_workspace_bytes.restype = c_size_t
    L.avdf_conv_gemm_workspace_bytes.argtypes = [POINTER(ConvGemmArgs)]
    L.avdf_conv_gemm.argtypes = [POINTER(ConvGemmArgs), c_void_p]
    L.avdf_mlp_fused.argtypes = [POINTER(MlpFusedArgs), c_void_p]
    L.avdf_ln_dwconv_ln.argtypes = [POINTER(LnDwconvLnArgs), c_void_p]
    L.avdf_attention.argtypes = [c_void_p] * 5 + [c_int32] * 8 + [c_void_p]
    L.avdf_ln_rows.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int64, c_int32, c_void_p]
    L.avdf_instnorm_lrelu.argtypes = [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_float, c_void_p]
    L.avdf_fpn_fuse.argtypes = [c_void_p] * 6 + [c_int32] * 4 + [POINTER(c_int32), c_void_p]
    L.avdf_head_final.argtypes = [c_void_p, c_void_p, c_int32] + [c_void_p] * 5 + [POINTER(c_float), c_void_p, c_void_p,
                                                                                  c_int32, c_int32, c_int32, POINTER(c_int32), c_void_p]
    L.avdf_head_combine.argtypes = [c_void_p] * 5 + [POINTER(c_float), c_void_p, c_void_p, c_int32, c_int32, POINTER(c_int32), c_void_p]
    L.avdf_vcls_exp12.argtypes = [c_void_p, c_int32] + [c_void_p] * 7 + [c_int32] * 3 + [c_void_p]
    L.avdf_vcls_exp13.argtypes = [c_void_p, c_int32] + [c_void_p] * 6 + [c_int32] * 3 + [c_void_p]
    L.avdf_host_pack.argtypes = [POINTER(c_void_p), POINTER(c_void_p), POINTER(c_size_t), c_int32, c_int32]
    L.avdf_host_all_pinned.argtypes = [POINTER(c_void_p), POINTER(c_size_t), c_int32]
    L.avdf_h2d_gather.argtypes = [POINTER(c_void_p), POINTER(c_void_p), POINTER(c_size_t), c_int32, c_void_p]
    L.avdf_logmel.argtypes = [c_void_p] * 4 + [c_int32] * 3 + [c_void_p] * 5 + [c_int32, c_float, c_float, c_void_p, c_void_p]
    L.avdf_byola_conv1_pool.argtypes = [c_void_p] * 6 + [c_int32, c_void_p, c_int32, c_void_p, c_void_p]
    L.avdf_byola_pool.argtypes = [c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_void_p]
    L.avdf_eval_workspace_bytes.restype = c_size_t
    L.avdf_eval_workspace_bytes.argtypes = [c_int64, c_int32]
    L.avdf_eval_detection.argtypes = [POINTER(EvalArgs), c_void_p]
    L.avdf_eval_proposal_workspace_bytes.restype = c_size_t
    L.avdf_eval_proposal_workspace_bytes.argtypes = [c_int32]
    L.avdf_eval_proposal.argtypes = [POINTER(EvalProposalArgs), c_void_p]
    L.avdf_plan_open.argtypes = [c_char_p, POINTER(c_void_p)]
    L.avdf_plan_get_info.argtypes = [c_void_p, POINTER(PlanInfo)]
    L.avdf_plan_upload.argtypes = [c_void_p, c_void_p, c_size_t, c_void_p]
    L.avdf_plan_close.argtypes = [c_void_p]
    L.avdf_plan_close.restype = None
    L.avdf_session_create.argtypes = [c_void_p, c_void_p, c_size_t, POINTER(c_void_p)]
    L.avdf_session_get_io.argtypes = [c_void_p, POINTER(SessionIO)]
    L.avdf_session_run.argtypes = [c_void_p, c_int32, POINTER(c_int64), c_void_p]
    L.avdf_session_destroy.argtypes = [c_void_p]
    L.avdf_session_destroy.restype = None
    L.avdf_plan_window_layout.argtypes = [c_void_p, c_double, POINTER(c_int64), c_double, c_double, c_int32, POINTER(c_int32),
                                          POINTER(c_int32), POINTER(c_float), POINTER(c_float)]
    L.avdf_session_window_bytes.restype = c_size_t
    L.avdf_session_window_bytes.argtypes = [c_void_p, c_int32, c_int32]
    L.avdf_session_attach_windows.argtypes = [c_void_p, c_void_p, c_size_t, c_int32, c_int32]
    L.avdf_session_run_windows.argtypes = [c_void_p, POINTER(WindowRunArgs), c_void_p]
    L.avdf_format_results_workspace_bytes.restype = c_size_t
    L.avdf_format_results_workspace_bytes.argtypes = [c_int32]
    L.avdf_format_results.argtypes = [POINTER(FormatArgs), c_void_p]
    for name in EXPORTS:
        fn = getattr(L, name)
        if name not in ("avdf_last_error", "avdf_nms_workspace_bytes", "avdf_postprocess_workspace_bytes",
                        "avdf_conv_gemm_workspace_bytes", "avdf_eval_workspace_bytes", "avdf_eval_proposal_workspace_bytes",
                        "avdf_window_merge_workspace_bytes", "avdf_abi_version", "avdf_plan_close", "avdf_session_destroy",
                        "avdf_session_window_bytes", "avdf_format_results_workspace_bytes",
                        "avdf_postprocess_sweep_workspace_bytes"):
            fn.restype = c_int32
    if L.avdf_abi_version() != 3:
        raise AvdfError("libavdf_sm100.so ABI version mismatch")
    _lib = L
    return L


def check(rc, what=""):
    if rc != 0:
        msg = lib().avdf_last_error()
        raise AvdfError("%s failed (%d): %s" % (what or "avdf call", rc, msg.decode() if msg else ""))


def ptr(t):
    """Raw device (or host) pointer of a torch tensor; None -> NULL."""
    if t is None:
        return None
    return c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return c_void_p(torch.cuda.current_stream().cuda_stream)


# launch counter: bench.py reports how many kernels of this library ran in the timed region
LAUNCHES = {"n": 0}


def count(n=1):
    LAUNCHES["n"] += n
