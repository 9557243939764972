/*
 * avdf.h — C-ABI of libavdf_sm100.so: the B200 (sm_100a) kernels behind the temporal-localization
 * inference path of audio-visual/Audio_Visual_Deepfake_Detection.
 *
 * Conventions
 *   - every entry point returns AVDF_OK (0) or a negative AVDF_ERR_* code and never throws;
 *     avdf_last_error() returns the message of the calling thread's last failure;
 *   - all pointers are DEVICE pointers owned by the caller unless a comment says "host";
 *     nothing is allocated behind the caller's back (scratch comes in through workspace
 *     pointers whose size is queried with the matching *_workspace_bytes function);
 *   - `stream` is a cudaStream_t passed as void*; calls are asynchronous on that stream;
 *   - activations are token-major ("channel-last"): [batch, rows_per_video, channels], channels
 *     contiguous; weights of a conv with k taps are [c_out, k * c_in] with the tap index outermost
 *     inside a row (W[co][j * c_in + ci] = reference weight[co][ci][j]).
 *
 * Reference interfaces replaced (paths relative to the reference root):
 *   avdf_nms_hard / avdf_nms_soft   pybind11 module nms_1d_cpu {nms, softnms},
 *                                   libs/utils/csrc/nms_cpu.cpp:19-58, 67-160, 172-182
 *   avdf_postprocess                libs/modeling/av_fd_no_recon.py:760-876 (inference_single_video,
 *                                   postprocessing) + libs/utils/nms.py:8-190 (NMSop, SoftNMSop,
 *                                   seg_voting, batched_nms)
 *   avdf_interp_concat              libs/datasets/deepfake_video_audio.py:513-547 (F.interpolate x3 + cat)
 *   avdf_interp_concat_ranges,      new: sliding windows over recordings longer than the training clips (the same
 *   avdf_window_merge               resampling on row ranges; the windows' results merged with batched_nms)
 *   avdf_host_pack                  HOST: DataLoader collate + pin of the raw stream arrays,
 *                                   libs/datasets/deepfake_video_audio.py:547-558 (dataset item) and the
 *                                   per-video `.to(device)` of libs/modeling/av_fd_no_recon.py:476-477
 *   avdf_pack_feats                 preprocessing, libs/modeling/av_fd_no_recon.py:431-479 (pad + batch layout)
 *   avdf_conv_gemm                  MaskedConv1D (libs/modeling/blocks.py:13-63) as used by the
 *                                   embedding (backbones.py:437-445), the 1x1 projections and MLP of the
 *                                   transformer blocks (blocks.py:1169-1171,1223,1291-1297), FPN laterals
 *                                   (necks.py:69-73), head towers (av_fd_no_recon.py:75-89,144-159) and
 *                                   DownBlock convs (blocks.py:1495-1516), with LayerNorm (blocks.py:70-112),
 *                                   activation, positional encoding and residual/AffineDropPath fused
 *   avdf_ln_dwconv_ln               LN -> depthwise MaskedConv1D(k3, stride) -> LN of LocalMaskedMHCA /
 *                                   LocalMaskedMMHCA (blocks.py:1159-1165, 726-741) incl. the nearest
 *                                   up/down-sampling of backbones.py:487,490 and MaxPool1d skip (blocks.py:1277-1281)
 *   avdf_attention                  banded / global softmax attention (blocks.py:977-1224, 274-313)
 *   avdf_ln_rows                    LayerNorm before the MLP (blocks.py:1311)
 *   avdf_instnorm_lrelu             InstanceNorm1d + LeakyReLU of DownBlock (blocks.py:1508-1515)
 *   avdf_fpn_fuse                   FPN1D top-down sum + depthwise conv + LN (necks.py:75-93)
 *   avdf_head_final                 last conv of the cls / reg heads + Scale + ReLU (av_fd_no_recon.py:82-89,152-159)
 *   avdf_vcls_exp12 / _exp13        video-level classifier tails (blocks.py:1608-1626, 1682-1700)
 *   avdf_eval_detection             libs/utils/metrics.py ANETdetection (AP and Recall@kx of one class), the evaluator
 *                                   valid_one_epoch calls (libs/utils/train_utils.py)
 *   avdf_eval_proposal              libs/utils/Evaluation/eval_proposal.py ANETproposal (ActivityNet AR vs. AN)
 */
#ifndef AVDF_H_
#define AVDF_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define AVDF_API __attribute__((visibility("default")))
#else
#define AVDF_API
#endif

/* 3: avdf_conv_gemm_args grew (dot_w / dot_n / dot_out, tap_rows); avdf_head_combine, avdf_logmel, avdf_byola_* added */
#define AVDF_ABI_VERSION 3
#define AVDF_MAX_LEVELS 8
#define AVDF_MAX_SEGS 1024

enum { AVDF_OK = 0, AVDF_ERR_INVALID = -1, AVDF_ERR_CUDA = -2, AVDF_ERR_UNSUPPORTED = -3 };
enum { AVDF_DTYPE_F32 = 0, AVDF_DTYPE_BF16 = 1, AVDF_DTYPE_F16 = 2 };
enum { AVDF_ACT_NONE = 0, AVDF_ACT_RELU = 1, AVDF_ACT_GELU = 2 };

/* ---- runtime ---- */
AVDF_API int avdf_abi_version(void);
AVDF_API const char* avdf_last_error(void);
/* fills SM count and compute capability of the current device */
AVDF_API int avdf_device_info(int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor);

/* ---- K1: per-stream linear resize to t_out + channel concat (video | byola | emo) ----
 * Streams are packed row-major [sum_b T_s(b), C_s] fp32 with per-stream prefix offsets [batch+1]
 * (rows). A stream with C_s == 0 is absent. out: [batch, t_out, c_video+c_byola+c_emo]. */
AVDF_API int avdf_interp_concat(const float* video, const float* byola, const float* emo,
                       const int32_t* video_off, const int32_t* byola_off, const int32_t* emo_off,
                       int32_t batch, int32_t c_video, int32_t c_byola, int32_t c_emo, int32_t t_out,
                       void* out, int32_t out_dtype, void* stream);

/* The same with the raw streams stored as bf16 (in_dtype = AVDF_DTYPE_BF16): the opt-in 16-bit feature-shard format of the
 * ingestion path (half the host -> device bytes per video; the interpolation arithmetic stays fp32). */
AVDF_API int avdf_interp_concat_in(const void* video, const void* byola, const void* emo, int32_t in_dtype,
                          const int32_t* video_off, const int32_t* byola_off, const int32_t* emo_off,
                          int32_t batch, int32_t c_video, int32_t c_byola, int32_t c_emo, int32_t t_out,
                          void* out, int32_t out_dtype, void* stream);

/* Row-range form (sliding windows over long recordings): video b of stream s is rows [start[s*batch + b],
 * start[s*batch + b] + count[s*batch + b]) of that stream's packed source; start / count are device int32 [3, batch]
 * (rows of absent streams are ignored). Windows may overlap and share rows, so overlapping windows of one recording
 * read one device copy of it. Every count must be >= 1 and every range inside the source. The arithmetic is
 * avdf_interp_concat's: a range equal to a video's CSR rows gives the same bits. */
AVDF_API int avdf_interp_concat_ranges(const void* video, const void* byola, const void* emo, int32_t in_dtype,
                              const int32_t* start, const int32_t* count,
                              int32_t batch, int32_t c_video, int32_t c_byola, int32_t c_emo, int32_t t_out,
                              void* out, int32_t out_dtype, void* stream);

/* ---- preprocessing (av_fd_no_recon.py:431-479): one video's feats [channels, t] fp32 (dataset item layout)
 * -> token-major rows out[t_padded, channels], zero-padded from t to t_padded. */
AVDF_API int avdf_pack_feats(const float* feats_ct, int32_t channels, int32_t t, int32_t t_padded, void* out,
                    int32_t out_dtype, void* stream);

/* ---- NMS: same contracts as nms_1d_cpu.nms / nms_1d_cpu.softnms, on device memory ----
 * segs [n,2], scores [n]; out_idx [n] int64 (kept input indices, descending score / pick order);
 * out_count [1]. max_num <= 0: run to completion (the reference's behaviour); max_num > 0: stop after
 * that many picks (the wrappers consume no more, nms.py:29-30,56-63). dets [n,3] is written in place
 * for the picks, like the reference. */
AVDF_API size_t avdf_nms_workspace_bytes(int32_t n);
AVDF_API int avdf_nms_hard(const float* segs, const float* scores, int32_t n, float iou_threshold, int32_t max_num,
                  int64_t* out_idx, int32_t* out_count, void* workspace, size_t workspace_bytes, void* stream);
AVDF_API int avdf_nms_soft(const float* segs, const float* scores, int32_t n, float* dets, float iou_threshold,
                  float sigma, float min_score, int32_t method, int32_t max_num, int64_t* out_idx,
                  int32_t* out_count, void* workspace, size_t workspace_bytes, void* stream);

/* ---- decode + batched_nms + seconds conversion, one CTA per video ---- */
typedef struct avdf_postprocess_args {
  int32_t batch;
  /* decode inputs (logits == NULL: candidates are provided in cand_* instead) */
  const float* logits;           /* [batch, P]      P = sum(level_len), level-major per video */
  const float* offsets;          /* [batch, P, 2]   */
  const uint8_t* mask;           /* [batch, P]      */
  int32_t n_levels;
  int32_t level_len[AVDF_MAX_LEVELS];
  float level_stride[AVDF_MAX_LEVELS];
  float pre_nms_thresh; int32_t pre_nms_topk; float duration_thresh;
  /* candidates: written by decode (and read by voting), or given */
  float* cand_segs;              /* [batch, cand_cap, 2] */
  float* cand_scores;            /* [batch, cand_cap]    */
  int32_t* cand_count;           /* [batch]              */
  int32_t cand_cap;
  /* batched_nms (class-agnostic path, nms.py:160-190) */
  float iou_threshold, min_score, sigma, voting_thresh;
  int32_t max_seg_num, use_soft_nms, soft_method;   /* use_soft_nms: 0 hard, 1 soft, -1 no NMS (test_cfg nms_method
                                                     * 'none', av_fd_no_recon.py:847: the decoded candidates go straight
                                                     * to the seconds conversion; out_* then hold cand_cap entries per video) */
  /* seconds conversion (all NULL: stay on the feature grid) */
  const float* vid_feat_stride;  /* [batch] */
  const float* vid_half_nframes; /* [batch] 0.5 * feat_num_frames */
  const float* vid_fps;          /* [batch] */
  const float* vid_duration;     /* [batch] */
  /* outputs, sorted by descending score */
  float* out_segs;               /* [batch, max_seg_num, 2] */
  float* out_scores;             /* [batch, max_seg_num]    */
  int32_t* out_count;            /* [batch]                 */
  void* workspace; size_t workspace_bytes;
  /* optional result records for the multi-GPU gather (SURVEY 8e; the reference's per-video JSON record,
   * libs/utils/train_utils.py:577-595): every video appends ONE fixed-size fp32 row
   *   [video index, count, video_cls, scores[max_seg_num], segs[max_seg_num][2]]
   * to rec_ring at row atomicAdd(rec_counter, 1) % rec_cap. All NULL / 0: no records. */
  float* rec_ring;               /* [rec_cap, 3 + 3 * max_seg_num] */
  uint32_t* rec_counter;         /* [1] device counter, owned by the caller */
  int32_t rec_cap;
  const int32_t* vid_index;      /* [batch] global video index of every row of the batch */
  const float* vid_cls;          /* [batch] video-level logit */
  /* optional: index (into the video's candidate list) of every returned segment, in output order - the label of a
   * pick in class-agnostic NMS over several classes is cls_idxs[index] (libs/utils/nms.py:159-180) */
  int32_t* out_index;            /* [batch, max_seg_num] */
} avdf_postprocess_args;          /* host struct */
AVDF_API size_t avdf_postprocess_workspace_bytes(int32_t batch, int32_t cand_cap);
AVDF_API int avdf_postprocess(const avdf_postprocess_args* args, void* stream);

/* ---- cross-window merge of the sliding-window path (csrc/window.cu) ----
 * Recording r owns window rows [rec_win[r], rec_win[r+1]) of the window outputs (the per-window postprocess results:
 * seconds within the window, sorted, win_count[w] <= max_seg_num of them). For a recording with more than one window:
 * candidates = fp32(win_start[w]) + segment (round to nearest) over its windows in ascending order, each window's
 * segments in output order; then the class-agnostic batched_nms of libs/utils/nms.py over that list (hard, or soft
 * method 2; seg_voting over the whole list when voting_thresh > 0, in the summation order of oracle/nms_ref.c; stable
 * sort by score; cap at max_seg_num); out_cls = max window logit. A recording with one window gets that window's
 * output unchanged. All of it is three launches on `stream`, no host synchronisation. Optional records: one row per
 * recording in the avdf_postprocess record layout. cand_cap >= max windows per recording * max_seg_num. */
typedef struct avdf_window_merge_args {
  int32_t n_rec;
  const int32_t* rec_win;        /* [n_rec + 1] device */
  const float* win_start;        /* [n_win] window start, seconds (fp32) */
  const float* win_segs;         /* [n_win, max_seg_num, 2] */
  const float* win_scores;       /* [n_win, max_seg_num] */
  const int32_t* win_count;      /* [n_win] */
  const float* win_cls;          /* [n_win] video-level logit of every window */
  int32_t cand_cap;
  float iou_threshold, min_score, sigma, voting_thresh;
  int32_t max_seg_num, use_soft_nms;   /* 0 hard, 1 soft */
  float* out_segs;               /* [n_rec, max_seg_num, 2] */
  float* out_scores;             /* [n_rec, max_seg_num] */
  int32_t* out_count;            /* [n_rec] */
  float* out_cls;                /* [n_rec] */
  void* workspace; size_t workspace_bytes;   /* avdf_window_merge_workspace_bytes(n_rec, cand_cap) */
  float* rec_ring; uint32_t* rec_counter; int32_t rec_cap; const int32_t* vid_index;   /* optional, as avdf_postprocess */
} avdf_window_merge_args;        /* host struct */
AVDF_API size_t avdf_window_merge_workspace_bytes(int32_t n_rec, int32_t cand_cap);
AVDF_API int avdf_window_merge(const avdf_window_merge_args* args, void* stream);

/* ---- conv-as-GEMM with fused epilogue ----
 * out[b, seg_o_row + t, n] = epi( sum_{j<taps} sum_{c<c_in} W[n, j*c_in + c] * A[b, seg_a_row + stride*t + j - taps/2, c] )
 * (rows outside [0, stride * seg_t_out) of the level read as zero), for every segment `seg`. Segments are levels of a
 * pyramid (shared weights) or independent problems stacked along the rows with their own weight block (seg_w_row):
 * e.g. the q, k, v projections of one attention block in a single launch.
 * epi(v): v += bias[n]; v *= mask[row]; v = LN_n(v) * ln_w + ln_b; v = act(v); v += pe[t, n] * mask[row];
 *         v = residual[row, n] * mask[row] + gamma[n] * v            (each step only if its pointer is set;
 *         ln_after_residual moves the LayerNorm behind the residual step, see the field below)
 * dtype F32 -> fp32 CUDA-core path (parity mode); BF16 / F16 -> TMA + tcgen05 tensor-core path (A and W in that
 * 16-bit format, fp32 accumulate in TMEM). out_h (optional) receives a 16-bit copy in out_h_dtype (BF16 | F16). */
#define AVDF_MAX_TAPS 9
typedef struct avdf_conv_gemm_args {
  int32_t batch, n_out, c_in, taps, stride, n_seg;
  int32_t seg_t_out[AVDF_MAX_LEVELS];
  int32_t seg_a_row[AVDF_MAX_LEVELS];
  int32_t seg_o_row[AVDF_MAX_LEVELS];
  int32_t seg_w_row[AVDF_MAX_LEVELS];  /* row offset into w / bias / ln_* / gamma for this segment (0: shared weights);
                                        * w then holds n_w_rows >= seg_w_row + n_out rows (0 means n_out) */
  int32_t n_w_rows;
  int64_t a_rows_per_video, o_rows_per_video;
  const void* a;                 /* [batch, a_rows_per_video, c_in] */
  const void* w;                 /* [n_out, taps * c_in] */
  int32_t dtype;
  const float* bias; const uint8_t* row_mask; const float* ln_w; const float* ln_b; int32_t act;
  const float* pe; const float* residual; const float* gamma;
  float* out_f32; void* out_h; int32_t out_h_dtype;   /* [batch, o_rows_per_video, n_out] */
  void* workspace; size_t workspace_bytes;
  /* ln_after_residual != 0 (16-bit path, n_out = 256, residual + ln_w + out_f32 + out_h all set): the LayerNorm is applied
   * AFTER the residual step instead of before it - out_f32 receives y = residual * mask + gamma * ((acc + bias) * mask)
   * (the block's residual stream, blocks.py:1309-1310 / 868-869) and out_h receives LN(y) * ln_w + ln_b, the operand of
   * the block's MLP (blocks.py:1311): the attention projection and LN2 in one launch. act must be NONE, pe NULL. */
  int32_t ln_after_residual;
  /* tap_mode 0: taps centred on the output position (offsets j - taps/2, MaskedConv1D); 1: forward taps (offsets
   * 0 .. taps-1, stride 1 only): the row pair (x[t], x[t+1]) a stride-2 ConvTranspose1d(k=3, padding=1, output_padding=1)
   * reads for its outputs 2t and 2t+1 (blocks.py:1443-1491) - see libs/modeling/engine.py `up_block` */
  int32_t tap_mode;
  /* Row dot products instead of (or next to) the output tensor (16-bit path, n_out = 256, wide configuration):
   * dot_out[row, j] = sum_n dot_w[j, n] * v[row, n] for j < dot_n <= 6, v = the epilogue's result. With dot_out set,
   * out_f32 and out_h may both be NULL: the last layer of the cls / reg towers then emits only the per-tap partial sums of
   * the heads' final k3 convolution (av_fd_no_recon.py:82-89, 152-159), which avdf_head_combine turns into logits / offsets. */
  const float* dot_w;            /* [dot_n, n_out] fp32 or NULL */
  int32_t dot_n;
  float* dot_out;                /* [batch, o_rows_per_video, dot_n] fp32 or NULL */
  /* Explicit tap table (stride 1, tap_mode 0, taps <= AVDF_MAX_TAPS): tap j reads input row t + tap_rows[j] instead of
   * t + j - taps/2. With the rows of a (time, mel) grid flattened and padded (csrc/byola.cu "grid layout") the nine offsets
   * {-1,0,1} * row_pitch + {-1,0,1} make the launch a 3x3 Conv2d (audio_feature/content_audio/byol_a/models.py:59, 64). */
  const int32_t* tap_rows;       /* host [taps] or NULL */
} avdf_conv_gemm_args;            /* host struct */
AVDF_API size_t avdf_conv_gemm_workspace_bytes(const avdf_conv_gemm_args* args);
AVDF_API int avdf_conv_gemm(const avdf_conv_gemm_args* args, void* stream);

/* ---- LN -> depthwise conv k3 (stride 1|2) * mask -> LN, for up to 3 streams sharing one source ----
 * src [batch, t_src, C] fp32. Virtual input position p in [0, t_virt) reads source row
 * (shift >= 0 ? p >> shift : p << -shift)  (nearest up / down-sampling of backbones.py:487,490).
 * out_s[b, t', :] = LN_out_s( (sum_j dw_s[:, j] * u_s[stride*t' + j - 1]) * mask_out[b, t'] ),
 * u_s[p] = LN(src[map(p)]) * ln_in_w_s + ln_in_b_s inside [0, t_virt), 0 outside.
 * skip_out (optional, stride 2): MaxPool1d(3, 2, 1) of the raw source rows. */
typedef struct avdf_ln_dwconv_ln_args {
  int32_t batch, channels, t_src, t_virt, shift, stride, n_streams;
  const float* src;
  const uint8_t* mask_out;       /* [batch, t_virt / stride] */
  const float* ln_in_w[3]; const float* ln_in_b[3];
  const float* dw_w[3];          /* [C, 3] */
  const float* ln_out_w[3]; const float* ln_out_b[3];
  void* out[3];                  /* [batch, out_rows_per_video, C], row t' of video b at b * out_rows_per_video + t' */
  int32_t out_dtype;
  int32_t out_rows_per_video;    /* 0: t_virt / stride (dense). Larger: several streams interleaved per video */
  float* skip_out;               /* [batch, t_virt / stride, C] fp32 or NULL */
  int32_t tile_rows;             /* output rows per warp tile: 0 = chosen from the problem size, or 2 / 4 / 8 */
} avdf_ln_dwconv_ln_args;
AVDF_API int avdf_ln_dwconv_ln(const avdf_ln_dwconv_ln_args* args, void* stream);

/* ---- fused transformer MLP (blocks.py:1236-1243 `self.mlp`, applied at blocks.py:1315-1316) ----
 * out = residual * mask + gamma * ((GELU(x W1^T + b1) W2^T + b2) * mask), exact-erf GELU, fp32 accumulate; the
 * [rows, hidden] activations stay on chip (16-bit, like the unfused path's intermediate tensor). channels = 256,
 * hidden = 1024, dtype = AVDF_DTYPE_F16 | AVDF_DTYPE_BF16 (x, w1, w2). Equivalent to two avdf_conv_gemm calls. */
typedef struct avdf_mlp_fused_args {
  int32_t rows, channels, hidden, dtype;
  const void* x;                 /* [rows, channels] */
  const void* w1; const float* b1;   /* [hidden, channels], [hidden] */
  const void* w2; const float* b2;   /* [channels, hidden], [channels] */
  const uint8_t* row_mask;       /* [rows] or NULL */
  const float* residual;         /* [rows, channels] fp32 */
  const float* gamma;            /* [channels] or NULL (AffineDropPath scale, blocks.py:1316) */
  float* out;                    /* [rows, channels] fp32 */
  void* out_h;                   /* optional 16-bit copy of out (same dtype as x) or NULL */
  int32_t out_h_t, out_h_pitch, out_h_row0;   /* 0: the copy is dense [rows, channels]; else rows = batch * out_h_t and row
                                               * b * out_h_t + t goes to row b * out_h_pitch + out_h_row0 + t (one level of
                                               * a [batch, P, channels] pyramid buffer, necks.py:62-93's input) */
  /* "block tail" (att != NULL): the attention output projection and LN2 of the block run in the same launch
   * (blocks.py:1223, 1309-1316 / 779, 868-872):
   *   y = skip * mask + gamma_attn * ((att w_o^T + b_o) * mask);  x = LN(y) * ln2_w + ln2_b (16-bit, never leaves the SM);
   *   out = (y + GELU(x w1^T + b1) w2^T + b2) * mask
   * y stays in the tensor-memory accumulator and the second GEMM accumulates on top of it, so the MLP's AffineDropPath
   * scale must be FOLDED by the caller: pass w2 = diag(scale) w2, b2 = scale * b2 and gamma = NULL. x and residual are
   * ignored; y (optional, may be NULL) receives a copy of the residual stream between the two halves of the block.
   * Equivalent to avdf_conv_gemm(ln_after_residual) followed by the plain avdf_mlp_fused. */
  const void* att;               /* [rows, channels] 16-bit (dtype) or NULL */
  const void* w_o; const float* b_o;   /* [channels, channels], [channels] */
  const float* gamma_attn;       /* [channels] or NULL */
  const float* ln2_w; const float* ln2_b;   /* [channels] */
  const float* skip;             /* [rows, channels] fp32: the block's input (or its max-pooled copy) */
  float* y;                      /* [rows, channels] fp32 or NULL */
} avdf_mlp_fused_args;
AVDF_API int avdf_mlp_fused(const avdf_mlp_fused_args* args, void* stream);

/* ---- multi-head attention over q,k,v [batch, t, C]; window > 1: band |i-j| <= window/2 with additive
 * -1e4 on masked keys and zeroed masked query rows (blocks.py:1152-1224); window <= 1: global with
 * -inf on masked keys (blocks.py:274-313). Row i of video b of q/k/v is at (b * qkv_rows_per_video + i) * C from the
 * respective pointer (qkv_rows_per_video 0 = t; 3t when q,k,v of a video are stacked in one buffer). out [batch, t, C]. */
AVDF_API int avdf_attention(const void* q, const void* k, const void* v, const uint8_t* kv_mask, void* out,
                   int32_t in_dtype, int32_t out_dtype, int32_t batch, int32_t t, int32_t qkv_rows_per_video,
                   int32_t channels, int32_t n_head, int32_t window, void* stream);

/* ---- LayerNorm over channels of fp32 rows -> fp32 or bf16 ---- */
AVDF_API int avdf_ln_rows(const float* x, const float* w, const float* b, void* out, int32_t out_dtype, int64_t rows,
                 int32_t channels, void* stream);

/* ---- InstanceNorm1d over T (per video, channel; eps 1e-5, biased) + LeakyReLU(slope) ---- */
AVDF_API int avdf_instnorm_lrelu(const float* x, void* out, int32_t out_dtype, int32_t batch, int32_t t, int32_t channels,
                        float slope, void* stream);

/* ---- FPN top-down fuse: L_l[t] = sum_{j>=l} lat_j[t >> (j-l)]; F_l = LN_l(dwconv3_l(L_l) * mask) ----
 * lat / out are pyramids [batch, P, C] with levels concatenated per video. dw_w [n_levels, C, 3],
 * ln_w / ln_b [n_levels, C]. */
AVDF_API int avdf_fpn_fuse(const float* lat, const uint8_t* mask, const float* dw_w, const float* ln_w, const float* ln_b,
                  void* out, int32_t out_dtype, int32_t batch, int32_t channels, int32_t n_levels,
                  const int32_t* level_len /* host */, void* stream);

/* ---- last conv (k3) of both heads: logits [batch,P] = cls_w . x_cls + cls_b (* mask);
 * offsets [batch,P,2] = relu((reg_w . x_reg + reg_b) * mask * scale_l). Towers are pyramids [batch,P,C]. */
AVDF_API int avdf_head_final(const void* cls_feat, const void* reg_feat, int32_t dtype, const uint8_t* mask,
                    const float* cls_w /* [1,3*C] */, const float* cls_b, const float* reg_w /* [2,3*C] */,
                    const float* reg_b, const float* level_scale /* host [n_levels] */, float* logits,
                    float* offsets, int32_t batch, int32_t channels, int32_t n_levels,
                    const int32_t* level_len /* host */, void* stream);

/* The same from per-tap partial sums (avdf_conv_gemm dot_out of the last tower layers): cls_dots [batch, P, 3] holds, for
 * every pyramid row, the dot products of its tower output with the three taps of cls_head.cls_head.conv.weight; reg_dots
 * [batch, P, 6] = (output o, tap j) at o * 3 + j. logit[t] = dots[t-1][0] + dots[t][1] + dots[t+1][2] + bias inside the level. */
AVDF_API int avdf_head_combine(const float* cls_dots, const float* reg_dots, const uint8_t* mask, const float* cls_b,
                      const float* reg_b, const float* level_scale /* host [n_levels] */, float* logits, float* offsets,
                      int32_t batch, int32_t n_levels, const int32_t* level_len /* host */, void* stream);

/* ---- video-level classifier tails ---- */
/* exp12 (blocks.py:1608-1626): z [batch, t <= 32, C] (after the last DownBlock) -> logit [batch]. The two dense
 * weights are passed TRANSPOSED ([in, out]: conv0_wt[k][c] = conv0.weight[c][k], lin1_wt[j][c] = conv1.weight[c][j]). */
AVDF_API int avdf_vcls_exp12(const void* z, int32_t dtype, const float* conv0_wt /* [C,C] */, const float* lin1_wt /* [2C,C] */,
                    const float* ln_w, const float* ln_b, const float* lin2_w /* [C] */, const float* lin2_b,
                    float* out, int32_t batch, int32_t t, int32_t channels, void* stream);
/* exp13 (blocks.py:1682-1700): z [batch, t, C] -> logit [batch] */
AVDF_API int avdf_vcls_exp13(const void* z, int32_t dtype, const float* conv0_w /* [C,C] */, const float* seg_w /* [C] */,
                    const float* seg_b, const float* cls_w /* [2] */, const float* cls_b, float* out,
                    int32_t batch, int32_t t, int32_t channels, void* stream);

/* ---- SURVEY 8(f).4: upstream BYOL-A feature extractor (audio_feature/content_audio) ----
 * A batch of clips is packed along time. frames(clip) = 1 + samples / 160 (centre = True); all index arrays are DEVICE
 * int arrays prepared by the host side (libs/features/byola.py `BatchPlan`). */
/* replaces torchaudio MelSpectrogram(16 kHz, n_fft = win = 1024, hop 160, 64 mels, 60-7800 Hz) + log(x + eps) +
 * PrecomputedNorm (extract_audio_feature_one.py:34-42, 66; byol_a/augmentations.py:218-219):
 * wav = the clips back to back, clip c = samples [clip_sample_off[c], clip_sample_off[c+1]) (each > 512 samples),
 * its frames are rows [clip_frame_off[c], clip_frame_off[c+1]) of lms [total_frames, 64] (time-major). One CTA transforms
 * frames 2j and 2j+1 of a clip together: clip_pair_off[c] = sum over earlier clips of ceil(frames / 2), total_pairs its end.
 * window [1024] (periodic Hann), twiddle [1024][2] = (cos, -sin)(2 pi j / 1024); the mel triangles in sparse form: filter m
 * weighs the power bins mel_lo[m] .. mel_lo[m] + mel_cnt[m] - 1 with mel_w[m * mel_stride + 0 ..] (all DEVICE arrays;
 * mel_lo[m] + mel_cnt[m] <= 513). */
AVDF_API int avdf_logmel(const float* wav, const int64_t* clip_sample_off, const int32_t* clip_frame_off,
                const int32_t* clip_pair_off, int32_t n_clips, int32_t total_frames, int32_t total_pairs, const float* window,
                const float* twiddle, const int32_t* mel_lo, const int32_t* mel_cnt, const float* mel_w, int32_t mel_stride,
                float mean, float std, float* lms, void* stream);
/* features.0-3 of AudioNTT2020Task6 (byol_a/models.py:54-57): Conv2d(1, 64, 3, padding 1) + BatchNorm2d (eval; folded by
 * the caller into w [64, 9] (mel tap major) and b [64]) + ReLU + MaxPool2d(2) -> level-1 grid layout
 * out [n_steps * 34, 64] (csrc/byola.cu): step s holds pooled time step t_of_step[s] of clip clip_of_step[s] (-1: an
 * all-zero separator step). mask_out (optional) [n_steps * 34] receives 1 for rows holding data, 0 for padding rows. */
AVDF_API int avdf_byola_conv1_pool(const float* lms, const int32_t* clip_frame_off, const float* w, const float* b,
                const int32_t* clip_of_step, const int32_t* t_of_step, int32_t n_steps, void* out, int32_t out_dtype,
                uint8_t* mask_out, void* stream);
/* MaxPool2d(2) (models.py:62, 67) from the grid layout with mel_in rows per step (clip c starts at step clip_step_in[c])
 * into the next grid layout (pad_out 1: [n_steps_out * (mel_in / 2 + 2), 64]) or into dense rows for the fc layers
 * (pad_out 0: [n_steps_out, (mel_in / 2) * 64], feature index = mel * 64 + channel as models.py:80-82 flattens it). */
AVDF_API int avdf_byola_pool(const void* in, int32_t dtype, int32_t mel_in, const int32_t* clip_step_in,
                const int32_t* clip_of_step, const int32_t* t_of_step, int32_t n_steps_out, int32_t pad_out, void* out,
                uint8_t* mask_out, void* stream);

/* ---- detection evaluation of ONE class: ActivityNet AP per tIoU threshold + Recall@kx (ActionFormer / UMMAFormer
 * libs/utils/metrics.py ANETdetection: compute_average_precision_detection, compute_topkx_recall_detection) ----
 * Videos in CSR form: video v owns predictions [pred_off[v], pred_off[v+1]) and GT rows [gt_off[v], gt_off[v+1]).
 * Prediction order is score descending, ties by smaller input index; within a video the GT rows are tried in tIoU-descending
 * order, ties by larger GT index. tIoU is fp64 in numpy's operation order. AP is the area under the monotone precision
 * envelope over npos = n_gt; recall_hits[t * n_topk + q] counts the GT rows whose best tIoU over their video's top
 * top_k[q] * n_gt(video) predictions is >= thresholds[t] (divide by n_gt for Recall@kx). Limits: n_thr <= 16, n_topk <= 4,
 * <= 8192 predictions and <= 64 GT rows per video. Per-video limits are checked on the device: a violation sets bits of
 * *status (AVDF_EVAL_*) and the call then writes none of ap / recall_hits / tp_mask. Deterministic (bit-identical runs). */
enum { AVDF_EVAL_PRED_LIMIT = 1, AVDF_EVAL_GT_LIMIT = 2, AVDF_EVAL_BAD_OFFSETS = 4 };
typedef struct avdf_eval_args {
  int64_t n_pred;                /* predictions (< 2^31) */
  int32_t n_video;               /* videos with GT or predictions of this class */
  int32_t n_gt;                  /* GT rows (npos >= 1) */
  const int64_t* pred_off;       /* [n_video + 1] */
  const double* pred_seg;        /* [n_pred, 2] (start, end), 16-byte aligned */
  const double* pred_score;      /* [n_pred] */
  const int32_t* gt_off;         /* [n_video + 1] */
  const double* gt_seg;          /* [n_gt, 2], 16-byte aligned */
  const double* thresholds;      /* HOST [n_thr] tIoU thresholds */
  int32_t n_thr;
  const int32_t* top_k;          /* HOST [n_topk] */
  int32_t n_topk;
  double* ap;                    /* [n_thr] */
  int64_t* recall_hits;          /* [n_thr * n_topk] */
  uint16_t* tp_mask;             /* [n_pred] or NULL: bit t = TP at thresholds[t], at the prediction's input position */
  const int32_t* pred_rank;      /* [n_pred] or NULL: a permutation of 0 .. n_pred - 1 that breaks score ties instead of the
                                  * position (must increase with the position inside every video); lets a caller whose
                                  * predictions are not grouped by video keep its own row order for the ties */
  int32_t* status;               /* [1] 0 on success, else AVDF_EVAL_* bits */
  void* workspace; size_t workspace_bytes;   /* 256-byte aligned */
} avdf_eval_args;                 /* host struct */
AVDF_API size_t avdf_eval_workspace_bytes(int64_t n_pred, int32_t n_video);
AVDF_API int avdf_eval_detection(const avdf_eval_args* args, void* stream);

/* ---- proposal evaluation: ActivityNet average recall vs. average number of proposals (eval_proposal.py
 * average_recall_vs_avg_nr_proposals, ANETproposal), class-agnostic ----
 * Videos in CSR form, normally the videos that have GT rows: video v owns proposals [prop_off[v], prop_off[v+1]) and GT rows
 * [gt_off[v], gt_off[v+1]). Walk order is score descending, ties by smaller row; a video walks its first keep[v] proposals
 * (the host's min(int(n_p * ratio), n_p)). With c = keep[v], or c = 1 and a tIoU of 0 for a video without proposals, point
 * j looks at the first cut_j = min(int(c * an_frac[j]), c) proposals (one fp64 product, truncated; an_frac = the host's
 * 100 pcn values, non-decreasing). matches[t * 100 + j] counts the GT rows with a proposal among those whose tIoU (fp64,
 * numpy's operation order) is >= thresholds[t]; recall = matches / n_gt. Limits: n_thr <= 16, <= 8192 proposals and <= 64 GT
 * rows per video, 0 <= keep[v] <= proposals of v; checked on the device: a violation sets bits of *status (AVDF_EVAL_*) and
 * the call then writes nothing to matches. Integer counts only: bit-identical runs. */
enum { AVDF_EVAL_BAD_KEEP = 8 };
typedef struct avdf_eval_proposal_args {
  int32_t n_video;               /* videos */
  int64_t n_prop;                /* proposal rows in the CSR */
  int32_t n_gt;                  /* GT rows */
  const int64_t* prop_off;       /* [n_video + 1] */
  const double* prop_seg;        /* [n_prop, 2] (start, end), 16-byte aligned */
  const double* prop_score;      /* [n_prop] */
  const int32_t* keep;           /* [n_video] proposals walked per video */
  const int32_t* gt_off;         /* [n_video + 1] */
  const double* gt_seg;          /* [n_gt, 2], 16-byte aligned */
  const double* thresholds;      /* HOST [n_thr] tIoU thresholds */
  int32_t n_thr;
  const double* an_frac;         /* HOST [100] */
  int64_t* matches;              /* [n_thr * 100] */
  int32_t* status;               /* [1] 0 on success, else AVDF_EVAL_* bits */
  void* workspace; size_t workspace_bytes;   /* 256-byte aligned */
} avdf_eval_proposal_args;        /* host struct */
AVDF_API size_t avdf_eval_proposal_workspace_bytes(int32_t n_video);
AVDF_API int avdf_eval_proposal(const avdf_eval_proposal_args* args, void* stream);

/* ---- HOST: gather n byte spans (src[i] -> dst[i], nbytes[i] bytes; all HOST pointers, any alignment; dst is normally
 * a slice of a pinned staging buffer) with up to n_threads threads of a pool that lives inside the library
 * (non-temporal stores). Synchronous; concurrent calls are serialised. No CUDA call is made. */
AVDF_API int avdf_host_pack(const void* const* src, void* const* dst, const size_t* nbytes, int32_t n, int32_t n_threads);

/* HOST: 1 when every span [src[i], src[i] + nbytes[i]) is page-locked host memory (cudaHostAlloc / cudaHostRegister), else 0. */
AVDF_API int avdf_host_all_pinned(const void* const* src, const size_t* nbytes, int32_t n);
/* n asynchronous copies src[i] (pinned HOST) -> dst[i] (DEVICE) on `stream`: ingestion without a staging copy. The sources
 * must stay alive and unchanged until the stream has passed the copies. */
AVDF_API int avdf_h2d_gather(const void* const* src, void* const* dst, const size_t* nbytes, int32_t n, void* stream);

/* ---- the whole model: launch plans (csrc/plan.cu) ----
 * A plan file holds the launch sequence of the raw-stream pass (resampling -> model -> decode / NMS) of one model at one
 * precision and test-time config, for a set of batch sizes, recorded by the Python side
 * (audio_visual_deepfake_detection_b200/libs/modeling/plan.py, `model.export_plan`), together with the packed constants
 * (weights, mask / positional-encoding tables). Replaying it calls the same entry points with the same arguments as the
 * Python path, so results are bit-identical to `model.forward_streams` on the same inputs.
 *
 *   avdf_plan* plan;  avdf_plan_info info;
 *   avdf_plan_open(path, &plan);  avdf_plan_get_info(plan, &info);          (host only, no CUDA call)
 *   cudaMalloc(&consts, info.const_bytes);  avdf_plan_upload(plan, consts, info.const_bytes, stream);
 *   cudaMalloc(&arena, info.session_bytes);  avdf_session_create(plan, arena, info.session_bytes, &s);
 *   avdf_session_get_io(s, &io);
 *   per batch: write io.streams / io.offsets / io.meta (cudaMemcpyAsync on `stream`), avdf_session_run(s, B, rows, stream),
 *              read io.segs / io.scores / io.counts / io.video_cls
 *   avdf_session_destroy(s);  avdf_plan_close(plan);  cudaFree(arena);  cudaFree(consts);
 *
 * Inputs (device, inside the session arena, sized for max_batch):
 *   streams[s]   [rows, channels[s]] of stream s (0 video, 1 byola, 2 emo; NULL when channels[s] == 0), the batch's
 *                recordings back to back, in_dtype (AVDF_DTYPE_F32, or AVDF_DTYPE_BF16 for 16-bit feature shards)
 *   offsets      int32 [3, max_batch + 1]: offsets[s * (max_batch + 1) + b] = first row of recording b in streams[s],
 *                offsets[s * (max_batch + 1) + B] = rows[s]
 *   meta         fp32 [4, B] contiguous (row r at meta + r * B): feat_stride, 0.5 * feat_num_frames, fps, duration.
 *                For a raw-stream item with T rows in its first stream (video if present, else byola), t_out = info.t_out
 *                and its duration in seconds, computed in double and then rounded to float:
 *                  feat_stride = (float)((double)T / t_out);  half_nframes = (float)(0.5 * ((double)T / t_out));
 *                  fps = (float)((double)T / duration);       duration = (float)duration
 * Outputs (device, at their max_batch allocations; rows b < B are written):
 *   segs [B, max_seg_num, 2] seconds, scores [B, max_seg_num] (descending), counts int32 [B], video_cls [B] (logit).
 * A session is one buffer set: it runs on one stream at a time. Concurrent batches use separate sessions of one plan
 * (they share its constants). The plan must stay open while it has sessions. Recordings longer than the model's
 * training clips run as sliding windows on a session: avdf_session_attach_windows / avdf_session_run_windows below. */
typedef struct avdf_plan avdf_plan;          /* parsed plan (host); its constants once uploaded */
typedef struct avdf_session avdf_session;    /* one buffer set = one batch in flight */
typedef struct avdf_plan_info {
  int32_t abi_version, cc_major, cc_minor, sm_count, max_batch, max_seg_num, t_out, in_dtype;
  int32_t channels[3];  int64_t stream_rows[3];    /* video, byola, emo; 0 channels = absent; rows = staging capacity */
  uint64_t batch_mask;                             /* bit b-1: a launch list for batch size b */
  size_t const_bytes, session_bytes;               /* device bytes of avdf_plan_upload / avdf_session_create (256-aligned) */
  char description[1024];                          /* model, precision, test config, switches */
} avdf_plan_info;
/* parse + validate the whole file; makes NO CUDA call. Fails (nothing allocated) on a bad magic / version, a truncated
 * file, an unknown entry point, a scalar type-tag mismatch, a relocation outside its allocation, a struct-size mismatch. */
AVDF_API int avdf_plan_open(const char* path, avdf_plan** out);
AVDF_API int avdf_plan_get_info(const avdf_plan* p, avdf_plan_info* info);
/* constants -> dev (const_bytes, 256-byte aligned) on `stream`, on the current device; refuses a device whose compute
 * capability or SM count differs from the recording device's (launch configurations depend on the SM count). */
AVDF_API int avdf_plan_upload(avdf_plan* p, void* dev, size_t bytes, void* stream);
AVDF_API void avdf_plan_close(avdf_plan* p);
/* dev: session_bytes of device memory (256-byte aligned) on the plan's device; zeroed here (synchronously). */
AVDF_API int avdf_session_create(const avdf_plan* p, void* dev, size_t bytes, avdf_session** out);
typedef struct avdf_session_io {
  void* streams[3]; int32_t* offsets; float* meta;
  float* segs; float* scores; int32_t* counts; float* video_cls;
} avdf_session_io;
AVDF_API int avdf_session_get_io(const avdf_session* s, avdf_session_io* io);
/* One batch of `batch` recordings with rows[s] rows per stream (checked against the staging capacity; nothing is launched
 * when a check fails). The first call for a batch size runs the launch list eagerly on `stream`, captures it (thread-local
 * capture mode) into a CUDA graph and launches that; later calls launch the graph. `stream` must be a created stream
 * (graph capture is not possible on the legacy default stream). Asynchronous; no host synchronisation. */
AVDF_API int avdf_session_run(avdf_session* s, int32_t batch, const int64_t rows[3], void* stream);
/* Releases the session's graphs and, when a window block is attached, its pinned parameter buffer and event. */
AVDF_API void avdf_session_destroy(avdf_session* s);

/* ---- sliding windows on a session (csrc/plan.cu; the C form of forward_streams(window=W, hop=H),
 * libs/modeling/windows.py) ----
 * A recording of D seconds longer than W is cut into n = (int)ceil((D - W) / H) + 1 windows (all in double):
 *   s_k = min(k * H, D - W); window k of stream s (T_s rows) covers rows [floor(s_k * T_s / D), + floor(W * T_s / D))
 *   and its meta is the session-run formula above with T = rows of the window in its first stream and duration W;
 *   win_start[k] = (float)s_k.
 * D <= W: one window covering every row, its meta from the recording's own T and duration D, win_start 0.
 * Every window runs through the plan's pass at the model's trained time scale (its first launch replaced by the row-range
 * resampling avdf_interp_concat_ranges); avdf_window_merge then turns the window results into one result per recording.
 * The first stream is video if present, else byola (else emo). */

/* HOST only, no CUDA call: the windows of one recording as plan p runs them. Returns n >= 1, or < 0 on bad input
 * (avdf_last_error: W not > 0 or NaN, hop not in (0, W], a duration that is not a positive finite number, rows for an
 * absent stream or none for a present one, a window that holds no row of a present stream). When cap >= n (and the
 * arrays are not NULL) it fills start / count [n][3] (rows relative to the recording, 0 for absent streams),
 * meta [n][4] (feat_stride, 0.5 * feat_num_frames, fps, duration) and win_start [n]. */
AVDF_API int32_t avdf_plan_window_layout(const avdf_plan* p, double duration, const int64_t rows[3], double window,
                                         double hop, int32_t cap, int32_t* start, int32_t* count, float* meta,
                                         float* win_start);
/* HOST only: device bytes of a session's window block for calls with at most max_windows windows in all and at most
 * max_windows_per_recording windows per recording (1 <= max_windows_per_recording <= max_windows <= 2^24). With
 * B = info.max_batch, K = info.max_seg_num, W = max_windows it is the sum of
 *   align256(4 * (12 W + 10 B))   window table (per batch [3, B] start, [3, B] count, [4, B] meta; win_start; rec_win)
 *   align256(24 B)                the fixed [3, B] start and count arrays the windowed graphs read
 *   align256(8 K W) + align256(4 K W) + align256(4 W) + align256(4 W)   every window's segs, scores, count, video_cls
 *   avdf_window_merge_workspace_bytes(W, K * max_windows_per_recording)
 * Returns 0 (avdf_last_error says why) when the limits are out of range or the plan cannot run windows: every launch
 * list must start with avdf_interp_concat_in reading the io offsets for its own batch size, and hold exactly one
 * avdf_postprocess that writes the io outputs, keeps no result records and runs hard or soft NMS. */
AVDF_API size_t avdf_session_window_bytes(const avdf_plan* p, int32_t max_windows, int32_t max_windows_per_recording);
/* dev: avdf_session_window_bytes of device memory (256-byte aligned) on the plan's device, owned by the caller and kept
 * until the session is destroyed. Allocates a small pinned host buffer and an event for the per-call parameters.
 * AVDF_ERR_UNSUPPORTED when the plan cannot run windows (see above); a session takes one window block. */
AVDF_API int avdf_session_attach_windows(avdf_session* s, void* dev, size_t bytes, int32_t max_windows,
                                         int32_t max_windows_per_recording);
typedef struct avdf_window_run_args {
  int32_t n_rec;                 /* recordings, >= 1 (may exceed max_batch) */
  const double* duration;        /* host [n_rec] seconds */
  const int64_t* rows;           /* host [n_rec][3]; the recordings lie back to back in io.streams, in this order */
  double window, hop;            /* W > 0, 0 < hop <= W (seconds) */
  float* out_segs;               /* [n_rec, max_seg_num, 2] seconds */
  float* out_scores;             /* [n_rec, max_seg_num] descending */
  int32_t* out_count;            /* [n_rec] */
  float* out_cls;                /* [n_rec] video-level logit (the largest of the recording's windows) */
} avdf_window_run_args;          /* host struct; out_* are device pointers */
/* One call over n_rec recordings staged in io.streams (written as for avdf_session_run; the rows of each stream must fit
 * its staging). Steps, all on `stream`: the windows of every recording (avdf_plan_window_layout) go up as one copy; they
 * run in recording order in batches of the plan's largest batch size - the last batch, when the plan has no list of its
 * size, as the smallest recorded size that holds it, its unused slots repeating its last window - each batch being a
 * device-to-device copy of its ranges and meta, the windowed launch list (eager and captured on the first call for a
 * size, a graph replay after that) and copies of its results aside; then avdf_window_merge with the NMS settings of the
 * plan's recorded postprocess and cand_cap = max_seg_num * (most windows of any recording in this call). No host
 * synchronisation (the pinned parameter buffer is rewritten after an event of the previous call's copy). Refused, with
 * nothing launched and the outputs untouched: no window block attached, n_rec < 1, bad W / hop or a window without a
 * row, rows for an absent stream or none for a present one, rows beyond the staging, more windows than max_windows or
 * more for one recording than max_windows_per_recording, the legacy default stream, another device than the plan's. */
AVDF_API int avdf_session_run_windows(avdf_session* s, const avdf_window_run_args* a, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AVDF_H_ */
