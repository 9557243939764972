// Cross-window merge of the sliding-window path (recordings longer than the window, libs/modeling/windows.py).
//
// Every window of a recording went through the ordinary pass (interp to max_seq_len -> model -> postprocess) as a
// video of its own; its output is seconds within the window. avdf_window_merge turns the window outputs of a call into
// one result per recording, in three launches and no host synchronisation:
//   gather    one CTA per recording: abs = fp32(s_k) + seg (round to nearest) for every segment of window k, windows in
//             ascending k, each window's segments in its output order -> the recording's candidate list
//   NMS       avdf_postprocess in candidate mode (logits == NULL): hard / soft NMS, stable sort by score, cap at
//             max_seg_num; no voting and no seconds conversion there
//   finalize  one CTA per recording: seg_voting of every pick against the whole candidate list in the order of
//             oracle/nms_ref.c (fp32 weights summed left to right, fp64 products accumulated left to right), so the
//             merge is bit-identical to the reference's batched_nms over the same list; video_cls = max window logit;
//             optional fixed-size result record per recording.
// A recording with one window is not merged: its window output is its result, bit for bit.
// Voting commutes with the sort: it rewrites segments only, and every pick's vote depends on that pick alone.
#include "common.cuh"

namespace avdf {

constexpr int WM_THREADS = 256;

struct WindowMergeParams {
  const int* rec_win; const float* win_start;
  const float* win_segs; const float* win_scores; const int* win_count; const float* win_cls;
  float* cand_segs; float* cand_scores; int* cand_count; int cand_cap;
  int K; float voting_thresh;
  float* out_segs; float* out_scores; int* out_count; float* out_cls;
  float* rec_ring; unsigned* rec_counter; int rec_cap; const int* vid_index;
};

__global__ void __launch_bounds__(WM_THREADS) window_gather_kernel(const WindowMergeParams p) {
  const int r = blockIdx.x;
  const int w0 = p.rec_win[r], w1 = p.rec_win[r + 1];
  __shared__ int s_base[WM_THREADS + 1];
  float* cs = p.cand_segs + (size_t)r * p.cand_cap * 2;
  float* cc = p.cand_scores + (size_t)r * p.cand_cap;
  if (w1 - w0 == 1) {                       // a single window is the recording's result as it is: nothing to merge
    if (threadIdx.x == 0) p.cand_count[r] = 0;
    return;
  }
  int base = 0;
  for (int c0 = w0; c0 < w1; c0 += WM_THREADS) {       // windows in chunks of WM_THREADS: prefix of their counts
    const int nw = min(WM_THREADS, w1 - c0);
    if (threadIdx.x == 0) {
      int acc = base;
      for (int i = 0; i < nw; ++i) { s_base[i] = acc; acc += p.win_count[c0 + i]; }
      s_base[nw] = acc;
    }
    __syncthreads();
    for (int i = 0; i < nw; ++i) {
      const int w = c0 + i, n = p.win_count[w], dst = s_base[i];
      const float s = p.win_start[w];
      const float* ws = p.win_segs + (size_t)w * p.K * 2;
      for (int q = threadIdx.x; q < n; q += WM_THREADS) {
        cs[2 * (dst + q)] = __fadd_rn(s, ws[2 * q]);
        cs[2 * (dst + q) + 1] = __fadd_rn(s, ws[2 * q + 1]);
        cc[dst + q] = p.win_scores[(size_t)w * p.K + q];
      }
    }
    base = s_base[nw];
    __syncthreads();
  }
  if (threadIdx.x == 0) p.cand_count[r] = base;
}

__global__ void __launch_bounds__(WM_THREADS) window_finalize_kernel(const WindowMergeParams p) {
  const int r = blockIdx.x, K = p.K;
  const int w0 = p.rec_win[r], w1 = p.rec_win[r + 1];
  float* os = p.out_segs + (size_t)r * K * 2;
  float* osc = p.out_scores + (size_t)r * K;
  __shared__ int s_k;
  __shared__ float s_cls;
  if (w1 - w0 == 1) {
    const int n = p.win_count[w0];
    for (int q = threadIdx.x; q < n; q += WM_THREADS) {
      os[2 * q] = p.win_segs[((size_t)w0 * K + q) * 2];
      os[2 * q + 1] = p.win_segs[((size_t)w0 * K + q) * 2 + 1];
      osc[q] = p.win_scores[(size_t)w0 * K + q];
    }
    if (threadIdx.x == 0) { s_k = n; s_cls = p.win_cls[w0]; }
  } else {
    const int k = p.out_count[r];
    const int n = p.cand_count[r];
    const float* cs = p.cand_segs + (size_t)r * p.cand_cap * 2;
    const float* cc = p.cand_scores + (size_t)r * p.cand_cap;
    if (p.voting_thresh > 0.f) {
      for (int q = threadIdx.x; q < k; q += WM_THREADS) {           // one thread per pick (ref_seg_voting, nms_ref.c)
        const float a0 = os[2 * q], a1 = os[2 * q + 1], la = __fsub_rn(a1, a0);
        float fsw = 0.f;
        for (int j = 0; j < n; ++j) {
          const float b0 = cs[2 * j], b1 = cs[2 * j + 1];
          const float inter = fmaxf(__fsub_rn(fminf(a1, b1), fmaxf(a0, b0)), 0.f);
          const float iou = __fdiv_rn(inter, __fsub_rn(__fadd_rn(la, __fsub_rn(b1, b0)), inter));
          fsw = __fadd_rn(fsw, __fmul_rn(__fmul_rn(iou >= p.voting_thresh ? 1.f : 0.f, cc[j]), iou));
        }
        double s0 = 0.0, s1 = 0.0;
        for (int j = 0; j < n; ++j) {
          const float b0 = cs[2 * j], b1 = cs[2 * j + 1];
          const float inter = fmaxf(__fsub_rn(fminf(a1, b1), fmaxf(a0, b0)), 0.f);
          const float iou = __fdiv_rn(inter, __fsub_rn(__fadd_rn(la, __fsub_rn(b1, b0)), inter));
          const float wgt = __fdiv_rn(__fmul_rn(__fmul_rn(iou >= p.voting_thresh ? 1.f : 0.f, cc[j]), iou), fsw);
          s0 = __dadd_rn(s0, __dmul_rn((double)wgt, (double)b0));
          s1 = __dadd_rn(s1, __dmul_rn((double)wgt, (double)b1));
        }
        os[2 * q] = __double2float_rn(s0);
        os[2 * q + 1] = __double2float_rn(s1);
      }
    }
    if (threadIdx.x == 0) {
      float m = p.win_cls[w0];
      for (int w = w0 + 1; w < w1; ++w) m = fmaxf(m, p.win_cls[w]);
      s_k = k; s_cls = m;
    }
  }
  __syncthreads();
  const int k = s_k;
  if (threadIdx.x == 0) { p.out_count[r] = k; p.out_cls[r] = s_cls; }
  if (p.rec_ring != nullptr) {
    // the record layout of avdf_postprocess: [index, count, video_cls, scores[K], segs[K][2]]
    __shared__ unsigned s_row;
    if (threadIdx.x == 0) s_row = atomicAdd(p.rec_counter, 1u) % (unsigned)p.rec_cap;
    __syncthreads();
    float* rec = p.rec_ring + (size_t)s_row * (3 + 3 * K);
    if (threadIdx.x == 0) {
      rec[0] = p.vid_index ? (float)p.vid_index[r] : (float)r;
      rec[1] = (float)k;
      rec[2] = s_cls;
    }
    for (int q = threadIdx.x; q < K; q += WM_THREADS) {
      const bool live = q < k;
      rec[3 + q] = live ? osc[q] : 0.f;
      rec[3 + K + 2 * q] = live ? os[2 * q] : 0.f;
      rec[3 + K + 2 * q + 1] = live ? os[2 * q + 1] : 0.f;
    }
  }
}

static size_t align256(size_t n) { return (n + 255) / 256 * 256; }

}  // namespace avdf

using namespace avdf;

extern "C" size_t avdf_window_merge_workspace_bytes(int32_t n_rec, int32_t cand_cap) {
  if (n_rec <= 0 || cand_cap <= 0) return 0;
  const size_t n = (size_t)n_rec * cand_cap;
  return align256(n * 2 * sizeof(float)) + align256(n * sizeof(float)) + align256((size_t)n_rec * sizeof(int)) +
         avdf_postprocess_workspace_bytes(n_rec, cand_cap);
}

extern "C" int avdf_window_merge(const avdf_window_merge_args* a, void* stream) {
  AVDF_CHECK_ARG(a != nullptr, "args is null");
  AVDF_CHECK_ARG(a->n_rec >= 0 && a->cand_cap > 0, "bad n_rec / cand_cap");
  AVDF_CHECK_ARG(a->max_seg_num > 0 && a->max_seg_num <= AVDF_MAX_SEGS, "max_seg_num out of range");
  AVDF_CHECK_ARG(a->use_soft_nms == 0 || a->use_soft_nms == 1, "use_soft_nms must be 0 (hard) or 1 (soft)");
  AVDF_CHECK_ARG(a->rec_win && a->win_start && a->win_segs && a->win_scores && a->win_count && a->win_cls, "null window input");
  AVDF_CHECK_ARG(a->out_segs && a->out_scores && a->out_count && a->out_cls, "null output");
  if (a->rec_ring) AVDF_CHECK_ARG(a->rec_counter && a->rec_cap > 0, "record ring needs a counter and a capacity");
  if (a->n_rec == 0) return AVDF_OK;
  const size_t need = avdf_window_merge_workspace_bytes(a->n_rec, a->cand_cap);
  AVDF_CHECK_ARG(a->workspace && a->workspace_bytes >= need, "workspace too small");
  const size_t n = (size_t)a->n_rec * a->cand_cap;
  unsigned char* ws = static_cast<unsigned char*>(a->workspace);
  WindowMergeParams p{};
  p.rec_win = a->rec_win; p.win_start = a->win_start;
  p.win_segs = a->win_segs; p.win_scores = a->win_scores; p.win_count = a->win_count; p.win_cls = a->win_cls;
  p.cand_segs = reinterpret_cast<float*>(ws); ws += align256(n * 2 * sizeof(float));
  p.cand_scores = reinterpret_cast<float*>(ws); ws += align256(n * sizeof(float));
  p.cand_count = reinterpret_cast<int*>(ws); ws += align256((size_t)a->n_rec * sizeof(int));
  p.cand_cap = a->cand_cap; p.K = a->max_seg_num; p.voting_thresh = a->voting_thresh;
  p.out_segs = a->out_segs; p.out_scores = a->out_scores; p.out_count = a->out_count; p.out_cls = a->out_cls;
  p.rec_ring = a->rec_ring; p.rec_counter = a->rec_counter; p.rec_cap = a->rec_cap; p.vid_index = a->vid_index;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  window_gather_kernel<<<a->n_rec, WM_THREADS, 0, st>>>(p);
  int rc = check_launch("window_gather_kernel");
  if (rc != AVDF_OK) return rc;
  avdf_postprocess_args pa{};
  pa.batch = a->n_rec;
  pa.cand_segs = p.cand_segs; pa.cand_scores = p.cand_scores; pa.cand_count = p.cand_count; pa.cand_cap = a->cand_cap;
  pa.iou_threshold = a->iou_threshold; pa.min_score = a->min_score; pa.sigma = a->sigma; pa.voting_thresh = 0.f;
  pa.max_seg_num = a->max_seg_num; pa.use_soft_nms = a->use_soft_nms; pa.soft_method = 2;
  pa.out_segs = a->out_segs; pa.out_scores = a->out_scores; pa.out_count = a->out_count;
  pa.workspace = ws; pa.workspace_bytes = avdf_postprocess_workspace_bytes(a->n_rec, a->cand_cap);
  rc = avdf_postprocess(&pa, stream);
  if (rc != AVDF_OK) return rc;
  window_finalize_kernel<<<a->n_rec, WM_THREADS, 0, st>>>(p);
  return check_launch("window_finalize_kernel");
}
