// ActivityNet-style detection evaluation (ActionFormer / UMMAFormer libs/utils/metrics.py `ANETdetection`):
// per-threshold TP/FP matching, average precision and Recall@kx of ONE class, on the GPU.
//
//   validate   one thread per video: CSR offsets well formed, <= EVAL_MAX_PRED predictions and <= EVAL_MAX_GT GT rows
//              per video; violations set bits of the caller's status word and every later kernel returns at once, so
//              nothing is written (the reference's pandas would be asked the same question row by row).
//   match      one warp per video (persistent). The predictions are walked in score-descending order (ties: smaller
//              input index first); a video whose rows are not already in that order (result records are) is queued for
//              match_sorted, which sorts it in shared memory first. Per prediction, lane j computes the tIoU with GT
//              rows j and j + 32 (fp64, -fmad=false: the same IEEE operations as numpy's segment_iou) and keeps their
//              running maximum for Recall@kx; lane t < n_thr then picks, among the GT rows not locked at threshold t,
//              the one with the largest tIoU (ties: larger GT index - numpy's argsort()[::-1]) and locks it when its
//              tIoU >= thr[t]. The TP bits of all thresholds form one uint16 per prediction (tp_mask, input position).
//              Recall hit counts are integers, summed per block and then with integer atomics: deterministic.
//   sort       stable LSD radix sort of all predictions by score (descending; payload: tp_mask), 8-bit digits. One
//              histogram pass over all eight digits first; a digit in which one bucket holds every key is skipped (the
//              plan kernel decides on the device, so the whole call stays asynchronous). Each remaining digit is
//              reduce-then-scan: tile histograms, a scan per bucket, a stable scatter (warp match_any ranks).
//   AP scan    per block TP counts per threshold, their scan, per block maximum precision over TP rows, a suffix maximum
//              over blocks, then sum_{i TP} max_{j >= i, j TP} prec_j per block and a fixed-order sum: AP = sum / npos.
//              The envelope max_{j>=i} prec_j of the reference's interpolated_prec_rec is attained at a TP row, so
//              only TP rows compute a precision. No floating-point atomics: bit-identical across runs.
//
// Proposal evaluation (ActivityNet eval_proposal.py `average_recall_vs_avg_nr_proposals`, avdf_eval_proposal) shares the
// per-video validation, the score key, the shared-memory sort and seg_tiou: one warp per GT video walks its first keep[v]
// proposals and turns each GT row's first rank at each threshold into one integer count (see eval_prop_match_kernel).
#include <algorithm>

#include "common.cuh"

namespace avdf {

constexpr int EVAL_MAX_THR = 16;
constexpr int EVAL_MAX_TOPK = 4;
constexpr int EVAL_MAX_PRED = 8192;     // predictions per video
constexpr int EVAL_MAX_GT = 64;         // GT rows per video (two per lane)

constexpr int MATCH_WARPS = 8;
constexpr int SORTV_THREADS = 256;      // match_sorted: bitonic sort of one video in shared memory
constexpr int RADIX_THREADS = 256;
constexpr int RADIX_ITEMS = 16;
constexpr int RADIX_TILE = RADIX_THREADS * RADIX_ITEMS;
constexpr int AP_THREADS = 256;
constexpr int AP_ITEMS = 16;
constexpr int AP_TILE = AP_THREADS * AP_ITEMS;
constexpr int SCAN_THREADS = 1024;

struct EvalParams {
  double thr[EVAL_MAX_THR];
  int32_t topk[EVAL_MAX_TOPK];
  int32_t n_thr, n_topk, n_video, n_gt;
  int64_t n_pred;
};

struct SortPlan {
  int32_t n_active;             // digit passes that move keys
  int32_t digit[8];             // their digit positions (0 = least significant byte)
  uint32_t base[8][256];        // exclusive bucket offsets of every digit position
};

// ---- score -> unsigned key whose ascending order is descending score (-0.0 and +0.0 are the same score) ----
__device__ __forceinline__ uint64_t score_key(double s) {
  uint64_t b = (uint64_t)__double_as_longlong(s == 0.0 ? 0.0 : s);
  b = (b >> 63) ? ~b : (b | 0x8000000000000000ull);     // ascending order-preserving
  return ~b;                                              // descending
}

// tIoU of prediction (ps, pe) against GT (gs, ge), numpy segment_iou's operation order (candidate = GT, target = pred)
__device__ __forceinline__ double seg_tiou(double ps, double pe, double gs, double ge) {
  double tt1 = fmax(ps, gs);
  double tt2 = fmin(pe, ge);
  double inter = fmax(__dsub_rn(tt2, tt1), 0.0);
  double uni = __dsub_rn(__dadd_rn(__dsub_rn(ge, gs), __dsub_rn(pe, ps)), inter);
  return __ddiv_rn(inter, uni);
}

// ---------------------------------------------------------------------------------------------
// keep (proposal evaluation, else nullptr): the walked prefix of every video, 0 <= keep[v] <= its row count
__global__ void eval_validate_kernel(const int64_t* __restrict__ pred_off, const int32_t* __restrict__ gt_off, int n_video,
                                     int64_t n_pred, int n_gt, int32_t* status, const int32_t* __restrict__ keep = nullptr) {
  int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v > n_video) return;
  int bad = 0;
  if (v == 0) bad |= (pred_off[0] != 0 || gt_off[0] != 0) ? AVDF_EVAL_BAD_OFFSETS : 0;
  if (v == n_video) bad |= (pred_off[n_video] != n_pred || gt_off[n_video] != n_gt) ? AVDF_EVAL_BAD_OFFSETS : 0;
  if (v < n_video) {
    int64_t np = pred_off[v + 1] - pred_off[v];
    int ng = gt_off[v + 1] - gt_off[v];
    if (np < 0 || ng < 0) bad |= AVDF_EVAL_BAD_OFFSETS;
    if (np > EVAL_MAX_PRED) bad |= AVDF_EVAL_PRED_LIMIT;
    if (ng > EVAL_MAX_GT) bad |= AVDF_EVAL_GT_LIMIT;
    if (keep && (keep[v] < 0 || keep[v] > np)) bad |= AVDF_EVAL_BAD_KEEP;
  }
  if (bad) atomicOr(status, bad);
}

// ---------------------------------------------------------------------------------------------
// The walk of one video by one warp. order == nullptr: the rows are already in walk order; else order[i] is the local
// row of rank i. acc[2]: lane l accumulates Recall hit counter l (acc[0]) and l + 32 (acc[1]), counter = t * n_topk + q.
__device__ __forceinline__ void walk_video(const EvalParams& P, const double2* __restrict__ seg, uint16_t* __restrict__ tp_mask, int64_t p0,
                           int n, const double2* __restrict__ gt, int g0, int n_gt, const uint16_t* order, double* tiou_sm,
                           uint32_t (&acc)[2]) {
  const int lane = threadIdx.x & 31;
  if (n_gt == 0) {                        // every prediction is a FP; Recall ignores the video
    for (int i = lane; i < n; i += 32) tp_mask[p0 + i] = 0;
    return;
  }
  double ga_s = 0, ga_e = 0, gb_s = 0, gb_e = 0;
  if (lane < n_gt) { double2 g = gt[g0 + lane]; ga_s = g.x; ga_e = g.y; }
  if (lane + 32 < n_gt) { double2 g = gt[g0 + lane + 32]; gb_s = g.x; gb_e = g.y; }
  double run_a = -1.0, run_b = -1.0;     // running maximum tIoU of GT rows lane, lane + 32 (numpy: any(tiou >= thr))
  const double my_thr = lane < P.n_thr ? P.thr[lane] : 2.0;
  uint64_t locked = 0;                    // lane t: GT rows locked at threshold t
  int pending = 0;                        // Recall snapshots not yet taken (bit q)
  for (int q = 0; q < P.n_topk; ++q) pending |= 1 << q;

  auto snapshot = [&](int q) {
    for (int t = 0; t < P.n_thr; ++t) {
      const double th = P.thr[t];
      int hits = __popc(__ballot_sync(0xffffffffu, lane < n_gt && run_a >= th)) +
                 __popc(__ballot_sync(0xffffffffu, lane + 32 < n_gt && run_b >= th));
      int c = t * P.n_topk + q;
      if (lane == (c & 31)) { if (c < 32) acc[0] += hits; else acc[1] += hits; }
    }
  };

  for (int base = 0; base < n; base += 32) {
    const int cnt = min(32, n - base);
    double ps = 0, pe = 0;
    int my_row = 0;
    if (lane < cnt) {
      my_row = order ? (int)order[base + lane] : base + lane;
      double2 s = seg[p0 + my_row]; ps = s.x; pe = s.y;
    }
    uint16_t my_mask = 0;
    for (int j = 0; j < cnt; ++j) {
      const double s = __shfl_sync(0xffffffffu, ps, j), e = __shfl_sync(0xffffffffu, pe, j);
      if (lane < n_gt) {
        double u = seg_tiou(s, e, ga_s, ga_e);
        run_a = fmax(run_a, u);
        tiou_sm[lane] = u;
      }
      if (lane + 32 < n_gt) {
        double u = seg_tiou(s, e, gb_s, gb_e);
        run_b = fmax(run_b, u);
        tiou_sm[lane + 32] = u;
      }
      __syncwarp();
      bool tp = false;
      if (lane < P.n_thr) {
        int best = -1; double bu = 0.0;
        for (int g = 0; g < n_gt; ++g) {
          double u = tiou_sm[g];
          if (!((locked >> g) & 1ull) && (best < 0 || u >= bu)) { best = g; bu = u; }
        }
        if (best >= 0 && bu >= my_thr) { tp = true; locked |= 1ull << best; }
      }
      const uint16_t m = (uint16_t)__ballot_sync(0xffffffffu, tp);
      if (lane == j) my_mask = m;
      __syncwarp();
      const int done = base + j + 1;       // predictions walked so far
      if (pending) {
        for (int q = 0; q < P.n_topk; ++q)
          if (((pending >> q) & 1) && P.topk[q] * n_gt == done) { snapshot(q); pending &= ~(1 << q); }
      }
    }
    if (lane < cnt) tp_mask[p0 + my_row] = my_mask;
  }
  for (int q = 0; q < P.n_topk; ++q)       // fewer than k * n_gt predictions: all of them count
    if ((pending >> q) & 1) snapshot(q);
}

__device__ void flush_hits(const EvalParams& P, uint32_t (&acc)[2], unsigned long long* hits_sm, unsigned long long* hits) {
  const int lane = threadIdx.x & 31, n_c = P.n_thr * P.n_topk;
  if (lane < n_c) atomicAdd(&hits_sm[lane], (unsigned long long)acc[0]);
  if (lane + 32 < n_c) atomicAdd(&hits_sm[lane + 32], (unsigned long long)acc[1]);
  __syncthreads();
  for (int c = threadIdx.x; c < n_c; c += blockDim.x)
    if (hits_sm[c]) atomicAdd(&hits[c], hits_sm[c]);
}

__global__ void __launch_bounds__(MATCH_WARPS * 32) eval_match_kernel(
    EvalParams P, const int64_t* __restrict__ pred_off, const double2* __restrict__ seg, const double* __restrict__ score,
    const int32_t* __restrict__ gt_off, const double2* __restrict__ gt, uint16_t* __restrict__ tp_mask,
    int32_t* __restrict__ unsorted, int32_t* __restrict__ n_unsorted, unsigned long long* __restrict__ hits,
    const int32_t* __restrict__ status) {
  __shared__ double tiou_sm[MATCH_WARPS][EVAL_MAX_GT];
  __shared__ unsigned long long hits_sm[EVAL_MAX_THR * EVAL_MAX_TOPK];
  if (*status) return;
  for (int c = threadIdx.x; c < EVAL_MAX_THR * EVAL_MAX_TOPK; c += blockDim.x) hits_sm[c] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  uint32_t acc[2] = {0, 0};
  for (int v = blockIdx.x * MATCH_WARPS + w; v < P.n_video; v += gridDim.x * MATCH_WARPS) {
    const int64_t p0 = pred_off[v];
    const int n = (int)(pred_off[v + 1] - p0);
    const int g0 = gt_off[v], n_gt = gt_off[v + 1] - g0;
    bool ok = true;
    if (n_gt > 0) {                       // walk order = input order iff the scores do not increase
      for (int i = lane; i + 1 < n && ok; i += 32) ok = score[p0 + i] >= score[p0 + i + 1];
      ok = __all_sync(0xffffffffu, ok);
    }
    if (!ok) {
      if (lane == 0) unsorted[atomicAdd(n_unsorted, 1)] = v;
      continue;
    }
    walk_video(P, seg, tp_mask, p0, n, gt, g0, n_gt, nullptr, tiou_sm[w], acc);
  }
  flush_hits(P, acc, hits_sm, hits);
}

// Block-wide: row[0 .. n) = the local rows of one video's n <= EVAL_MAX_PRED entries of `score`, score descending, equal
// scores by smaller row (bitonic sort of the unique (score key, row) pairs in shared memory, so the order is exactly the
// stable one). Starts and ends with a barrier.
__device__ void sort_video_rows(const double* __restrict__ score, int n, uint64_t* key, uint16_t* row) {
  int m = 1;
  while (m < n) m <<= 1;
  __syncthreads();
  for (int i = threadIdx.x; i < m; i += blockDim.x) {
    key[i] = i < n ? score_key(score[i]) : ~0ull;
    row[i] = (uint16_t)(i < n ? i : 0xffff);
  }
  for (int size = 2; size <= m; size <<= 1)
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      __syncthreads();
      for (int i = threadIdx.x; i < m; i += blockDim.x) {
        const int j = i ^ stride;
        if (j > i) {
          const bool up = (i & size) == 0;
          const uint64_t ki = key[i], kj = key[j];
          const uint16_t ri = row[i], rj = row[j];
          const bool gt_ = ki > kj || (ki == kj && ri > rj);
          if (gt_ == up) { key[i] = kj; key[j] = ki; row[i] = rj; row[j] = ri; }
        }
      }
    }
  __syncthreads();
}

// Videos whose predictions are out of order: one CTA sorts them (sort_video_rows), then its first warp walks them.
__global__ void __launch_bounds__(SORTV_THREADS) eval_match_sorted_kernel(
    EvalParams P, const int64_t* __restrict__ pred_off, const double2* __restrict__ seg, const double* __restrict__ score,
    const int32_t* __restrict__ gt_off, const double2* __restrict__ gt, uint16_t* __restrict__ tp_mask,
    const int32_t* __restrict__ unsorted, const int32_t* __restrict__ n_unsorted, unsigned long long* __restrict__ hits,
    const int32_t* __restrict__ status) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint64_t* key = reinterpret_cast<uint64_t*>(smem_raw);                        // [EVAL_MAX_PRED]
  uint16_t* row = reinterpret_cast<uint16_t*>(key + EVAL_MAX_PRED);             // [EVAL_MAX_PRED]
  __shared__ double tiou_sm[EVAL_MAX_GT];
  __shared__ unsigned long long hits_sm[EVAL_MAX_THR * EVAL_MAX_TOPK];
  if (*status) return;
  const int count = *n_unsorted;
  if ((int)blockIdx.x >= count) return;
  for (int c = threadIdx.x; c < EVAL_MAX_THR * EVAL_MAX_TOPK; c += blockDim.x) hits_sm[c] = 0;
  uint32_t acc[2] = {0, 0};
  for (int k = blockIdx.x; k < count; k += gridDim.x) {
    const int v = unsorted[k];
    const int64_t p0 = pred_off[v];
    const int n = (int)(pred_off[v + 1] - p0);
    sort_video_rows(score + p0, n, key, row);
    if (threadIdx.x < 32) {
      const int g0 = gt_off[v], n_gt = gt_off[v + 1] - g0;
      walk_video(P, seg, tp_mask, p0, n, gt, g0, n_gt, row, tiou_sm, acc);
    }
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    const int lane = threadIdx.x, n_c = P.n_thr * P.n_topk;
    if (lane < n_c) hits_sm[lane] += acc[0];
    if (lane + 32 < n_c) hits_sm[lane + 32] += acc[1];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < P.n_thr * P.n_topk; c += blockDim.x)
    if (hits_sm[c]) atomicAdd(&hits[c], hits_sm[c]);
}

// ---------------------------------------------------------------------------------------------
// radix sort
__global__ void __launch_bounds__(256) eval_key_hist_kernel(const double* __restrict__ score, int64_t n,
                                                            uint32_t* __restrict__ hist /*[8][256]*/, const int32_t* status) {
  __shared__ uint32_t h[8][256];
  if (*status) return;
  for (int i = threadIdx.x; i < 8 * 256; i += blockDim.x) (&h[0][0])[i] = 0;
  __syncthreads();
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const uint64_t k = score_key(score[i]);
#pragma unroll
    for (int d = 0; d < 8; ++d) atomicAdd(&h[d][(k >> (8 * d)) & 255], 1u);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 8 * 256; i += blockDim.x) {
    const uint32_t c = (&h[0][0])[i];
    if (c) atomicAdd(&hist[i], c);
  }
}

__global__ void eval_plan_kernel(const uint32_t* __restrict__ hist, int64_t n, SortPlan* plan, const int32_t* status) {
  __shared__ int trivial[8];
  if (*status) return;
  const int d = threadIdx.x >> 5, lane = threadIdx.x & 31;    // 8 warps: warp d scans digit position d
  uint32_t run = 0;
  bool triv = false;
  for (int b0 = 0; b0 < 256; b0 += 32) {
    const uint32_t c = hist[d * 256 + b0 + lane];
    triv |= (uint64_t)c == (uint64_t)n;
    uint32_t x = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    plan->base[d][b0 + lane] = run + x - c;
    run += __shfl_sync(0xffffffffu, x, 31);
  }
  triv = __any_sync(0xffffffffu, triv);
  if (lane == 0) trivial[d] = triv;
  __syncthreads();
  if (threadIdx.x == 0) {
    int a = 0;
    for (int k = 0; k < 8; ++k)
      if (!trivial[k]) plan->digit[a++] = k;
    plan->n_active = a;
  }
}

// tile histograms of the digit of pass `slot`: cnt[bucket * n_tiles + tile]
template <bool FROM_SCORE>
__global__ void __launch_bounds__(RADIX_THREADS) eval_radix_upsweep_kernel(const double* __restrict__ score,
    const uint64_t* __restrict__ keys, int64_t n, int slot, const SortPlan* __restrict__ plan, uint32_t* __restrict__ cnt,
    int n_tiles, const int32_t* status) {
  __shared__ uint32_t h[256];
  if (*status || slot >= plan->n_active) return;
  const int shift = 8 * plan->digit[slot];
  h[threadIdx.x] = 0;
  __syncthreads();
  const int64_t t0 = (int64_t)blockIdx.x * RADIX_TILE;
#pragma unroll 4
  for (int r = 0; r < RADIX_ITEMS; ++r) {
    const int64_t i = t0 + r * RADIX_THREADS + threadIdx.x;
    if (i < n) {
      const uint64_t k = FROM_SCORE ? score_key(score[i]) : keys[i];
      atomicAdd(&h[(k >> shift) & 255], 1u);
    }
  }
  __syncthreads();
  cnt[(size_t)threadIdx.x * n_tiles + blockIdx.x] = h[threadIdx.x];
}

// exclusive scan of one bucket's tile counts (block b = bucket b), plus the bucket's base offset
__global__ void __launch_bounds__(SCAN_THREADS) eval_radix_scan_kernel(uint32_t* __restrict__ cnt, int n_tiles, int slot,
                                                                       const SortPlan* __restrict__ plan, const int32_t* status) {
  __shared__ uint32_t wsum[SCAN_THREADS / 32];
  __shared__ uint32_t carry;
  if (*status || slot >= plan->n_active) return;
  uint32_t* row = cnt + (size_t)blockIdx.x * n_tiles;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (threadIdx.x == 0) carry = plan->base[plan->digit[slot]][blockIdx.x];
  for (int b0 = 0; b0 < n_tiles; b0 += SCAN_THREADS) {
    const int i = b0 + threadIdx.x;
    const uint32_t c = i < n_tiles ? row[i] : 0;
    uint32_t x = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    if (lane == 31) wsum[w] = x;
    __syncthreads();
    if (w == 0) {
      uint32_t s = wsum[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, s, o); if (lane >= o) s += y; }
      wsum[lane] = s;
    }
    __syncthreads();
    const uint32_t before = carry + (w ? wsum[w - 1] : 0u);
    if (i < n_tiles) row[i] = before + x - c;
    __syncthreads();
    if (threadIdx.x == 0) carry += wsum[SCAN_THREADS / 32 - 1];
    __syncthreads();
  }
}

// stable scatter of one tile: 16 rounds of 256 consecutive keys; within a round, warp w's keys of a bucket follow those
// of warps < w, ranks inside a warp come from match_any
template <bool FROM_SCORE>
__global__ void __launch_bounds__(RADIX_THREADS) eval_radix_scatter_kernel(const double* __restrict__ score,
    const uint64_t* __restrict__ keys_in, const uint16_t* __restrict__ pay_in, uint64_t* __restrict__ keys_out,
    uint16_t* __restrict__ pay_out, int64_t n, int slot, const SortPlan* __restrict__ plan, const uint32_t* __restrict__ cnt,
    int n_tiles, const int32_t* status) {
  constexpr int W = RADIX_THREADS / 32;
  __shared__ uint32_t wcnt[W][256], wpre[W][256], run[256];
  if (*status || slot >= plan->n_active) return;
  const int shift = 8 * plan->digit[slot];
  const bool write_keys = slot + 1 < plan->n_active;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  run[threadIdx.x] = cnt[(size_t)threadIdx.x * n_tiles + blockIdx.x];
  for (int k = 0; k < W; ++k) wcnt[k][threadIdx.x] = 0;
  __syncthreads();
  const int64_t t0 = (int64_t)blockIdx.x * RADIX_TILE;
  const uint32_t lt = (1u << lane) - 1u;
  for (int r = 0; r < RADIX_ITEMS; ++r) {
    const int64_t i = t0 + r * RADIX_THREADS + threadIdx.x;
    const bool valid = i < n;
    uint64_t k = 0; uint16_t p = 0;
    if (valid) { k = FROM_SCORE ? score_key(score[i]) : keys_in[i]; p = pay_in[i]; }
    const int d = valid ? (int)((k >> shift) & 255) : 256 + lane;
    const uint32_t peers = __match_any_sync(0xffffffffu, d);
    const int rank = __popc(peers & lt);
    if (valid && rank == 0) wcnt[w][d] = __popc(peers);
    __syncthreads();
    {
      const int b = threadIdx.x;
      uint32_t s = run[b];
#pragma unroll
      for (int q = 0; q < W; ++q) { const uint32_t c = wcnt[q][b]; wpre[q][b] = s; s += c; wcnt[q][b] = 0; }
      run[b] = s;
    }
    __syncthreads();
    if (valid) {
      const uint32_t pos = wpre[w][d] + rank;
      if (write_keys) keys_out[pos] = k;
      pay_out[pos] = p;
    }
  }
}

// pred_rank given: scores and tp masks are first scattered into rank order, so that the stable sort breaks ties by rank
__global__ void eval_permute_kernel(const int32_t* __restrict__ rank, const double* __restrict__ score,
                                    const uint16_t* __restrict__ tp, double* __restrict__ score_r, uint16_t* __restrict__ tp_r,
                                    int64_t n, const int32_t* status) {
  if (*status) return;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int32_t r = rank[i];
    score_r[r] = score[i];
    tp_r[r] = tp[i];
  }
}

// ---------------------------------------------------------------------------------------------
// AP scan over the sorted tp masks
__device__ __forceinline__ const uint16_t* sorted_tp(const SortPlan* plan, const uint16_t* p_in, const uint16_t* p0,
                                                     const uint16_t* p1) {
  const int a = plan->n_active;
  return a == 0 ? p_in : ((a - 1) & 1 ? p1 : p0);
}

// the AP_ITEMS masks of this thread (consecutive rows), zero beyond n
__device__ __forceinline__ void load_masks(const uint16_t* tp, int64_t n, int64_t i0, uint16_t (&m)[AP_ITEMS]) {
  if (i0 + AP_ITEMS <= n) {
    const uint4* q = reinterpret_cast<const uint4*>(tp + i0);
    uint4 a = q[0], b = q[1];
    const uint32_t u[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
    for (int k = 0; k < 8; ++k) { m[2 * k] = (uint16_t)(u[k] & 0xffff); m[2 * k + 1] = (uint16_t)(u[k] >> 16); }
  } else {
#pragma unroll
    for (int k = 0; k < AP_ITEMS; ++k) m[k] = i0 + k < n ? tp[i0 + k] : 0;
  }
}

__global__ void __launch_bounds__(AP_THREADS) eval_ap_count_kernel(const SortPlan* plan, const uint16_t* p_in,
    const uint16_t* p0, const uint16_t* p1, int64_t n, int n_thr, int32_t* __restrict__ blk_cnt, const int32_t* status) {
  __shared__ int32_t ws[AP_THREADS / 32][EVAL_MAX_THR];
  if (*status) return;
  const uint16_t* tp = sorted_tp(plan, p_in, p0, p1);
  uint16_t m[AP_ITEMS];
  load_masks(tp, n, (int64_t)blockIdx.x * AP_TILE + threadIdx.x * AP_ITEMS, m);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int t = 0; t < n_thr; ++t) {
    int c = 0;
#pragma unroll
    for (int k = 0; k < AP_ITEMS; ++k) c += (m[k] >> t) & 1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if (lane == 0) ws[w][t] = c;
  }
  __syncthreads();
  if (threadIdx.x < n_thr) {
    int c = 0;
    for (int q = 0; q < AP_THREADS / 32; ++q) c += ws[q][threadIdx.x];
    blk_cnt[(size_t)blockIdx.x * EVAL_MAX_THR + threadIdx.x] = c;
  }
}

// one CTA: exclusive scan of the block TP counts (blk_cnt -> blk_off, in place) per threshold
__global__ void __launch_bounds__(SCAN_THREADS) eval_ap_offsets_kernel(int32_t* __restrict__ blk, int n_blk, int n_thr,
                                                                       const int32_t* status) {
  __shared__ int32_t wsum[SCAN_THREADS / 32];
  __shared__ int32_t carry;
  if (*status) return;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int t = 0; t < n_thr; ++t) {
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int b0 = 0; b0 < n_blk; b0 += SCAN_THREADS) {
      const int i = b0 + threadIdx.x;
      const int32_t c = i < n_blk ? blk[(size_t)i * EVAL_MAX_THR + t] : 0;
      int32_t x = c;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { int32_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
      if (lane == 31) wsum[w] = x;
      __syncthreads();
      if (w == 0) {
        int32_t s = wsum[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int32_t y = __shfl_up_sync(0xffffffffu, s, o); if (lane >= o) s += y; }
        wsum[lane] = s;
      }
      __syncthreads();
      if (i < n_blk) blk[(size_t)i * EVAL_MAX_THR + t] = carry + (w ? wsum[w - 1] : 0) + x - c;
      __syncthreads();
      if (threadIdx.x == 0) carry += wsum[SCAN_THREADS / 32 - 1];
      __syncthreads();
    }
  }
}

// exclusive prefix of this thread's TP count at threshold t inside the block (collective: every thread calls it)
__device__ __forceinline__ int thread_prefix(int c, int32_t* ws /*[AP_THREADS / 32]*/) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int x = c;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
  if (lane == 31) ws[w] = x;
  __syncthreads();
  int before = 0;
  for (int q = 0; q < w; ++q) before += ws[q];
  __syncthreads();
  return before + x - c;
}

// pass 1: maximum precision over the TP rows of every block. pass 2: sum over TP rows of max(prec over later TP rows)
template <bool SUM>
__global__ void __launch_bounds__(AP_THREADS) eval_ap_block_kernel(const SortPlan* plan, const uint16_t* p_in,
    const uint16_t* p0, const uint16_t* p1, int64_t n, int n_thr, const int32_t* __restrict__ blk_off,
    const double* __restrict__ carry_in /*[n_blk][16] max over later blocks*/, double* __restrict__ out /*[n_blk][16]*/,
    const int32_t* status) {
  constexpr int W = AP_THREADS / 32;
  __shared__ int32_t wsi[W];
  __shared__ double wsd[W];
  if (*status) return;
  const uint16_t* tp = sorted_tp(plan, p_in, p0, p1);
  uint16_t m[AP_ITEMS];
  const int64_t i0 = (int64_t)blockIdx.x * AP_TILE + threadIdx.x * AP_ITEMS;
  load_masks(tp, n, i0, m);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int t = 0; t < n_thr; ++t) {
    int c = 0;
#pragma unroll
    for (int k = 0; k < AP_ITEMS; ++k) c += (m[k] >> t) & 1;
    const int start = blk_off[(size_t)blockIdx.x * EVAL_MAX_THR + t] + thread_prefix(c, wsi);
    // forward: precision at this thread's TP rows, their maximum
    double mx = 0.0;
    int cc = start;
#pragma unroll
    for (int k = 0; k < AP_ITEMS; ++k)
      if ((m[k] >> t) & 1) { ++cc; mx = fmax(mx, __ddiv_rn((double)cc, (double)(i0 + k + 1))); }
    if (!SUM) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      if (lane == 0) wsd[w] = mx;
      __syncthreads();
      if (threadIdx.x == 0) {
        double b = 0.0;
        for (int q = 0; q < W; ++q) b = fmax(b, wsd[q]);
        out[(size_t)blockIdx.x * EVAL_MAX_THR + t] = b;
      }
      __syncthreads();
      continue;
    }
    // maximum over the rows of later threads of the block and of later blocks
    double later = mx;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { double y = __shfl_down_sync(0xffffffffu, later, o); if (lane + o < 32) later = fmax(later, y); }
    if (lane == 0) wsd[w] = later;                   // warp maximum
    __syncthreads();
    double run = carry_in[(size_t)blockIdx.x * EVAL_MAX_THR + t];
    for (int q = w + 1; q < W; ++q) run = fmax(run, wsd[q]);
    const double nxt = __shfl_down_sync(0xffffffffu, later, 1);
    if (lane < 31) run = fmax(run, nxt);
    __syncthreads();
    // backward over this thread's rows
    double sum = 0.0;
    cc = start + c;
#pragma unroll
    for (int k = AP_ITEMS - 1; k >= 0; --k)
      if ((m[k] >> t) & 1) { run = fmax(run, __ddiv_rn((double)cc, (double)(i0 + k + 1))); sum += run; --cc; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lane == 0) wsd[w] = sum;
    __syncthreads();
    if (threadIdx.x == 0) {
      double b = 0.0;
      for (int q = 0; q < W; ++q) b += wsd[q];
      out[(size_t)blockIdx.x * EVAL_MAX_THR + t] = b;
    }
    __syncthreads();
  }
}

// one CTA, one warp per threshold: carry[b] = max of blk_max over blocks > b
__global__ void eval_ap_carry_kernel(const double* __restrict__ blk_max, double* __restrict__ carry, int n_blk, int n_thr,
                                     const int32_t* status) {
  if (*status) return;
  const int lane = threadIdx.x & 31, t = threadIdx.x >> 5;
  if (t >= n_thr) return;
  double run = 0.0;
  for (int b1 = n_blk; b1 > 0; b1 -= 32) {              // chunks of 32 blocks from the end
    const int b = b1 - 32 + lane;
    const double v = b >= 0 ? blk_max[(size_t)b * EVAL_MAX_THR + t] : 0.0;
    double s = v;                                        // inclusive suffix maximum inside the chunk
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { double y = __shfl_down_sync(0xffffffffu, s, o); if (lane + o < 32) s = fmax(s, y); }
    double excl = __shfl_down_sync(0xffffffffu, s, 1);
    if (lane == 31) excl = 0.0;
    if (b >= 0) carry[(size_t)b * EVAL_MAX_THR + t] = fmax(run, excl);
    run = fmax(run, __shfl_sync(0xffffffffu, s, 0));
  }
}

// one CTA: fixed-order sums of the block sums -> ap[t]; hit counts -> recall_hits. Nothing is written on a bad status.
__global__ void eval_finish_kernel(const double* __restrict__ blk_sum, int n_blk, int n_thr, int n_topk, int npos,
                                   const unsigned long long* __restrict__ hits, double* __restrict__ ap,
                                   int64_t* __restrict__ recall_hits, const int32_t* status) {
  if (*status) return;
  const int lane = threadIdx.x & 31, t = threadIdx.x >> 5;
  if (t < n_thr) {
    double s = 0.0;
    for (int b = lane; b < n_blk; b += 32) s += blk_sum[(size_t)b * EVAL_MAX_THR + t];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) ap[t] = s / (double)npos;
  }
  if (threadIdx.x < n_thr * n_topk) recall_hits[threadIdx.x] = (int64_t)hits[threadIdx.x];
}

// ---------------------------------------------------------------------------------------------
// Proposal evaluation (ActivityNet eval_proposal.py, average_recall_vs_avg_nr_proposals), class-agnostic: per tIoU
// threshold t and point j, the number of GT rows matched by their video's first cut_j(c) proposals in walk order, where
// c = keep[v] (the video's walked prefix) or 1 for a video without proposals (upstream's zeros((n_gt, 1)) column) and
// cut_j(c) = min(int(c * an_frac[j]), c). cut_j does not decrease in j, so a GT row whose first rank reaching t is r is
// matched at exactly the points j >= j0, j0 = the first point with cut_j > r: one integer count into hist[t][j0], and a
// prefix over j gives the matches. The walk stops once every (row, threshold) has its first rank, or at cut_99.
constexpr int PROP_POINTS = 100;

struct PropParams {
  double thr[EVAL_MAX_THR];
  double frac[PROP_POINTS];      // the host's pcn: one fp64 product c * frac[j] per cut, never recomputed here
  int32_t n_thr, n_video;
};

// cut[j] = min(int(c * frac[j]), c) (one fp64 product truncated toward zero, numpy's astype(int)); returns cut[99], the
// most ranks any point looks at. Warp-collective; the first barrier lets the warp's previous walk finish reading cut.
__device__ __forceinline__ int prop_cuts(const PropParams& P, int c, int32_t* cut) {
  __syncwarp();
  for (int j = threadIdx.x & 31; j < PROP_POINTS; j += 32)
    cut[j] = (int)min(__double2ll_rz(__dmul_rn((double)c, P.frac[j])), (long long)c);
  __syncwarp();
  return cut[PROP_POINTS - 1];
}

// The walk of one video by one warp over its first lim proposals (order == nullptr: input order, else order[r] is the
// local row of rank r; virt: no proposals, the one column is a tIoU of 0). Lane l owns GT rows l and l + 32 and, per row,
// the bit set of thresholds not reached yet. A rank whose tIoU does not exceed the row's running maximum reaches nothing
// new, so the thresholds are only tried when the maximum grows.
__device__ __forceinline__ void walk_proposals(const PropParams& P, const double2* __restrict__ seg, int64_t p0, int lim,
                                               bool virt, const double2* __restrict__ gt, int g0, int n_gt,
                                               const uint16_t* order, const int32_t* cut, uint32_t* hist_sm) {
  const int lane = threadIdx.x & 31;
  const uint32_t all = (1u << P.n_thr) - 1u;
  double ga_s = 0, ga_e = 0, gb_s = 0, gb_e = 0;
  uint32_t pend_a = 0, pend_b = 0;
  if (lane < n_gt) { double2 g = gt[g0 + lane]; ga_s = g.x; ga_e = g.y; pend_a = all; }
  if (lane + 32 < n_gt) { double2 g = gt[g0 + lane + 32]; gb_s = g.x; gb_e = g.y; pend_b = all; }
  const double nan = __longlong_as_double(0x7ff8000000000000ll);
  double run_a = nan, run_b = nan;         // NaN: the first rank is always tried; a NaN tIoU reaches nothing
  auto reach = [&](uint32_t& pend, double& run, double u, int r) {
    if (u <= run) return;
    run = fmax(run, u);
    for (uint32_t m = pend; m; m &= m - 1) {
      const int t = __ffs(m) - 1;
      if (u >= P.thr[t]) {
        pend &= ~(1u << t);
        int lo = 0, hi = PROP_POINTS - 1;      // first j with cut[j] > r; cut[99] = lim > r
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (cut[mid] > r) hi = mid; else lo = mid + 1; }
        atomicAdd(&hist_sm[t * PROP_POINTS + lo], 1u);
      }
    }
  };
  for (int base = 0; base < lim; base += 32) {
    if (!__any_sync(0xffffffffu, pend_a | pend_b)) break;
    const int cnt = min(32, lim - base);
    double ps = 0, pe = 0;
    if (lane < cnt && !virt) {
      const double2 s = seg[p0 + (order ? (int)order[base + lane] : base + lane)];
      ps = s.x; pe = s.y;
    }
    for (int j = 0; j < cnt; ++j) {
      const double s = __shfl_sync(0xffffffffu, ps, j), e = __shfl_sync(0xffffffffu, pe, j);
      if (pend_a) reach(pend_a, run_a, virt ? 0.0 : seg_tiou(s, e, ga_s, ga_e), base + j);
      if (pend_b) reach(pend_b, run_b, virt ? 0.0 : seg_tiou(s, e, gb_s, gb_e), base + j);
    }
  }
}

__device__ __forceinline__ void prop_flush(const PropParams& P, const uint32_t* hist_sm, unsigned long long* hist) {
  __syncthreads();
  for (int i = threadIdx.x; i < P.n_thr * PROP_POINTS; i += blockDim.x)
    if (hist_sm[i]) atomicAdd(&hist[i], (unsigned long long)hist_sm[i]);
}

__global__ void __launch_bounds__(MATCH_WARPS * 32) eval_prop_match_kernel(
    PropParams P, const int64_t* __restrict__ prop_off, const double2* __restrict__ seg, const double* __restrict__ score,
    const int32_t* __restrict__ keep, const int32_t* __restrict__ gt_off, const double2* __restrict__ gt,
    int32_t* __restrict__ unsorted, int32_t* __restrict__ n_unsorted, unsigned long long* __restrict__ hist,
    const int32_t* __restrict__ status) {
  __shared__ int32_t cut_sm[MATCH_WARPS][PROP_POINTS];
  __shared__ uint32_t hist_sm[EVAL_MAX_THR * PROP_POINTS];
  if (*status) return;
  for (int i = threadIdx.x; i < EVAL_MAX_THR * PROP_POINTS; i += blockDim.x) hist_sm[i] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int v = blockIdx.x * MATCH_WARPS + w; v < P.n_video; v += gridDim.x * MATCH_WARPS) {
    const int64_t p0 = prop_off[v];
    const int n = (int)(prop_off[v + 1] - p0);
    const int g0 = gt_off[v], n_gt = gt_off[v + 1] - g0;
    if (n_gt == 0) continue;
    const int lim = prop_cuts(P, n ? keep[v] : 1, cut_sm[w]);
    if (lim == 0) continue;
    bool ok = true;                       // walk order = input order iff the scores do not increase
    for (int i = lane; i + 1 < n && ok; i += 32) ok = score[p0 + i] >= score[p0 + i + 1];
    if (!__all_sync(0xffffffffu, ok)) {
      if (lane == 0) unsorted[atomicAdd(n_unsorted, 1)] = v;
      continue;
    }
    walk_proposals(P, seg, p0, lim, n == 0, gt, g0, n_gt, nullptr, cut_sm[w], hist_sm);
  }
  prop_flush(P, hist_sm, hist);
}

// the videos eval_prop_match_kernel queued: one CTA sorts one video's rows (sort_video_rows), its first warp walks them
__global__ void __launch_bounds__(SORTV_THREADS) eval_prop_match_sorted_kernel(
    PropParams P, const int64_t* __restrict__ prop_off, const double2* __restrict__ seg, const double* __restrict__ score,
    const int32_t* __restrict__ keep, const int32_t* __restrict__ gt_off, const double2* __restrict__ gt,
    const int32_t* __restrict__ unsorted, const int32_t* __restrict__ n_unsorted, unsigned long long* __restrict__ hist,
    const int32_t* __restrict__ status) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint64_t* key = reinterpret_cast<uint64_t*>(smem_raw);                        // [EVAL_MAX_PRED]
  uint16_t* row = reinterpret_cast<uint16_t*>(key + EVAL_MAX_PRED);             // [EVAL_MAX_PRED]
  __shared__ int32_t cut_sm[PROP_POINTS];
  __shared__ uint32_t hist_sm[EVAL_MAX_THR * PROP_POINTS];
  if (*status) return;
  const int count = *n_unsorted;
  if ((int)blockIdx.x >= count) return;
  for (int i = threadIdx.x; i < EVAL_MAX_THR * PROP_POINTS; i += blockDim.x) hist_sm[i] = 0;
  for (int k = blockIdx.x; k < count; k += gridDim.x) {
    const int v = unsorted[k];
    const int64_t p0 = prop_off[v];
    sort_video_rows(score + p0, (int)(prop_off[v + 1] - p0), key, row);
    if (threadIdx.x < 32) {
      const int g0 = gt_off[v], n_gt = gt_off[v + 1] - g0;
      const int lim = prop_cuts(P, keep[v], cut_sm);
      walk_proposals(P, seg, p0, lim, false, gt, g0, n_gt, row, cut_sm, hist_sm);
    }
  }
  prop_flush(P, hist_sm, hist);
}

// matches[t][j] = sum over j' <= j of hist[t][j']. Nothing is written on a bad status.
__global__ void eval_prop_finish_kernel(const unsigned long long* __restrict__ hist, int n_thr, int64_t* __restrict__ matches,
                                        const int32_t* status) {
  if (*status) return;
  const int t = threadIdx.x;
  if (t >= n_thr) return;
  unsigned long long run = 0;
  for (int j = 0; j < PROP_POINTS; ++j) {
    run += hist[t * PROP_POINTS + j];
    matches[t * PROP_POINTS + j] = (int64_t)run;
  }
}

struct PropWs {
  int32_t* unsorted; int32_t* n_unsorted; unsigned long long* hist;
  size_t bytes;
};

static PropWs prop_layout(char* base, int32_t n_video) {
  PropWs w;
  size_t off = 0;
  auto take = [&](size_t bytes) { char* p = base ? base + off : nullptr; off += (bytes + 255) & ~size_t(255); return p; };
  w.unsorted = (int32_t*)take(4 * (size_t)(n_video > 0 ? n_video : 1)); w.n_unsorted = (int32_t*)take(4);
  w.hist = (unsigned long long*)take(8 * EVAL_MAX_THR * PROP_POINTS);
  w.bytes = off;
  return w;
}

// ---------------------------------------------------------------------------------------------
struct EvalWs {
  uint64_t* keys[2]; uint16_t* pay[2]; uint16_t* tp;
  uint32_t* hist; SortPlan* plan; uint32_t* tile_cnt; int32_t* unsorted; int32_t* n_unsorted;
  unsigned long long* hits; int32_t* blk_cnt; double* blk_max; double* carry; double* blk_sum;
  size_t bytes;
};

static EvalWs eval_layout(char* base, int64_t n_pred, int32_t n_video) {
  EvalWs w;
  size_t off = 0;
  auto take = [&](size_t bytes) { char* p = base ? base + off : nullptr; off += (bytes + 255) & ~size_t(255); return p; };
  const int64_t n = n_pred > 0 ? n_pred : 1;
  const int64_t n_tiles = (n + RADIX_TILE - 1) / RADIX_TILE, n_blk = (n + AP_TILE - 1) / AP_TILE;
  w.keys[0] = (uint64_t*)take(8 * n); w.keys[1] = (uint64_t*)take(8 * n);
  w.pay[0] = (uint16_t*)take(2 * n); w.pay[1] = (uint16_t*)take(2 * n); w.tp = (uint16_t*)take(2 * n);
  w.hist = (uint32_t*)take(8 * 256 * 4); w.plan = (SortPlan*)take(sizeof(SortPlan));
  w.tile_cnt = (uint32_t*)take(256 * 4 * n_tiles);
  w.unsorted = (int32_t*)take(4 * (size_t)(n_video > 0 ? n_video : 1)); w.n_unsorted = (int32_t*)take(4);
  w.hits = (unsigned long long*)take(8 * EVAL_MAX_THR * EVAL_MAX_TOPK);
  w.blk_cnt = (int32_t*)take(4 * EVAL_MAX_THR * n_blk);
  w.blk_max = (double*)take(8 * EVAL_MAX_THR * n_blk); w.carry = (double*)take(8 * EVAL_MAX_THR * n_blk);
  w.blk_sum = (double*)take(8 * EVAL_MAX_THR * n_blk);
  w.bytes = off;
  return w;
}

}  // namespace avdf

using namespace avdf;

extern "C" AVDF_API size_t avdf_eval_workspace_bytes(int64_t n_pred, int32_t n_video) {
  if (n_pred < 0 || n_video < 0) return 0;
  return eval_layout(nullptr, n_pred, n_video).bytes;
}

extern "C" AVDF_API int avdf_eval_detection(const avdf_eval_args* a, void* stream) {
  AVDF_CHECK_ARG(a != nullptr, "args is NULL");
  AVDF_CHECK_ARG(a->n_thr >= 1 && a->n_thr <= EVAL_MAX_THR, "n_thr must be 1..16");
  AVDF_CHECK_ARG(a->n_topk >= 0 && a->n_topk <= EVAL_MAX_TOPK, "n_topk must be 0..4");
  AVDF_CHECK_ARG(a->thresholds != nullptr && (a->n_topk == 0 || a->top_k != nullptr), "thresholds / top_k are NULL");
  for (int t = 0; t < a->n_thr; ++t) AVDF_CHECK_ARG(a->thresholds[t] == a->thresholds[t], "threshold is NaN");
  for (int q = 0; q < a->n_topk; ++q) AVDF_CHECK_ARG(a->top_k[q] >= 1 && a->top_k[q] <= EVAL_MAX_PRED, "top_k must be 1..8192");
  AVDF_CHECK_ARG(a->n_pred >= 0 && a->n_pred < (int64_t)1 << 31, "n_pred must be 0 .. 2^31 - 1");
  AVDF_CHECK_ARG(a->n_video >= 0 && a->n_gt >= 1, "n_video >= 0 and n_gt >= 1 (a class without GT has no AP)");
  AVDF_CHECK_ARG(a->pred_off && a->gt_off && a->gt_seg, "CSR offsets / GT segments are NULL");
  AVDF_CHECK_ARG(a->n_pred == 0 || (a->pred_seg && a->pred_score), "prediction arrays are NULL");
  AVDF_CHECK_ARG(a->pred_rank == nullptr || ((uintptr_t)a->pred_rank & 3) == 0, "pred_rank must be 4-byte aligned");
  AVDF_CHECK_ARG(a->ap && a->status && (a->n_topk == 0 || a->recall_hits), "outputs are NULL");
  AVDF_CHECK_ARG(((uintptr_t)a->pred_seg & 15) == 0 && ((uintptr_t)a->gt_seg & 15) == 0 && ((uintptr_t)a->tp_mask & 15) == 0,
                 "segments and tp_mask must be 16-byte aligned");
  const EvalWs need = eval_layout(nullptr, a->n_pred, a->n_video);
  AVDF_CHECK_ARG(a->workspace && a->workspace_bytes >= need.bytes && ((uintptr_t)a->workspace & 255) == 0,
                 "workspace too small or not 256-byte aligned (avdf_eval_workspace_bytes)");

  cudaStream_t st = (cudaStream_t)stream;
  EvalWs w = eval_layout((char*)a->workspace, a->n_pred, a->n_video);
  EvalParams P = {};
  for (int t = 0; t < a->n_thr; ++t) P.thr[t] = a->thresholds[t];
  for (int q = 0; q < a->n_topk; ++q) P.topk[q] = a->top_k[q];
  P.n_thr = a->n_thr; P.n_topk = a->n_topk; P.n_video = a->n_video; P.n_gt = a->n_gt; P.n_pred = a->n_pred;
  const int64_t n = a->n_pred;
  const int n_tiles = (int)((n + RADIX_TILE - 1) / RADIX_TILE), n_blk = (int)((n + AP_TILE - 1) / AP_TILE);
  uint16_t* tp = a->tp_mask ? a->tp_mask : w.tp;
  const double2* seg = reinterpret_cast<const double2*>(a->pred_seg);
  const double2* gt = reinterpret_cast<const double2*>(a->gt_seg);
  const int sms = device_sm_count();

  AVDF_CUDA(cudaMemsetAsync(a->status, 0, sizeof(int32_t), st));
  AVDF_CUDA(cudaMemsetAsync(w.hist, 0, 8 * 256 * 4, st));
  AVDF_CUDA(cudaMemsetAsync(w.n_unsorted, 0, 4, st));
  AVDF_CUDA(cudaMemsetAsync(w.hits, 0, 8 * EVAL_MAX_THR * EVAL_MAX_TOPK, st));
  eval_validate_kernel<<<(a->n_video + 1 + 255) / 256, 256, 0, st>>>(a->pred_off, a->gt_off, a->n_video, n, a->n_gt, a->status);
  if (a->n_video > 0) {
    const int grid = (int)std::min<int64_t>((a->n_video + MATCH_WARPS - 1) / MATCH_WARPS, (int64_t)sms * 8);
    eval_match_kernel<<<grid, MATCH_WARPS * 32, 0, st>>>(P, a->pred_off, seg, a->pred_score, a->gt_off, gt, tp, w.unsorted,
                                                        w.n_unsorted, w.hits, a->status);
    const size_t smem = (size_t)EVAL_MAX_PRED * (8 + 2);
    AVDF_SMEM_ATTR_ONCE(eval_match_sorted_kernel, smem);
    eval_match_sorted_kernel<<<std::min(a->n_video, 2 * sms), SORTV_THREADS, smem, st>>>(
        P, a->pred_off, seg, a->pred_score, a->gt_off, gt, tp, w.unsorted, w.n_unsorted, w.hits, a->status);
  }
  if (n > 0) {
    eval_key_hist_kernel<<<(int)std::min<int64_t>((n + 255) / 256, (int64_t)sms * 4), 256, 0, st>>>(a->pred_score, n, w.hist, a->status);
    // sort input: (scores, tp) in position order, or scattered into pred_rank order (keys[0] / pay[1] are free until
    // slot 0 has read them: slot 0 writes keys[1] and pay[0])
    const double* sc_in = a->pred_score;
    const uint16_t* tp_in = tp;
    if (a->pred_rank) {
      double* sc_r = reinterpret_cast<double*>(w.keys[0]);
      eval_permute_kernel<<<(int)std::min<int64_t>((n + 255) / 256, (int64_t)sms * 8), 256, 0, st>>>(a->pred_rank, a->pred_score, tp,
                                                                                                    sc_r, w.pay[1], n, a->status);
      sc_in = sc_r; tp_in = w.pay[1];
    }
    eval_plan_kernel<<<1, 256, 0, st>>>(w.hist, n, w.plan, a->status);
    for (int slot = 0; slot < 8; ++slot) {     // passes beyond plan->n_active return at once
      const uint64_t* kin = w.keys[slot & 1];
      uint64_t* kout = w.keys[(slot + 1) & 1];
      const uint16_t* pin = slot == 0 ? tp_in : w.pay[(slot - 1) & 1];
      uint16_t* pout = w.pay[slot & 1];
      if (slot == 0)
        eval_radix_upsweep_kernel<true><<<n_tiles, RADIX_THREADS, 0, st>>>(sc_in, kin, n, slot, w.plan, w.tile_cnt, n_tiles, a->status);
      else
        eval_radix_upsweep_kernel<false><<<n_tiles, RADIX_THREADS, 0, st>>>(sc_in, kin, n, slot, w.plan, w.tile_cnt, n_tiles, a->status);
      eval_radix_scan_kernel<<<256, SCAN_THREADS, 0, st>>>(w.tile_cnt, n_tiles, slot, w.plan, a->status);
      if (slot == 0)
        eval_radix_scatter_kernel<true><<<n_tiles, RADIX_THREADS, 0, st>>>(sc_in, kin, pin, kout, pout, n, slot, w.plan, w.tile_cnt, n_tiles, a->status);
      else
        eval_radix_scatter_kernel<false><<<n_tiles, RADIX_THREADS, 0, st>>>(sc_in, kin, pin, kout, pout, n, slot, w.plan, w.tile_cnt, n_tiles, a->status);
    }
    eval_ap_count_kernel<<<n_blk, AP_THREADS, 0, st>>>(w.plan, tp_in, w.pay[0], w.pay[1], n, a->n_thr, w.blk_cnt, a->status);
    eval_ap_offsets_kernel<<<1, SCAN_THREADS, 0, st>>>(w.blk_cnt, n_blk, a->n_thr, a->status);
    eval_ap_block_kernel<false><<<n_blk, AP_THREADS, 0, st>>>(w.plan, tp_in, w.pay[0], w.pay[1], n, a->n_thr, w.blk_cnt, nullptr, w.blk_max, a->status);
    eval_ap_carry_kernel<<<1, 32 * EVAL_MAX_THR, 0, st>>>(w.blk_max, w.carry, n_blk, a->n_thr, a->status);
    eval_ap_block_kernel<true><<<n_blk, AP_THREADS, 0, st>>>(w.plan, tp_in, w.pay[0], w.pay[1], n, a->n_thr, w.blk_cnt, w.carry, w.blk_sum, a->status);
  }
  eval_finish_kernel<<<1, 32 * EVAL_MAX_THR, 0, st>>>(w.blk_sum, n > 0 ? n_blk : 0, a->n_thr, a->n_topk, a->n_gt, w.hits, a->ap,
                                                   a->recall_hits, a->status);
  return check_launch("avdf_eval_detection");
}

extern "C" AVDF_API size_t avdf_eval_proposal_workspace_bytes(int32_t n_video) {
  if (n_video < 0) return 0;
  return prop_layout(nullptr, n_video).bytes;
}

extern "C" AVDF_API int avdf_eval_proposal(const avdf_eval_proposal_args* a, void* stream) {
  AVDF_CHECK_ARG(a != nullptr, "args is NULL");
  AVDF_CHECK_ARG(a->n_thr >= 1 && a->n_thr <= EVAL_MAX_THR, "n_thr must be 1..16");
  AVDF_CHECK_ARG(a->thresholds != nullptr && a->an_frac != nullptr, "thresholds / an_frac are NULL");
  for (int t = 0; t < a->n_thr; ++t) AVDF_CHECK_ARG(a->thresholds[t] == a->thresholds[t], "threshold is NaN");
  for (int j = 0; j < PROP_POINTS; ++j)
    AVDF_CHECK_ARG(a->an_frac[j] >= 0.0 && a->an_frac[j] <= 1e12 && (j == 0 || a->an_frac[j] >= a->an_frac[j - 1]),
                   "an_frac must be non-decreasing values in [0, 1e12]");
  AVDF_CHECK_ARG(a->n_video >= 0 && a->n_prop >= 0 && a->n_gt >= 0, "n_video, n_prop and n_gt must be >= 0");
  AVDF_CHECK_ARG(a->prop_off && a->gt_off && a->keep, "CSR offsets / keep are NULL");
  AVDF_CHECK_ARG(a->n_prop == 0 || (a->prop_seg && a->prop_score), "proposal arrays are NULL");
  AVDF_CHECK_ARG(a->n_gt == 0 || a->gt_seg, "GT segments are NULL");
  AVDF_CHECK_ARG(a->matches && a->status, "outputs are NULL");
  AVDF_CHECK_ARG(((uintptr_t)a->prop_seg & 15) == 0 && ((uintptr_t)a->gt_seg & 15) == 0, "segments must be 16-byte aligned");
  const PropWs need = prop_layout(nullptr, a->n_video);
  AVDF_CHECK_ARG(a->workspace && a->workspace_bytes >= need.bytes && ((uintptr_t)a->workspace & 255) == 0,
                 "workspace too small or not 256-byte aligned (avdf_eval_proposal_workspace_bytes)");

  cudaStream_t st = (cudaStream_t)stream;
  PropWs w = prop_layout((char*)a->workspace, a->n_video);
  PropParams P = {};
  for (int t = 0; t < a->n_thr; ++t) P.thr[t] = a->thresholds[t];
  for (int j = 0; j < PROP_POINTS; ++j) P.frac[j] = a->an_frac[j];
  P.n_thr = a->n_thr; P.n_video = a->n_video;
  const double2* seg = reinterpret_cast<const double2*>(a->prop_seg);
  const double2* gt = reinterpret_cast<const double2*>(a->gt_seg);
  const int sms = device_sm_count();

  AVDF_CUDA(cudaMemsetAsync(a->status, 0, sizeof(int32_t), st));
  AVDF_CUDA(cudaMemsetAsync(w.n_unsorted, 0, 4, st));
  AVDF_CUDA(cudaMemsetAsync(w.hist, 0, 8 * EVAL_MAX_THR * PROP_POINTS, st));
  eval_validate_kernel<<<(a->n_video + 1 + 255) / 256, 256, 0, st>>>(a->prop_off, a->gt_off, a->n_video, a->n_prop, a->n_gt,
                                                                     a->status, a->keep);
  if (a->n_video > 0) {
    const int grid = (int)std::min<int64_t>((a->n_video + MATCH_WARPS - 1) / MATCH_WARPS, (int64_t)sms * 8);
    eval_prop_match_kernel<<<grid, MATCH_WARPS * 32, 0, st>>>(P, a->prop_off, seg, a->prop_score, a->keep, a->gt_off, gt,
                                                             w.unsorted, w.n_unsorted, w.hist, a->status);
    const size_t smem = (size_t)EVAL_MAX_PRED * (8 + 2);
    AVDF_SMEM_ATTR_ONCE(eval_prop_match_sorted_kernel, smem);
    eval_prop_match_sorted_kernel<<<std::min(a->n_video, 2 * sms), SORTV_THREADS, smem, st>>>(
        P, a->prop_off, seg, a->prop_score, a->keep, a->gt_off, gt, w.unsorted, w.n_unsorted, w.hist, a->status);
  }
  eval_prop_finish_kernel<<<1, 32, 0, st>>>(w.hist, a->n_thr, a->matches, a->status);
  return check_launch("avdf_eval_proposal");
}
