// Result files on the GPU: the JSON text of fixed-size result records (libs/utils/sharding.py layout), byte for byte
// what Python's json writes for the same values (libs/utils/result_writer.py drives it):
//   AVDF_FORMAT_RECORDS      data_left.json items: json.dump([result_item(id, rec), ...], ensure_ascii=False, indent=4)
//   AVDF_FORMAT_PREDICTIONS  prediction.json entries: merge_results' json.dump(segs, sort_keys=True, ensure_ascii=False,
//                            indent=4) with filter_segments(min_score)
// One call formats the output positions [pos_begin, pos_begin + n_rows) into `out` in three launches: one warp per position
// measures its text (a lane per item, the numbers through json_format.cuh), one block scans the lengths in position order
// (integer sums: runs are deterministic), one warp per position writes its text at its offset.
#include "common.cuh"
#include "json_format.cuh"

namespace {

using avdf_json::format_f32;

constexpr int FMT_WARPS = 8;
constexpr int SCAN_THREADS = 1024;

// the fixed text around the numbers (json.dump, indent=4); L(s) is its length without the terminator
#define L(s) ((int)sizeof(s) - 1)
#define R_HEAD "    {\n        \"video_id\": "
#define R_CLS ",\n        \"video_cls\": [\n            "
#define R_SCORES "\n        ],\n        \"scores\": ["
#define R_EMPTY "],\n        \"segments\": []\n    }"
#define R_SCORE "\n            "
#define R_SEGS "\n        ],\n        \"segments\": ["
#define R_PAIR_A "\n            [\n                "
#define R_PAIR_B ",\n                "
#define R_PAIR_C "\n            ]"
#define R_TAIL "\n        ]\n    }"
#define P_HEAD "    "
#define P_OPEN ": ["
#define P_NONE "\n        [\n            0,\n            0,\n            0\n        ]"
#define P_ITEM_A "\n        [\n            "
#define P_ITEM_B ",\n            "
#define P_ITEM_C "\n        ]"
#define P_TAIL "\n    ]"

// Longest text of one position (separator included) for an id of id_bytes bytes; the entry point refuses a buffer that
// cannot hold n_rows of them. libs/utils/result_writer.py row_bytes_max() restates it.
__host__ int64_t row_bytes_max(int mode, int K, int64_t id_bytes) {
  const int64_t N = AVDF_JSON_NUM_MAX;
  if (mode == AVDF_FORMAT_RECORDS)
    return 2 + L(R_HEAD) + id_bytes + L(R_CLS) + N + L(R_SCORES) + L(R_EMPTY) +
           (int64_t)K * (L(R_SCORE) + N + 1) + L(R_SEGS) + (int64_t)K * (L(R_PAIR_A) + N + L(R_PAIR_B) + N + L(R_PAIR_C) + 1) + L(R_TAIL);
  return 2 + L(P_HEAD) + id_bytes + L(P_OPEN) + L(P_NONE) + (int64_t)K * (L(P_ITEM_A) + 3 * N + 2 * L(P_ITEM_B) + L(P_ITEM_C) + 1) + L(P_TAIL);
}

__device__ __forceinline__ uint32_t fbits(const float* p) { return __float_as_uint(__ldg(p)); }

__device__ __forceinline__ int put(char* dst, const char* s, int n) {
  for (int i = 0; i < n; ++i) dst[i] = s[i];
  return n;
}

struct Row {
  const float* rec;     // the record
  int n;                // records: segments; predictions: candidates (the kept ones are those with score > min_score)
  bool ok;
};

__device__ __forceinline__ Row load_row(const avdf_format_args& a, int64_t p) {
  Row r{nullptr, 0, false};
  const int32_t row = __ldg(a.order + p);
  if (row < 0 || (int64_t)row >= a.n_records) return r;
  r.rec = a.records + (int64_t)row * (3 + 3 * (int64_t)a.K);
  const float nf = __ldg(r.rec + 1);
  if (!(nf >= 0.f && nf <= (float)a.K) || nf != truncf(nf)) return r;
  r.n = (int)nf;
  r.ok = true;
  return r;
}

__device__ __forceinline__ bool kept(const avdf_format_args& a, const Row& r, int j) {
  return (double)__ldg(r.rec + 3 + j) > a.min_score;
}

// Length of item t of a record and, when dst is not NULL, its text: t < n is score t, else segment pair t - n.
__device__ __forceinline__ int record_item(const avdf_format_args& a, const Row& r, int t, char* dst) {
  const int n = r.n;
  if (t < n) {
    int len = L(R_SCORE);
    if (dst) put(dst, R_SCORE, L(R_SCORE));
    len += format_f32(fbits(r.rec + 3 + t), dst ? dst + len : nullptr);
    if (t < n - 1) { if (dst) dst[len] = ','; ++len; }
    return len;
  }
  const int j = t - n;             // pair 0 carries the "segments" opener
  const float* s = r.rec + 3 + a.K + 2 * j;
  int len = j == 0 ? L(R_SEGS) : 0;
  if (dst && j == 0) put(dst, R_SEGS, L(R_SEGS));
  if (dst) put(dst + len, R_PAIR_A, L(R_PAIR_A));
  len += L(R_PAIR_A);
  len += format_f32(fbits(s), dst ? dst + len : nullptr);
  if (dst) put(dst + len, R_PAIR_B, L(R_PAIR_B));
  len += L(R_PAIR_B);
  len += format_f32(fbits(s + 1), dst ? dst + len : nullptr);
  if (dst) put(dst + len, R_PAIR_C, L(R_PAIR_C));
  len += L(R_PAIR_C);
  if (j < n - 1) { if (dst) dst[len] = ','; ++len; }
  return len;
}

// The same for candidate j of a prediction entry, a kept segment (`last`: the entry's final kept one).
__device__ __forceinline__ int prediction_item(const avdf_format_args& a, const Row& r, int j, bool last, char* dst) {
  const float* s = r.rec + 3 + a.K + 2 * j;
  int len = L(P_ITEM_A);
  if (dst) put(dst, P_ITEM_A, L(P_ITEM_A));
  len += format_f32(fbits(r.rec + 3 + j), dst ? dst + len : nullptr);
  if (dst) put(dst + len, P_ITEM_B, L(P_ITEM_B));
  len += L(P_ITEM_B);
  len += format_f32(fbits(s), dst ? dst + len : nullptr);
  if (dst) put(dst + len, P_ITEM_B, L(P_ITEM_B));
  len += L(P_ITEM_B);
  len += format_f32(fbits(s + 1), dst ? dst + len : nullptr);
  if (dst) put(dst + len, P_ITEM_C, L(P_ITEM_C));
  len += L(P_ITEM_C);
  if (!last) { if (dst) dst[len] = ','; ++len; }
  return len;
}

__device__ __forceinline__ int warp_incl_scan(int v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int u = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += u;
  }
  return v;
}

// Text of one position. Pass 1 (dst == NULL) returns its length on every lane; pass 2 writes it at dst.
__device__ int64_t format_row(const avdf_format_args& a, int64_t p, const Row& r, char* dst, int lane) {
  const int64_t id0 = __ldg(a.id_off + p), id_len = __ldg(a.id_off + p + 1) - id0;
  int64_t len = p > 0 ? 2 : 0;
  if (dst && lane == 0 && p > 0) { dst[0] = ','; dst[1] = '\n'; }
  if (a.mode == AVDF_FORMAT_RECORDS) {
    if (dst && lane == 0) put(dst + len, R_HEAD, L(R_HEAD));
    len += L(R_HEAD);
    if (dst) for (int64_t c = lane; c < id_len; c += 32) dst[len + c] = (char)__ldg(a.ids + id0 + c);
    len += id_len;
    if (dst && lane == 0) put(dst + len, R_CLS, L(R_CLS));
    len += L(R_CLS);
    len += format_f32(fbits(r.rec + 2), dst && lane == 0 ? dst + len : nullptr);
    if (dst && lane == 0) put(dst + len, R_SCORES, L(R_SCORES));
    len += L(R_SCORES);
    if (r.n == 0) {
      if (dst && lane == 0) put(dst + len, R_EMPTY, L(R_EMPTY));
      return len + L(R_EMPTY);
    }
    for (int base = 0; base < 2 * r.n; base += 32) {
      const int t = base + lane;
      const int il = t < 2 * r.n ? record_item(a, r, t, nullptr) : 0;
      const int incl = warp_incl_scan(il, lane);
      if (dst && t < 2 * r.n) record_item(a, r, t, dst + len + incl - il);
      len += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (dst && lane == 0) put(dst + len, R_TAIL, L(R_TAIL));
    return len + L(R_TAIL);
  }
  if (dst && lane == 0) put(dst + len, P_HEAD, L(P_HEAD));
  len += L(P_HEAD);
  if (dst) for (int64_t c = lane; c < id_len; c += 32) dst[len + c] = (char)__ldg(a.ids + id0 + c);
  len += id_len;
  if (dst && lane == 0) put(dst + len, P_OPEN, L(P_OPEN));
  len += L(P_OPEN);
  int m = 0;                        // kept segments of the row
  for (int base = 0; base < r.n; base += 32) {
    const int j = base + lane;
    m += __popc(__ballot_sync(0xffffffffu, j < r.n && kept(a, r, j)));
  }
  if (m == 0) {
    if (dst && lane == 0) put(dst + len, P_NONE, L(P_NONE));
    len += L(P_NONE);
  } else {
    int k0 = 0;
    for (int base = 0; base < r.n; base += 32) {
      const int j = base + lane;
      const bool keep = j < r.n && kept(a, r, j);
      const unsigned bal = __ballot_sync(0xffffffffu, keep);
      const int k = k0 + __popc(bal & ((1u << lane) - 1));
      const int il = keep ? prediction_item(a, r, j, k == m - 1, nullptr) : 0;
      const int incl = warp_incl_scan(il, lane);
      if (dst && keep) prediction_item(a, r, j, k == m - 1, dst + len + incl - il);
      len += __shfl_sync(0xffffffffu, incl, 31);
      k0 += __popc(bal);
    }
  }
  if (dst && lane == 0) put(dst + len, P_TAIL, L(P_TAIL));
  return len + L(P_TAIL);
}

__global__ void __launch_bounds__(FMT_WARPS * 32) format_len_kernel(avdf_format_args a, uint32_t* lens, int32_t* bad) {
  const int w = (blockIdx.x * FMT_WARPS) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (w >= a.n_rows) return;
  const int64_t p = a.pos_begin + w;
  const Row r = load_row(a, p);
  const int64_t id_len = __ldg(a.id_off + p + 1) - __ldg(a.id_off + p);
  if (!r.ok || id_len < 0 || id_len > a.id_bytes_max) {
    if (lane == 0) { atomicOr(bad, 1); lens[w] = 0; }
    return;
  }
  const int64_t len = format_row(a, p, r, nullptr, lane);
  if (lane == 0) lens[w] = (uint32_t)len;
}

// exclusive scan of the chunk's lengths in position order; *out_bytes = total, or -1 when a row was invalid
__global__ void __launch_bounds__(SCAN_THREADS) format_scan_kernel(const uint32_t* lens, int32_t n, uint64_t* offs,
                                                                   const int32_t* bad, int64_t* out_bytes) {
  __shared__ uint64_t warp_tot[SCAN_THREADS / 32];
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  const int per = (n + SCAN_THREADS - 1) / SCAN_THREADS;
  const int lo = min(n, t * per), hi = min(n, lo + per);
  uint64_t s = 0;
  for (int i = lo; i < hi; ++i) s += lens[i];
  uint64_t incl = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint64_t u = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += u;
  }
  if (lane == 31) warp_tot[wid] = incl;
  __syncthreads();
  if (wid == 0) {
    uint64_t v = warp_tot[lane], x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint64_t u = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += u;
    }
    warp_tot[lane] = x - v;
  }
  __syncthreads();
  uint64_t run = warp_tot[wid] + incl - s;
  for (int i = lo; i < hi; ++i) { offs[i] = run; run += lens[i]; }
  if (t == SCAN_THREADS - 1) *out_bytes = *bad ? -1 : (int64_t)run;
}

__global__ void __launch_bounds__(FMT_WARPS * 32) format_write_kernel(avdf_format_args a, const uint64_t* offs, const int32_t* bad) {
  const int w = (blockIdx.x * FMT_WARPS) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (w >= a.n_rows || *bad) return;
  const int64_t p = a.pos_begin + w;
  format_row(a, p, load_row(a, p), reinterpret_cast<char*>(a.out) + offs[w], lane);
}

struct FormatWs {
  int32_t* bad; uint32_t* lens; uint64_t* offs; size_t bytes;
};

FormatWs format_layout(char* base, int64_t n_rows) {
  FormatWs w;
  size_t o = 0;
  auto take = [&](size_t b) { size_t at = o; o += (b + 255) & ~(size_t)255; return base ? base + at : nullptr; };
  w.bad = reinterpret_cast<int32_t*>(take(4));
  w.lens = reinterpret_cast<uint32_t*>(take(4 * (size_t)n_rows));
  w.offs = reinterpret_cast<uint64_t*>(take(8 * (size_t)n_rows));
  w.bytes = o;
  return w;
}

}  // namespace

using namespace avdf;

extern "C" AVDF_API size_t avdf_format_results_workspace_bytes(int32_t n_rows) {
  if (n_rows < 0) return 0;
  return format_layout(nullptr, n_rows).bytes;
}

extern "C" AVDF_API int avdf_format_results(const avdf_format_args* a, void* stream) {
  AVDF_CHECK_ARG(a != nullptr, "args is NULL");
  AVDF_CHECK_ARG(a->mode == AVDF_FORMAT_RECORDS || a->mode == AVDF_FORMAT_PREDICTIONS, "mode must be AVDF_FORMAT_RECORDS or AVDF_FORMAT_PREDICTIONS");
  AVDF_CHECK_ARG(a->K >= 1 && a->K <= (1 << 20), "K must be 1 .. 2^20");
  AVDF_CHECK_ARG(a->n_records >= 0 && a->n_pos >= 0, "n_records / n_pos must be >= 0");
  AVDF_CHECK_ARG(a->n_rows >= 1 && a->pos_begin >= 0 && a->pos_begin + a->n_rows <= a->n_pos, "rows must lie inside 0 .. n_pos");
  AVDF_CHECK_ARG(a->records && a->order && a->ids && a->id_off, "records / order / ids / id_off are NULL");
  AVDF_CHECK_ARG(a->out && a->out_bytes, "out / out_bytes are NULL");
  AVDF_CHECK_ARG(a->id_bytes_max >= 0, "id_bytes_max must be >= 0");
  AVDF_CHECK_ARG(a->min_score == a->min_score, "min_score is NaN");
  const int64_t row_max = row_bytes_max(a->mode, a->K, a->id_bytes_max);
  AVDF_CHECK_ARG(row_max <= (int64_t)UINT32_MAX, "a row's text would exceed 4 GiB");
  AVDF_CHECK_ARG((uint64_t)row_max * (uint64_t)a->n_rows <= a->out_capacity,
                 "out_capacity is below n_rows times the longest row text (result_writer.row_bytes_max)");
  const FormatWs need = format_layout(nullptr, a->n_rows);
  AVDF_CHECK_ARG(a->workspace && a->workspace_bytes >= need.bytes && ((uintptr_t)a->workspace & 255) == 0,
                 "workspace too small or not 256-byte aligned (avdf_format_results_workspace_bytes)");
  cudaStream_t st = (cudaStream_t)stream;
  const FormatWs w = format_layout((char*)a->workspace, a->n_rows);
  const int grid = (a->n_rows + FMT_WARPS - 1) / FMT_WARPS;
  AVDF_CUDA(cudaMemsetAsync(w.bad, 0, 4, st));
  format_len_kernel<<<grid, FMT_WARPS * 32, 0, st>>>(*a, w.lens, w.bad);
  format_scan_kernel<<<1, SCAN_THREADS, 0, st>>>(w.lens, a->n_rows, w.offs, w.bad, a->out_bytes);
  format_write_kernel<<<grid, FMT_WARPS * 32, 0, st>>>(*a, w.offs, w.bad);
  return check_launch("avdf_format_results");
}
