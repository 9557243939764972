/* Plain-C restatement of the reference's 1-D NMS path. TEST INFRASTRUCTURE:
 * the parity checker for the CUDA kernels, never linked into the product.
 *
 * Follows (paths relative to the reference root):
 *   libs/utils/csrc/nms_cpu.cpp:19-58   nms_1d_cpu      -> ref_nms_1d
 *   libs/utils/csrc/nms_cpu.cpp:67-160  softnms_1d_cpu  -> ref_softnms_1d
 *   libs/utils/nms.py:67-101            seg_voting      -> ref_seg_voting
 * Pinned against the reference's compiled extension (oracle/_ref) and the
 * known answers in tests/golden/nms_kat.json (tests/test_oracle_golden.py).
 *
 * Build: gcc -O2 -ffp-contract=off -shared -fPIC (no FMA contraction, so the
 * float arithmetic is the same sequence of IEEE ops the reference's g++ build
 * performs). Tie rule where the reference leaves it to the sort
 * implementation: equal scores keep ascending input order.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

static const float *g_key;
static int cmp_desc(const void *a, const void *b) {
  int64_t ia = *(const int64_t *)a, ib = *(const int64_t *)b;
  float sa = g_key[ia], sb = g_key[ib];
  if (sa > sb) return -1;
  if (sa < sb) return 1;
  return (ia > ib) - (ia < ib);
}

/* order[] <- indices sorted by descending score, ties by ascending index */
static void argsort_desc(const float *scores, int64_t n, int64_t *order) {
  for (int64_t i = 0; i < n; i++) order[i] = i;
  g_key = scores;
  qsort(order, (size_t)n, sizeof(int64_t), cmp_desc);
}

/* nms_cpu.cpp:19-58. segs [n,2], scores [n]; out_idx gets the kept input
 * indices in descending-score order; returns their count. */
int64_t ref_nms_1d(const float *segs, const float *scores, int64_t n,
                   float iou_threshold, int64_t *out_idx) {
  if (n == 0) return 0;
  int64_t *order = (int64_t *)malloc(sizeof(int64_t) * n);
  float *areas = (float *)malloc(sizeof(float) * n);
  unsigned char *sel = (unsigned char *)malloc((size_t)n);
  for (int64_t i = 0; i < n; i++) {
    areas[i] = (segs[2 * i + 1] - segs[2 * i]) + 1e-6f; /* :27 float + (float)1e-6 */
    sel[i] = 1;
  }
  argsort_desc(scores, n, order);
  for (int64_t _i = 0; _i < n; _i++) {
    if (!sel[_i]) continue;
    int64_t i = order[_i];
    float ix1 = segs[2 * i], ix2 = segs[2 * i + 1], ia = areas[i];
    for (int64_t _j = _i + 1; _j < n; _j++) {
      if (!sel[_j]) continue;
      int64_t j = order[_j];
      float xx1 = fmaxf(ix1, segs[2 * j]);
      float xx2 = fminf(ix2, segs[2 * j + 1]);
      float inter = fmaxf(0.f, xx2 - xx1);
      float ovr = inter / (ia + areas[j] - inter);
      if (ovr >= iou_threshold) sel[_j] = 0;
    }
  }
  int64_t k = 0;
  for (int64_t _i = 0; _i < n; _i++)
    if (sel[_i]) out_idx[k++] = order[_i];
  free(order); free(areas); free(sel);
  return k;
}

/* nms_cpu.cpp:67-160. dets [n,3] is written in place (x1, x2, score per
 * pick); out_inds gets the original indices in pick order; returns count.
 * max_num > 0 stops after that many picks: pick i depends on picks 0..i-1
 * only, so the result is the prefix of the full run (what the kernels'
 * max_num returns), at a fraction of the O(n * picks) cost. */
int64_t ref_softnms_1d_capped(const float *segs, const float *scores, float *dets,
                              int64_t n, float iou_threshold, float sigma,
                              float min_score, int method, int64_t max_num,
                              int64_t *out_inds) {
  if (n == 0) return 0;
  float *x1 = (float *)malloc(sizeof(float) * n), *x2 = (float *)malloc(sizeof(float) * n);
  float *sc = (float *)malloc(sizeof(float) * n), *ar = (float *)malloc(sizeof(float) * n);
  int64_t *inds = (int64_t *)malloc(sizeof(int64_t) * n);
  for (int64_t i = 0; i < n; i++) {
    x1[i] = segs[2 * i]; x2[i] = segs[2 * i + 1]; sc[i] = scores[i];
    ar[i] = (x2[i] - x1[i]) + 1e-6f; inds[i] = i;
  }
  int64_t nsegs = n;
  for (int64_t i = 0; i < nsegs; i++) {
    if (max_num > 0 && i >= max_num) { nsegs = i; break; }
    float max_score = sc[i];
    int64_t max_pos = i;
    for (int64_t pos = i + 1; pos < nsegs; pos++)
      if (max_score < sc[pos]) { max_score = sc[pos]; max_pos = pos; }
    float ix1 = dets[i * 3 + 0] = x1[max_pos];
    float ix2 = dets[i * 3 + 1] = x2[max_pos];
    float isc = dets[i * 3 + 2] = sc[max_pos];
    float iar = ar[max_pos];
    int64_t iind = inds[max_pos];
    x1[max_pos] = x1[i]; x2[max_pos] = x2[i]; sc[max_pos] = sc[i];
    ar[max_pos] = ar[i]; inds[max_pos] = inds[i];
    x1[i] = ix1; x2[i] = ix2; sc[i] = isc; ar[i] = iar; inds[i] = iind;
    int64_t pos = i + 1;
    while (pos < nsegs) {
      float xx1 = fmaxf(ix1, x1[pos]);
      float xx2 = fminf(ix2, x2[pos]);
      float inter = fmaxf(0.f, xx2 - xx1);
      float ovr = inter / (iar + ar[pos] - inter);
      float weight = 1.f;
      if (method == 0) { if (ovr >= iou_threshold) weight = 0.f; }
      else if (method == 1) { if (ovr >= iou_threshold) weight = 1.f - ovr; }
      else if (method == 2) { weight = expf(-(ovr * ovr) / sigma); }
      sc[pos] *= weight;
      if (sc[pos] < min_score) {
        x1[pos] = x1[nsegs - 1]; x2[pos] = x2[nsegs - 1]; sc[pos] = sc[nsegs - 1];
        ar[pos] = ar[nsegs - 1]; inds[pos] = inds[nsegs - 1];
        nsegs--; pos--;
      }
      pos++;
    }
  }
  memcpy(out_inds, inds, sizeof(int64_t) * nsegs);
  free(x1); free(x2); free(sc); free(ar); free(inds);
  return nsegs;
}

int64_t ref_softnms_1d(const float *segs, const float *scores, float *dets,
                       int64_t n, float iou_threshold, float sigma,
                       float min_score, int method, int64_t *out_inds) {
  return ref_softnms_1d_capped(segs, scores, dets, n, iou_threshold, sigma,
                               min_score, method, 0, out_inds);
}

/* nms.py:67-101 (score_offset is computed but unused there). nms_segs [k,2]
 * refined in `out` [k,2] against ALL candidates; fp32, sums accumulated in
 * candidate order (the reference uses a matmul, so agreement is to rounding,
 * not bitwise). */
void ref_seg_voting(const float *nms_segs, int64_t k, const float *all_segs,
                    const float *all_scores, int64_t n, float iou_threshold, float *out) {
  for (int64_t i = 0; i < k; i++) {
    float a0 = nms_segs[2 * i], a1 = nms_segs[2 * i + 1], la = a1 - a0;
    double sw = 0.0, s0 = 0.0, s1 = 0.0;
    float fsw = 0.f;
    for (int64_t j = 0; j < n; j++) {
      float b0 = all_segs[2 * j], b1 = all_segs[2 * j + 1];
      float left = fmaxf(a0, b0), right = fminf(a1, b1);
      float inter = fmaxf(right - left, 0.f);
      float iou = inter / (la + (b1 - b0) - inter);
      float w = (iou >= iou_threshold ? 1.f : 0.f) * all_scores[j] * iou;
      fsw += w;
      sw += w;
    }
    (void)sw;
    for (int64_t j = 0; j < n; j++) {
      float b0 = all_segs[2 * j], b1 = all_segs[2 * j + 1];
      float left = fmaxf(a0, b0), right = fminf(a1, b1);
      float inter = fmaxf(right - left, 0.f);
      float iou = inter / (la + (b1 - b0) - inter);
      float w = (iou >= iou_threshold ? 1.f : 0.f) * all_scores[j] * iou;
      w = w / fsw;
      s0 += (double)w * b0;
      s1 += (double)w * b1;
    }
    out[2 * i] = (float)s0;
    out[2 * i + 1] = (float)s1;
  }
}
