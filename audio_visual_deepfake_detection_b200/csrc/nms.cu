// 1-D hard / soft NMS, segment voting, decode and the fused per-video postprocess kernel.
//
// Replaces the reference's only native component, libs/utils/csrc/nms_cpu.cpp
// (nms_1d_cpu :19-58, softnms_1d_cpu :67-160), plus the python glue around it:
// libs/utils/nms.py (NMSop :8-35, SoftNMSop :38-64, seg_voting :67-101, batched_nms :103-190),
// and libs/modeling/av_fd_no_recon.py inference_single_video :760-825 / postprocessing :827-876.
//
// One CTA per video. Candidates live in shared memory (<= NMS_SMEM_CAP) or in a caller-provided
// global workspace (the 100k sweep). Bit-level parity rules:
//   * every float expression is the same sequence of IEEE ops as the g++ build of the reference
//     (compiled with -fmad=false; IEEE division), areas = (x2 - x1) + 1e-6f;
//   * hard NMS: greedy over descending score, ties by ascending input index (stable sort);
//   * soft NMS: the reference's in-place selection / swap-with-last bookkeeping is emulated
//     exactly (array positions decide ties), including "first pick is emitted even if it is
//     below min_score";
//   * the gaussian weight uses a restatement of glibc's expf (double polynomial + table),
//     which is what std::exp(float) resolves to in the reference build.
#include <stdlib.h>
#include <algorithm>
#include <cmath>
#include "common.cuh"

namespace avdf {

constexpr int NMS_THREADS = 512;
constexpr int NMS_WARPS = NMS_THREADS / 32;
constexpr int NMS_SMEM_CAP = 6144;   // candidates kept in shared memory (6 arrays * 4 B * cap = 144 KB)

// ---------------------------------------------------------------------------------------------
// glibc expf (sysdeps/ieee754/flt-32/e_expf.c, exp2f_data N=32) restated; bit-identical to the
// host libm on 2e8 random inputs (see DESIGN.md). |x| >= 88 falls back to CUDA expf.
// ---------------------------------------------------------------------------------------------
__constant__ unsigned long long c_exp2f_tab[32] = {
    0x3ff0000000000000ull, 0x3fefd9b0d3158574ull, 0x3fefb5586cf9890full, 0x3fef9301d0125b51ull,
    0x3fef72b83c7d517bull, 0x3fef54873168b9aaull, 0x3fef387a6e756238ull, 0x3fef1e9df51fdee1ull,
    0x3fef06fe0a31b715ull, 0x3feef1a7373aa9cbull, 0x3feedea64c123422ull, 0x3feece086061892dull,
    0x3feebfdad5362a27ull, 0x3feeb42b569d4f82ull, 0x3feeab07dd485429ull, 0x3feea47eb03a5585ull,
    0x3feea09e667f3bcdull, 0x3fee9f75e8ec5f74ull, 0x3feea11473eb0187ull, 0x3feea589994cce13ull,
    0x3feeace5422aa0dbull, 0x3feeb737b0cdc5e5ull, 0x3feec49182a3f090ull, 0x3feed503b23e255dull,
    0x3feee89f995ad3adull, 0x3feeff76f2fb5e47ull, 0x3fef199bdd85529cull, 0x3fef3720dcef9069ull,
    0x3fef5818dcfba487ull, 0x3fef7c97337b9b5full, 0x3fefa4afa2a490daull, 0x3fefd0765b6e4540ull};

__device__ __forceinline__ float expf_glibc(float x) {
  if (!(fabsf(x) < 88.0f)) return expf(x);
  const double kInvLn2N = 0x1.71547652b82fep+0 * 32.0;
  const double kShift = 0x1.8p+52;
  const double C0 = 0x1.c6af84b912394p-5 / 32.0 / 32.0 / 32.0;
  const double C1 = 0x1.ebfce50fac4f3p-3 / 32.0 / 32.0;
  const double C2 = 0x1.62e42ff0c52d6p-1 / 32.0;
  double z = __dmul_rn(kInvLn2N, (double)x);
  double kd = __dadd_rn(z, kShift);
  unsigned long long ki = (unsigned long long)__double_as_longlong(kd);
  kd = __dsub_rn(kd, kShift);
  double r = __dsub_rn(z, kd);
  unsigned long long t = c_exp2f_tab[ki & 31ull] + (ki << 47);
  double s = __longlong_as_double((long long)t);
  double p = __fma_rn(C0, r, C1);
  double r2 = __dmul_rn(r, r);
  double y = __fma_rn(C2, r, 1.0);
  y = __fma_rn(p, r2, y);
  y = __dmul_rn(y, s);
  return (float)y;
}

// IoU with the reference's epsilon'd areas (nms_cpu.cpp:27,51-53 / :77,124-128)
__device__ __forceinline__ float ovr_eps(float ix1, float ix2, float iar, float jx1, float jx2, float jar) {
  float xx1 = fmaxf(ix1, jx1);
  float xx2 = fminf(ix2, jx2);
  float inter = fmaxf(0.f, __fsub_rn(xx2, xx1));
  return __fdiv_rn(inter, __fsub_rn(__fadd_rn(iar, jar), inter));
}

struct Cand {          // struct-of-arrays working set of one video
  float* x1; float* x2; float* sc; float* ar; int* id; int* hole;
};

// key for argmax: larger score wins; equal score -> smaller tie index wins
struct Best { float s; int tie; int pos; };
__device__ __forceinline__ bool better(float s, int tie, const Best& b) {
  return (b.pos < 0) || (s > b.s) || (s == b.s && tie < b.tie);
}
__device__ __forceinline__ Best warp_best(Best b) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    Best c;
    c.s = __shfl_xor_sync(0xffffffffu, b.s, o);
    c.tie = __shfl_xor_sync(0xffffffffu, b.tie, o);
    c.pos = __shfl_xor_sync(0xffffffffu, b.pos, o);
    if (c.pos >= 0 && better(c.s, c.tie, b)) b = c;
  }
  return b;
}
// Block argmax; `slot` alternates 0/1 between consecutive calls so one barrier suffices.
__device__ __forceinline__ Best block_best(Best b, Best* sh /*[2][NMS_WARPS]*/, int slot) {
  b = warp_best(b);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) sh[slot * NMS_WARPS + w] = b;
  __syncthreads();
  Best c;
  c.pos = -1; c.s = 0.f; c.tie = 0;
  if (lane < NMS_WARPS) c = sh[slot * NMS_WARPS + lane];
  return warp_best(c);
}
__device__ __forceinline__ int block_sum(int v, int* sh /*[2][NMS_WARPS]*/, int slot) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) sh[slot * NMS_WARPS + w] = v;
  __syncthreads();
  int c = (lane < NMS_WARPS) ? sh[slot * NMS_WARPS + lane] : 0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  return c;
}

struct NmsShared {
  Best best[2 * NMS_WARPS];
  int sum[2 * NMS_WARPS];
  int scan[NMS_WARPS];
};

// ---------------------------------------------------------------------------------------------
// hard NMS (nms_cpu.cpp:19-58). Candidates c.{x1,x2,sc,ar}[0..n); c.id[i] >= 0 alive.
// Emits kept ORIGINAL positions (0..n) in descending score order; stops after max_num (>0).
// ---------------------------------------------------------------------------------------------
__device__ int hard_nms_block(const Cand& c, int n, float thr, int max_num, int* out_pos, NmsShared& sh) {
  int k = 0, slot = 0;
  while (max_num <= 0 || k < max_num) {
    Best b; b.pos = -1; b.s = 0.f; b.tie = 0;
    for (int p = threadIdx.x; p < n; p += NMS_THREADS)
      if (c.id[p] >= 0 && better(c.sc[p], p, b)) { b.s = c.sc[p]; b.tie = p; b.pos = p; }
    b = block_best(b, sh.best, slot);
    slot ^= 1;
    if (b.pos < 0) break;
    const float ix1 = c.x1[b.pos], ix2 = c.x2[b.pos], iar = c.ar[b.pos];
    if (threadIdx.x == 0) out_pos[k] = b.pos;
    for (int p = threadIdx.x; p < n; p += NMS_THREADS) {
      if (c.id[p] < 0) continue;
      if (p == b.pos) { c.id[p] = ~c.id[p]; continue; }
      float ovr = ovr_eps(ix1, ix2, iar, c.x1[p], c.x2[p], c.ar[p]);
      if (ovr >= thr) c.id[p] = ~c.id[p];
    }
    ++k;
  }
  return k;
}

// ---------------------------------------------------------------------------------------------
// soft NMS (nms_cpu.cpp:67-160) with exact emulation of the reference's array bookkeeping.
// c.* are the reference's working arrays in POSITION order; c.id[] holds original indices.
// dets (x1,x2,score per pick) and out_idx are written for picks [0, K). Returns K.
// ---------------------------------------------------------------------------------------------
__device__ int soft_nms_block(const Cand& c, int n, float thr, float sigma, float min_score, int method,
                              int max_num, float* dets, int* out_idx, NmsShared& sh) {
  int nsegs = n, slot = 0, sslot = 0;
  int i = 0;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (; i < nsegs; ++i) {
    if (max_num > 0 && i >= max_num) break;
    // 1. first maximum in position order over [i, nsegs)  (:92-103, strict '<')
    Best b; b.pos = -1; b.s = 0.f; b.tie = 0;
    {
      int p0 = i + ((threadIdx.x - i) % NMS_THREADS + NMS_THREADS) % NMS_THREADS;   // p === tid (mod T), p >= i
      for (int p = p0; p < nsegs; p += NMS_THREADS)
        if (better(c.sc[p], p, b)) { b.s = c.sc[p]; b.tie = p; b.pos = p; }
    }
    b = block_best(b, sh.best, slot);
    slot ^= 1;
    const int mp = b.pos;
    // 2. read the pick and the element it is swapped with (:105-122)
    const float ix1 = c.x1[mp], ix2 = c.x2[mp], isc = c.sc[mp], iar = c.ar[mp];
    const int iid = c.id[mp];
    const float ox1 = c.x1[i], ox2 = c.x2[i], osc = c.sc[i], oar = c.ar[i];
    const int oid = c.id[i];
    if (threadIdx.x == 0) {
      dets[3 * i + 0] = ix1; dets[3 * i + 1] = ix2; dets[3 * i + 2] = isc;
      out_idx[i] = iid;
    }
    __syncthreads();            // all reads of [mp] and [i] done before [mp] is overwritten
    // 3. decay every position in (i, nsegs) (:125-146); the slot mp now holds the old element i
    int nfail = 0;
    {
      int p0 = (i + 1) + ((threadIdx.x - (i + 1)) % NMS_THREADS + NMS_THREADS) % NMS_THREADS;
      for (int p = p0; p < nsegs; p += NMS_THREADS) {
        float jx1, jx2, jsc, jar;
        if (p == mp) {
          jx1 = ox1; jx2 = ox2; jsc = osc; jar = oar;
          c.x1[p] = ox1; c.x2[p] = ox2; c.ar[p] = oar; c.id[p] = oid;
        } else {
          jx1 = c.x1[p]; jx2 = c.x2[p]; jsc = c.sc[p]; jar = c.ar[p];
        }
        float ovr = ovr_eps(ix1, ix2, iar, jx1, jx2, jar);
        float weight = 1.f;
        if (method == 0) { if (ovr >= thr) weight = 0.f; }
        else if (method == 1) { if (ovr >= thr) weight = __fsub_rn(1.f, ovr); }
        else if (method == 2) { weight = expf_glibc(__fdiv_rn(-__fmul_rn(ovr, ovr), sigma)); }
        jsc = __fmul_rn(jsc, weight);
        c.sc[p] = jsc;
        nfail += (jsc < min_score) ? 1 : 0;
      }
    }
    const int F = block_sum(nfail, sh.sum, sslot);   // barrier inside: decay writes are visible
    sslot ^= 1;
    if (F == 0) continue;
    // 4. emulate "swap with last, shrink" (:150-157): after the pass the first nsegs-F positions
    //    hold the survivors; the k-th failed slot below the new end receives the k-th survivor
    //    counted from the old end backwards.
    const int lo = i + 1, L = nsegs - lo, new_n = nsegs - F;
    const int chunk = (L + NMS_THREADS - 1) / NMS_THREADS;
    const int cb = lo + threadIdx.x * chunk;
    const int ce = min(cb + chunk, nsegs);
    int cnt = 0;
    for (int p = cb; p < ce; ++p) cnt += (c.sc[p] < min_score) ? 1 : 0;
    // block exclusive scan of cnt
    int inc = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
    if (lane == 31) sh.scan[w] = inc;
    __syncthreads();
    int wbase = 0;
    for (int q = 0; q < w; ++q) wbase += sh.scan[q];
    int run = wbase + inc - cnt;                     // failures strictly before this chunk
    int run_hi = run;                                // ... and strictly before max(cb, new_n)
    for (int p = cb; p < ce; ++p) {
      bool fail = c.sc[p] < min_score;
      if (fail && p < new_n) c.hole[run] = p;        // ascending rank among failures == rank among holes
      run += fail ? 1 : 0;
      if (p < new_n) run_hi = run;
    }
    __syncthreads();
    // the moves below fill holes (< new_n) while other threads still scan their chunks: read positions >= new_n only
    run = run_hi;
    for (int p = max(cb, new_n); p < ce; ++p) {
      bool fail = c.sc[p] < min_score;
      run += fail ? 1 : 0;                           // inclusive failure count through p
      if (!fail && p >= new_n) {
        int rank_desc = (nsegs - 1 - p) - (F - run); // survivors at positions > p
        int dst = c.hole[rank_desc];
        c.x1[dst] = c.x1[p]; c.x2[dst] = c.x2[p]; c.sc[dst] = c.sc[p]; c.ar[dst] = c.ar[p]; c.id[dst] = c.id[p];
      }
    }
    __syncthreads();
    nsegs = new_n;
  }
  return i;
}

// ---------------------------------------------------------------------------------------------
// standalone kernels behind avdf_nms_hard / avdf_nms_soft (same contract as nms_1d_cpu.{nms,softnms})
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ Cand carve(void* base, int cap) {
  Cand c;
  float* f = reinterpret_cast<float*>(base);
  c.x1 = f; c.x2 = f + cap; c.sc = f + 2 * cap; c.ar = f + 3 * cap;
  c.id = reinterpret_cast<int*>(f + 4 * cap);
  c.hole = reinterpret_cast<int*>(f + 5 * cap);
  return c;
}

__global__ void __launch_bounds__(NMS_THREADS, 1)
nms_standalone_kernel(const float* __restrict__ segs, const float* __restrict__ scores, int n,
                      float thr, float sigma, float min_score, int method /* -1 = hard */, int max_num,
                      float* dets, long long* out_idx, int* out_count, void* gws, int use_gws) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ NmsShared sh;
  Cand c = use_gws ? carve(gws, n) : carve(smem_raw, NMS_SMEM_CAP);
  for (int p = threadIdx.x; p < n; p += NMS_THREADS) {
    float a = segs[2 * p], b = segs[2 * p + 1];
    c.x1[p] = a; c.x2[p] = b; c.sc[p] = scores[p];
    c.ar[p] = __fadd_rn(__fsub_rn(b, a), 1e-6f);
    c.id[p] = p;
  }
  __syncthreads();
  int* tmp_idx = c.hole;      // hard: kept positions; soft: original ids (hole[] is also scratch there -> use gws tail)
  int k;
  if (method < 0) {
    k = hard_nms_block(c, n, thr, max_num, tmp_idx, sh);
    __syncthreads();
    for (int q = threadIdx.x; q < k; q += NMS_THREADS) out_idx[q] = tmp_idx[q];
  } else {
    // out ids go straight to global as int32 scratch placed in dets' tail is not available: use out_idx as int32 scratch
    int* oi = reinterpret_cast<int*>(out_idx);       // 2n ints available; widened in place below
    k = soft_nms_block(c, n, thr, sigma, min_score, method, max_num, dets, oi, sh);
    __syncthreads();
    // widen int32 -> int64 in place, back to front, single thread-block ordered by chunks
    for (int base = ((k - 1) / NMS_THREADS) * NMS_THREADS; base >= 0; base -= NMS_THREADS) {
      int q = base + threadIdx.x;
      int v = (q < k) ? oi[q] : 0;
      __syncthreads();
      if (q < k) out_idx[q] = v;
      __syncthreads();
    }
  }
  if (threadIdx.x == 0) *out_count = k;
}

// ---------------------------------------------------------------------------------------------
// Large candidate lists (n > NMS_SMEM_CAP: the 10k / 100k points of the NMS sweep): one CLUSTER of NMS_CL CTAs. The
// reference's working arrays are distributed by POSITION - position p lives in CTA p / S at offset p % S of that CTA's
// shared memory - so every pick is: local argmax over the CTA's slice -> the CTA's best (with the candidate's data) is
// written into every CTA's exchange table through distributed shared memory -> barrier.cluster -> every CTA reduces the
// NMS_CL records to the same global pick and decays / suppresses its own slice. The soft-NMS bookkeeping (swap the pick
// to the front, swap failed candidates with the last one and shrink, nms_cpu.cpp:105-157) is emulated exactly as in
// soft_nms_block above: fail counts are exchanged the same way, holes are ranked through a cluster-wide prefix, the hole
// list lives in the global workspace, survivors beyond the new end are moved into the holes with remote stores.
// One CTA walking a 100k list from global memory takes ~70-80 us per pick; here a pick costs 2-4 cluster barriers.
// ---------------------------------------------------------------------------------------------
constexpr int NMS_CL = 16;                      // CTAs per cluster (non-portable size: needs the launch attribute)
constexpr int NMS_CL_SLICE_MAX = 11264;         // positions per CTA: 5 arrays x 4 B x 11264 = 220 KB
struct ClRec { float s; int pos; float x1, x2, ar; int id; };       // a CTA's best candidate (pos < 0: none)
struct ClSwap { float x1, x2, sc, ar; int id; int pad; };            // the element at position i (it moves to the pick's slot)
struct ClShared {
  ClRec rec[2][NMS_CL];
  ClSwap swp[2];
  int cnt[NMS_CL];
};
__device__ __forceinline__ uint32_t smem_addr_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t cl_map(uint32_t addr, int rank) {
  uint32_t r; asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank)); return r;
}
__device__ __forceinline__ void cl_st(uint32_t cluster_addr, uint32_t v) {
  asm volatile("st.shared::cluster.b32 [%0], %1;" ::"r"(cluster_addr), "r"(v) : "memory");
}
__device__ __forceinline__ void cl_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ int cl_rank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return (int)r; }

__global__ void __launch_bounds__(NMS_THREADS, 1)
nms_cluster_kernel(const float* __restrict__ segs, const float* __restrict__ scores, int n, int S,
                   float thr, float sigma, float min_score, int method /* -1 = hard */, int max_num,
                   float* dets, long long* out_idx, int* out_count, int* hole /* global, n ints */) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ NmsShared sh;
  __shared__ ClShared cs;
  float* x1 = reinterpret_cast<float*>(smem_raw);
  float* x2 = x1 + S; float* sc = x2 + S; float* ar = sc + S;
  int* id = reinterpret_cast<int*>(ar + S);
  const int rank = cl_rank();
  const int base = rank * S;                       // first position of this CTA's slice
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int o = threadIdx.x; o < S; o += NMS_THREADS) {
    const int p = base + o;
    if (p < n) {
      float a = segs[2 * p], b = segs[2 * p + 1];
      x1[o] = a; x2[o] = b; sc[o] = scores[p];
      ar[o] = __fadd_rn(__fsub_rn(b, a), 1e-6f);
      id[o] = p;
    }
  }
  __syncthreads();
  // publish this CTA's best candidate (threads 0..NMS_CL-1: one remote CTA each)
  auto publish_best = [&](const Best& b, int buf) {
    if (threadIdx.x < NMS_CL) {
      ClRec r; r.s = b.s; r.pos = b.pos;
      if (b.pos >= 0) { const int o = b.pos - base; r.x1 = x1[o]; r.x2 = x2[o]; r.ar = ar[o]; r.id = id[o]; }
      else { r.x1 = r.x2 = r.ar = 0.f; r.id = 0; }
      const uint32_t dst = cl_map(smem_addr_u32(&cs.rec[buf][rank]), (int)threadIdx.x);
      cl_st(dst, __float_as_uint(r.s)); cl_st(dst + 4, (uint32_t)r.pos); cl_st(dst + 8, __float_as_uint(r.x1));
      cl_st(dst + 12, __float_as_uint(r.x2)); cl_st(dst + 16, __float_as_uint(r.ar)); cl_st(dst + 20, (uint32_t)r.id);
    }
  };
  auto global_best = [&](int buf) -> ClRec {      // the same record in every thread of every CTA
    ClRec g = cs.rec[buf][0];
#pragma unroll
    for (int c = 1; c < NMS_CL; ++c) {
      const ClRec r = cs.rec[buf][c];
      if (r.pos >= 0 && (g.pos < 0 || r.s > g.s || (r.s == g.s && r.pos < g.pos))) g = r;
    }
    return g;
  };
  int k = 0;
  if (method < 0) {
    // ---- hard NMS (nms_cpu.cpp:19-58): greedy over descending score, ties by ascending index; id < 0 = suppressed
    int slot = 0, buf = 0;
    const int cnt_own = min(S, n - base);
    while (max_num <= 0 || k < max_num) {
      Best b; b.pos = -1; b.s = 0.f; b.tie = 0;
      for (int o = threadIdx.x; o < cnt_own; o += NMS_THREADS)
        if (id[o] >= 0 && better(sc[o], base + o, b)) { b.s = sc[o]; b.tie = base + o; b.pos = base + o; }
      b = block_best(b, sh.best, slot);
      slot ^= 1;
      publish_best(b, buf);
      cl_sync();
      const ClRec g = global_best(buf);
      buf ^= 1;
      if (g.pos < 0) break;
      if (rank == 0 && threadIdx.x == 0) out_idx[k] = g.pos;
      for (int o = threadIdx.x; o < cnt_own; o += NMS_THREADS) {
        if (id[o] < 0) continue;
        if (base + o == g.pos) { id[o] = ~id[o]; continue; }
        float ovr = ovr_eps(g.x1, g.x2, g.ar, x1[o], x2[o], ar[o]);
        if (ovr >= thr) id[o] = ~id[o];
      }
      __syncthreads();
      ++k;
    }
  } else {
    // ---- soft NMS (nms_cpu.cpp:67-160), positions [0, nsegs) distributed over the cluster
    int nsegs = n, slot = 0, sslot = 0;
    int i = 0;
    for (; i < nsegs; ++i) {
      if (max_num > 0 && i >= max_num) break;
      const int hi = min(nsegs, base + S);       // this CTA's positions are [base, hi)
      // 1. first maximum in position order over [i, nsegs): local part, then the exchange
      Best b; b.pos = -1; b.s = 0.f; b.tie = 0;
      for (int p = max(i, base) + threadIdx.x; p < hi; p += NMS_THREADS)
        if (better(sc[p - base], p, b)) { b.s = sc[p - base]; b.tie = p; b.pos = p; }
      b = block_best(b, sh.best, slot);
      slot ^= 1;
      publish_best(b, 0);
      if (i >= base && i < base + S && threadIdx.x >= 32 && threadIdx.x < 32 + NMS_CL) {   // the owner of position i
        const int o = i - base;
        const uint32_t dst = cl_map(smem_addr_u32(&cs.swp[0]), (int)threadIdx.x - 32);
        cl_st(dst, __float_as_uint(x1[o])); cl_st(dst + 4, __float_as_uint(x2[o])); cl_st(dst + 8, __float_as_uint(sc[o]));
        cl_st(dst + 12, __float_as_uint(ar[o])); cl_st(dst + 16, (uint32_t)id[o]);
      }
      cl_sync();
      const ClRec g = global_best(0);
      const ClSwap o_ = cs.swp[0];
      const int mp = g.pos;
      if (rank == 0 && threadIdx.x == 0) {
        dets[3 * i + 0] = g.x1; dets[3 * i + 1] = g.x2; dets[3 * i + 2] = g.s;
        out_idx[i] = g.id;
      }
      // 3. decay every position in (i, nsegs); the slot mp now holds the old element i
      int nfail = 0;
      for (int p = max(i + 1, base) + threadIdx.x; p < hi; p += NMS_THREADS) {
        const int o = p - base;
        float jx1, jx2, jsc, jar;
        if (p == mp) {
          jx1 = o_.x1; jx2 = o_.x2; jsc = o_.sc; jar = o_.ar;
          x1[o] = o_.x1; x2[o] = o_.x2; ar[o] = o_.ar; id[o] = o_.id;
        } else {
          jx1 = x1[o]; jx2 = x2[o]; jsc = sc[o]; jar = ar[o];
        }
        float ovr = ovr_eps(g.x1, g.x2, g.ar, jx1, jx2, jar);
        float weight = 1.f;
        if (method == 0) { if (ovr >= thr) weight = 0.f; }
        else if (method == 1) { if (ovr >= thr) weight = __fsub_rn(1.f, ovr); }
        else if (method == 2) { weight = expf_glibc(__fdiv_rn(-__fmul_rn(ovr, ovr), sigma)); }
        jsc = __fmul_rn(jsc, weight);
        sc[o] = jsc;
        nfail += (jsc < min_score) ? 1 : 0;
      }
      const int Fc = block_sum(nfail, sh.sum, sslot);   // barrier inside: decay writes are visible in the CTA
      sslot ^= 1;
      if (threadIdx.x < NMS_CL) cl_st(cl_map(smem_addr_u32(&cs.cnt[rank]), (int)threadIdx.x), (uint32_t)Fc);
      cl_sync();
      int F = 0, before = 0;
#pragma unroll
      for (int c = 0; c < NMS_CL; ++c) { const int v = cs.cnt[c]; F += v; before += (c < rank) ? v : 0; }
      if (F == 0) continue;                            // (uniform over the cluster)
      // 4. "swap with last, shrink": holes = failed positions below the new end, ranked in ascending order; the k-th hole
      //    receives the k-th survivor counted from the old end backwards
      const int lo = max(i + 1, base), L = max(hi - lo, 0), new_n = nsegs - F;
      const int chunk = (L + NMS_THREADS - 1) / NMS_THREADS;
      const int cb = lo + threadIdx.x * chunk;
      const int ce = min(cb + chunk, hi);
      int cnt = 0;
      for (int p = cb; p < ce; ++p) cnt += (sc[p - base] < min_score) ? 1 : 0;
      int inc = cnt;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
      if (lane == 31) sh.scan[w] = inc;
      __syncthreads();
      int wbase = before;
      for (int q = 0; q < w; ++q) wbase += sh.scan[q];
      int run = wbase + inc - cnt;                     // failures strictly before this chunk, over the whole list
      int run_hi = run;                                // ... and strictly before max(cb, new_n)
      for (int p = cb; p < ce; ++p) {
        const bool fail = sc[p - base] < min_score;
        if (fail && p < new_n) hole[run] = p;
        run += fail ? 1 : 0;
        if (p < new_n) run_hi = run;
      }
      cl_sync();                                       // the hole list (global memory) is complete
      // remote stores fill holes (< new_n) while other threads still scan: read positions >= new_n only
      run = run_hi;
      for (int p = max(cb, new_n); p < ce; ++p) {
        const int o = p - base;
        const bool fail = sc[o] < min_score;
        run += fail ? 1 : 0;                           // inclusive failure count through p
        if (!fail && p >= new_n) {
          const int rank_desc = (nsegs - 1 - p) - (F - run);
          const int dst = __ldcg(hole + rank_desc);    // (written by another SM: bypass L1)
          const int dr = dst / S, dof = dst - dr * S;
          cl_st(cl_map(smem_addr_u32(x1 + dof), dr), __float_as_uint(x1[o]));
          cl_st(cl_map(smem_addr_u32(x2 + dof), dr), __float_as_uint(x2[o]));
          cl_st(cl_map(smem_addr_u32(sc + dof), dr), __float_as_uint(sc[o]));
          cl_st(cl_map(smem_addr_u32(ar + dof), dr), __float_as_uint(ar[o]));
          cl_st(cl_map(smem_addr_u32(id + dof), dr), (uint32_t)id[o]);
        }
      }
      cl_sync();                                       // moves have landed before the next argmax
      nsegs = new_n;
    }
    k = i;
  }
  if (rank == 0 && threadIdx.x == 0) *out_count = k;
  cl_sync();                                           // no CTA exits while its shared memory may still be written remotely
}

// ---------------------------------------------------------------------------------------------
// decode (av_fd_no_recon.py:775-823), one CTA per video; levels are processed in order.
// logits [B, P] (P = sum of T_l, level-major within a video), offsets [B, P, 2], mask [B, P] (u8).
// Output candidates in the reference's order: level by level, within a level by descending
// probability (ties by ascending point index), after the pre_nms_topk cut and the duration cut.
// ---------------------------------------------------------------------------------------------
constexpr int DEC_MAX_T = 2048;        // largest level length handled by the in-smem bitonic sort

struct DecodeParams {
  const float* logits; const float* offsets; const unsigned char* mask;
  const int* valid_len;            // [B], used when mask == nullptr: point t of level l is kept iff t * stride_l < valid
  int B, P, n_levels;
  int lvl_off[AVDF_MAX_LEVELS]; int lvl_len[AVDF_MAX_LEVELS]; float lvl_stride[AVDF_MAX_LEVELS];
  float pre_nms_thresh; int pre_nms_topk; float duration_thresh;
  float* cand_segs; float* cand_scores; int* cand_count;   // [B,P,2], [B,P], [B]
};

__device__ int decode_block(const DecodeParams& d, int b, float* key, int* val, float* o_segs, float* o_scores) {
  // key/val: smem [DEC_MAX_T]; returns candidate count
  __shared__ int s_count, s_base;
  if (threadIdx.x == 0) s_base = 0;
  __syncthreads();
  for (int l = 0; l < d.n_levels; ++l) {
    const int T = d.lvl_len[l], off = d.lvl_off[l];
    int npow = 1; while (npow < T) npow <<= 1;
    const float stride = d.lvl_stride[l];
    for (int t = threadIdx.x; t < npow; t += blockDim.x) {
      float p = -1.f;        // sentinel below any probability
      if (t < T) {
        float lg = d.logits[(size_t)b * d.P + off + t];
        const bool keep = d.mask ? d.mask[(size_t)b * d.P + off + t] != 0 : __fmul_rn((float)t, stride) < (float)d.valid_len[b];
        float m = keep ? 1.f : 0.f;
        float pr = __fmul_rn(__fdiv_rn(1.f, __fadd_rn(1.f, expf(-lg))), m);
        p = (pr > d.pre_nms_thresh) ? pr : -1.f;
      }
      key[t] = p; val[t] = t;
    }
    __syncthreads();
    // bitonic sort, descending by key then ascending by val
    for (int k = 2; k <= npow; k <<= 1) {
      for (int j = k >> 1; j > 0; j >>= 1) {
        for (int t = threadIdx.x; t < npow; t += blockDim.x) {
          int u = t ^ j;
          if (u > t) {
            float ka = key[t], kb = key[u]; int va = val[t], vb = val[u];
            bool a_first = (ka > kb) || (ka == kb && va < vb);     // a precedes b in the wanted order
            bool up = ((t & k) == 0);
            if (up ? !a_first : a_first) { key[t] = kb; key[u] = ka; val[t] = vb; val[u] = va; }
          }
        }
        __syncthreads();
      }
    }
    // keep the first min(topk, #valid) entries, then the duration filter, in order (stable compaction)
    if (threadIdx.x == 0) s_count = 0;
    __syncthreads();
    const int base = s_base;
    for (int t0 = 0; t0 < npow; t0 += blockDim.x) {
      int t = t0 + threadIdx.x;
      bool ok = false; float left = 0.f, right = 0.f, pr = 0.f;
      if (t < npow && t < d.pre_nms_topk && key[t] > 0.f) {
        int pt = val[t];
        pr = key[t];
        float o0 = d.offsets[((size_t)b * d.P + off + pt) * 2 + 0];
        float o1 = d.offsets[((size_t)b * d.P + off + pt) * 2 + 1];
        float tt = __fmul_rn((float)pt, stride);
        left = __fsub_rn(tt, __fmul_rn(o0, stride));
        right = __fadd_rn(tt, __fmul_rn(o1, stride));
        ok = __fsub_rn(right, left) > d.duration_thresh;
      }
      // ordered compaction: warp ballot + per-chunk running base
      unsigned bal = __ballot_sync(0xffffffffu, ok);
      __shared__ int wcnt[32];
      const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
      if (lane == 0) wcnt[w] = __popc(bal);
      __syncthreads();
      int before = 0;
      for (int q = 0; q < w; ++q) before += wcnt[q];
      int total = 0;
      for (int q = 0; q < (int)(blockDim.x >> 5); ++q) total += wcnt[q];
      int cur = s_count;
      if (ok) {
        int dst = base + cur + before + __popc(bal & ((1u << lane) - 1u));
        o_segs[2 * dst] = left; o_segs[2 * dst + 1] = right; o_scores[dst] = pr;
      }
      __syncthreads();
      if (threadIdx.x == 0) s_count = cur + total;
      __syncthreads();
    }
    if (threadIdx.x == 0) s_base = base + s_count;
    __syncthreads();
  }
  return s_base;
}

// ---------------------------------------------------------------------------------------------
// batched_nms of one video (nms.py:103-190, class-agnostic) from its decoded candidates: hard NMS (with NMSop's score
// filter) or soft NMS, then seg_voting against ALL candidates. Shared by postprocess_kernel and postprocess_sweep_kernel.
// ---------------------------------------------------------------------------------------------
struct PickShared {    // the picks of one video: boundaries (voted when voting is on), scores, candidate index
  float p_x1[AVDF_MAX_SEGS], p_x2[AVDF_MAX_SEGS], p_sc[AVDF_MAX_SEGS];
  float dets[3 * AVDF_MAX_SEGS];
  int idx[AVDF_MAX_SEGS];
};

// c: working arrays (shared memory or global workspace) of capacity >= n; all_segs / all_scores [n]: the candidates.
// Returns the number of picks k <= K in ps (in pick order).
__device__ int nms_vote_block(const Cand& c, const float* all_segs, const float* all_scores, int n, bool soft, int method,
                              float iou_thr, float min_score, float sigma, float voting_thresh, int K, PickShared& ps,
                              NmsShared& sh) {
  float* p_x1 = ps.p_x1; float* p_x2 = ps.p_x2; float* p_sc = ps.p_sc;
  float* dets_sh = ps.dets; int* idx_sh = ps.idx;
  int k = 0;
  if (n > 0) {
    if (!soft) {
      // NMSop: score filter first (nms.py:15-21), order preserved
      for (int p = threadIdx.x; p < n; p += NMS_THREADS) {
        float a = all_segs[2 * p], e = all_segs[2 * p + 1], s = all_scores[p];
        c.x1[p] = a; c.x2[p] = e; c.sc[p] = s; c.ar[p] = __fadd_rn(__fsub_rn(e, a), 1e-6f);
        bool keep = (min_score > 0.f) ? (s > min_score) : true;
        c.id[p] = keep ? p : ~p;
      }
      __syncthreads();
      k = hard_nms_block(c, n, iou_thr, K, idx_sh, sh);
      __syncthreads();
      for (int q = threadIdx.x; q < k; q += NMS_THREADS) {
        int p = idx_sh[q];
        p_x1[q] = c.x1[p]; p_x2[q] = c.x2[p]; p_sc[q] = c.sc[p];
      }
    } else {
      for (int p = threadIdx.x; p < n; p += NMS_THREADS) {
        float a = all_segs[2 * p], e = all_segs[2 * p + 1];
        c.x1[p] = a; c.x2[p] = e; c.sc[p] = all_scores[p]; c.ar[p] = __fadd_rn(__fsub_rn(e, a), 1e-6f);
        c.id[p] = p;
      }
      __syncthreads();
      k = soft_nms_block(c, n, iou_thr, sigma, min_score, method, K, dets_sh, idx_sh, sh);
      __syncthreads();
      for (int q = threadIdx.x; q < k; q += NMS_THREADS) {
        p_x1[q] = dets_sh[3 * q]; p_x2[q] = dets_sh[3 * q + 1]; p_sc[q] = dets_sh[3 * q + 2];
      }
    }
    __syncthreads();
    // seg_voting (nms.py:67-101) against ALL candidates, one warp per pick
    if (voting_thresh > 0.f && k > 0) {
      const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
      for (int q = w; q < k; q += NMS_WARPS) {
        const float a0 = p_x1[q], a1 = p_x2[q], la = __fsub_rn(a1, a0);
        float sw = 0.f;
        for (int j = lane; j < n; j += 32) {
          float b0 = all_segs[2 * j], b1 = all_segs[2 * j + 1];
          float inter = fmaxf(__fsub_rn(fminf(a1, b1), fmaxf(a0, b0)), 0.f);
          float iou = __fdiv_rn(inter, __fsub_rn(__fadd_rn(la, __fsub_rn(b1, b0)), inter));
          float wgt = __fmul_rn(__fmul_rn((iou >= voting_thresh) ? 1.f : 0.f, all_scores[j]), iou);
          sw += wgt;
        }
        sw = warp_sum(sw);
        float s0 = 0.f, s1 = 0.f;
        for (int j = lane; j < n; j += 32) {
          float b0 = all_segs[2 * j], b1 = all_segs[2 * j + 1];
          float inter = fmaxf(__fsub_rn(fminf(a1, b1), fmaxf(a0, b0)), 0.f);
          float iou = __fdiv_rn(inter, __fsub_rn(__fadd_rn(la, __fsub_rn(b1, b0)), inter));
          float wgt = __fmul_rn(__fmul_rn((iou >= voting_thresh) ? 1.f : 0.f, all_scores[j]), iou);
          wgt = __fdiv_rn(wgt, sw);
          s0 = fmaf(wgt, b0, s0); s1 = fmaf(wgt, b1, s1);
        }
        s0 = warp_sum(s0); s1 = warp_sum(s1);
        __syncwarp();
        if (lane == 0) { dets_sh[3 * q] = s0; dets_sh[3 * q + 1] = s1; }
      }
      __syncthreads();
      for (int q = threadIdx.x; q < k; q += NMS_THREADS) { p_x1[q] = dets_sh[3 * q]; p_x2[q] = dets_sh[3 * q + 1]; }
      __syncthreads();
    }
  }
  return k;
}

struct VideoMeta { bool to_sec; float st, hn, fps, dur; };
__device__ __forceinline__ VideoMeta video_meta(const float* stride, const float* half_nframes, const float* fps,
                                                const float* duration, int b) {
  VideoMeta m; m.to_sec = fps != nullptr; m.st = 1.f; m.hn = 0.f; m.fps = 1.f; m.dur = 0.f;
  if (m.to_sec) { m.st = stride[b]; m.hn = half_nframes[b]; m.fps = fps[b]; m.dur = duration[b]; }
  return m;
}

// final stable sort by score desc + cap (nms.py:184-189): rank by counting (k <= AVDF_MAX_SEGS), then feature grid ->
// seconds with the reference's clamping (av_fd_no_recon.py:860-865). o_segs [k, 2] / o_scores [k] in output order.
__device__ void rank_seconds_block(const PickShared& ps, int k, const VideoMeta& m, float* o_segs, float* o_scores,
                                   int* out_index) {
  const float* p_sc = ps.p_sc;
  for (int q = threadIdx.x; q < k; q += NMS_THREADS) {
    float s = p_sc[q];
    int rank = 0;
    for (int r = 0; r < k; ++r) rank += (p_sc[r] > s || (p_sc[r] == s && r < q)) ? 1 : 0;
    float v0 = ps.p_x1[q], v1 = ps.p_x2[q];
    if (m.to_sec) {
      v0 = __fdiv_rn(__fadd_rn(__fmul_rn(v0, m.st), m.hn), m.fps);
      v1 = __fdiv_rn(__fadd_rn(__fmul_rn(v1, m.st), m.hn), m.fps);
      if (v0 <= 0.f) v0 = __fmul_rn(v0, 0.f);
      if (v1 <= 0.f) v1 = __fmul_rn(v1, 0.f);
      if (v0 >= m.dur) v0 = __fadd_rn(__fmul_rn(v0, 0.f), m.dur);
      if (v1 >= m.dur) v1 = __fadd_rn(__fmul_rn(v1, 0.f), m.dur);
    }
    o_segs[2 * rank] = v0; o_segs[2 * rank + 1] = v1; o_scores[rank] = s;
    if (out_index) out_index[rank] = ps.idx[q];
  }
}

// ---------------------------------------------------------------------------------------------
// fused postprocess: [decode ->] hard/soft NMS -> voting -> sort desc + cap -> seconds + clamp
// ---------------------------------------------------------------------------------------------
struct PostParams {
  DecodeParams dec;                // dec.logits == nullptr: candidates are given
  const float* cand_segs; const float* cand_scores; const int* cand_count; int cand_cap;   // [B,cap,2],[B,cap],[B]
  float iou_thr, min_score, sigma, voting_thresh; int max_num, soft, method;
  const float* vid_stride; const float* vid_half_nframes; const float* vid_fps; const float* vid_duration;  // [B] or null
  float* out_segs; float* out_scores; int* out_count;   // [B,max_num,2], [B,max_num], [B]
  void* gws; size_t gws_per_video;                       // used when candidates exceed NMS_SMEM_CAP
  float* rec_ring; unsigned* rec_counter; int rec_cap; const int* vid_index; const float* vid_cls;   // optional result records
  int* out_index;                                        // optional [B, max_num]: candidate index of every output
};

__global__ void __launch_bounds__(NMS_THREADS, 1) postprocess_kernel(const PostParams prm) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ NmsShared sh;
  __shared__ int s_n;
  const int b = blockIdx.x;
  const int cap = prm.cand_cap;
  float* all_segs; float* all_scores; int n;
  if (prm.dec.logits != nullptr) {
    // decode into the global candidate buffers (they are also the voting set)
    all_segs = prm.dec.cand_segs + (size_t)b * cap * 2;
    all_scores = prm.dec.cand_scores + (size_t)b * cap;
    float* key = reinterpret_cast<float*>(smem_raw);
    int* val = reinterpret_cast<int*>(key + DEC_MAX_T);
    int cnt = decode_block(prm.dec, b, key, val, all_segs, all_scores);
    if (threadIdx.x == 0) { prm.dec.cand_count[b] = cnt; s_n = cnt; }
    __syncthreads();
    n = s_n;
    __threadfence_block();
  } else {
    all_segs = const_cast<float*>(prm.cand_segs) + (size_t)b * cap * 2;
    all_scores = const_cast<float*>(prm.cand_scores) + (size_t)b * cap;
    n = prm.cand_count[b];
  }
  __syncthreads();
  const bool big = n > NMS_SMEM_CAP;
  Cand c = big ? carve(reinterpret_cast<unsigned char*>(prm.gws) + (size_t)b * prm.gws_per_video, n)
               : carve(smem_raw, NMS_SMEM_CAP);
  if (prm.soft < 0) {
    // nms_method 'none' (av_fd_no_recon.py:847-858): every decoded candidate, in decode order, to seconds
    float st = 1.f, hn = 0.f, fps = 1.f, dur = 0.f;
    const bool to_sec = prm.vid_fps != nullptr;
    if (to_sec) { st = prm.vid_stride[b]; hn = prm.vid_half_nframes[b]; fps = prm.vid_fps[b]; dur = prm.vid_duration[b]; }
    for (int q = threadIdx.x; q < n; q += NMS_THREADS) {
      float v0 = all_segs[2 * q], v1 = all_segs[2 * q + 1];
      if (to_sec) {
        v0 = __fdiv_rn(__fadd_rn(__fmul_rn(v0, st), hn), fps);
        v1 = __fdiv_rn(__fadd_rn(__fmul_rn(v1, st), hn), fps);
        if (v0 <= 0.f) v0 = __fmul_rn(v0, 0.f);
        if (v1 <= 0.f) v1 = __fmul_rn(v1, 0.f);
        if (v0 >= dur) v0 = __fadd_rn(__fmul_rn(v0, 0.f), dur);
        if (v1 >= dur) v1 = __fadd_rn(__fmul_rn(v1, 0.f), dur);
      }
      prm.out_segs[((size_t)b * cap + q) * 2] = v0; prm.out_segs[((size_t)b * cap + q) * 2 + 1] = v1;
      prm.out_scores[(size_t)b * cap + q] = all_scores[q];
    }
    if (threadIdx.x == 0) prm.out_count[b] = n;
    return;
  }
  const int K = prm.max_num;
  // pick buffers live after the candidate arrays' hole[] region is no longer needed -> use out_* directly
  float* o_segs = prm.out_segs + (size_t)b * K * 2;
  float* o_scores = prm.out_scores + (size_t)b * K;
  __shared__ PickShared ps;
  const int k = nms_vote_block(c, all_segs, all_scores, n, prm.soft != 0, prm.method, prm.iou_thr, prm.min_score, prm.sigma,
                               prm.voting_thresh, K, ps, sh);
  VideoMeta vm = video_meta(prm.vid_stride, prm.vid_half_nframes, prm.vid_fps, prm.vid_duration, b);
  rank_seconds_block(ps, k, vm, o_segs, o_scores, prm.out_index ? prm.out_index + (size_t)b * K : nullptr);
  if (threadIdx.x == 0) prm.out_count[b] = k;
  if (prm.rec_ring != nullptr) {
    // one fixed-size record per video into the ring: [index, count, video_cls, scores[K], segs[K][2]]
    __shared__ unsigned s_row;
    __syncthreads();                                   // this CTA's o_segs / o_scores writes are visible to the block
    if (threadIdx.x == 0) s_row = atomicAdd(prm.rec_counter, 1u) % (unsigned)prm.rec_cap;
    __syncthreads();
    float* rec = prm.rec_ring + (size_t)s_row * (3 + 3 * K);
    if (threadIdx.x == 0) {
      rec[0] = prm.vid_index ? (float)prm.vid_index[b] : (float)b;
      rec[1] = (float)k;
      rec[2] = prm.vid_cls ? prm.vid_cls[b] : 0.f;
    }
    for (int q = threadIdx.x; q < K; q += NMS_THREADS) {
      const bool live = q < k;
      rec[3 + q] = live ? o_scores[q] : 0.f;
      rec[3 + K + 2 * q] = live ? o_segs[2 * q] : 0.f;
      rec[3 + K + 2 * q + 1] = live ? o_segs[2 * q + 1] : 0.f;
    }
  }
}

static size_t nms_smem_bytes() { return (size_t)NMS_SMEM_CAP * 6 * sizeof(float); }

// ---------------------------------------------------------------------------------------------
// postprocess sweep: many test_cfg settings over the same dense outputs. One CTA per video (persistent over the batch);
// the settings arrive sorted by decode group (equal pre_nms_thresh / pre_nms_topk / duration_thresh): the CTA decodes
// once per group into its workspace slice and runs every NMS setting of the group from that list, with the same device
// functions as postprocess_kernel. The candidate arrays are sized to the pyramid (not NMS_SMEM_CAP), so two CTAs fit on
// an SM where postprocess_kernel fits one. A decoded list never exceeds the shared-memory capacity: decode takes levels
// of <= DEC_MAX_T points, and a pyramid of halving levels holds < 2 * DEC_MAX_T points.
// ---------------------------------------------------------------------------------------------
constexpr int SWEEP_MAX = 64;            // settings per launch
constexpr int SWEEP_MAX_CTAS = 1024;     // persistent grid: the workspace holds one candidate list per CTA
constexpr int SWEEP_MIN_BLOCKS = 2;
struct SweepDecode { float pre_nms_thresh; int pre_nms_topk; float duration_thresh; };
struct SweepSetting { float iou_thr, min_score, sigma, voting_thresh; int max_num, soft, group, row; };
struct SweepParams {
  DecodeParams dec;                      // logits / offsets / valid_len / levels (thresholds come from grp[])
  SweepDecode grp[SWEEP_MAX]; int n_groups;
  SweepSetting set[SWEEP_MAX]; int n_set;        // sorted by group; set[i].row = the setting's index in the caller's table
  const float* vid_stride; const float* vid_half_nframes; const float* vid_fps; const float* vid_duration;
  const float* vid_cls; const int* vid_index;
  float* out_rows; long long rows_per_setting; int row_k;
  void* ws; size_t ws_per_cta; int cap_sh;       // cap_sh: capacity of the shared-memory candidate arrays (>= P)
};
static_assert(2 * DEC_MAX_T <= NMS_SMEM_CAP, "a decoded pyramid must fit the shared-memory candidate arrays");

static size_t sweep_ws_per_cta(int P) { return ((size_t)P * 3 * sizeof(float) + 255) / 256 * 256; }   // segments [P, 2] + scores [P]

__global__ void __launch_bounds__(NMS_THREADS, SWEEP_MIN_BLOCKS) postprocess_sweep_kernel(const SweepParams prm) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ NmsShared sh;
  __shared__ PickShared ps;
  __shared__ int s_n;
  const int P = prm.dec.P, K = prm.row_k, rec_len = 3 + 3 * prm.row_k;
  unsigned char* ws = reinterpret_cast<unsigned char*>(prm.ws) + (size_t)blockIdx.x * prm.ws_per_cta;
  float* all_segs = reinterpret_cast<float*>(ws);
  float* all_scores = all_segs + 2 * (size_t)P;
  float* key = reinterpret_cast<float*>(smem_raw);
  int* val = reinterpret_cast<int*>(key + DEC_MAX_T);
  for (int b = blockIdx.x; b < prm.dec.B; b += gridDim.x) {
    const long long row = prm.vid_index ? prm.vid_index[b] : b;
    const bool row_ok = row >= 0 && row < prm.rows_per_setting;
    const VideoMeta vm = video_meta(prm.vid_stride, prm.vid_half_nframes, prm.vid_fps, prm.vid_duration, b);
    const float vcls = prm.vid_cls ? prm.vid_cls[b] : 0.f;
    int si = 0;
    for (int g = 0; g < prm.n_groups; ++g) {
      DecodeParams d = prm.dec;
      d.pre_nms_thresh = prm.grp[g].pre_nms_thresh; d.pre_nms_topk = prm.grp[g].pre_nms_topk;
      d.duration_thresh = prm.grp[g].duration_thresh;
      __syncthreads();                                 // the previous setting is done with smem_raw / the candidates
      const int cnt = decode_block(d, b, key, val, all_segs, all_scores);
      if (threadIdx.x == 0) s_n = cnt;
      __syncthreads();
      const int n = s_n;
      __threadfence_block();
      const Cand c = carve(smem_raw, prm.cap_sh);
      for (; si < prm.n_set && prm.set[si].group == g; ++si) {
        const SweepSetting& st = prm.set[si];
        __syncthreads();                               // the previous setting's tail is done with ps
        const int k = nms_vote_block(c, all_segs, all_scores, n, st.soft != 0, 2, st.iou_thr, st.min_score, st.sigma,
                                     st.voting_thresh, st.max_num, ps, sh);
        if (!row_ok) continue;
        float* rec = prm.out_rows + ((size_t)st.row * prm.rows_per_setting + row) * rec_len;
        rank_seconds_block(ps, k, vm, rec + 3 + K, rec + 3, nullptr);
        if (threadIdx.x == 0) { rec[0] = (float)row; rec[1] = (float)k; rec[2] = vcls; }
        for (int q = k + threadIdx.x; q < K; q += NMS_THREADS) { rec[3 + q] = 0.f; rec[3 + K + 2 * q] = 0.f; rec[3 + K + 2 * q + 1] = 0.f; }
      }
    }
  }
}

}  // namespace avdf

using namespace avdf;

static bool g_nms_cluster = !(getenv("AVDF_NMS_CLUSTER") && atoi(getenv("AVDF_NMS_CLUSTER")) == 0);
// Debug / test hook: lists longer than the shared-memory capacity run on a cluster of CTAs (1, default) or on one CTA from
// the global workspace (0). Returns the previous setting.
extern "C" __attribute__((visibility("default"))) int avdf_debug_nms_cluster(int on) {
  const int prev = g_nms_cluster ? 1 : 0;
  g_nms_cluster = on != 0;
  return prev;
}

extern "C" size_t avdf_nms_workspace_bytes(int32_t n) {
  return n > NMS_SMEM_CAP ? (size_t)n * 6 * sizeof(float) : 0;
}

static int launch_standalone(const float* segs, const float* scores, int32_t n, float thr, float sigma,
                             float min_score, int method, int32_t max_num, float* dets, int64_t* out_idx,
                             int32_t* out_count, void* ws, size_t ws_bytes, void* stream) {
  AVDF_CHECK_ARG(n >= 0, "n < 0");
  AVDF_CHECK_ARG(out_count != nullptr, "out_count is null");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (n == 0) { AVDF_CUDA(cudaMemsetAsync(out_count, 0, sizeof(int32_t), st)); return AVDF_OK; }
  AVDF_CHECK_ARG(segs && scores && out_idx, "null pointer");
  const int use_gws = n > NMS_SMEM_CAP;
  if (use_gws) AVDF_CHECK_ARG(ws != nullptr && ws_bytes >= avdf_nms_workspace_bytes(n), "workspace too small");
  if (use_gws && g_nms_cluster && n <= NMS_CL * NMS_CL_SLICE_MAX) {
    // one cluster of NMS_CL CTAs, the working arrays distributed over their shared memory
    const int S = ((n + NMS_CL - 1) / NMS_CL + 31) / 32 * 32;
    const size_t smem = (size_t)S * 5 * sizeof(float);
    static avdf::DeviceOnce once;
    const int dev = avdf::current_device();
    if (!once.done(dev)) {
      AVDF_CUDA(cudaFuncSetAttribute(nms_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)((size_t)NMS_CL_SLICE_MAX * 5 * sizeof(float))));
      AVDF_CUDA(cudaFuncSetAttribute(nms_cluster_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
      once.mark(dev);
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(NMS_CL); cfg.blockDim = dim3(NMS_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = NMS_CL; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    // a device (or partition) that cannot co-schedule NMS_CL such CTAs in one cluster takes the single-CTA path below
    // (asked once per device, for the largest slice: the query is a host-side driver call of its own)
    static int cluster_ok[64];              // 0 unknown, 1 yes, -1 no
    int max_clusters = dev >= 0 && dev < 64 ? cluster_ok[dev] : 0;
    if (max_clusters == 0) {
      cudaLaunchConfig_t probe = cfg;
      probe.dynamicSmemBytes = (size_t)NMS_CL_SLICE_MAX * 5 * sizeof(float);
      int n_cl = 0;
      if (cudaOccupancyMaxActiveClusters(&n_cl, nms_cluster_kernel, &probe) != cudaSuccess) { n_cl = 0; (void)cudaGetLastError(); }
      max_clusters = n_cl >= 1 ? 1 : -1;
      if (dev >= 0 && dev < 64) cluster_ok[dev] = max_clusters;
    }
    if (max_clusters >= 1) {
      const cudaError_t e = cudaLaunchKernelEx(&cfg, nms_cluster_kernel, segs, scores, (int)n, S, thr, sigma, min_score, method, (int)max_num,
                                               dets, reinterpret_cast<long long*>(out_idx), out_count, reinterpret_cast<int*>(ws));
      if (e != cudaSuccess) { set_error("nms_cluster_kernel: launch failed: %s", cudaGetErrorString(e)); return AVDF_ERR_CUDA; }
      return check_launch("nms_cluster_kernel");
    }
  }
  AVDF_SMEM_ATTR_ONCE(nms_standalone_kernel, nms_smem_bytes());
  nms_standalone_kernel<<<1, NMS_THREADS, use_gws ? 0 : nms_smem_bytes(), st>>>(
      segs, scores, n, thr, sigma, min_score, method, max_num, dets, reinterpret_cast<long long*>(out_idx),
      out_count, ws, use_gws);
  return check_launch("nms_standalone_kernel");
}

extern "C" int avdf_nms_hard(const float* segs, const float* scores, int32_t n, float iou_threshold,
                             int32_t max_num, int64_t* out_idx, int32_t* out_count, void* workspace,
                             size_t workspace_bytes, void* stream) {
  return launch_standalone(segs, scores, n, iou_threshold, 0.f, 0.f, -1, max_num, nullptr, out_idx, out_count,
                           workspace, workspace_bytes, stream);
}

extern "C" int avdf_nms_soft(const float* segs, const float* scores, int32_t n, float* dets, float iou_threshold,
                             float sigma, float min_score, int32_t method, int32_t max_num, int64_t* out_idx,
                             int32_t* out_count, void* workspace, size_t workspace_bytes, void* stream) {
  AVDF_CHECK_ARG(method >= 0 && method <= 2, "method must be 0, 1 or 2");
  AVDF_CHECK_ARG(n == 0 || dets != nullptr, "dets is null");
  return launch_standalone(segs, scores, n, iou_threshold, sigma, min_score, method, max_num, dets, out_idx,
                           out_count, workspace, workspace_bytes, stream);
}

extern "C" size_t avdf_postprocess_workspace_bytes(int32_t batch, int32_t cand_cap) {
  return cand_cap > NMS_SMEM_CAP ? (size_t)batch * cand_cap * 6 * sizeof(float) : 0;
}

extern "C" int avdf_postprocess(const avdf_postprocess_args* a, void* stream) {
  AVDF_CHECK_ARG(a != nullptr, "args is null");
  AVDF_CHECK_ARG(a->batch >= 0, "batch < 0");
  AVDF_CHECK_ARG(a->max_seg_num > 0 && a->max_seg_num <= AVDF_MAX_SEGS, "max_seg_num out of range");
  AVDF_CHECK_ARG(a->out_segs && a->out_scores && a->out_count, "null output");
  if (a->batch == 0) return AVDF_OK;
  PostParams p{};
  p.cand_cap = a->cand_cap;
  if (a->logits != nullptr) {
    AVDF_CHECK_ARG(a->offsets && a->mask && a->cand_segs && a->cand_scores && a->cand_count, "decode needs offsets/mask/cand buffers");
    AVDF_CHECK_ARG(a->n_levels > 0 && a->n_levels <= AVDF_MAX_LEVELS, "n_levels out of range");
    DecodeParams& d = p.dec;
    d.logits = a->logits; d.offsets = a->offsets; d.mask = a->mask;
    d.B = a->batch; d.n_levels = a->n_levels;
    int off = 0;
    for (int l = 0; l < a->n_levels; ++l) {
      AVDF_CHECK_ARG(a->level_len[l] > 0 && a->level_len[l] <= DEC_MAX_T, "level length out of range");
      d.lvl_off[l] = off; d.lvl_len[l] = a->level_len[l]; d.lvl_stride[l] = a->level_stride[l];
      off += a->level_len[l];
    }
    d.P = off;
    AVDF_CHECK_ARG(a->cand_cap >= off, "cand_cap smaller than the number of points");
    d.pre_nms_thresh = a->pre_nms_thresh; d.pre_nms_topk = a->pre_nms_topk; d.duration_thresh = a->duration_thresh;
    d.cand_segs = a->cand_segs; d.cand_scores = a->cand_scores; d.cand_count = a->cand_count;
  } else {
    AVDF_CHECK_ARG(a->cand_segs && a->cand_scores && a->cand_count, "null candidate buffers");
    p.cand_segs = a->cand_segs; p.cand_scores = a->cand_scores; p.cand_count = a->cand_count;
  }
  p.iou_thr = a->iou_threshold; p.min_score = a->min_score; p.sigma = a->sigma; p.voting_thresh = a->voting_thresh;
  p.max_num = a->max_seg_num; p.soft = a->use_soft_nms; p.method = a->soft_method;
  AVDF_CHECK_ARG(a->use_soft_nms >= -1 && a->use_soft_nms <= 1, "use_soft_nms must be 0 (hard), 1 (soft) or -1 (no NMS)");
  if (a->rec_ring) {
    AVDF_CHECK_ARG(a->rec_counter && a->rec_cap > 0, "record ring needs a counter and a capacity");
    AVDF_CHECK_ARG(a->use_soft_nms >= 0, "records are written after NMS only");
    p.rec_ring = a->rec_ring; p.rec_counter = a->rec_counter; p.rec_cap = a->rec_cap; p.vid_index = a->vid_index; p.vid_cls = a->vid_cls;
  }
  p.vid_stride = a->vid_feat_stride; p.vid_half_nframes = a->vid_half_nframes; p.vid_fps = a->vid_fps;
  p.vid_duration = a->vid_duration;
  if (p.vid_fps) AVDF_CHECK_ARG(p.vid_stride && p.vid_half_nframes && p.vid_duration, "incomplete video meta arrays");
  p.out_segs = a->out_segs; p.out_scores = a->out_scores; p.out_count = a->out_count;
  p.out_index = a->out_index;
  p.gws = a->workspace;
  p.gws_per_video = (size_t)a->cand_cap * 6 * sizeof(float);
  if (a->cand_cap > NMS_SMEM_CAP)
    AVDF_CHECK_ARG(a->workspace && a->workspace_bytes >= avdf_postprocess_workspace_bytes(a->batch, a->cand_cap), "workspace too small");
  AVDF_SMEM_ATTR_ONCE(postprocess_kernel, nms_smem_bytes());
  postprocess_kernel<<<a->batch, NMS_THREADS, nms_smem_bytes(), reinterpret_cast<cudaStream_t>(stream)>>>(p);
  return check_launch("postprocess_kernel");
}

static int sweep_points(int32_t n_levels, const int32_t* level_len) {
  if (n_levels <= 0 || n_levels > AVDF_MAX_LEVELS) return -1;
  int P = 0;
  for (int l = 0; l < n_levels; ++l) {
    if (level_len[l] <= 0 || level_len[l] > DEC_MAX_T) return -1;
    P += level_len[l];
  }
  return P;
}

extern "C" size_t avdf_postprocess_sweep_workspace_bytes(int32_t batch, int32_t n_points) {
  if (batch <= 0 || n_points <= 0) return 0;
  return (size_t)std::min(batch, SWEEP_MAX_CTAS) * sweep_ws_per_cta(n_points);
}

extern "C" int avdf_postprocess_sweep(const avdf_postprocess_sweep_args* a, void* stream) {
  AVDF_CHECK_ARG(a != nullptr, "args is null");
  AVDF_CHECK_ARG(a->batch >= 0, "batch < 0");
  AVDF_CHECK_ARG(a->n_settings >= 1 && a->n_settings <= SWEEP_MAX, "n_settings must be 1..64");
  AVDF_CHECK_ARG(a->settings != nullptr, "settings is null");
  AVDF_CHECK_ARG(a->row_k >= 1 && a->row_k <= AVDF_MAX_SEGS, "row_k out of range");
  const int P = sweep_points(a->n_levels, a->level_len);
  AVDF_CHECK_ARG(P > 0 && P <= NMS_SMEM_CAP, "n_levels or a level length out of range");
  for (int l = 0; l < a->n_levels; ++l)
    AVDF_CHECK_ARG(std::isfinite(a->level_stride[l]) && a->level_stride[l] > 0.f, "level_stride must be finite and > 0");
  SweepParams p{};
  for (int i = 0; i < a->n_settings; ++i) {
    const avdf_sweep_setting& s = a->settings[i];
    AVDF_CHECK_ARG(std::isfinite(s.pre_nms_thresh) && std::isfinite(s.duration_thresh) && std::isfinite(s.iou_threshold) &&
                   std::isfinite(s.min_score) && std::isfinite(s.sigma) && std::isfinite(s.voting_thresh),
                   "a setting holds a non-finite value");
    AVDF_CHECK_ARG(s.use_soft_nms == 0 || s.use_soft_nms == 1, "use_soft_nms must be 0 (hard) or 1 (soft)");
    AVDF_CHECK_ARG(s.max_seg_num >= 1 && s.max_seg_num <= a->row_k, "max_seg_num must be 1..row_k");
    AVDF_CHECK_ARG(s.pre_nms_topk >= 0, "pre_nms_topk < 0");
    AVDF_CHECK_ARG(!s.use_soft_nms || s.sigma > 0.f, "soft NMS needs sigma > 0");
  }
  AVDF_CHECK_ARG(a->rows_per_setting >= 1 && (a->vid_index != nullptr || a->rows_per_setting >= a->batch),
                 "rows_per_setting smaller than the batch");
  AVDF_CHECK_ARG(a->out_rows != nullptr, "out_rows is null");
  if (a->vid_fps) AVDF_CHECK_ARG(a->vid_feat_stride && a->vid_half_nframes && a->vid_duration, "incomplete video meta arrays");
  if (a->batch == 0) return AVDF_OK;
  AVDF_CHECK_ARG(a->logits && a->offsets && a->valid_len, "logits, offsets and valid_len are required");
  const size_t need = avdf_postprocess_sweep_workspace_bytes(a->batch, P);
  AVDF_CHECK_ARG(a->workspace != nullptr && a->workspace_bytes >= need, "workspace too small");
  // decode groups in order of first appearance; the settings of a group run one after the other from its candidate list
  int n_groups = 0;
  int grp_of[SWEEP_MAX];
  for (int i = 0; i < a->n_settings; ++i) {
    const avdf_sweep_setting& s = a->settings[i];
    int g = 0;
    for (; g < n_groups; ++g)
      if (p.grp[g].pre_nms_thresh == s.pre_nms_thresh && p.grp[g].pre_nms_topk == s.pre_nms_topk &&
          p.grp[g].duration_thresh == s.duration_thresh) break;
    if (g == n_groups) { p.grp[g] = SweepDecode{s.pre_nms_thresh, s.pre_nms_topk, s.duration_thresh}; ++n_groups; }
    grp_of[i] = g;
  }
  p.n_groups = n_groups;
  for (int g = 0; g < n_groups; ++g)
    for (int i = 0; i < a->n_settings; ++i) {
      if (grp_of[i] != g) continue;
      const avdf_sweep_setting& s = a->settings[i];
      p.set[p.n_set++] = SweepSetting{s.iou_threshold, s.min_score, s.sigma, s.voting_thresh, s.max_seg_num, s.use_soft_nms, g, i};
    }
  DecodeParams& d = p.dec;
  d.logits = a->logits; d.offsets = a->offsets; d.mask = nullptr; d.valid_len = a->valid_len;
  d.B = a->batch; d.n_levels = a->n_levels; d.P = P;
  int off = 0;
  for (int l = 0; l < a->n_levels; ++l) {
    d.lvl_off[l] = off; d.lvl_len[l] = a->level_len[l]; d.lvl_stride[l] = a->level_stride[l];
    off += a->level_len[l];
  }
  p.vid_stride = a->vid_feat_stride; p.vid_half_nframes = a->vid_half_nframes; p.vid_fps = a->vid_fps;
  p.vid_duration = a->vid_duration; p.vid_cls = a->vid_cls; p.vid_index = a->vid_index;
  p.out_rows = a->out_rows; p.rows_per_setting = a->rows_per_setting; p.row_k = a->row_k;
  p.ws = a->workspace; p.ws_per_cta = sweep_ws_per_cta(P);
  p.cap_sh = P;
  int max_t = 1;
  for (int l = 0; l < a->n_levels; ++l) { int np2 = 1; while (np2 < a->level_len[l]) np2 <<= 1; max_t = std::max(max_t, np2); }
  // the decode's sort keys (key / val) and the candidate arrays share the dynamic shared memory
  const size_t smem = std::max((size_t)p.cap_sh * 6 * sizeof(float), (size_t)(DEC_MAX_T + max_t) * sizeof(float));
  AVDF_SMEM_ATTR_ONCE(postprocess_sweep_kernel, nms_smem_bytes());
  const int grid = std::min(a->batch, SWEEP_MAX_CTAS);
  postprocess_sweep_kernel<<<grid, NMS_THREADS, smem, reinterpret_cast<cudaStream_t>(stream)>>>(p);
  return check_launch("postprocess_sweep_kernel");
}
