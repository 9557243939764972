// K1: fixed-length linear resampling + channel concat of the per-stream features.
//
// Replaces libs/datasets/deepfake_video_audio.py:513-547 (DeepFakeVideoAudioDatasetInfer3.__getitem__:
// F.interpolate(size=max_seq_len, mode='linear', align_corners=False) per stream, torch.cat along C)
// and the [C,T] -> device copy of av_fd_no_recon.py:431-479. Output is token-major [B, T_out, C_total]
// (channel-last: what the conv-GEMM's TMA boxes want), bf16 or fp32.
//
// Index math is ATen's area_pixel_compute_source_index with the two FMAs its vectorised CPU kernel
// executes, so fp32 output is bit-identical to F.interpolate (oracle/interp_ref.py):
//   scale = T_in / T_out (fp32);  src = max(0, fma(scale, t + 0.5, -0.5));  i0 = (int)src
//   i1 = i0 + (i0 < T_in - 1);  l1 = src - i0;  l0 = 1 - l1;  out = fma(l0, x[i0], l1 * x[i1])
//
// HBM-bound streaming kernel: one thread = 8 consecutive channels of a run of output rows (2x float4 loads
// per NEW source row, one 16 B (bf16) or two 16 B (fp32) stores per output row); the threads of a warp are
// contiguous in C so every access is a fully coalesced 128 B+ line. Algorithmic bytes per video:
// 4 * sum_s(T_s * C_s) read + T_out * C_total * sizeof(out) written.
//
// avdf_interp_concat_ranges runs the same kernel on (start, count) row ranges instead of CSR offsets: the overlapping
// windows of a long recording (libs/modeling/windows.py) read one device copy of it.
#include "common.cuh"

namespace avdf {

struct InterpParams {
  const void* src[3];          // packed rows of all videos, per stream: [sum_b T_s(b), C_s], fp32 or bf16 (16-bit feature shards)
  const int* row_off[3];       // [B+1] prefix offsets (rows) per stream, or with row_cnt: [B] first rows
  const int* row_cnt[3];       // null: CSR (rows of video b = [row_off[b], row_off[b+1])); else [B] row counts
  int c[3];                    // channels per stream (0 = stream absent)
  int c_off[3];                // channel offset in the concatenated output
  int c_total, t_out, B;
};

// A thread walks INTERP_ROWS consecutive output rows of its 8-channel group and keeps the two source rows of the current
// interval in registers: with the 2-8x up-sampling of the audio streams (T_in ~ 90-400 -> 768) consecutive output rows
// share their source rows, so a source row is fetched once per run instead of twice per output row. (One thread per
// output row re-read every source row ~2 * 768 / T_in times through L2: 0.55 GB of L2 -> SM traffic for 70 MB of
// sources per 32-video batch, which is what bounded the kernel at 45 % of the HBM roofline.)
constexpr int INTERP_ROWS = 16;

template <typename InT, typename OutT>
__global__ void __launch_bounds__(256) interp_concat_kernel(const InterpParams p, OutT* __restrict__ out) {
  const int groups_per_row = p.c_total >> 3;
  const int chunks_per_video = (p.t_out + INTERP_ROWS - 1) / INTERP_ROWS;
  const long long total = (long long)p.B * chunks_per_video * groups_per_row;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (long long)gridDim.x * blockDim.x) {
    const int cg = (int)(g % groups_per_row);
    const long long chunk = g / groups_per_row;
    const int t_first = (int)(chunk % chunks_per_video) * INTERP_ROWS;
    const int b = (int)(chunk / chunks_per_video);
    const int t_end = min(t_first + INTERP_ROWS, p.t_out);
    const int ch = cg << 3;
    const int s = (ch >= p.c_off[2] && p.c[2] > 0) ? 2 : ((ch >= p.c_off[1] && p.c[1] > 0) ? 1 : 0);
    const int cs = ch - p.c_off[s];
    const int r0 = p.row_off[s][b];
    const int t_in = p.row_cnt[s] ? p.row_cnt[s][b] : p.row_off[s][b + 1] - r0;
    const int cstride = p.c[s];
    const InT* base = static_cast<const InT*>(p.src[s]) + (size_t)r0 * cstride + cs;
    OutT* orow = out + ((size_t)b * p.t_out + t_first) * p.c_total + ch;
    if (t_in == p.t_out) {
      for (int t = t_first; t < t_end; ++t, orow += p.c_total) {
        float v[8];
        Row8<InT>::load(base + (size_t)t * cstride, v);
        Row8<OutT>::store(orow, v);
      }
      continue;
    }
    const float scale = __fdiv_rn((float)t_in, (float)p.t_out);
    float a[8], c[8];
    int h0 = -1, h1 = -1;                 // source rows held in a / c
    for (int t = t_first; t < t_end; ++t, orow += p.c_total) {
      float src = __fmaf_rn(scale, __fadd_rn((float)t, 0.5f), -0.5f);
      src = src < 0.f ? 0.f : src;
      const int i0 = (int)src;
      const int i1 = i0 + (i0 < t_in - 1 ? 1 : 0);
      const float l1 = __fsub_rn(src, (float)i0);
      const float l0 = __fsub_rn(1.f, l1);
      if (i0 != h0) {
        if (i0 == h1) {
#pragma unroll
          for (int k = 0; k < 8; ++k) a[k] = c[k];
        } else {
          Row8<InT>::load(base + (size_t)i0 * cstride, a);
        }
        h0 = i0;
      }
      if (i1 != h1) {
        if (i1 == i0) {
#pragma unroll
          for (int k = 0; k < 8; ++k) c[k] = a[k];
        } else {
          Row8<InT>::load(base + (size_t)i1 * cstride, c);
        }
        h1 = i1;
      }
      float v[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] = __fmaf_rn(l0, a[k], __fmul_rn(l1, c[k]));
      Row8<OutT>::store(orow, v);
    }
  }
}

// preprocessing (libs/modeling/av_fd_no_recon.py:431-479): one video's feats [C, T] fp32 (the dataset item
// layout) -> token-major [L, C] rows of the batch buffer, zero-padded from T to L. 32x32 smem tile transpose:
// reads coalesced along T, writes coalesced along C.
template <typename OutT>
__global__ void __launch_bounds__(256) pack_feats_kernel(const float* __restrict__ in, int C, int T, int L, OutT* __restrict__ out) {
  __shared__ float tile[32][33];
  const int t0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int c = c0 + i, t = t0 + threadIdx.x;
    tile[i][threadIdx.x] = (c < C && t < T) ? in[(size_t)c * T + t] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int t = t0 + i, c = c0 + threadIdx.x;
    if (t < L && c < C) {
      store1(out + (size_t)t * C + c, tile[threadIdx.x][i]);
    }
  }
}

}  // namespace avdf

using namespace avdf;

extern "C" int avdf_pack_feats(const float* feats_ct, int32_t channels, int32_t t, int32_t t_padded, void* out,
                               int32_t out_dtype, void* stream) {
  AVDF_CHECK_ARG(feats_ct && out, "null pointer");
  AVDF_CHECK_ARG(channels > 0 && t > 0 && t_padded >= t, "bad sizes");
  AVDF_CHECK_DTYPE(out_dtype, "out_dtype");
  dim3 grid((t_padded + 31) / 32, (channels + 31) / 32), block(32, 8);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  AVDF_DISPATCH_DTYPE(out_dtype, OutT, (pack_feats_kernel<OutT><<<grid, block, 0, st>>>(feats_ct, channels, t, t_padded, reinterpret_cast<OutT*>(out))));
  return check_launch("pack_feats_kernel");
}

extern "C" int avdf_interp_concat(const float* video, const float* byola, const float* emo,
                                  const int32_t* video_off, const int32_t* byola_off, const int32_t* emo_off,
                                  int32_t batch, int32_t c_video, int32_t c_byola, int32_t c_emo, int32_t t_out,
                                  void* out, int32_t out_dtype, void* stream) {
  return avdf_interp_concat_in(video, byola, emo, AVDF_DTYPE_F32, video_off, byola_off, emo_off, batch, c_video, c_byola, c_emo, t_out,
                               out, out_dtype, stream);
}

static int launch_interp(InterpParams& p, int32_t in_dtype, void* out, int32_t out_dtype, void* stream) {
  const long long total = (long long)p.B * ((p.t_out + INTERP_ROWS - 1) / INTERP_ROWS) * (p.c_total / 8);
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  long long want = (total + 255) / 256;
  int grid = (int)(want < (long long)sms * 16 ? want : (long long)sms * 16);   // grid-stride, 16 CTAs of 256 per SM
  if (grid < 1) grid = 1;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (in_dtype == AVDF_DTYPE_F32) {
    AVDF_DISPATCH_DTYPE(out_dtype, OutT, (interp_concat_kernel<float, OutT><<<grid, 256, 0, st>>>(p, reinterpret_cast<OutT*>(out))));
  } else {
    AVDF_DISPATCH_DTYPE(out_dtype, OutT, (interp_concat_kernel<__nv_bfloat16, OutT><<<grid, 256, 0, st>>>(p, reinterpret_cast<OutT*>(out))));
  }
  return check_launch("interp_concat_kernel");
}

static int interp_params(InterpParams& p, const void* video, const void* byola, const void* emo, int32_t in_dtype,
                         int32_t batch, int32_t c_video, int32_t c_byola, int32_t c_emo, int32_t t_out, void* out, int32_t out_dtype) {
  AVDF_CHECK_ARG(batch >= 0 && t_out > 0, "bad batch / t_out");
  AVDF_CHECK_ARG(in_dtype == AVDF_DTYPE_F32 || in_dtype == AVDF_DTYPE_BF16, "in_dtype must be F32 or BF16");
  AVDF_CHECK_ARG(c_video >= 0 && c_byola >= 0 && c_emo >= 0, "negative channel count");
  AVDF_CHECK_ARG((c_video % 8 | c_byola % 8 | c_emo % 8) == 0, "channel counts must be multiples of 8");
  AVDF_CHECK_ARG(c_video + c_byola + c_emo > 0, "no stream");
  AVDF_CHECK_DTYPE(out_dtype, "out_dtype");
  AVDF_CHECK_ARG((c_video == 0 || video) && (c_byola == 0 || byola) && (c_emo == 0 || emo), "null stream pointer");
  AVDF_CHECK_ARG(out != nullptr, "out is null");
  p.src[0] = video; p.src[1] = byola; p.src[2] = emo;
  p.c[0] = c_video; p.c[1] = c_byola; p.c[2] = c_emo;
  p.c_off[0] = 0; p.c_off[1] = c_video; p.c_off[2] = c_video + c_byola;
  p.c_total = c_video + c_byola + c_emo; p.t_out = t_out; p.B = batch;
  return AVDF_OK;
}

extern "C" int avdf_interp_concat_in(const void* video, const void* byola, const void* emo, int32_t in_dtype,
                                     const int32_t* video_off, const int32_t* byola_off, const int32_t* emo_off,
                                     int32_t batch, int32_t c_video, int32_t c_byola, int32_t c_emo, int32_t t_out,
                                     void* out, int32_t out_dtype, void* stream) {
  InterpParams p{};
  const int rc = interp_params(p, video, byola, emo, in_dtype, batch, c_video, c_byola, c_emo, t_out, out, out_dtype);
  if (rc != AVDF_OK) return rc;
  AVDF_CHECK_ARG((c_video == 0 || video_off) && (c_byola == 0 || byola_off) && (c_emo == 0 || emo_off), "null stream pointer");
  if (batch == 0) return AVDF_OK;
  p.row_off[0] = video_off; p.row_off[1] = byola_off; p.row_off[2] = emo_off;
  return launch_interp(p, in_dtype, out, out_dtype, stream);
}

extern "C" int avdf_interp_concat_ranges(const void* video, const void* byola, const void* emo, int32_t in_dtype,
                                         const int32_t* start, const int32_t* count,
                                         int32_t batch, int32_t c_video, int32_t c_byola, int32_t c_emo, int32_t t_out,
                                         void* out, int32_t out_dtype, void* stream) {
  InterpParams p{};
  const int rc = interp_params(p, video, byola, emo, in_dtype, batch, c_video, c_byola, c_emo, t_out, out, out_dtype);
  if (rc != AVDF_OK) return rc;
  AVDF_CHECK_ARG(start != nullptr && count != nullptr, "null start / count");
  if (batch == 0) return AVDF_OK;
  for (int s = 0; s < 3; ++s) {
    p.row_off[s] = start + (size_t)s * batch;
    p.row_cnt[s] = count + (size_t)s * batch;
  }
  return launch_interp(p, in_dtype, out, out_dtype, stream);
}
