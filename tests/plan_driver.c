/* A C caller of a launch plan, with no Python in the process: include/avdf.h and the CUDA runtime only.
 *
 *   plan_driver PLAN INPUT OUTPUT
 *
 * INPUT (little-endian): int32 B; per recording: float64 duration, int64 rows[3]; then per present stream (video, byola,
 * emo; channels > 0 in the plan) the rows of all B recordings back to back, in the plan's input dtype.
 * OUTPUT: int32 B, int32 max_seg_num; fp32 segs [B, K, 2]; fp32 scores [B, K]; int32 counts [B]; fp32 video_cls [B].
 * meta is computed with the formula documented in avdf.h. */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <cuda_runtime.h>

#include "avdf.h"

#define CHECK_AVDF(call)                                                        \
  do {                                                                          \
    int rc_ = (call);                                                           \
    if (rc_ != AVDF_OK) {                                                       \
      fprintf(stderr, "%s failed (%d): %s\n", #call, rc_, avdf_last_error());   \
      return 1;                                                                 \
    }                                                                           \
  } while (0)
#define CHECK_CUDA(call)                                                                 \
  do {                                                                                   \
    cudaError_t e_ = (call);                                                             \
    if (e_ != cudaSuccess) {                                                             \
      fprintf(stderr, "%s failed: %s\n", #call, cudaGetErrorString(e_));                 \
      return 1;                                                                          \
    }                                                                                    \
  } while (0)
#define READ(ptr, size, n)                                                   \
  do {                                                                       \
    if (fread(ptr, size, n, in) != (size_t)(n)) {                            \
      fprintf(stderr, "short read of %s\n", #ptr);                           \
      return 1;                                                              \
    }                                                                        \
  } while (0)

int main(int argc, char** argv) {
  if (argc != 4) {
    fprintf(stderr, "usage: %s PLAN INPUT OUTPUT\n", argv[0]);
    return 2;
  }
  avdf_plan* plan = NULL;
  avdf_plan_info info;
  CHECK_AVDF(avdf_plan_open(argv[1], &plan));
  CHECK_AVDF(avdf_plan_get_info(plan, &info));

  FILE* in = fopen(argv[2], "rb");
  if (!in) return 1;
  int32_t B = 0;
  READ(&B, 4, 1);
  if (B < 1 || B > info.max_batch) return 1;
  double* duration = (double*)malloc(sizeof(double) * B);
  int64_t(*rows)[3] = malloc(sizeof(int64_t[3]) * B);
  for (int b = 0; b < B; ++b) {
    READ(&duration[b], 8, 1);
    READ(rows[b], 8, 3);
  }
  const size_t es = info.in_dtype == AVDF_DTYPE_F32 ? 4 : 2;
  int64_t total[3] = {0, 0, 0};
  void* host[3] = {NULL, NULL, NULL};
  int32_t* offsets = (int32_t*)calloc(3 * (info.max_batch + 1), sizeof(int32_t));
  for (int s = 0; s < 3; ++s) {
    if (info.channels[s] == 0) continue;
    for (int b = 0; b < B; ++b) {
      offsets[s * (info.max_batch + 1) + b] = (int32_t)total[s];
      total[s] += rows[b][s];
    }
    offsets[s * (info.max_batch + 1) + B] = (int32_t)total[s];
    host[s] = malloc((size_t)total[s] * info.channels[s] * es);
    READ(host[s], es * info.channels[s], total[s]);
  }
  fclose(in);

  /* meta [4, B]: the documented formula, T = rows of the first present stream among video / byola */
  float* meta = (float*)malloc(sizeof(float) * 4 * B);
  const int first = info.channels[0] ? 0 : 1;
  for (int b = 0; b < B; ++b) {
    const double T = (double)rows[b][first];
    meta[0 * B + b] = (float)(T / info.t_out);
    meta[1 * B + b] = (float)(0.5 * (T / info.t_out));
    meta[2 * B + b] = (float)(T / duration[b]);
    meta[3 * B + b] = (float)duration[b];
  }

  cudaStream_t stream;
  CHECK_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
  void *consts = NULL, *arena = NULL;
  CHECK_CUDA(cudaMalloc(&consts, info.const_bytes ? info.const_bytes : 1));
  CHECK_CUDA(cudaMalloc(&arena, info.session_bytes));
  CHECK_AVDF(avdf_plan_upload(plan, consts, info.const_bytes, stream));
  avdf_session* session = NULL;
  avdf_session_io io;
  CHECK_AVDF(avdf_session_create(plan, arena, info.session_bytes, &session));
  CHECK_AVDF(avdf_session_get_io(session, &io));
  for (int s = 0; s < 3; ++s)
    if (host[s])
      CHECK_CUDA(cudaMemcpyAsync(io.streams[s], host[s], (size_t)total[s] * info.channels[s] * es, cudaMemcpyHostToDevice, stream));
  CHECK_CUDA(cudaMemcpyAsync(io.offsets, offsets, sizeof(int32_t) * 3 * (info.max_batch + 1), cudaMemcpyHostToDevice, stream));
  CHECK_CUDA(cudaMemcpyAsync(io.meta, meta, sizeof(float) * 4 * B, cudaMemcpyHostToDevice, stream));
  CHECK_AVDF(avdf_session_run(session, B, total, stream));

  const int K = info.max_seg_num;
  float* segs = (float*)malloc(sizeof(float) * B * K * 2);
  float* scores = (float*)malloc(sizeof(float) * B * K);
  int32_t* counts = (int32_t*)malloc(sizeof(int32_t) * B);
  float* vcls = (float*)malloc(sizeof(float) * B);
  CHECK_CUDA(cudaMemcpyAsync(segs, io.segs, sizeof(float) * B * K * 2, cudaMemcpyDeviceToHost, stream));
  CHECK_CUDA(cudaMemcpyAsync(scores, io.scores, sizeof(float) * B * K, cudaMemcpyDeviceToHost, stream));
  CHECK_CUDA(cudaMemcpyAsync(counts, io.counts, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, stream));
  CHECK_CUDA(cudaMemcpyAsync(vcls, io.video_cls, sizeof(float) * B, cudaMemcpyDeviceToHost, stream));
  CHECK_CUDA(cudaStreamSynchronize(stream));

  FILE* out = fopen(argv[3], "wb");
  if (!out) return 1;
  fwrite(&B, 4, 1, out);
  fwrite(&K, 4, 1, out);
  fwrite(segs, sizeof(float), (size_t)B * K * 2, out);
  fwrite(scores, sizeof(float), (size_t)B * K, out);
  fwrite(counts, sizeof(int32_t), B, out);
  fwrite(vcls, sizeof(float), B, out);
  fclose(out);

  avdf_session_destroy(session);
  avdf_plan_close(plan);
  CHECK_CUDA(cudaFree(arena));
  CHECK_CUDA(cudaFree(consts));
  CHECK_CUDA(cudaStreamDestroy(stream));
  printf("plan_driver: %d recordings, %s\n", B, info.description);
  return 0;
}
