/* A C caller of sliding windows on a launch plan, with no Python in the process: include/avdf.h and the CUDA runtime only.
 *
 *   plan_window_driver PLAN INPUT OUTPUT
 *
 * INPUT (little-endian): int32 R; float64 window, hop; per recording: float64 duration, int64 rows[3]; then per present
 * stream (video, byola, emo; channels > 0 in the plan) the rows of all R recordings back to back, in the plan's input dtype.
 * OUTPUT: int32 R, int32 max_seg_num; fp32 segs [R, K, 2]; fp32 scores [R, K]; int32 counts [R]; fp32 video_cls [R].
 * The window block is sized from avdf_plan_window_layout: the windows of this call and the most of any recording. */
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
  int32_t R = 0;
  double window = 0, hop = 0;
  READ(&R, 4, 1);
  READ(&window, 8, 1);
  READ(&hop, 8, 1);
  if (R < 1) return 1;
  double* duration = (double*)malloc(sizeof(double) * R);
  int64_t* rows = (int64_t*)malloc(sizeof(int64_t) * 3 * R);
  for (int r = 0; r < R; ++r) {
    READ(&duration[r], 8, 1);
    READ(&rows[3 * r], 8, 3);
  }
  const size_t es = info.in_dtype == AVDF_DTYPE_F32 ? 4 : 2;
  int64_t total[3] = {0, 0, 0};
  void* host[3] = {NULL, NULL, NULL};
  for (int s = 0; s < 3; ++s) {
    if (info.channels[s] == 0) continue;
    for (int r = 0; r < R; ++r) total[s] += rows[3 * r + s];
    host[s] = malloc((size_t)total[s] * info.channels[s] * es);
    READ(host[s], es * info.channels[s], total[s]);
  }
  fclose(in);

  /* size the window block for this call */
  int32_t n_windows = 0, most = 0;
  for (int r = 0; r < R; ++r) {
    const int32_t n = avdf_plan_window_layout(plan, duration[r], &rows[3 * r], window, hop, 0, NULL, NULL, NULL, NULL);
    if (n < 0) {
      fprintf(stderr, "recording %d: %s\n", r, avdf_last_error());
      return 1;
    }
    n_windows += n;
    if (n > most) most = n;
  }
  const size_t win_bytes = avdf_session_window_bytes(plan, n_windows, most);
  if (win_bytes == 0) {
    fprintf(stderr, "avdf_session_window_bytes: %s\n", avdf_last_error());
    return 1;
  }

  cudaStream_t stream;
  CHECK_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
  void *consts = NULL, *arena = NULL, *win = NULL;
  CHECK_CUDA(cudaMalloc(&consts, info.const_bytes ? info.const_bytes : 1));
  CHECK_CUDA(cudaMalloc(&arena, info.session_bytes));
  CHECK_CUDA(cudaMalloc(&win, win_bytes));
  CHECK_AVDF(avdf_plan_upload(plan, consts, info.const_bytes, stream));
  avdf_session* session = NULL;
  avdf_session_io io;
  CHECK_AVDF(avdf_session_create(plan, arena, info.session_bytes, &session));
  CHECK_AVDF(avdf_session_get_io(session, &io));
  CHECK_AVDF(avdf_session_attach_windows(session, win, win_bytes, n_windows, most));
  for (int s = 0; s < 3; ++s)
    if (host[s])
      CHECK_CUDA(cudaMemcpyAsync(io.streams[s], host[s], (size_t)total[s] * info.channels[s] * es, cudaMemcpyHostToDevice, stream));

  const int K = info.max_seg_num;
  void *d_segs = NULL, *d_scores = NULL, *d_counts = NULL, *d_cls = NULL;
  CHECK_CUDA(cudaMalloc(&d_segs, sizeof(float) * R * K * 2));
  CHECK_CUDA(cudaMalloc(&d_scores, sizeof(float) * R * K));
  CHECK_CUDA(cudaMalloc(&d_counts, sizeof(int32_t) * R));
  CHECK_CUDA(cudaMalloc(&d_cls, sizeof(float) * R));
  avdf_window_run_args a;
  memset(&a, 0, sizeof(a));
  a.n_rec = R;
  a.duration = duration;
  a.rows = rows;
  a.window = window;
  a.hop = hop;
  a.out_segs = (float*)d_segs;
  a.out_scores = (float*)d_scores;
  a.out_count = (int32_t*)d_counts;
  a.out_cls = (float*)d_cls;
  CHECK_AVDF(avdf_session_run_windows(session, &a, stream));

  float* segs = (float*)malloc(sizeof(float) * R * K * 2);
  float* scores = (float*)malloc(sizeof(float) * R * K);
  int32_t* counts = (int32_t*)malloc(sizeof(int32_t) * R);
  float* vcls = (float*)malloc(sizeof(float) * R);
  CHECK_CUDA(cudaMemcpyAsync(segs, d_segs, sizeof(float) * R * K * 2, cudaMemcpyDeviceToHost, stream));
  CHECK_CUDA(cudaMemcpyAsync(scores, d_scores, sizeof(float) * R * K, cudaMemcpyDeviceToHost, stream));
  CHECK_CUDA(cudaMemcpyAsync(counts, d_counts, sizeof(int32_t) * R, cudaMemcpyDeviceToHost, stream));
  CHECK_CUDA(cudaMemcpyAsync(vcls, d_cls, sizeof(float) * R, cudaMemcpyDeviceToHost, stream));
  CHECK_CUDA(cudaStreamSynchronize(stream));

  FILE* out = fopen(argv[3], "wb");
  if (!out) return 1;
  fwrite(&R, 4, 1, out);
  fwrite(&K, 4, 1, out);
  fwrite(segs, sizeof(float), (size_t)R * K * 2, out);
  fwrite(scores, sizeof(float), (size_t)R * K, out);
  fwrite(counts, sizeof(int32_t), R, out);
  fwrite(vcls, sizeof(float), R, out);
  fclose(out);

  avdf_session_destroy(session);
  avdf_plan_close(plan);
  CHECK_CUDA(cudaFree(d_segs));
  CHECK_CUDA(cudaFree(d_scores));
  CHECK_CUDA(cudaFree(d_counts));
  CHECK_CUDA(cudaFree(d_cls));
  CHECK_CUDA(cudaFree(win));
  CHECK_CUDA(cudaFree(arena));
  CHECK_CUDA(cudaFree(consts));
  CHECK_CUDA(cudaStreamDestroy(stream));
  printf("plan_window_driver: %d recordings, %d windows, %s\n", R, n_windows, info.description);
  return 0;
}
