// Host build of the JSON number formatter (csrc/json_format.cuh) for tests/test_json_format.py:
//   json_format_driver <in.u32> <out.txt>
// reads little-endian fp32 bit patterns and writes them as json.dumps writes the list of their float64 widenings:
// "[x, y, ...]".
#include <stdio.h>
#include <stdlib.h>
#include "../audio_visual_deepfake_detection_b200/csrc/json_format.cuh"

int main(int argc, char** argv) {
  if (argc != 3) { fprintf(stderr, "usage: %s in.u32 out.txt\n", argv[0]); return 2; }
  FILE* fi = fopen(argv[1], "rb");
  FILE* fo = fopen(argv[2], "wb");
  if (!fi || !fo) { perror("open"); return 2; }
  static uint32_t in[1 << 16];
  static char buf[(1 << 16) * (AVDF_JSON_NUM_MAX + 2)];
  size_t n, total = 0;
  fputc('[', fo);
  while ((n = fread(in, 4, 1 << 16, fi)) > 0) {
    size_t p = 0;
    for (size_t i = 0; i < n; ++i) {
      if (total + i > 0) { buf[p++] = ','; buf[p++] = ' '; }
      p += avdf_json::format_f32(in[i], buf + p);
    }
    fwrite(buf, 1, p, fo);
    total += n;
  }
  fputc(']', fo);
  fclose(fi);
  return fclose(fo) == 0 ? 0 : 1;
}
