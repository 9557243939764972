"""Exhaustive check of the JSON number formatter (csrc/json_format.cuh) over all 2^32 fp32 bit patterns.

    python scripts/json_float_sweep.py [--procs N] [--out result.json]

Builds a small C harness host-side with nvcc that, for every bit pattern, formats the value with the formatter and
with CPython's own `PyOS_double_to_string(x, 'r', 0, Py_DTSF_ADD_DOT_0, NULL)` (the routine behind `float.__repr__`,
through libpython3.12) with json's spelling of the non-finite values, and compares the bytes. The range is split over
N processes, each with its own interpreter. Prints one JSON line: patterns checked, mismatches (with the first few),
the longest finite text and the run time.
"""
import argparse
import json
import os
import subprocess
import sys
import sysconfig
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

HARNESS = r'''
#include <Python.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "json_format.cuh"

int main(int argc, char** argv) {
  const uint64_t lo = strtoull(argv[1], 0, 0), hi = strtoull(argv[2], 0, 0);
  Py_Initialize();
  uint64_t bad = 0;
  int longest = 0;
  char mine[64];
  for (uint64_t b = lo; b < hi; ++b) {
    const uint32_t bits = (uint32_t)b;
    float f;
    memcpy(&f, &bits, 4);
    const double d = (double)f;
    char* ref = NULL;
    const char* want;
    if (d != d) want = "NaN";
    else if (d == 1.0 / 0.0) want = "Infinity";
    else if (d == -1.0 / 0.0) want = "-Infinity";
    else want = ref = PyOS_double_to_string(d, 'r', 0, Py_DTSF_ADD_DOT_0, NULL);
    const int n = avdf_json::format_f32(bits, mine);
    mine[n] = 0;
    if (d == d && d - d == 0 && n > longest) longest = n;
    if (strcmp(mine, want) != 0) {
      if (bad < 8) fprintf(stderr, "0x%08x: got %s want %s\n", bits, mine, want);
      ++bad;
    }
    if (ref) PyMem_Free(ref);
  }
  printf("%llu %d\n", (unsigned long long)bad, longest);
  return 0;
}
'''


def build(tmp):
    src = os.path.join(tmp, "sweep.cu")
    with open(src, "w") as f:
        f.write(HARNESS)
    exe = os.path.join(tmp, "sweep")
    inc = sysconfig.get_paths()["include"]
    libdir = sysconfig.get_config_var("LIBDIR")
    ver = sysconfig.get_config_var("LDVERSION")
    cmd = ["nvcc", "-O2", "-std=c++17", "-I", inc, "-I", os.path.join(ROOT, "audio_visual_deepfake_detection_b200", "csrc"),
           src, "-o", exe, "-L", libdir, "-lpython" + ver, "-Xlinker", "-rpath=" + libdir]
    subprocess.run(cmd, check=True)
    return exe


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--procs", type=int, default=os.cpu_count() or 1)
    ap.add_argument("--lo", type=lambda s: int(s, 0), default=0)
    ap.add_argument("--hi", type=lambda s: int(s, 0), default=1 << 32)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    t0 = time.time()
    with tempfile.TemporaryDirectory() as tmp:
        exe = build(tmp)
        span = args.hi - args.lo
        cuts = [args.lo + span * k // args.procs for k in range(args.procs + 1)]
        procs = [subprocess.Popen([exe, str(cuts[k]), str(cuts[k + 1])], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
                 for k in range(args.procs)]
        bad, longest, errs = 0, 0, []
        for p in procs:
            out, err = p.communicate()
            if p.returncode != 0:
                raise RuntimeError("harness failed: " + err)
            b, n = out.split()
            bad += int(b)
            longest = max(longest, int(n))
            errs += err.splitlines()
    res = {"patterns": span, "range": [hex(args.lo), hex(args.hi)], "mismatches": bad, "first_mismatches": errs[:16],
           "longest_finite_bytes": longest, "procs": args.procs, "seconds": round(time.time() - t0, 1),
           "reference": "CPython %s PyOS_double_to_string(x, 'r', 0, Py_DTSF_ADD_DOT_0)" % sys.version.split()[0]}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    return 0 if bad == 0 else 1


if __name__ == "__main__":
    sys.exit(main())
