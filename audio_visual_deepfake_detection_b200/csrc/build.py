"""Build libavdf_sm100.so (the C-ABI library, include/avdf.h) in-tree with nvcc for sm_100a.

    python -m audio_visual_deepfake_detection_b200.csrc.build [--force] [--verbose]

Objects are compiled in parallel (one nvcc per .cu) and linked into
audio_visual_deepfake_detection_b200/csrc/libavdf_sm100.so. The library links the CUDA runtime
statically and resolves the one driver entry point it needs (cuTensorMapEncodeTiled) at run time,
so it loads on a machine without a GPU driver (the CPU test box checks its exported symbols).
"""
import concurrent.futures
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = ["runtime.cu", "interp.cu", "nms.cu", "gemm_simt.cu", "gemm_tc.cu", "mlp_fused.cu", "blocks.cu", "host_pack.cu", "attention_mma.cu", "byola.cu", "eval.cu", "window.cu", "plan.cu", "results.cu"]
LIB = os.path.join(HERE, "libavdf_sm100.so")
OBJ_DIR = os.path.join(HERE, "build")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
          "--expt-relaxed-constexpr", "-Xptxas", "-v"]
# nms.cu restates g++-compiled float code: no fused multiply-add contraction, IEEE div/sqrt; eval.cu restates numpy's fp64
# segment_iou, whose TP / FP decisions must come out bit-identical
PER_FILE = {"nms.cu": ["-fmad=false", "-prec-div=true", "-prec-sqrt=true"], "eval.cu": ["-fmad=false"], "window.cu": ["-fmad=false", "-prec-div=true"],"gemm_tc.cu": (["-DAVDF_GEMM_TIMELINE"] if os.environ.get("AVDF_GEMM_TIMELINE") else []),
            "blocks.cu": os.environ.get("AVDF_BLOCKS_FLAGS", "").split()}


def nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found")
    return exe


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    os.makedirs(OBJ_DIR, exist_ok=True)
    headers = [os.path.join(HERE, f) for f in os.listdir(HERE) if f.endswith(".cuh")]
    headers.append(os.path.join(os.path.dirname(os.path.dirname(HERE)), "include", "avdf.h"))
    jobs = []
    for src in SOURCES:
        s = os.path.join(HERE, src)
        o = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
        if force or _stale(o, [s] + headers):
            jobs.append((s, o, [nvcc(), *ARCH, *COMMON, *PER_FILE.get(src, []), "-c", s, "-o", o]))
    logs = {}

    def run(job):
        s, o, cmd = job
        r = subprocess.run(cmd, capture_output=True, text=True)
        return s, r

    with concurrent.futures.ThreadPoolExecutor(max_workers=max(1, min(len(jobs), os.cpu_count() or 1))) as ex:
        for s, r in ex.map(run, jobs):
            logs[s] = r.stderr + r.stdout
            if r.returncode != 0:
                sys.stderr.write(logs[s])
                raise RuntimeError("nvcc failed on %s" % s)
            if verbose:
                sys.stderr.write(logs[s])
    with open(os.path.join(OBJ_DIR, "ptxas.log"), "a" if not force else "w") as f:
        for s, l in logs.items():
            f.write("==== %s\n%s\n" % (s, l))
    objs = [os.path.join(OBJ_DIR, src.replace(".cu", ".o")) for src in SOURCES]
    if force or jobs or _stale(LIB, objs):
        cmd = [nvcc(), *ARCH, "-shared", "-o", LIB, *objs, "-Xcompiler", "-fPIC", "-cudart", "static"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stderr + r.stdout)
            raise RuntimeError("link failed")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
