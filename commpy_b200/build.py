"""In-tree build of libcommpy_b200.so for sm_100a (nvcc cross-compiles without a GPU).

    python -m commpy_b200.build [--force] [--verbose]

Objects go to build/, the shared library to commpy_b200/libcommpy_b200.so (git-ignored, but it travels
to the GPU box with the gpurun snapshot)."""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
OBJDIR = os.path.join(ROOT, "build")
LIB = os.path.join(HERE, "libcommpy_b200.so")
SOURCES = ["common.cu", "viterbi.cu", "bcjr.cu", "ldpc.cu", "demap.cu", "count.cu", "pipeline.cu", "hostapi.cu", "txlink.cu", "turbolink.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
         "-Xcompiler", "-fPIC", "--fmad=true"]


def _newer(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    os.makedirs(OBJDIR, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(ROOT, "include", "commpy_b200.h"))
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    objs = []
    jobs = []
    for s in srcs:
        src = os.path.join(CSRC, s)
        obj = os.path.join(OBJDIR, s.replace(".cu", ".o"))
        objs.append(obj)
        if force or _newer(obj, [src] + headers):
            cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
            jobs.append(cmd)

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        if verbose or r.returncode != 0:
            sys.stderr.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed: " + " ".join(cmd))

    with ThreadPoolExecutor(max(1, min(len(jobs), os.cpu_count() or 1))) as ex:
        list(ex.map(run, jobs))
    if force or jobs or _newer(LIB, objs):
        cmd = [NVCC, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a",
                                                     "-Xcompiler", "-fPIC", "-lcudart"]
        run(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
