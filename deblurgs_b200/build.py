"""Build libdgs_b200.so in-tree with plain nvcc for sm_100a (no torch headers, no JIT cache).

The library is the product's only native component: hand-written CUDA kernels plus the C-ABI
declared in include/dgs_b200.h.  It is compiled here (nvcc cross-compiles without a GPU) and
travels to the GPU box with the repository snapshot.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "build")
LIB = os.path.join(HERE, "libdgs_b200.so")
SOURCES = ["dgs_forward.cu", "dgs_backward.cu", "dgs_binning.cu", "dgs_api.cu", "dgs_pose.cu", "dgs_knn.cu", "dgs_loss.cu", "dgs_params.cu",
           "dgs_ssim.cu", "dgs_mcmc.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-O3", "-std=c++17", "-Xcompiler", "-fPIC", "-gencode", "arch=compute_100a,code=sm_100a",
         "-lineinfo", "-I" + os.path.join(ROOT, "include"), "-I" + CSRC]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    headers = [os.path.join(CSRC, "dgs_internal.cuh"), os.path.join(ROOT, "include", "dgs_b200.h")]
    jobs = []
    objs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + headers):
            jobs.append([NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o])

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed: %s\n%s\n%s" % (" ".join(cmd), r.stdout, r.stderr))
        if verbose:
            sys.stderr.write(r.stderr)

    if jobs:
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
            list(ex.map(run, jobs))
    if jobs or force or _stale(LIB, objs):
        run([NVCC, "-shared", "-o", LIB] + objs)
    return LIB


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
