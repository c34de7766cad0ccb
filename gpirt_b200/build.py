"""Builds gpirt_b200/libgpirt_b200.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python -m gpirt_b200.build          # incremental
    python -m gpirt_b200.build --force

nvcc cross-compiles without a GPU, so this runs in the build container; the .so travels to the GPU box."""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "_obj")
LIB = os.path.join(HERE, "libgpirt_b200.so")
SOURCES = ["gemm.cu", "linalg.cu", "kernels.cu", "softplus_table.cu", "theta_int8.cu", "dgemm_i8.cu", "ppc.cu", "comm.cu", "sampler.cu", "capi.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
         "--cudart", "static"]


def _deps():
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hdrs.append(os.path.join(HERE, "..", "include", "gpirt_b200.h"))
    return max(os.path.getmtime(h) for h in hdrs)


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    hdr_time = _deps()
    jobs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, src.replace(".cu", ".o"))
        if force or not os.path.exists(o) or os.path.getmtime(o) < max(os.path.getmtime(s), hdr_time):
            jobs.append([NVCC] + FLAGS + ["-c", s, "-o", o])

    def run(cmd):
        if verbose:
            print(" ".join(cmd))
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode:
            raise RuntimeError("nvcc failed:\n%s\n%s" % (" ".join(cmd), r.stderr))
        return r.stderr

    with ThreadPoolExecutor(max_workers=6) as ex:
        list(ex.map(run, jobs))
    objs = [os.path.join(OBJ, src.replace(".cu", ".o")) for src in SOURCES]
    if jobs or force or not os.path.exists(LIB):
        run([NVCC, "-shared", "--cudart", "static", "-o", LIB] + objs + ["-ldl", "-lpthread"])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
