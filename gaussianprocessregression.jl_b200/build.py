"""Build libgpr_sm100a.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python gaussianprocessregression.jl_b200/build.py [--force]

The library is a plain CUDA-runtime shared object with a C ABI (include/gpr_sm100a.h);
it does not link against torch.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libgpr_sm100a.so")
SOURCES = ["gpr_api.cu"]
DEPS = ["gpr_api.cu", "kbuild_tma.cuh", "dgemm_tma.cuh", "ozaki_i8.cuh", "fastexp.cuh", "mgpu_api.inl", "dist_blocked.hpp", "blocked.hpp", "cov_kernels.cuh", "grad_wide.cuh", "dgemm_sm100.cuh", "leaf_kernels.cuh",
        os.path.join(ROOT, "include", "gpr_sm100a.h")]
NVCC_FLAGS = ["-shared", "-Xcompiler", "-fPIC", "-O3", "-std=c++17",
              "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    for d in DEPS:
        p = d if os.path.isabs(d) else os.path.join(CSRC, d)
        if os.path.exists(p) and os.path.getmtime(p) > t:
            return True
    return False


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + \
          [os.path.join(CSRC, s) for s in SOURCES]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
