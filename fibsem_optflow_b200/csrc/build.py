"""Builds libtvl1_b200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels to
the GPU box with the snapshot).

-fmad=false and no --use_fast_math are REQUIRED: parity with the CPU path needs one rounding
per fp32 operation (SURVEY.md H2).  -lineinfo keeps ncu's source page usable.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "libtvl1_b200.so")
SOURCES = ["tvl1_engine.cu", "tvl1_sampler.cu", "tvl1_features.cu"]
DEPS = SOURCES + ["tvl1_kernels.cuh", "tvl1_batch.cuh", "tvl1_internal.h", os.path.join("..", "..", "include", "tvl1_b200.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-fmad=false", "-prec-div=true", "-prec-sqrt=true", "-ftz=false",
    "-ccbin", "/usr/bin/g++",
    "-Xcompiler", "-fPIC,-ffp-contract=off,-O2",
    "-shared", "-cudart", "static",
]


def stale():
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    return any(os.path.getmtime(os.path.join(HERE, d)) > t for d in DEPS)


def build(force=False, verbose=False):
    if not force and not stale():
        return SO
    cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", SO] + [os.path.join(HERE, s) for s in SOURCES]
    subprocess.check_call(cmd, cwd=HERE)
    return SO


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(SO)
