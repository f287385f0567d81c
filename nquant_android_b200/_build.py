"""Builds libnquant_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "libnquant_b200.so")
SOURCES = ["nq_api.cu"]
DEPS = ["nq_api.cu", "nq_types.h", "nq_math.h", "nq_math_tables.h", "nq_color.h", "nq_bluenoise_table.h",
        "nq_hist.cuh", "nq_pnn.cuh", "nq_dither.cuh", "nq_dither_spec.cuh", "nq_fastmath.cuh", "nq_gilbert.h", os.path.join("..", "..", "include", "nquant_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    # Java arithmetic has no fused multiply-add: contraction off on both sides of the compiler
    "-fmad=false", "-Xcompiler", "-fPIC,-ffp-contract=off,-fno-fast-math",
    "-shared",
]


def is_stale():
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    return any(os.path.getmtime(os.path.join(CSRC, d)) > t for d in DEPS)


def build(force=False, verbose=False):
    if not force and not is_stale():
        return SO
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + ["-o", SO] + [os.path.join(CSRC, s) for s in SOURCES]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    subprocess.check_call(cmd)
    return SO


if __name__ == "__main__":
    print(build(force=True, verbose=True))
