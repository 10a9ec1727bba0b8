"""Builds librepose_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "librepose_b200.so")
# (source, extra flags): the LM kernels are built with FMA contraction, everything else without
SOURCES = [("repose_b200.cu", ["-fmad=false", "-DRP_SOLVE_MIN_BLOCKS=" + os.environ.get("RP_SOLVE_MIN_BLOCKS", "1"),
                               "-DRP_SOLVE2_MIN_BLOCKS=" + os.environ.get("RP_SOLVE2_MIN_BLOCKS", "3")] + os.environ.get("RP_MAIN_EXTRA", "").split()), ("repose_lm.cu", ["-fmad=true", "-DRP_LM_MIN_BLOCKS=" + os.environ.get("RP_LM_MIN_BLOCKS", "3")] + os.environ.get("RP_LM_EXTRA", "").split())]
HEADERS = ["rp_common.cuh", "rp_types.cuh", "rp_solvers.cuh", "rp_score.cuh", "rp_lm.cuh", "rp_lm_kernel.cuh", "rp_kernels.cuh", "rp_tc.cuh", "rp_order.cuh",
           "../../include/repose_b200.h"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
]
# repose_b200.cu: -fmad=false, `a*b+c` rounds twice like the reference's SSE2 build (FMAs explicit)


def stale() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in [s for s, _ in SOURCES] + HEADERS)


def build_native(force: bool = False, verbose: bool = False) -> str:
    if not force and not stale():
        return OUT
    nvcc = os.environ.get("NVCC", "nvcc")
    objs = []
    for src, extra in SOURCES:
        obj = os.path.join(CSRC, src.replace(".cu", ".o"))
        subprocess.check_call([nvcc] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) +
                              ["-c", "-o", obj, os.path.join(CSRC, src)])
        objs.append(obj)
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-Xcompiler", "-fPIC",
                           "-o", OUT] + objs)
    return OUT


if __name__ == "__main__":
    print(build_native(force="--force" in sys.argv, verbose="-v" in sys.argv))
