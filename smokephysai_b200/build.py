"""Build libsmoke_sm100.so in-tree with nvcc for sm_100a (no torch headers, no libtorch link).

    python -m smokephysai_b200.build [--force] [--verbose]

-fmad=false is part of the arithmetic contract (no FMA contraction: SURVEY.md s8a parity traps), not a
tuning knob; -lineinfo keeps ncu's source page usable.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "libsmoke_sm100.so")
SOURCES = ["abi.cu", "jacobi.cu", "stencil.cu", "features.cu", "fused.cu", "nccl_halo.cu", "peer_halo.cu", "adjoint.cu"]
HEADERS = ["common.cuh", "jacobi_core.cuh", os.path.join("..", "..", "include", "smoke_b200.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-fmad=false", "-prec-div=true", "-prec-sqrt=true",
    "-Xcompiler", "-fPIC,-fvisibility=hidden", "-shared",
    "-cudart", "static", "-ldl",
]


def nvcc_path():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libsmoke_sm100.so cannot be built")


def stale():
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not stale():
        return SO
    extra = os.environ.get("SMK_NVCC_EXTRA", "").split()          # e.g. -DSMK_FZ_ELEM=float2 for an A/B build of a kernel variant
    cmd = [nvcc_path()] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + \
          ["-o", SO] + [os.path.join(CSRC, s) for s in SOURCES]
    if verbose:
        print(" ".join(cmd))
    subprocess.check_call(cmd)
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
