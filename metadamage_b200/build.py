"""Build libmdgb200.so in-tree with nvcc for sm_100a (B200). No other architecture is built."""
import glob
import os
import shutil
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
LIB_PATH = os.path.join(_HERE, "libmdgb200.so")
SOURCES = [os.path.join(_HERE, "csrc", "mdg_api.cu")]
HEADERS = [os.path.join(_ROOT, "include", "mdg.h")] + sorted(glob.glob(os.path.join(_HERE, "csrc", "*.cuh")))
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    # no implicit mul+add contraction: every kernel variant (MAP's 1, 2 or 4 positions per lane)
    # must give bit-identical results; fused operations are written as fma() explicitly
    "-fmad=false",
    "-Xcompiler", "-fPIC", "-shared", "-cudart", "static",
]


def find_nvcc():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: libmdgb200.so cannot be built")
    return nvcc


def is_stale():
    if not os.path.exists(LIB_PATH):
        return True
    built = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(f) > built for f in SOURCES + HEADERS)


def build(force=False, verbose=False):
    """Compile the CUDA library if it is missing or older than its sources. Returns its path."""
    if not force and not is_stale():
        return LIB_PATH
    cmd = [find_nvcc(), *NVCC_FLAGS, "-I", os.path.join(_ROOT, "include"), "-o", LIB_PATH, *SOURCES]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
        print(" ".join(cmd), file=sys.stderr)
    subprocess.run(cmd, check=True)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
