"""Build the CUDA library in-tree: therldaisyworld_b200/libdaisyworld_b200.so (sm_100a only).

nvcc cross-compiles without a GPU.  -fmad=false is part of the numerical contract: the literal
kernels must round a*b+c twice like NumPy; fused multiply-adds are written out (__fma_rn) where the
fast lattice path wants them."""
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(PKG, "csrc", "dw_api.cu")
OUT = os.path.join(PKG, "libdaisyworld_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-fmad=false", "-lineinfo", "-std=c++17",
         "-Xcompiler", "-fPIC", "-shared", "-cudart", "static"]


def sources():
    d = os.path.join(PKG, "csrc")
    inc = os.path.join(PKG, "..", "include", "daisyworld_b200.h")
    return [os.path.join(d, f) for f in os.listdir(d)] + [inc]


def build(force=False, verbose=False):
    if not force and os.path.exists(OUT) and all(os.path.getmtime(OUT) >= os.path.getmtime(s) for s in sources()):
        return OUT
    cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", OUT, SRC]
    subprocess.check_call(cmd)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
