"""Build libbwgr_b200.so (CUDA kernels + C ABI) in-tree for sm_100a.

nvcc cross-compiles without a GPU.  The shared object stays in bwgr_b200/lib/ (git-ignored, but it
travels to the GPU box with the repo snapshot).  Rebuilds only what changed.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "lib", "obj")
LIB = os.path.join(HERE, "lib", "libbwgr_b200.so")
SOURCES = ["handle.cu", "store.cu", "fit.cu", "solvers.cu", "mrr_host.cu", "geno.cu", "small_n.cu", "grid_sweep.cu", "epilogue.cu", "gram_tc.cu", "gram_fp4.cu", "sweep_pipe.cu", "mrr.cu", "mrr_gen.cu", "block_inv.cu", "host_narrow.cpp"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
         "--expt-relaxed-constexpr"]


def _newest_header():
    hs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    hs.append(os.path.join(HERE, "..", "include", "bwgr_b200.h"))
    return max(os.path.getmtime(h) for h in hs)


def _compile(src):
    obj = os.path.join(OBJ, src.replace(".cu", ".o").replace(".cpp", ".o"))
    path = os.path.join(CSRC, src)
    if os.path.exists(obj) and os.path.getmtime(obj) >= max(os.path.getmtime(path), _newest_header()):
        return obj, False
    subprocess.check_call([NVCC] + FLAGS + ["-c", path, "-o", obj])
    return obj, True


def build(verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        res = list(ex.map(_compile, SOURCES))
    objs = [o for o, _ in res]
    if any(c for _, c in res) or not os.path.exists(LIB):
        subprocess.check_call([NVCC, "-shared", "-o", LIB] + objs + ["-cudart", "static"])
        if verbose:
            print("linked", LIB)
    return LIB


if __name__ == "__main__":
    print(build(verbose=True))
    sys.exit(0)
