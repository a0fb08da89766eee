"""Builds libctd_b200.so (the C-ABI kernel library) in-tree with nvcc for sm_100a.

No torch involvement: the library is plain CUDA C++ behind `extern "C"` (include/ctd_b200.h).
`python -m connecting_the_dots_b200._build` or `__graft_entry__.build()` runs this; nvcc
cross-compiles without a GPU.  The .so is git-ignored but travels to the GPU box with gpurun.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
OBJ = os.path.join(CSRC, "build")
LIB = os.path.join(PKG, "libctd_b200.so")
SOURCES = ["ctd_core.cu", "photometric.cu", "photometric_tma.cu", "census_sym.cu", "lcn.cu", "lcn_extra.cu", "xcorrvol.cu", "index_ops.cu", "reduce.cu", "warp.cu", "geometric.cu", "disparity_loss.cu", "ssim.cu", "sgm.cu", "census_match.cu", "disparity_check.cu", "speckle.cu", "corr_softargmax.cu", "host_api.cu"]
HEADERS = [os.path.join(CSRC, "ctd_common.cuh"), os.path.join(CSRC, "ctd_tma.cuh"), os.path.join(PKG, "..", "include", "ctd_b200.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
# -fmad=false: the reference's CPU build has no fused multiply-adds and the index ops must match it
# bit for bit; the hot kernels spell their FMAs out with fmaf().
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-fmad=false",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "-Xptxas", "-v"] + os.environ.get("CTD_NVCC_EXTRA", "").split()


def _stale(target, deps):
    return not os.path.exists(target) or any(os.path.getmtime(d) > os.path.getmtime(target) for d in deps)


def _compile(src):
    obj = os.path.join(OBJ, src.replace(".cu", ".o"))
    path = os.path.join(CSRC, src)
    if _stale(obj, [path] + HEADERS):
        r = subprocess.run([NVCC] + FLAGS + ["-c", path, "-o", obj], capture_output=True, text=True)
        with open(obj + ".log", "w") as f:
            f.write(r.stdout + r.stderr)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed on %s:\n%s" % (src, r.stderr[-4000:]))
    return obj


def build(verbose=False):
    """Compile what is stale and link libctd_b200.so; returns its path."""
    os.makedirs(OBJ, exist_ok=True)
    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(_compile, SOURCES))
    if _stale(LIB, objs):
        r = subprocess.run([NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs + ["-Xcompiler", "-fPIC"], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n" + r.stderr[-4000:])
    if verbose:
        print("built", LIB)
    return LIB


if __name__ == "__main__":
    build(verbose=True)
    sys.exit(0)
