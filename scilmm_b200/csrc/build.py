"""Builds libscilmm_b200.so in-tree with nvcc for sm_100a (no torch dependency in the library)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.dirname(HERE)
LIB = os.path.join(PKG, "libscilmm_b200.so")
CUDA_HOME = os.environ.get("CUDA_HOME", "/usr/local/cuda")
NVCC = os.path.join(CUDA_HOME, "bin", "nvcc")
METIS = os.path.join(CUDA_HOME, "lib64", "libmetis_static.a")
SOURCES_CU = ["chol.cu", "sparse_ops.cu", "ibd.cu", "quadform_tiled.cu", "assoc.cu", "blup.cu", "glmm.cu"]
SOURCES_CPP = ["symbolic.cpp"]
HEADERS = ["common.h", "dense_tiles.cuh", "potrf_block.cuh", "symbolic.h", "skinny_ops.cuh", "matset.h", "dense_tiles_tma.cuh"]


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    for f in SOURCES_CU + SOURCES_CPP + HEADERS + ["build.py"]:
        if os.path.getmtime(os.path.join(HERE, f)) > t:
            return True
    return False


def build(force=False, verbose=False):
    if not force and not _stale():
        return LIB
    if not os.path.exists(NVCC):
        raise RuntimeError("nvcc not found at %s" % NVCC)
    objs = []
    for src in SOURCES_CPP:
        obj = os.path.join(HERE, src.replace(".cpp", ".o"))
        cmd = ["g++", "-O2", "-fPIC", "-std=c++17", "-c", os.path.join(HERE, src), "-o", obj]
        subprocess.check_call(cmd)
        objs.append(obj)
    cmd = [NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
           "-Xcompiler", "-fPIC", "-shared"]
    if verbose:
        cmd += ["-Xptxas", "-v"]
    cmd += [os.path.join(HERE, s) for s in SOURCES_CU] + objs + [METIS, "-o", LIB]
    out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or out.returncode != 0:
        sys.stderr.write(out.stdout)
    if out.returncode != 0:
        raise RuntimeError("nvcc failed")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
