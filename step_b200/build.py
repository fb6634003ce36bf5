"""Builds step_b200/libstep_b200.so (hand-written sm_100a CUDA behind the C ABI of include/step_b200.h).

    python -m step_b200.build            # incremental
nvcc cross-compiles without a GPU; the .so is built in-tree so it travels with the gpurun snapshot.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "_obj")
LIB = os.path.join(HERE, "libstep_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
SOURCES = ["api.cu", "nms.cu", "roi.cu", "tubes.cu", "pool_layout.cu", "conv_simt.cu", "conv_umma.cu", "conv_halo.cu", "bottleneck_exit.cu", "train.cu", "frames.cu"]
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
         "-Xcompiler", "-fPIC", "--use_fast_math=false" if False else "-Xptxas", "-v"]
# nms/roi/tubes/frames rely on explicitly rounded intrinsics; -fmad=false additionally forbids contraction
NO_FMAD = {"nms.cu", "roi.cu", "tubes.cu", "train.cu", "frames.cu"}


def _deps(src):
    return [os.path.join(CSRC, src), os.path.join(CSRC, "common.cuh"), os.path.join(CSRC, "umma_ptx.cuh"),
            os.path.join(os.path.dirname(HERE), "include", "step_b200.h")]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def _compile(src, verbose):
    obj = os.path.join(OBJ, src.replace(".cu", ".o"))
    if not _stale(obj, _deps(src)):
        return obj, ""
    cmd = [NVCC] + FLAGS + (["-fmad=false"] if src in NO_FMAD else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
    return obj, r.stderr


def build(verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        res = list(ex.map(lambda s: _compile(s, verbose), SOURCES))
    objs = [o for o, _ in res]
    if verbose:
        for _, log in res:
            if log:
                print(log)
    if _stale(LIB, objs):
        cmd = [NVCC, "-shared", "-o", LIB] + objs + ["-lcudart"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    return LIB


if __name__ == "__main__":
    print(build(verbose="-v" in sys.argv))
