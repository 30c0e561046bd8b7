"""Builds libvbmf_b200.so (sm_100a only) in-tree with nvcc.  No torch, no JIT cache: the .so travels with the repo snapshot."""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libvbmf_b200.so")
SOURCES = ["gemm_dmma.cu", "gemm_int8.cu", "kernels.cu", "batched.cu", "capi.cu", "multi.cu"]
HEADERS = ["common.cuh", "elbo.cuh", "gemm.cuh", "kernels.cuh", "linalg.cuh", os.path.join("..", "..", "include", "vbmf_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    os.makedirs(LIBDIR, exist_ok=True)
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    hdrs = [os.path.join(CSRC, h) for h in HEADERS]
    nvcc = _nvcc()

    def compile_one(src):
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        path = os.path.join(CSRC, src)
        if force or _stale(obj, [path] + hdrs):
            cmd = [nvcc] + NVCC_FLAGS + ["-c", path, "-o", obj]
            if verbose:
                print(" ".join(cmd))
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    if force or _stale(LIB, objs):
        cmd = [nvcc, "-shared", "-cudart", "static", "-o", LIB] + objs + ["-ldl", "-lpthread"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
