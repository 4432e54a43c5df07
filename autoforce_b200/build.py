"""Build libsgpr_b200.so in-tree with nvcc for sm_100a (no JIT cache: the built .so
travels with the repository snapshot to the GPU box)."""
from __future__ import annotations

import os
import shutil
import subprocess
from concurrent.futures import ThreadPoolExecutor

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
LIBDIR = os.path.join(PKG, "lib")
LIBPATH = os.path.join(LIBDIR, "libsgpr_b200.so")
SOURCES = ["api.cu", "nl.cu", "descriptor.cu", "gemm.cu", "i8gemm.cu", "md.cu", "relax.cu"]
HEADERS = ["sgpr_internal.cuh", "sgpr_math.cuh", "gemm_kernel.cuh", "i8gemm_kernel.cuh", "i8gemm2_kernel.cuh", os.path.join("..", "..", "include", "sgpr_b200.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
]


def _nvcc():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: cannot build libsgpr_b200.so")
    return nvcc


def needs_build():
    if not os.path.exists(LIBPATH):
        return True
    t = os.path.getmtime(LIBPATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force=False, verbose=False):
    """Compile every .cu for sm_100a and link the shared library. Returns its path."""
    if not force and not needs_build():
        return LIBPATH
    nvcc = _nvcc()
    os.makedirs(LIBDIR, exist_ok=True)
    objdir = os.path.join(LIBDIR, "obj")
    os.makedirs(objdir, exist_ok=True)

    def compile_one(src):
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            print(" ".join(cmd), flush=True)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    # dynamic cudart so that the library shares the CUDA runtime instance (context, streams)
    # with the torch process that loads it; rpaths cover the venv wheel and the toolkit
    rpaths = ["/usr/local/cuda/lib64"]
    try:
        import nvidia.cuda_runtime as _cr  # the wheel torch links against

        rpaths.insert(0, os.path.join(os.path.dirname(_cr.__file__), "lib"))
    except Exception:
        pass
    cmd = [nvcc, "-shared", "-cudart", "shared", "-o", LIBPATH] + objs
    for rp in rpaths:
        cmd += ["-Xlinker", "-rpath", "-Xlinker", rp]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIBPATH


if __name__ == "__main__":
    print(build_library(force=True, verbose=True))
