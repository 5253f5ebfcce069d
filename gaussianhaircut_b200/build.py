"""Build libgh_raster.so (the C-ABI CUDA library) in-tree for sm_100a.

    python -m gaussianhaircut_b200.build [--force]

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels to the GPU box with the
gpurun snapshot.  No torch headers are involved: the library is plain CUDA C++ behind `extern "C"`.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
OBJ_DIR = os.path.join(LIB_DIR, "obj")
LIB_PATH = os.path.join(LIB_DIR, "libgh_raster.so")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")

SOURCES = ["gh_api.cu", "gh_preprocess.cu", "gh_binning.cu", "gh_blend.cu", "gh_preprocess_bwd.cu", "gh_adam.cu", "gh_image_loss.cu", "gh_allreduce.cu", "gh_project.cu", "gh_densify.cu"]
HEADERS = ["gh_common.cuh", "gh_kernels.h", "gh_project_math.h"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def needs_build() -> bool:
    if not os.path.isfile(LIB_PATH):
        return True
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [
        os.path.join(INCLUDE, "gh_rasterizer.h"), os.path.abspath(__file__)]
    return os.path.getmtime(LIB_PATH) < max(os.path.getmtime(p) for p in deps)


def build(force: bool = False, verbose: bool = True) -> str:
    if not force and not needs_build():
        return LIB_PATH
    os.makedirs(OBJ_DIR, exist_ok=True)
    nvcc = _nvcc()

    def compile_one(src: str) -> str:
        obj = os.path.join(OBJ_DIR, src + ".o")
        cmd = [nvcc, "-c", os.path.join(CSRC, src), "-o", obj, f"-I{INCLUDE}", f"-I{CSRC}"] + NVCC_FLAGS
        if verbose:
            print("[gh build]", " ".join(cmd), flush=True)
        subprocess.run(cmd, check=True)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [nvcc, "-shared", "-o", LIB_PATH] + objs + ["-gencode", "arch=compute_100a,code=sm_100a",
                                                       "-cudart", "static", "-Xcompiler", "-fPIC"]
    if verbose:
        print("[gh build]", " ".join(cmd), flush=True)
    subprocess.run(cmd, check=True)
    return LIB_PATH


if __name__ == "__main__":
    build(force="--force" in sys.argv)
    print(LIB_PATH)
