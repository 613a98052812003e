"""Builds libvidc_b200.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python -m vi_depth_completion_b200.build [--force]

-fmad=false is REQUIRED: the kernels restate the reference's fp32 roundings and write every fused
multiply-add explicitly (csrc/exact_math.cuh).  No fast-math, IEEE division and square root.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libvidc_b200.so")
SOURCES = [os.path.join(CSRC, "vidc_kernels.cu")]
DEPS = SOURCES + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh")] + [
    os.path.join(os.path.dirname(HERE), "include", "vidc_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-fmad=false", "-prec-div=true", "-prec-sqrt=true", "-ftz=false",
    "-shared", "-Xcompiler", "-fPIC",
    "-cudart", "static",
]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; libvidc_b200.so cannot be built")


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(d) > t for d in DEPS)


def build(force: bool = False, verbose: bool = False) -> str:
    if force or needs_build():
        extra = os.environ.get("VIDC_NVCC_EXTRA", "").split()
        cmd = [nvcc_path()] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + SOURCES
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
        if verbose:
            print(res.stderr)
    return LIB


# ---- the thin torch C++ extension in front of the C ABI (csrc/torch_ops.cpp): plain g++, in-tree, links libvidc_b200.so ------
TORCH_OPS_SRC = os.path.join(CSRC, "torch_ops.cpp")
TORCH_OPS_LIB = os.path.join(HERE, "_vidc_torch_ops.so")


def torch_ops_needs_build() -> bool:
    if not os.path.exists(TORCH_OPS_LIB):
        return True
    t = os.path.getmtime(TORCH_OPS_LIB)
    return any(os.path.getmtime(d) > t for d in (TORCH_OPS_SRC, os.path.join(os.path.dirname(HERE), "include", "vidc_b200.h")))


def build_torch_ops(force: bool = False) -> str:
    """g++ -shared csrc/torch_ops.cpp against the torch of this interpreter and libvidc_b200.so (rpath $ORIGIN)."""
    build(force=False)
    if force or torch_ops_needs_build():
        import torch
        from torch.utils import cpp_extension as ce
        tlib = os.path.join(os.path.dirname(torch.__file__), "lib")
        cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
        cmd = (["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-deprecated-declarations",
                f"-D_GLIBCXX_USE_CXX11_ABI={int(torch._C._GLIBCXX_USE_CXX11_ABI)}", "-DTORCH_API_INCLUDE_EXTENSION_H"] +
               [f"-I{p}" for p in ce.include_paths()] + [f"-I{cuda_inc}", TORCH_OPS_SRC, "-o", TORCH_OPS_LIB,
               f"-L{tlib}", "-ltorch", "-ltorch_cpu", "-ltorch_cuda", "-lc10", "-lc10_cuda", f"-L{HERE}", "-l:libvidc_b200.so",
               "-Wl,-rpath,$ORIGIN", f"-Wl,-rpath,{tlib}"])
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("g++ failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    return TORCH_OPS_LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
    print(build_torch_ops(force="--force" in sys.argv))
