"""In-tree build of libsplash_cuda.so for sm_100a (nvcc cross-compiles without a GPU)."""
from __future__ import annotations

import os
import shutil
import subprocess

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
# SPLASH_CUDA_LIB: development override to load/build a variant of the library (e.g. another SPLASH_LEVEL)
LIB_PATH = os.environ.get("SPLASH_CUDA_LIB") or os.path.join(PKG_DIR, "libsplash_cuda.so")
SOURCES = [os.path.join(CSRC, "splash_cuda.cu")]
HEADERS = [os.path.join(CSRC, "splash_model.cuh"), os.path.join(CSRC, "splash_math.cuh"), os.path.join(CSRC, "splash_consts.cuh"), os.path.join(CSRC, "splash_host_tables.h"), os.path.join(CSRC, "splash_upslope.cuh"),os.path.join(PKG_DIR, "..", "include", "splash_cuda.h")]

# -fmad=false: the reference build has no FMA contraction (R's default x86-64 flags); the day step
# mirrors its evaluation order, explicit fma() is used only where glibc's expf does.
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-fmad=false",
    "-shared", "-Xcompiler", "-fPIC", "-Xcompiler", "-pthread", "-Xptxas", "-v",
]


def nvcc_path() -> str:
    p = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(p):
        raise RuntimeError("nvcc not found: libsplash_cuda cannot be built")
    return p


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(f) > t for f in SOURCES + HEADERS if os.path.exists(f))


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile rsplash_b200/libsplash_cuda.so; returns the ptxas resource report."""
    if not force and not needs_build():
        return ""
    extra = os.environ.get("SPLASH_NVCC_EXTRA", "").split()  # e.g. -DSPLASH_LEVEL=0 for the literal-order day step
    cmd = [nvcc_path(), *NVCC_FLAGS, *extra, "-o", LIB_PATH, *SOURCES]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stderr)
    return r.stderr


if __name__ == "__main__":
    print(build(force=True))
