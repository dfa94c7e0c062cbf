"""In-tree build of libcsnappy_b200.so: plain-C shim (gcc) + sm_100a kernels (nvcc).

    python -m csnappy_b200.build            # incremental
    python -m csnappy_b200.build --force

The .so lands next to this file (git-ignored, travels to the GPU box with the
snapshot).  cudart is linked statically, so the library has no dependency on
torch's or the system's libcudart.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
TAG = os.environ.get("CSB_BUILD_TAG", "")  # experiments: a variant library next to the product one (see CSNAPPY_B200_LIB)
OBJ = os.path.join(HERE, "build" + ("_" + TAG if TAG else ""))
LIB = os.path.join(HERE, "libcsnappy_b200" + ("_" + TAG if TAG else "") + ".so")
CUDA_HOME = os.environ.get("CUDA_HOME", "/usr/local/cuda")
NVCC = shutil.which("nvcc") or os.path.join(CUDA_HOME, "bin", "nvcc")

CU = ["compress_kernel.cu", "decompress_kernel.cu", "decompress_lane_kernel.cu", "stream_kernel.cu", "pack_kernel.cu",
      "framed_kernel.cu", "bc_kernel.cu"]
C = ["csnappy_shim.c"]
HEADERS = [os.path.join(CSRC, h) for h in ("kernels.h", "device_common.cuh")] + [
    os.path.join(HERE, "..", "include", h) for h in ("csnappy.h", "csnappy_batch.h")
]

NVCC_FLAGS = [
    "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
    "-Xcompiler", "-fPIC,-fvisibility=hidden", "-Xptxas", "-v", "--expt-relaxed-constexpr",
]
NVCC_FLAGS += os.environ.get("CSB_NVCC_EXTRA", "").split()  # experiments: e.g. -DCSB_CUT_MIN=20
CC_FLAGS = ["-O2", "-std=gnu11", "-Wall", "-Wextra", "-fPIC", "-I" + os.path.join(CUDA_HOME, "include")]


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    objs = []
    log = []
    for src in CU:
        s, o = os.path.join(CSRC, src), os.path.join(OBJ, src + ".o")
        objs.append(o)
        if force or _stale(o, [s] + HEADERS):
            r = subprocess.run([NVCC] + NVCC_FLAGS + ["-c", s, "-o", o], capture_output=True, text=True)
            log.append(r.stderr)
            if r.returncode:
                raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
    for src in C:
        s, o = os.path.join(CSRC, src), os.path.join(OBJ, src + ".o")
        objs.append(o)
        if force or _stale(o, [s] + HEADERS):
            r = subprocess.run(["gcc"] + CC_FLAGS + ["-c", s, "-o", o], capture_output=True, text=True)
            log.append(r.stderr)
            if r.returncode:
                raise RuntimeError(f"gcc failed on {src}:\n{r.stdout}\n{r.stderr}")
    if force or _stale(LIB, objs):
        r = subprocess.run([NVCC, "-shared", "-o", LIB] + objs + ["-lpthread", "-Xlinker", "--exclude-libs,ALL"], capture_output=True, text=True)
        if r.returncode:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    if verbose:
        print("".join(log))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
