"""In-tree build of libtsgu_b200.so with nvcc for sm_100a (no torch headers, no JIT cache).

    python -m torchsparsegradutils_b200.csrc.build [--force]

The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import concurrent.futures as cf
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
SOURCES = ["api.cu", "spmm.cu", "sddmm.cu", "index.cu", "merge.cu", "window.cu", "trisolve.cu"]
HEADERS = ["common.cuh", "tile.cuh", os.path.join(ROOT, "include", "tsgu_b200.h")]
LIB = os.path.join(os.path.dirname(HERE), "libtsgu_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC,-fvisibility=hidden", "--expt-relaxed-constexpr", "-Xptxas", "-v",
    "-DTSGU_BUILD",
] + os.environ.get("TSGU_EXTRA_NVCC_FLAGS", "").split()


def _stale(target: str, deps: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def _compile(src: str, force: bool) -> str:
    obj = os.path.join(HERE, "_obj", src.replace(".cu", ".o"))
    os.makedirs(os.path.dirname(obj), exist_ok=True)
    deps = [os.path.join(HERE, src)] + [h if os.path.isabs(h) else os.path.join(HERE, h) for h in HEADERS]
    if force or _stale(obj, deps):
        log = obj + ".log"
        with open(log, "w") as fh:
            subprocess.check_call([NVCC, *FLAGS, "-c", os.path.join(HERE, src), "-o", obj], stdout=fh, stderr=fh)
    return obj


def build(force: bool = False, verbose: bool = False) -> str:
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(HERE, s))]
    with cf.ThreadPoolExecutor(max_workers=min(len(srcs), os.cpu_count() or 4)) as ex:
        objs = list(ex.map(lambda s: _compile(s, force), srcs))
    if force or _stale(LIB, objs):
        subprocess.check_call([NVCC, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a"])
    if verbose:
        print("built", LIB)
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose=True)
