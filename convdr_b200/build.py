"""In-tree build of the CUDA library (sm_100a only).

`python -m convdr_b200.build` or `__graft_entry__.build()`.  nvcc cross-compiles without a GPU.
The built `.so` files are git-ignored but travel with the repo snapshot to the GPU box.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "convdr_b200", "csrc")
LIB = os.path.join(CSRC, "libb2f.so")
SOURCES = ["b2f_api.cu"]
HEADERS = ["common.cuh", "kernels_scan.cuh", "kernels_select.cuh", "kernels_selector.cuh", "kernels_umma.cuh", "kernels_umma_qs.cuh", "kernels_util.cuh",
           os.path.join("..", "..", "include", "b2f.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
]


def _stale(target: str, deps: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build_cuda(force: bool = False, verbose: bool = False) -> str:
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS]
    if not force and not _stale(LIB, deps):
        return LIB
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    cmd = [nvcc, *NVCC_FLAGS, "-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return LIB


def main() -> None:
    force = "--force" in sys.argv
    print(build_cuda(force=force, verbose="-v" in sys.argv))


if __name__ == "__main__":
    main()
