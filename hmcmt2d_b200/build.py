"""Builds libhmcmt_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).  The translation units are
compiled in parallel and only when one of their dependencies changed."""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libhmcmt_b200.so")
OBJDIR = os.path.join(HERE, "build")
HDR = os.path.join("..", "..", "include", "hmcmt_b200.h")
# translation unit -> headers it includes
SOURCES = {
    "hmcmt_b200.cu": ["common.cuh", "band_factor.cuh", "band_solve.cuh", "mt_kernels.cuh", "mf_solver.cuh", "mf_symbolic.h", HDR],
    "mumps_shim.cu": ["common.cuh", "band_factor.cuh", "band_solve.cuh", "mf_solver.cuh", "mf_symbolic.h", HDR],
    "mf_solver.cu": ["common.cuh", "band_factor.cuh", "mf_kernels.cuh", "mf_selinv.cuh", "mf_solver.cuh", "mf_symbolic.h"],
}
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC"]


def _newer(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def _obj(src: str) -> str:
    return os.path.join(OBJDIR, os.path.splitext(src)[0] + ".o")


def build(force: bool = False, verbose: bool = False) -> str:
    nvcc = os.environ.get("NVCC", "nvcc")
    os.makedirs(OBJDIR, exist_ok=True)
    todo = [s for s, hdrs in SOURCES.items()
            if force or _newer(_obj(s), [os.path.join(CSRC, s)] + [os.path.join(CSRC, h) for h in hdrs])]

    def compile_one(src):
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", _obj(src)]
        return src, subprocess.run(cmd, capture_output=True, text=True)

    with ThreadPoolExecutor(max_workers=max(1, len(todo))) as ex:
        for src, res in ex.map(compile_one, todo):
            if res.returncode != 0:
                sys.stderr.write(res.stdout + res.stderr)
                raise RuntimeError(f"nvcc failed compiling {src}")
            if verbose:
                sys.stderr.write(res.stderr)
    objs = [_obj(s) for s in SOURCES]
    if todo or _newer(LIB, objs):
        res = subprocess.run([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs + ["-ldl"], capture_output=True, text=True)
        if res.returncode != 0:
            sys.stderr.write(res.stdout + res.stderr)
            raise RuntimeError("nvcc failed linking libhmcmt_b200.so")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
