"""Builds libmultimm_b200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels
with the repo snapshot to the GPU box).

    python -m multimm_b200.build [--force] [--verbose]
"""
from __future__ import annotations

import glob
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_PATH = os.path.join(HERE, os.environ.get("MMM_LIB_NAME", "libmultimm_b200.so"))

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC", "-shared",
    "-ccbin", "/usr/bin/g++",
    "--threads", "0",  # the .cu files compile side by side (same SASS, half the wall time)
]


def cuda_tool(name: str) -> str:
    """A CUDA toolkit program (nvcc, cuobjdump): from PATH, else the toolkit's default location."""
    for cand in (shutil.which(name), os.path.join("/usr/local/cuda/bin", name)):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError(f"{name} not found (neither on PATH nor in /usr/local/cuda/bin)")


def sources() -> list[str]:
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def _stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = sources() + glob.glob(os.path.join(CSRC, "*.cuh")) + [
        os.path.join(HERE, "..", "include", "multimm_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB_PATH
    # link into a private name and rename: a concurrent reader (another test worker, an ensemble
    # worker) sees either the old library or the complete new one, never a half-written file
    tmp = f"{LIB_PATH}.{os.getpid()}.tmp"
    cmd = [cuda_tool("nvcc"), *NVCC_FLAGS, *os.environ.get("MMM_EXTRA_NVCC_FLAGS", "").split(), "-o", tmp, *sources()]
    if verbose:
        cmd[1:1] = ["-Xptxas", "-v"]
    try:
        res = subprocess.run(cmd, capture_output=True, text=True)
        if verbose or res.returncode != 0:
            sys.stderr.write(res.stdout + res.stderr)
        if res.returncode != 0:
            raise RuntimeError("nvcc failed building libmultimm_b200.so")
        os.replace(tmp, LIB_PATH)
    finally:
        if os.path.exists(tmp):
            os.remove(tmp)
    return LIB_PATH


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(LIB_PATH)
