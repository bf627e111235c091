"""Build libmgb200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import glob
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libmgb200.so")
TOOL = os.path.join(HERE, "multigrid_b200")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC,-ffp-contract=off,-O2", "-shared", "-cudart", "static",
]


def sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = sources() + glob.glob(os.path.join(CSRC, "*.cuh")) + [os.path.join(HERE, "..", "include", "mgb200.h")]
    return any(os.path.getmtime(p) > t for p in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: libmgb200.so cannot be built and there is no CPU path")
    cmd = [nvcc, *NVCC_FLAGS, "-o", LIB, *sources()]
    if verbose:
        print(" ".join(cmd))
    env = dict(os.environ)
    env.pop("CC", None); env.pop("CXX", None)
    subprocess.run(cmd, check=True, env=env)
    # the command-line front end (tools/multigrid_b200.cpp): plain C++ over the C ABI
    tool_src = os.path.join(HERE, "..", "tools", "multigrid_b200.cpp")
    if os.path.exists(tool_src):
        subprocess.run(["g++", "-O2", "-std=c++17", "-o", TOOL, tool_src, "-L" + HERE, "-lmgb200", "-Wl,-rpath,$ORIGIN"],
                       check=True, env=env)
    return LIB


if __name__ == "__main__":
    print(build(force=True, verbose=True))
