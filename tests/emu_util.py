"""Helpers shared by the host-model tests of the streaming pass: the solver's split layout in numpy, seeded
fields, and the loader of the model library (tests/emu/syst_emu.cpp, built on demand)."""
import ctypes as C
import os
import subprocess

import numpy as np

from conftest import ROOT

EMU_DIR = os.path.join(ROOT, "tests", "emu")
_dp = C.POINTER(C.c_double)
SRC = [os.path.join(EMU_DIR, "syst_emu.cpp"),
       os.path.join(ROOT, "hpcclassmultigridproject_b200", "csrc", "syst_pass_body.cuh"),
       os.path.join(ROOT, "hpcclassmultigridproject_b200", "csrc", "common.cuh")]
SO = os.path.join(EMU_DIR, "libsystemu.so")
CUDA_INCLUDE = os.path.join(os.environ.get("CUDA_HOME") or "/usr/local/cuda", "include")    # cuda_runtime.h (vector types)


def env_without_cc():
    return {k: v for k, v in os.environ.items() if k not in ("CC", "CXX")}


def stale(out, extra=()):
    deps = list(SRC) + list(extra)
    return not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in deps)


def load_model():
    """build (if stale) and load the host model of the kernel"""
    if stale(SO):
        # built under a name of this process and renamed into place: test processes running side by side (pytest -n)
        # may build it at the same time, and none may load a half-written file
        tmp = SO[: -len(".so")] + f".{os.getpid()}.so"
        subprocess.run(["g++", "-O2", "-ffp-contract=off", "-std=c++17", "-fPIC", "-shared", "-pthread",
                        "-I" + CUDA_INCLUDE, "-o", tmp, SRC[0]], check=True, env=env_without_cc())
        os.replace(tmp, SO)
    lib = C.CDLL(SO)
    lib.syst_emu_run.restype = C.c_long
    lib.syst_emu_run.argtypes = [C.c_long] * 5 + [_dp] * 8 + [C.c_int] * 3 + [C.c_double] * 3 + [C.c_int] * 3 + [C.c_long] * 6
    return lib


def layout(n):
    odd = (n // 2 + 1 + 15) // 16 * 16 + 32          # split_layout() of common.cuh
    return 2 * odd, odd


def to_split(a, fill=np.nan):
    n = a.shape[0] - 1
    pitch, odd = layout(n)
    s = np.full((n + 1, pitch), fill)
    s[:, : n // 2 + 1] = a[:, 0::2]
    s[:, odd: odd + n // 2] = a[:, 1::2]
    return s


def from_split(s, n):
    pitch, odd = layout(n)
    a = np.empty((n + 1, n + 1))
    a[:, 0::2] = s[:, : n // 2 + 1]
    a[:, 1::2] = s[:, odd: odd + n // 2]
    return a


def ptr(a):
    return None if a is None else a.ctypes.data_as(_dp)


def fields(n, seed):
    rng = np.random.default_rng(seed)
    return [rng.standard_normal((n + 1, n + 1)) for _ in range(4)]
