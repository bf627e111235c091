"""Host model of the streaming pass (tests/emu) on the smallest levels a pass runs on, n = 8 and n = 16, with random
fields whose four boundary lines are nonzero and a diffusion number D = 2 dt |nu| / dx^2 = 8, where the operator is far
from the identity.  Every flavour -- injection, residual norm, full weighting, plain smoothing, and the up leg's
prolongation followed by injection -- is compared bit for bit with the oracle's operator sequence, for K = 1..3
iterations and every strip/band geometry of the other host-model tests.  These levels are the coarse end of the deep
hierarchies the GPU level tests run (tests/test_gpu_levels.py); here their strip and ring index logic is checked
node by node."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from emu_util import CUDA_INCLUDE, EMU_DIR, env_without_cc, from_split, layout, load_model, ptr, stale, to_split

GEOMS = [(0, 0), (24, 1), (24, 3), (56, 2), (120, 2)]      # (owned pairs per strip = SWK - 8, bands); 0: the planner's
JITTER = (0, 4, 8, 2, 0)
POST_NONE, POST_INJECT, POST_NORM2 = 0, 1, 2
D = 8.0
FW_SRC = os.path.join(EMU_DIR, "syst_emu_fw.cpp")
FW_SO = os.path.join(EMU_DIR, "libsystemu_fw.so")


@pytest.fixture(scope="module")
def emu():
    return load_model()


@pytest.fixture(scope="module")
def emu_fw():
    if stale(FW_SO, [FW_SRC]):
        tmp = FW_SO[: -len(".so")] + f".{os.getpid()}.so"          # renamed into place: parallel test processes
        subprocess.run(["g++", "-O2", "-ffp-contract=off", "-std=c++17", "-fPIC", "-shared", "-pthread",
                        "-I" + CUDA_INCLUDE, "-o", tmp, FW_SRC], check=True, env=env_without_cc())
        os.replace(tmp, FW_SO)
    lib = C.CDLL(FW_SO)
    dp = C.POINTER(C.c_double)
    lib.syst_emu_fw_run.restype = C.c_long
    lib.syst_emu_fw_run.argtypes = [C.c_long] * 5 + [dp] * 6 + [C.c_int] * 2 + [C.c_double] * 3 + [C.c_int] * 3 + [C.c_long] * 6
    return lib


def problem(n, seed):
    """u, rhs, v1, v2 with O(1) values everywhere (all four boundary lines nonzero), dt = dx/10, nu for D = 8"""
    rng = np.random.default_rng(seed)
    u, rhs, v1, v2 = (rng.uniform(-1.0, 1.0, (n + 1, n + 1)) + s for s in (0.5, 0.0, 0.0, 0.0))
    for a in (u, v1, v2):
        assert a[0, :].all() and a[-1, :].all() and a[:, 0].all() and a[:, -1].all()
    dx = 1.0 / n; dt = dx / 10
    nu = -D * dx * dx / (2 * dt)
    return u, rhs, v1, v2, dt, nu, dx


def coarse_correction(n, seed):
    cu = np.random.default_rng(seed).uniform(-1.0, 1.0, (n // 2 + 1, n // 2 + 1))
    cu[0, :] = cu[-1, :] = 0; cu[:, 0] = cu[:, -1] = 0           # a coarse correction has a zero boundary
    return cu


def run(emu, n, u, rhs, v1, v2, K, post, dt, nu, dx, cu=None, wk=0, nbands=0, jitter=0):
    pitch, odd = layout(n)
    cp, co = layout(n // 2)
    out = np.full((n + 1, pitch), np.nan)
    crhs = np.zeros((n // 2 + 1, cp))
    partials = np.zeros(4096)
    cus = None if cu is None else to_split(cu)
    nt = emu.syst_emu_run(n, pitch, odd, cp, co, ptr(to_split(u)), ptr(out), ptr(to_split(rhs)), ptr(to_split(v1)),
                          ptr(to_split(v2)), ptr(cus), ptr(crhs), ptr(partials), K, post, 1, dt, nu, dx, wk, nbands,
                          jitter, 0, 0, 0, 0, 0, 0)
    assert nt > 0
    return from_split(out, n), from_split(crhs, n // 2), partials[:nt]


def boundary_kept(got, u):
    return (np.array_equal(got[0, :], u[0, :]) and np.array_equal(got[-1, :], u[-1, :])
            and np.array_equal(got[:, 0], u[:, 0]) and np.array_equal(got[:, -1], u[:, -1]))


@pytest.mark.parametrize("n", [8, 16])
@pytest.mark.parametrize("K", [1, 2, 3])
def test_down_leg_injection_and_plain_smoothing(emu, oracle, n, K):
    u, rhs, v1, v2, dt, nu, dx = problem(n, 31 * n + K)
    want_u = oracle.gauss_seidel(u.copy(), rhs, n, v1, v2, dt, nu, dx, K)
    want_c = oracle.restriction(oracle.residual(want_u, rhs, n, v1, v2, dt, nu, dx), n)
    for (wk, nb), jit in zip(GEOMS, JITTER):
        got_u, got_c, _ = run(emu, n, u, rhs, v1, v2, K, POST_INJECT, dt, nu, dx, wk=wk, nbands=nb, jitter=jit)
        assert np.array_equal(got_u, want_u), (wk, nb)
        assert boundary_kept(got_u, u), (wk, nb)
        assert np.array_equal(got_c[1:-1, 1:-1], want_c[1:-1, 1:-1]), (wk, nb)
        assert not got_c[0, :].any() and not got_c[-1, :].any() and not got_c[:, 0].any() and not got_c[:, -1].any()
        got_u, got_c, parts = run(emu, n, u, rhs, v1, v2, K, POST_NONE, dt, nu, dx, wk=wk, nbands=nb, jitter=jit)
        assert np.array_equal(got_u, want_u), (wk, nb)
        assert not got_c.any() and not parts.any(), (wk, nb)


@pytest.mark.parametrize("n", [8, 16])
@pytest.mark.parametrize("K", [1, 2, 3])
def test_up_leg_norm(emu, oracle, n, K):
    """u += P(coarse) ; K iterations ; per-tile sums of squares of the residual"""
    u, rhs, v1, v2, dt, nu, dx = problem(n, 37 * n + K)
    cu = coarse_correction(n, 5 * n + K)
    want_u = oracle.gauss_seidel(u + oracle.prolongation(cu, n // 2), rhs, n, v1, v2, dt, nu, dx, K)
    res = oracle.residual(want_u, rhs, n, v1, v2, dt, nu, dx)
    want_r2 = oracle.norm(res, n) ** 2
    for (wk, nb), jit in zip(GEOMS, JITTER):
        got_u, _, parts = run(emu, n, u, rhs, v1, v2, K, POST_NORM2, dt, nu, dx, cu=cu, wk=wk, nbands=nb, jitter=jit)
        assert np.array_equal(got_u, want_u), (wk, nb)
        assert boundary_kept(got_u, u), (wk, nb)
        # the tiles sum the same squares in another order: a few ulp of the total
        assert abs(parts.sum() - want_r2) <= 1e-13 * want_r2, (wk, nb)


@pytest.mark.parametrize("n", [8, 16])
@pytest.mark.parametrize("K", [1, 2, 3])
def test_up_leg_with_injection(emu, oracle, n, K):
    """an up-leg chunk followed by a restriction (the W-cycle's inner repetitions): prolongation + K iterations +
    residual + injection"""
    u, rhs, v1, v2, dt, nu, dx = problem(n, 41 * n + K)
    cu = coarse_correction(n, 7 * n + K)
    want_u = oracle.gauss_seidel(u + oracle.prolongation(cu, n // 2), rhs, n, v1, v2, dt, nu, dx, K)
    want_c = oracle.restriction(oracle.residual(want_u, rhs, n, v1, v2, dt, nu, dx), n)
    for (wk, nb), jit in zip(GEOMS, JITTER):
        got_u, got_c, _ = run(emu, n, u, rhs, v1, v2, K, POST_INJECT, dt, nu, dx, cu=cu, wk=wk, nbands=nb, jitter=jit)
        assert np.array_equal(got_u, want_u), (wk, nb)
        assert np.array_equal(got_c[1:-1, 1:-1], want_c[1:-1, 1:-1]), (wk, nb)


@pytest.mark.parametrize("n", [8, 16])
@pytest.mark.parametrize("K", [1, 2, 3])
def test_down_leg_full_weighting(emu_fw, oracle, n, K):
    u, rhs, v1, v2, dt, nu, dx = problem(n, 43 * n + K)
    want_u = oracle.gauss_seidel(u.copy(), rhs, n, v1, v2, dt, nu, dx, K)
    want_c = oracle.restriction_fw(oracle.residual(want_u, rhs, n, v1, v2, dt, nu, dx), n)
    pitch, odd = layout(n)
    cp, co = layout(n // 2)
    for (wk, nb), jit in zip(GEOMS, JITTER):
        out = np.full((n + 1, pitch), np.nan)
        crhs = np.zeros((n // 2 + 1, cp))
        nt = emu_fw.syst_emu_fw_run(n, pitch, odd, cp, co, ptr(to_split(u)), ptr(out), ptr(to_split(rhs)),
                                    ptr(to_split(v1)), ptr(to_split(v2)), ptr(crhs), K, 1, dt, nu, dx, wk, nb, jit,
                                    0, 0, 0, 0, 0, 0)
        assert nt > 0
        got_u, got_c = from_split(out, n), from_split(crhs, n // 2)
        assert np.array_equal(got_u, want_u), (wk, nb)
        assert boundary_kept(got_u, u), (wk, nb)
        assert np.array_equal(got_c[1:-1, 1:-1], want_c[1:-1, 1:-1]), (wk, nb)
        assert not got_c[0, :].any() and not got_c[-1, :].any() and not got_c[:, 0].any() and not got_c[:, -1].any()
