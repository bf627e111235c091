"""Host model (tests/emu/syst_emu_batched.cpp over the kernel's own per-thread code) of the batched streaming pass:
three members with different seeded fields in one launch, every flavour of the pass, K = 1..3 and several strip
geometries.  Each member must equal the oracle's operator sequence bit for bit (and its partial sums the
single-problem pass's); a member whose active flag is 0 must keep its NaN-filled outputs and partials.  The
planner with a member count of 1 must give the plan of one problem."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from emu_util import CUDA_INCLUDE, EMU_DIR, env_without_cc, fields, from_split, layout, load_model, ptr, stale, to_split

B_SRC = os.path.join(EMU_DIR, "syst_emu_batched.cpp")
B_SO = os.path.join(EMU_DIR, "libsystemu_batched.so")
GEOMS = [(0, 0), (24, 3), (56, 2)]       # (owned pairs per strip = SWK - 8, bands); (0, 0): the planner's
POST_NONE, POST_INJECT, POST_NORM2, POST_FW = 0, 1, 2, 3
B = 3


@pytest.fixture(scope="module")
def emu():
    """build (if stale) and load the model with the batched entry point"""
    if stale(B_SO, [B_SRC, os.path.join(EMU_DIR, "syst_emu_fw.cpp")]):
        tmp = B_SO[: -len(".so")] + f".{os.getpid()}.so"          # renamed into place: parallel test processes
        subprocess.run(["g++", "-O2", "-ffp-contract=off", "-std=c++17", "-fPIC", "-shared", "-pthread",
                        "-I" + CUDA_INCLUDE, "-o", tmp, B_SRC], check=True, env=env_without_cc())
        os.replace(tmp, B_SO)
    lib = C.CDLL(B_SO)
    dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int)
    lib.syst_emu_batched_run.restype = C.c_long
    lib.syst_emu_batched_run.argtypes = ([C.c_long] * 5 + [C.c_int, C.c_long, C.c_long, ip] + [dp] * 8 + [C.c_long]
                                         + [C.c_int] * 3 + [C.c_double] * 3 + [C.c_int] * 3)
    lib.syst_emu_plan.restype = C.c_long
    lib.syst_emu_plan.argtypes = [C.c_long, C.c_long, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_long * 5)]
    return lib


def run_batched(emu, n, us, rhs, v1, v2, K, post, arith, dt, nu, dx, cus=None, active=(1, 1, 1), wk=0, nbands=0, jitter=0):
    """us / cus: lists of B fields (us None: zero iterate).  Returns per member (u, coarse rhs, partials)."""
    pitch, odd = layout(n)
    cp, co = layout(n // 2)
    ms, cms = (n + 1) * pitch, (n // 2 + 1) * cp
    stack = lambda arrs: np.ascontiguousarray(np.stack([to_split(a) for a in arrs]))
    u_in = None if us is None else stack(us)
    out = np.full((B, n + 1, pitch), np.nan)
    crhs = np.zeros((B, n // 2 + 1, cp))
    for m in range(B):
        if not active[m]:
            crhs[m] = np.nan
    pstride = 512
    partials = np.full(B * pstride, np.nan)
    cu = None if cus is None else stack(cus)
    act = (C.c_int * B)(*active)
    nt = emu.syst_emu_batched_run(n, pitch, odd, cp, co, B, ms, cms, act, ptr(u_in), ptr(out), ptr(stack(rhs)), ptr(stack(v1)),
                                  ptr(stack(v2)), ptr(cu), ptr(crhs), ptr(partials), pstride, K, post, arith, dt, nu, dx,
                                  wk, nbands, jitter)
    assert nt > 0
    return [(out[m], crhs[m], partials[m * pstride: m * pstride + nt]) for m in range(B)]


def member_fields(n, seed):
    return [fields(n, seed + 101 * m) for m in range(B)]


def coarse(n, seed):
    c = np.random.default_rng(seed).standard_normal((n // 2 + 1, n // 2 + 1))
    c[0, :] = c[-1, :] = 0; c[:, 0] = c[:, -1] = 0             # a coarse correction has a zero boundary
    return c


FLAVOURS = [(POST_NONE, False), (POST_INJECT, False), (POST_NORM2, False), (POST_FW, False),
            (POST_NONE, True), (POST_INJECT, True), (POST_NORM2, True)]


@pytest.mark.timeout(1800)
@pytest.mark.parametrize("post,pre", FLAVOURS)
@pytest.mark.parametrize("K", [1, 2, 3])
def test_batched_pass_equals_oracle(emu, oracle, post, pre, K):
    n = 64
    fl = member_fields(n, 31 * K + 7 * post + pre)
    us = [f[0] for f in fl]; rhs = [f[1] for f in fl]; v1 = [f[2] for f in fl]; v2 = [f[3] for f in fl]
    cus = [coarse(n, 5 * m + K) for m in range(B)] if pre else None
    dx = 1.0 / n; dt = dx / 10; nu = -4e-4
    solo = load_model()
    for gi, ((wk, nb), jit) in enumerate(zip(GEOMS, (0, 4, 2))):
        active = (1, 0, 1) if gi == 1 else (1, 1, 1)
        got = run_batched(emu, n, us, rhs, v1, v2, K, post, 1, dt, nu, dx, cus=cus, active=active, wk=wk, nbands=nb, jitter=jit)
        for m in range(B):
            gu, gc, gp = got[m]
            if not active[m]:
                assert np.isnan(gu).all() and np.isnan(gc).all() and np.isnan(gp).all(), "a frozen member was written"
                continue
            want_u = us[m] + oracle.prolongation(cus[m], n // 2) if pre else us[m].copy()
            want_u = oracle.gauss_seidel(want_u, rhs[m], n, v1[m], v2[m], dt, nu, dx, K)
            assert np.array_equal(from_split(gu, n), want_u), (m, wk, nb)
            c = from_split(gc, n // 2)
            if post in (POST_INJECT, POST_FW):
                res = oracle.residual(want_u, rhs[m], n, v1[m], v2[m], dt, nu, dx)
                want_c = oracle.restriction(res, n) if post == POST_INJECT else oracle.restriction_fw(res, n)
                assert np.array_equal(c[1:-1, 1:-1], want_c[1:-1, 1:-1]), (m, wk, nb)
                assert not c[0, :].any() and not c[:, 0].any()
            else:
                assert not c.any()
            if post == POST_NORM2:
                # the same tiles as the single-problem pass of that geometry: the same partial sums
                pitch, odd = layout(n)
                cp, co = layout(n // 2)
                sp = np.zeros(4096)
                nt = solo.syst_emu_run(n, pitch, odd, cp, co, ptr(to_split(us[m])), ptr(np.full((n + 1, pitch), np.nan)),
                                       ptr(to_split(rhs[m])), ptr(to_split(v1[m])), ptr(to_split(v2[m])),
                                       ptr(to_split(cus[m]) if pre else None), ptr(np.zeros((n // 2 + 1, cp))), ptr(sp), K,
                                       POST_NORM2, 1, dt, nu, dx, wk, nb, 0, 0, 0, 0, 0, 0, 0)
                if wk or nb:
                    assert np.array_equal(gp, sp[:nt]), (m, wk, nb)
                want_r2 = oracle.norm(oracle.residual(want_u, rhs[m], n, v1[m], v2[m], dt, nu, dx), n) ** 2
                assert abs(gp.sum() - want_r2) <= 1e-12 * want_r2


@pytest.mark.timeout(900)
def test_batched_zero_iterate_and_small_level(emu, oracle):
    """u_in == NULL (a fresh coarse level): every member's rows come from an out-of-bounds box of its own; n = 8"""
    for n in (8, 32):
        fl = member_fields(n, 900 + n)
        rhs = [f[1] for f in fl]; v1 = [f[2] for f in fl]; v2 = [f[3] for f in fl]
        dx = 1.0 / n; dt = dx / 10; nu = -4e-4 * n          # a diffusion number where the coarse grid matters
        got = run_batched(emu, n, None, rhs, v1, v2, 3, POST_INJECT, 1, dt, nu, dx, jitter=4)
        for m in range(B):
            want_u = oracle.gauss_seidel(np.zeros((n + 1, n + 1)), rhs[m], n, v1[m], v2[m], dt, nu, dx, 3)
            want_c = oracle.restriction(oracle.residual(want_u, rhs[m], n, v1[m], v2[m], dt, nu, dx), n)
            assert np.array_equal(from_split(got[m][0], n), want_u), (n, m)
            assert np.array_equal(from_split(got[m][1], n // 2)[1:-1, 1:-1], want_c[1:-1, 1:-1]), (n, m)


def plan_model(n, nrows, K, sms):
    """make_plan of the parent commit (before the member count), restated"""
    HK, GROUP = 4, 4
    npairs = n // 2 + 1
    best, best_cost = None, 1e300
    for SWK in range(32, 129, 16):
        WK = SWK - 2 * HK
        nstrips = (npairs + WK - 1) // WK
        nb = 1
        while nb <= 4096:
            RB = (nrows + nb - 1) // nb
            if nb > 1 and RB < 8:
                break
            nbands = (nrows + RB - 1) // RB
            waves = (nstrips * nbands + sms - 1) // sms
            cost = waves * (RB + 2.0 * (2 * K + 1) + 4.0 * K + 2.0 * GROUP) * (96.0 + SWK)
            if cost < best_cost:
                best_cost, best = cost, (WK, SWK, nstrips, nbands, RB)
            nb = nb + 1 if nb < 16 else nb * 2
    return best


def test_plan_of_one_member_is_the_single_problem_plan(emu):
    for lg in range(3, 17):
        n = 1 << lg
        for K in (1, 2, 3):
            one, dflt = (C.c_long * 5)(), (C.c_long * 5)()
            emu.syst_emu_plan(n, n + 1, K, 148, 1, C.byref(one))
            emu.syst_emu_plan(n, n + 1, K, 148, 0, C.byref(dflt))
            assert list(one) == list(dflt) == list(plan_model(n, n + 1, K, 148)), (n, K)


def test_plan_counts_waves_over_members(emu):
    """at N = 256 one problem fills a wave with small tiles; 64 members take the widest strips and fewest bands"""
    one, many = (C.c_long * 5)(), (C.c_long * 5)()
    t1 = emu.syst_emu_plan(256, 257, 3, 148, 1, C.byref(one))
    t64 = emu.syst_emu_plan(256, 257, 3, 148, 64, C.byref(many))
    assert t64 < t1
