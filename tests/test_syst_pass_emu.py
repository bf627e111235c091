"""Host model of the systolic streaming kernel (tests/emu/syst_emu.cpp compiles the SAME per-thread
code as the CUDA kernel, csrc/syst_pass_body.cuh, and runs every lane of a block as a real thread
with the hardware's mbarrier semantics) against the oracle: ring / pipeline / halo index logic and
the barrier protocol, checked bit-for-bit with NaN-poisoned shared memory; a ThreadSanitizer build
of the same model reports every pair of conflicting shared-memory accesses the protocol leaves
unordered."""
import os
import subprocess

import numpy as np
import pytest

from emu_util import CUDA_INCLUDE, EMU_DIR, SRC, env_without_cc, fields, from_split, layout, load_model, ptr, stale, to_split


@pytest.fixture(scope="module")
def emu():
    return load_model()


def run(emu, n, u, rhs, v1, v2, K, post, arith, dt, nu, dx, cu=None, wk=0, nbands=0, jitter=0):
    pitch, odd = layout(n)
    cp, co = layout(n // 2)
    us = None if u is None else to_split(u)
    out = np.full((n + 1, pitch), np.nan)
    crhs = np.zeros((n // 2 + 1, cp))
    partials = np.zeros(4096)
    cus = None if cu is None else to_split(cu)
    nt = emu.syst_emu_run(n, pitch, odd, cp, co, ptr(us), ptr(out), ptr(to_split(rhs)), ptr(to_split(v1)),
                          ptr(to_split(v2)), ptr(cus), ptr(crhs), ptr(partials), K, post, arith, dt, nu, dx, wk, nbands,
                          jitter, 0, 0, 0, 0, 0, 0)
    assert nt > 0
    return from_split(out, n), from_split(crhs, n // 2), partials[:nt]


GEOMS = [(0, 0), (24, 1), (24, 3), (56, 2), (120, 2)]      # (owned pairs per strip = SWK - 8, bands)


@pytest.mark.timeout(900)
@pytest.mark.parametrize("n", [32, 64, 200])
@pytest.mark.parametrize("K", [1, 2, 3])
def test_down_leg(emu, oracle, n, K):
    """K RB iterations + residual + injection in one pass == oracle operator sequence, bitwise"""
    u, rhs, v1, v2 = fields(n, 7 * n + K)
    dx = 1.0 / n; dt = dx / 10; nu = -4e-4
    want_u = oracle.gauss_seidel(u.copy(), rhs, n, v1, v2, dt, nu, dx, K)
    want_c = oracle.restriction(oracle.residual(want_u, rhs, n, v1, v2, dt, nu, dx), n)
    for (wk, nb), jit in zip(GEOMS, (0, 4, 8, 2, 0)):
        got_u, got_c, _ = run(emu, n, u, rhs, v1, v2, K, 1, 1, dt, nu, dx, wk=wk, nbands=nb, jitter=jit)
        assert np.array_equal(got_u, want_u), (wk, nb)
        assert np.array_equal(got_c[1:-1, 1:-1], want_c[1:-1, 1:-1]), (wk, nb)
        assert not got_c[0, :].any() and not got_c[:, 0].any()       # coarse rhs boundary untouched


@pytest.mark.timeout(900)
@pytest.mark.parametrize("n", [32, 64, 200])
@pytest.mark.parametrize("K", [1, 3])
def test_up_leg(emu, oracle, n, K):
    """u += P(coarse) ; K RB iterations ; sum of squares of the residual"""
    u, rhs, v1, v2 = fields(n, 11 * n + K)
    cu = np.random.default_rng(n).standard_normal((n // 2 + 1, n // 2 + 1))
    cu[0, :] = cu[-1, :] = 0; cu[:, 0] = cu[:, -1] = 0           # a coarse correction has a zero boundary
    dx = 1.0 / n; dt = dx / 10; nu = -4e-4
    want_u = u + oracle.prolongation(cu, n // 2)
    want_u = oracle.gauss_seidel(want_u, rhs, n, v1, v2, dt, nu, dx, K)
    want_r2 = oracle.norm(oracle.residual(want_u, rhs, n, v1, v2, dt, nu, dx), n) ** 2
    for (wk, nb), jit in zip(GEOMS, (8, 0, 4, 2, 0)):
        got_u, _, parts = run(emu, n, u, rhs, v1, v2, K, 2, 1, dt, nu, dx, cu=cu, wk=wk, nbands=nb, jitter=jit)
        assert np.array_equal(got_u, want_u), (wk, nb)
        assert abs(parts.sum() - want_r2) <= 1e-12 * want_r2


@pytest.mark.timeout(900)
def test_plain_smoothing_zero_input_and_fast_arithmetic(emu, oracle):
    n = 128
    u, rhs, v1, v2 = fields(n, 5)
    dx = 1.0 / n; dt = dx / 10; nu = -4e-4
    want = oracle.gauss_seidel(np.zeros((n + 1, n + 1)), rhs, n, v1, v2, dt, nu, dx, 3)
    got, _, _ = run(emu, n, None, rhs, v1, v2, 3, 1, 1, dt, nu, dx)          # u_in == NULL: u is zero
    assert np.array_equal(got, want)
    gotf, _, _ = run(emu, n, None, rhs, v1, v2, 3, 1, 0, dt, nu, dx, wk=40, nbands=3, jitter=4)
    assert np.linalg.norm(gotf - want) <= 1e-13 * np.linalg.norm(want)
    want2 = oracle.gauss_seidel(u.copy(), rhs, n, v1, v2, dt, nu, dx, 2)     # no epilogue at all
    got2, crhs, parts = run(emu, n, u, rhs, v1, v2, 2, 0, 1, dt, nu, dx, wk=56, nbands=2)
    assert np.array_equal(got2, want2) and not crhs.any() and not parts.any()


@pytest.mark.timeout(1800)
@pytest.mark.parametrize("wk,nb", [(56, 3), (120, 2)])
def test_interior_strips_run_the_mask_free_step(emu, oracle, wk, nb):
    """n = 512: the middle strips touch neither side of the domain and run the step without masks (every lane stores,
    the strip's outermost pairs hold halo garbage); both legs must still equal the oracle bit for bit"""
    n = 512
    u, rhs, v1, v2 = fields(n, 77)
    cu = np.random.default_rng(8).standard_normal((n // 2 + 1, n // 2 + 1))
    cu[0, :] = cu[-1, :] = 0; cu[:, 0] = cu[:, -1] = 0
    dx = 1.0 / n; dt = dx / 10; nu = -4e-4
    want_u = oracle.gauss_seidel(u.copy(), rhs, n, v1, v2, dt, nu, dx, 3)
    want_c = oracle.restriction(oracle.residual(want_u, rhs, n, v1, v2, dt, nu, dx), n)
    got_u, got_c, _ = run(emu, n, u, rhs, v1, v2, 3, 1, 1, dt, nu, dx, wk=wk, nbands=nb, jitter=2)
    assert np.array_equal(got_u, want_u)
    assert np.array_equal(got_c[1:-1, 1:-1], want_c[1:-1, 1:-1])
    want_u = oracle.gauss_seidel(u + oracle.prolongation(cu, n // 2), rhs, n, v1, v2, dt, nu, dx, 3)
    want_r2 = oracle.norm(oracle.residual(want_u, rhs, n, v1, v2, dt, nu, dx), n) ** 2
    got_u, _, parts = run(emu, n, u, rhs, v1, v2, 3, 2, 1, dt, nu, dx, cu=cu, wk=wk, nbands=nb, jitter=0)
    assert np.array_equal(got_u, want_u)
    assert abs(parts.sum() - want_r2) <= 1e-12 * want_r2


@pytest.mark.timeout(900)
def test_pre_with_injection(emu, oracle):
    """an up-leg chunk that is followed by nothing (W-cycle inner repetitions): prolongation + smoothing + injection"""
    n = 64
    u, rhs, v1, v2 = fields(n, 21)
    cu = np.random.default_rng(4).standard_normal((n // 2 + 1, n // 2 + 1))
    cu[0, :] = cu[-1, :] = 0; cu[:, 0] = cu[:, -1] = 0
    dx = 1.0 / n; dt = dx / 10; nu = -4e-4
    want_u = oracle.gauss_seidel(u + oracle.prolongation(cu, n // 2), rhs, n, v1, v2, dt, nu, dx, 3)
    want_c = oracle.restriction(oracle.residual(want_u, rhs, n, v1, v2, dt, nu, dx), n)
    got_u, got_c, _ = run(emu, n, u, rhs, v1, v2, 3, 1, 1, dt, nu, dx, cu=cu, wk=24, nbands=2, jitter=4)
    assert np.array_equal(got_u, want_u)
    assert np.array_equal(got_c[1:-1, 1:-1], want_c[1:-1, 1:-1])


@pytest.mark.timeout(900)
@pytest.mark.parametrize("P", [2, 4])
def test_row_slabs(emu, oracle, P):
    """the same pass on row slabs (own rows + 8 halo rows held, like the sharded solver's windows): every slab is
    computed from its own window only and the pieces equal the unsharded oracle result"""
    n, K, HALO = 128, 3, 8
    u, rhs, v1, v2 = fields(n, 99)
    cu = np.random.default_rng(3).standard_normal((n // 2 + 1, n // 2 + 1))
    cu[0, :] = cu[-1, :] = 0; cu[:, 0] = cu[:, -1] = 0
    dx = 1.0 / n; dt = dx / 10; nu = -4e-4
    start = u + oracle.prolongation(cu, n // 2)
    want_u = oracle.gauss_seidel(start.copy(), rhs, n, v1, v2, dt, nu, dx, K)
    want_c = oracle.restriction(oracle.residual(want_u, rhs, n, v1, v2, dt, nu, dx), n)
    pitch, odd = layout(n); cp, co = layout(n // 2)
    S = [to_split(a) for a in (u, rhs, v1, v2)]
    CU = to_split(cu)
    got_u = np.full((n + 1, n + 1), np.nan)
    got_c = np.zeros((n // 2 + 1, n // 2 + 1))
    per = n // P
    for r in range(P):
        own_lo, own_hi = r * per, (r + 1) * per - 1 + (1 if r == P - 1 else 0)
        mem_lo, mem_hi = max(0, own_lo - HALO), min(n, own_hi + HALO)
        clo, chi = max(0, (own_lo + 1) // 2 - HALO), min(n // 2, own_hi // 2 + HALO)
        win = [np.ascontiguousarray(a[mem_lo:mem_hi + 1]) for a in S]
        cwin = np.ascontiguousarray(CU[clo:chi + 1])
        out = np.full((mem_hi - mem_lo + 1, pitch), np.nan)
        crhs = np.zeros((chi - clo + 1, cp))
        parts = np.zeros(4096)
        nt = emu.syst_emu_run(n, pitch, odd, cp, co, ptr(win[0]), ptr(out), ptr(win[1]), ptr(win[2]), ptr(win[3]), ptr(cwin),
                              ptr(crhs), ptr(parts), K, 1, 1, dt, nu, dx, 56, 2, 2, own_lo, own_hi, mem_lo, mem_hi - mem_lo + 1,
                              clo, chi - clo + 1)
        assert nt > 0
        full = np.full((n + 1, pitch), np.nan); full[mem_lo:mem_hi + 1] = out
        got_u[own_lo:own_hi + 1] = from_split(full, n)[own_lo:own_hi + 1]
        cfull = np.zeros((n // 2 + 1, cp)); cfull[clo:chi + 1] = crhs
        c = from_split(cfull, n // 2)
        ilo, ihi = (own_lo + 1) // 2, own_hi // 2
        got_c[ilo:ihi + 1] = c[ilo:ihi + 1]
    assert np.array_equal(got_u, want_u)
    assert np.array_equal(got_c[1:-1, 1:-1], want_c[1:-1, 1:-1])


@pytest.mark.timeout(1800)
def test_barrier_protocol_under_thread_sanitizer():
    """The same model built with -fsanitize=thread, driven by tests/emu/syst_tsan_main.cpp over the pass flavours
    (both legs, K = 1..3, one and two warps per stage, several bands): no unordered conflicting access."""
    exe = os.path.join(EMU_DIR, "syst_tsan")
    main = os.path.join(EMU_DIR, "syst_tsan_main.cpp")
    if stale(exe, [main]):
        r = subprocess.run(["g++", "-O1", "-g", "-fsanitize=thread", "-ffp-contract=off", "-std=c++17", "-pthread",
                            "-I" + CUDA_INCLUDE, "-o", exe, main, SRC[0]], capture_output=True, text=True, env=env_without_cc())
        assert r.returncode == 0, r.stderr[-3000:]
    env = dict(env_without_cc(), TSAN_OPTIONS="halt_on_error=0 report_signal_unsafe=0 history_size=4")
    r = subprocess.run([exe], capture_output=True, text=True, env=env, timeout=1700)
    assert "ThreadSanitizer" not in r.stderr, r.stderr[:6000]
    assert r.returncode == 0, (r.returncode, r.stdout[-2000:], r.stderr[-2000:])
    assert "all passes done" in r.stdout
