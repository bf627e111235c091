"""Host model (tests/emu/syst_emu_fw.cpp over syst_emu.cpp, the kernel's own per-thread code) of the full-weighting
down-leg pass,
POST_FW: K RB iterations, the residual, and its full-weighting restriction onto the coarse interior in one pass.
Checked bit for bit against the oracle's operator sequence, on whole levels and on row slabs, and under
ThreadSanitizer for the protocol of the residual rows the last stage and the EPI role share."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from emu_util import CUDA_INCLUDE, EMU_DIR, env_without_cc, fields, from_split, layout, ptr, stale, to_split

FW_SRC = os.path.join(EMU_DIR, "syst_emu_fw.cpp")
FW_SO = os.path.join(EMU_DIR, "libsystemu_fw.so")
GEOMS = [(0, 0), (24, 1), (24, 3), (56, 2), (120, 2)]      # (owned pairs per strip = SWK - 8, bands)


@pytest.fixture(scope="module")
def emu():
    """build (if stale) and load the model with the POST_FW entry point"""
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


def run_fw(emu, n, u, rhs, v1, v2, K, arith, dt, nu, dx, wk=0, nbands=0, jitter=0):
    pitch, odd = layout(n)
    cp, co = layout(n // 2)
    out = np.full((n + 1, pitch), np.nan)
    crhs = np.zeros((n // 2 + 1, cp))
    nt = emu.syst_emu_fw_run(n, pitch, odd, cp, co, ptr(to_split(u)), ptr(out), ptr(to_split(rhs)), ptr(to_split(v1)),
                             ptr(to_split(v2)), ptr(crhs), K, arith, dt, nu, dx, wk, nbands, jitter, 0, 0, 0, 0, 0, 0)
    assert nt > 0
    return from_split(out, n), from_split(crhs, n // 2)


def want_fw(oracle, n, u, rhs, v1, v2, K, dt, nu, dx):
    want_u = oracle.gauss_seidel(u.copy(), rhs, n, v1, v2, dt, nu, dx, K)
    return want_u, oracle.restriction_fw(oracle.residual(want_u, rhs, n, v1, v2, dt, nu, dx), n)


@pytest.mark.timeout(900)
@pytest.mark.parametrize("n", [32, 64, 200])
@pytest.mark.parametrize("K", [1, 2, 3])
def test_down_leg_full_weighting(emu, oracle, n, K):
    """K RB iterations + residual + full weighting in one pass == gauss_seidel x K ; residual ; restriction_fw"""
    u, rhs, v1, v2 = fields(n, 13 * n + K)
    dx = 1.0 / n; dt = dx / 10; nu = -4e-4
    want_u, want_c = want_fw(oracle, n, u, rhs, v1, v2, K, dt, nu, dx)
    for (wk, nb), jit in zip(GEOMS, (0, 4, 8, 2, 0)):
        got_u, got_c = run_fw(emu, n, u, rhs, v1, v2, K, 1, dt, nu, dx, wk=wk, nbands=nb, jitter=jit)
        assert np.array_equal(got_u, want_u), (wk, nb)
        assert np.array_equal(got_c[1:-1, 1:-1], want_c[1:-1, 1:-1]), (wk, nb)
        assert not got_c[0, :].any() and not got_c[-1, :].any() and not got_c[:, 0].any() and not got_c[:, -1].any()


@pytest.mark.timeout(1800)
@pytest.mark.parametrize("wk,nb", [(56, 3), (120, 2)])
def test_interior_strips_mask_free(emu, oracle, wk, nb):
    """n = 512: the middle strips run the mask-free step in the last stage, whose residual feeds the restriction"""
    n, K = 512, 3
    u, rhs, v1, v2 = fields(n, 78)
    dx = 1.0 / n; dt = dx / 10; nu = -4e-4
    want_u, want_c = want_fw(oracle, n, u, rhs, v1, v2, K, dt, nu, dx)
    got_u, got_c = run_fw(emu, n, u, rhs, v1, v2, K, 1, dt, nu, dx, wk=wk, nbands=nb, jitter=2)
    assert np.array_equal(got_u, want_u)
    assert np.array_equal(got_c[1:-1, 1:-1], want_c[1:-1, 1:-1])


@pytest.mark.timeout(900)
def test_fast_arithmetic_close(emu, oracle):
    n = 128
    u, rhs, v1, v2 = fields(n, 6)
    dx = 1.0 / n; dt = dx / 10; nu = -4e-4
    want_u, want_c = want_fw(oracle, n, u, rhs, v1, v2, 3, dt, nu, dx)
    got_u, got_c = run_fw(emu, n, u, rhs, v1, v2, 3, 0, dt, nu, dx, wk=40, nbands=3, jitter=4)
    assert np.linalg.norm(got_u - want_u) <= 1e-13 * np.linalg.norm(want_u)
    assert np.linalg.norm(got_c[1:-1, 1:-1] - want_c[1:-1, 1:-1]) <= 1e-9 * np.linalg.norm(want_c[1:-1, 1:-1])   # (the residual cancels: relative error above u's)


@pytest.mark.timeout(900)
@pytest.mark.parametrize("P", [2, 4])
@pytest.mark.parametrize("K", [1, 3])
def test_row_slabs(emu, oracle, P, K):
    """row slabs holding own rows + 8 halo rows (the sharded solver's windows): each slab restricts the coarse rows
    under its own even rows from its window alone, and the union equals the unsharded result"""
    n, HALO = 128, 8
    u, rhs, v1, v2 = fields(n, 101 + K)
    dx = 1.0 / n; dt = dx / 10; nu = -4e-4
    want_u, want_c = want_fw(oracle, n, u, rhs, v1, v2, K, dt, nu, dx)
    pitch, odd = layout(n); cp, co = layout(n // 2)
    S = [to_split(a) for a in (u, rhs, v1, v2)]
    got_u = np.full((n + 1, n + 1), np.nan)
    got_c = np.full((n // 2 + 1, n // 2 + 1), np.nan)
    per = n // P
    for r in range(P):
        own_lo, own_hi = r * per, (r + 1) * per - 1 + (1 if r == P - 1 else 0)
        mem_lo, mem_hi = max(0, own_lo - HALO), min(n, own_hi + HALO)
        clo, chi = max(0, (own_lo + 1) // 2 - HALO), min(n // 2, own_hi // 2 + HALO)
        win = [np.ascontiguousarray(a[mem_lo:mem_hi + 1]) for a in S]
        out = np.full((mem_hi - mem_lo + 1, pitch), np.nan)
        crhs = np.zeros((chi - clo + 1, cp))
        nt = emu.syst_emu_fw_run(n, pitch, odd, cp, co, ptr(win[0]), ptr(out), ptr(win[1]), ptr(win[2]), ptr(win[3]),
                                 ptr(crhs), K, 1, dt, nu, dx, 56, 2, 2, own_lo, own_hi, mem_lo, mem_hi - mem_lo + 1,
                                 clo, chi - clo + 1)
        assert nt > 0
        full = np.full((n + 1, pitch), np.nan); full[mem_lo:mem_hi + 1] = out
        got_u[own_lo:own_hi + 1] = from_split(full, n)[own_lo:own_hi + 1]
        cfull = np.zeros((n // 2 + 1, cp)); cfull[clo:chi + 1] = crhs
        ilo, ihi = (own_lo + 1) // 2, own_hi // 2
        got_c[ilo:ihi + 1] = from_split(cfull, n // 2)[ilo:ihi + 1]
    assert np.array_equal(got_u, want_u)
    assert np.array_equal(got_c[1:-1, 1:-1], want_c[1:-1, 1:-1])


@pytest.mark.timeout(1800)
def test_residual_rows_protocol_under_thread_sanitizer():
    """the model built with -fsanitize=thread over the POST_FW pass (K = 1..3, one and two warps per stage, several
    bands, the mask-free step): no unordered conflicting access"""
    exe = os.path.join(EMU_DIR, "syst_tsan_fw")
    main = os.path.join(EMU_DIR, "syst_tsan_fw_main.cpp")
    if stale(exe, [main, FW_SRC]):
        r = subprocess.run(["g++", "-O1", "-g", "-fsanitize=thread", "-ffp-contract=off", "-std=c++17", "-pthread",
                            "-I" + CUDA_INCLUDE, "-o", exe, main, FW_SRC], capture_output=True, text=True, env=env_without_cc())
        assert r.returncode == 0, r.stderr[-3000:]
    env = dict(env_without_cc(), TSAN_OPTIONS="halt_on_error=0 report_signal_unsafe=0 history_size=4")
    r = subprocess.run([exe], capture_output=True, text=True, env=env, timeout=1700)
    assert "ThreadSanitizer" not in r.stderr, r.stderr[:6000]
    assert r.returncode == 0, (r.returncode, r.stdout[-2000:], r.stderr[-2000:])
    assert "all passes done" in r.stdout
