"""The oracle restatement (oracle/mg_oracle.c) against every known answer we hold:
golden vectors generated from the compiled reference (tests/golden/make_golden.py) and the
stdout of the reference's own print tests.  Bit-for-bit wherever the data is binary."""
import json
import math
import os
import re

import numpy as np
import pytest

from conftest import GOLDEN, golden
from oracle.oracle import OracleSolver


@pytest.mark.parametrize("name", ["ops_n32.npz", "ops_n64.npz"])
def test_operators_bitwise(oracle, name):
    g = golden(name)
    n = int(g["n"]); dx, dt, nu = float(g["dx"]), float(g["dt"]), float(g["nu"])
    u, rhs, v1, v2 = g["u"], g["rhs"], g["v1"], g["v2"]
    assert np.array_equal(oracle.compute_rhs(u, n, v1, v2, dt, nu, dx), g["compute_rhs"])
    res = oracle.residual(u, rhs, n, v1, v2, dt, nu, dx)
    assert np.array_equal(res, g["residual"])
    assert oracle.norm(res, n) == float(g["norm"])
    assert np.array_equal(oracle.gauss_seidel(u.copy(), rhs, n, v1, v2, dt, nu, dx, 1), g["gs1"])
    assert np.array_equal(oracle.gauss_seidel(u.copy(), rhs, n, v1, v2, dt, nu, dx, 3), g["gs3"])
    assert np.array_equal(oracle.restriction(u, n), g["restriction"])
    assert np.array_equal(oracle.prolongation(u, n), g["prolongation"])


SOLVES = ["solve_n32", "solve_n64", "solve_n128", "solve_n256", "solve_cfg_wcycle_n128",
          "solve_cfg_tight_n256", "solve_cfg_adv_n256", "solve_cfg_diff_n256", "solve_cfg_n512",
          "solve_cfg_n1024"]


def exact_norm(a):
    """||a||_2 from the correctly rounded sum of the squares: the same bits on every host, unlike np.linalg.norm,
    whose summation order follows the BLAS kernel and its thread count"""
    return math.sqrt(math.fsum(np.square(a).ravel()))


@pytest.mark.parametrize("tag", SOLVES)
def test_time_steps_bitwise(oracle, tag):
    g = golden(tag + ".npz")
    n, steps = int(g["n"]), int(g["steps"])
    u0, v1, v2 = oracle.initial_conditions(n, float(g["vscale"]))
    s = OracleSolver(n, u0, v1, v2, float(g["nu"]), float(g["dt"]), float(g["dx"]), float(g["tol"]),
                     int(g["shape"]))
    for k in range(steps):
        s.form_rhs()
        it, hist = s.solve()
        assert it == int(g["cycles"][k])
        assert np.array_equal(hist, g["hist"][k][: it + 1])      # norms bit-for-bit (same serial sum)
    uT = s.u(0)
    # the npz's norm_uT carries the rounding of the BLAS that computed it.  With a stored field the norm is taken from
    # it (the array_equal below already implies this check); without one, from tests/golden/make_golden_norms.py
    if "uT" in g:
        want_norm = exact_norm(g["uT"])
    else:
        want_norm = json.load(open(os.path.join(GOLDEN, "solve_norms.json")))[tag]
    assert exact_norm(uT) == want_norm
    assert uT[n // 2, n // 2] == float(g["mid"])
    if "uT" in g:
        assert np.array_equal(uT, g["uT"])
    s.close()


def test_reference_main_output(oracle):
    """multigrid.cpp main(): N=256, 100 steps, its own inline ICs -> uT.txt (6 decimals)."""
    g = golden("refmain_uT_n256_100steps.npz")
    n = 256; dx = 1.0 / n; dt = dx / 10
    u0, v1, v2 = oracle.initial_conditions(n)
    uT = oracle.timestepper(u0, v1, v2, -4e-4, n, dt, 100, dx, 1e-6)
    assert np.abs(uT - g["uT"].astype(np.float64)).max() < 6e-7     # %f rounding + float32 storage


def _blocks(path):
    out, cur, key = {}, None, None
    for line in open(path):
        line = line.rstrip("\n")
        if re.match(r"^[A-Za-z]", line) and not line.startswith("res norm"):
            key = line.strip(); out[key] = []
        elif line.startswith("res norm"):
            out["res norm"] = float(line.split(":")[1])
        elif line.strip() and key:
            out[key].append([float(x) for x in line.split()])
    return {k: (np.array(v) if isinstance(v, list) else v) for k, v in out.items()}


def test_known_answer_prolrestest(oracle):
    """prolrestest.cpp:76-118 -- ramp i+j on 6x6 prolongs to (I+J)/2 on 11x11; restriction undoes it."""
    b = _blocks(os.path.join(GOLDEN, "prolrestest_stdout.txt"))
    n = 5
    up = np.add.outer(np.arange(n + 1.0), np.arange(n + 1.0))
    assert np.array_equal(up, b["Original matrix"])
    fine = oracle.prolongation(up, n)
    assert np.array_equal(fine, b["Prolongated matrix"])
    assert np.array_equal(fine, np.add.outer(np.arange(2 * n + 1.0), np.arange(2 * n + 1.0)) / 2)
    assert np.array_equal(oracle.restriction(fine, 2 * n), b["Restriction matrix"])


def test_known_answer_resnormtest(oracle):
    """resnormtest.cpp:210-283 -- N=5 Gaussian/vortex (boundary of u NOT zeroed there):
    rhs, residual (4 decimals), 'res norm: 0.149437', and u after one RB iteration."""
    b = _blocks(os.path.join(GOLDEN, "resnormtest_stdout.txt"))
    n = 5; dx = 1.0 / n; dt = dx / 10; nu = -4e-4
    PI = 3.1415926535897932
    i = np.arange(n + 1.0)[:, None]; j = np.arange(n + 1.0)[None, :]
    u = np.exp(-100.0 * ((i * dx - 0.2) ** 2 + (j * dx - 0.4) ** 2))
    v1 = -PI * np.sin(PI * i * dx) * np.cos(PI * j * dx)
    v2 = PI * np.cos(PI * i * dx) * np.sin(PI * j * dx)
    rhs = oracle.compute_rhs(u, n, v1, v2, dt, nu, dx)
    res = oracle.residual(u, rhs, n, v1, v2, dt, nu, dx)
    assert np.abs(rhs - b["rhs matrix"]).max() <= 5.01e-5
    assert np.abs(res - b["res matrix"]).max() <= 5.01e-5
    assert abs(oracle.norm(res, n) - b["res norm"]) <= 5.01e-7
    # the reference test then calls gauss_seidel2 (summation order c,d,a,b: gs.cpp:209), ours is
    # gauss_seidel's c,a,d,b (gs.cpp:130): equal to print precision
    u1 = oracle.gauss_seidel(u.copy(), rhs, n, v1, v2, dt, nu, dx, 1)
    assert np.abs(u1 - b["u matrix"]).max() <= 5.01e-5


def test_initial_condition_quirks(oracle):
    """multigrid.cpp:227-233: boundary zeroed with i < N, so node (N,0) keeps exp(-80)."""
    n = 64
    u0, v1, v2 = oracle.initial_conditions(n)
    assert u0[0, :].max() == 0 and u0[:, n].max() == 0 and u0[n, 1:].max() == 0 and u0[:n, 0].max() == 0
    assert u0[n, 0] > 0 and abs(u0[n, 0] / np.exp(-80.0) - 1) < 1e-12
    u0s, v1s, v2s = oracle.initial_conditions(n, 3.0)
    assert np.array_equal(u0s, u0) and np.array_equal(v1s, v1 * 3.0) and np.array_equal(v2s, v2 * 3.0)


def test_coarse_velocity_tower_quirk(oracle):
    """SURVEY.md section 8 P1 (multigrid.cpp:148-160): every coarse velocity level is filled by
    restriction(dst, src, N/2) on zero-filled (N/2+1)^2 buffers, read back with the true stride."""
    n = 128
    u0, v1, v2 = oracle.initial_conditions(n)
    s = OracleSolver(n, u0, v1, v2, -4e-4, 1.0 / n / 10, 1.0 / n, 1e-6)
    nh, nq = n // 2, n // 4
    flat1 = np.zeros((nh + 1) ** 2)
    src = v1.reshape(-1)
    for i in range(nq + 1):
        for j in range(nq + 1):
            flat1[i * (nq + 1) + j] = src[2 * i * (nh + 1) + 2 * j]
    assert np.array_equal(s.v1(1).reshape(-1), flat1)
    flat2 = np.zeros((nh + 1) ** 2)
    for i in range(nq + 1):
        for j in range(nq + 1):
            flat2[i * (nq + 1) + j] = flat1[2 * i * (nh + 1) + 2 * j]
    assert np.array_equal(s.v1(2).reshape(-1), flat2[: (nq + 1) ** 2])
    s.close()


def test_full_weighting_restatement(oracle):
    """orc_restriction_fw restates lines the reference keeps commented out (gs.cpp:277-280), so there is
    no compiled twin to pin it to: check it against the written formula and its defining properties"""
    rng = np.random.default_rng(7)
    nf = 16
    f = rng.standard_normal((nf + 1, nf + 1))
    c = oracle.restriction_fw(f, nf)
    I, J = 3, 5
    want = (f[2*I-1, 2*J-1] + 2*f[2*I-1, 2*J] + f[2*I-1, 2*J+1]) / 16
    want += (2*f[2*I, 2*J-1] + 4*f[2*I, 2*J] + 2*f[2*I, 2*J+1]) / 16
    want += (f[2*I+1, 2*J-1] + 2*f[2*I+1, 2*J] + f[2*I+1, 2*J+1]) / 16
    assert c[I, J] == want
    assert np.array_equal(c[0, :], f[0, ::2]) and np.array_equal(c[:, -1], f[::2, -1])      # boundary: injection
    assert np.array_equal(oracle.restriction_fw(np.ones_like(f), nf), np.ones((nf // 2 + 1, nf // 2 + 1)))   # weights sum to 1
    ramp = np.add.outer(np.arange(nf + 1.0), 2.0 * np.arange(nf + 1.0))
    assert np.array_equal(oracle.restriction_fw(ramp, nf), ramp[::2, ::2])                   # exact on linear functions
