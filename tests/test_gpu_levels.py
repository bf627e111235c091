"""The solver at every level count it accepts, on random fields with nonzero Dirichlet boundaries, at diffusion numbers
where the coarse grid does work.

The diffusion number is D = 2 dt |nu| / dx^2.  With the reference's dt = dx/10 and nu = -4e-4 it stays below 0.1 for
every n <= 1024: the operator is then almost the identity and a wrong coarse-grid correction barely shows in the
converged field.  Here nu is chosen per case from a target D in {0.02, 1, 8} (plus dt = dx at D = 1), and the fields are
seeded random numbers, O(1) everywhere including all four boundary lines, so that every kernel that reads a boundary
value has to read the right one.

Covered: every (n, maxlvl) with n in 4..256 whose coarsest level has 4 <= n_c <= 64 (25 pairs) plus two deep and
shallow hierarchies at n = 1024; both plans; EXACT arithmetic bit for bit against the oracle on every level after
every cycle; FAST fused = unfused bit for bit, and FAST against the EXACT oracle; the restriction, coarse_exact,
correct_towers and niter options at the edge levels; the reported residual norms against a long-double
restatement of the operator; the drop-in entry points (mg_inner / mg_outer on caller-owned towers, the gs.h host
operators, the one-call timestepper and its handle cache) and their argument checks; row slabs on 2 and 4 GPUs."""
import ctypes as C
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from oracle.oracle import OracleSolver, _p
from oracle_fw import FwOracleSolver

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

EPS = np.finfo(np.float64).eps
LD = np.longdouble


@pytest.fixture(scope="module")
def mg():
    import hpcclassmultigridproject_b200 as m
    m.lib()
    assert torch.cuda.is_available()
    return m


# ---- inputs -------------------------------------------------------------------------------------------------------
def valid_pairs(n):
    """every maxlvl the solver accepts at n: the coarsest level n >> (maxlvl-1) has 4..64 nodes per side"""
    return [(n, m) for m in range(1, int(math.log2(n)) + 1) if 4 <= n >> (m - 1) <= 64]


PAIRS = [p for n in (4, 8, 16, 32, 64, 128, 256) for p in valid_pairs(n)] + [(1024, 5), (1024, 9)]
assert len(PAIRS) == 27
# (D, dt/dx): the reference's dt = dx/10 at three diffusion numbers, and dt = dx
REGIMES = [(0.02, 0.1), (1.0, 0.1), (8.0, 0.1), (1.0, 1.0)]
PLANS = ["unfused", "fused"]


def pair_id(p):
    return f"n{p[0]}-m{p[1]}"


def regime_id(r):
    return f"D{r[0]:g}-dt{r[1]:g}dx"


def plan_id(mg, name):
    return mg.PLAN_UNFUSED if name == "unfused" else mg.PLAN_FUSED


def problem(n, D, dtfac=0.1, seed=0):
    """seeded u0, v1, v2 of shape (n+1)^2, O(1) and nonzero on all four boundary lines; dt = dtfac*dx and nu for the
    target diffusion number D = 2 dt |nu| / dx^2"""
    rng = np.random.default_rng(seed * 1000003 + n)
    u0 = rng.uniform(0.25, 1.25, (n + 1, n + 1)) * rng.choice([-1.0, 1.0], (n + 1, n + 1))
    v1 = rng.uniform(-1.0, 1.0, (n + 1, n + 1))
    v2 = rng.uniform(-1.0, 1.0, (n + 1, n + 1))
    for a in (u0, v1, v2):
        assert a[0, :].all() and a[-1, :].all() and a[:, 0].all() and a[:, -1].all()
    dx = 1.0 / n
    dt = dtfac * dx
    nu = -D * dx * dx / (2.0 * dt)
    return u0, v1, v2, nu, dt, dx


# ---- the high-precision reference: A and B of orc_residual / orc_compute_rhs (mg_oracle.c:53-83) in long double ----
def _apply(u, v1, v2, nu, dt, dx, sign):
    """A u (sign = +1) or B u (sign = -1) on the interior, (1 - sign*4 r nu) u + sign*(north, west, south and east
    terms) as in mg_oracle.c; and the scale of its rounding error, every term of the formula in absolute value (a
    coefficient r (+-v dx/2 + nu) is rounded relative to r (|v| dx/2 + |nu|), not to its possibly cancelled value)"""
    r = LD(0.5) * LD(dt) / (LD(dx) * LD(dx))
    h, nu = LD(dx) / LD(2), LD(nu)
    a, b = v2[1:-1, 1:-1].astype(LD), v1[1:-1, 1:-1].astype(LD)
    # west (u[i][j-1]), east (u[i][j+1]) from v2; north (u[i-1][j]), south (u[i+1][j]) from v1
    w, e, no, so = r * (-a * h + nu), r * (a * h + nu), r * (-b * h + nu), r * (b * h + nu)
    U = u.astype(LD)
    c, up, dn, lf, rt = U[1:-1, 1:-1], U[:-2, 1:-1], U[2:, 1:-1], U[1:-1, :-2], U[1:-1, 2:]
    diag = LD(1) - LD(sign) * LD(4) * r * nu
    val = diag * c + LD(sign) * (no * up + w * lf + so * dn + e * rt)
    ka, kb = r * (abs(a) * h + abs(nu)), r * (abs(b) * h + abs(nu))
    mag = (LD(1) + LD(4) * r * abs(nu)) * abs(c) + kb * (abs(up) + abs(dn)) + ka * (abs(lf) + abs(rt))
    return val, mag


def fsum_norm(a):
    return math.sqrt(math.fsum((np.asarray(a, dtype=LD) ** 2).astype(np.float64).ravel()))


def true_residual(u, f, v1, v2, nu, dt, dx):
    """(||f - A u||_2 over the interior, || |f| + |A| |u| ||_2): the residual norm and the scale of its rounding error"""
    au, mag = _apply(u, v1, v2, nu, dt, dx, +1)
    F = f[1:-1, 1:-1].astype(LD)
    return fsum_norm(F - au), fsum_norm(abs(F) + mag)


def true_rhs(u, v1, v2, nu, dt, dx):
    """B u on the interior and |B| |u| (long double)"""
    return _apply(u, v1, v2, nu, dt, dx, -1)


# A residual norm of n^2 nodes, each a handful of double operations away from the truth (the coefficients included),
# differs from the exact value by at most C_NORM * eps * || |f| + |A| |u| ||: that term covers the cancellation once
# the iterate has converged.  The relative term covers the summation order of the sum of squares.
C_NORM = 16.0


def norm_ok(reported, true, scale):
    return abs(reported - true) <= 1e-12 * true + C_NORM * EPS * scale


def assert_norm(reported, u, f, v1, v2, nu, dt, dx, what):
    true, scale = true_residual(u, f, v1, v2, nu, dt, dx)
    assert norm_ok(reported, true, scale), (what, reported, true, scale)
    return true, scale


# ---- one solver and the oracle side by side -----------------------------------------------------------------------
def side_by_side(mg, n, maxlvl, D, dtfac, shape, plan, ncyc=3, oracle_cls=OracleSolver, oracle_kw=None, seed=0, **opts):
    """form_rhs and ncyc cycles on the GPU (EXACT) and in the oracle from the same random state: the level-0 rhs,
    then u on every level and the coarse right-hand sides after every cycle, bit for bit; the boundaries; and each
    reported norm against the long-double truth"""
    u0, v1, v2, nu, dt, dx = problem(n, D, dtfac, seed)
    o = oracle_cls(n, u0, v1, v2, nu, dt, dx, 1e-12, shape, maxlvl=maxlvl, **(oracle_kw or {}))
    try:
        with mg.Solver(n, nu, dt, dx, 1e-12, maxlvl=maxlvl, shape=shape, arith=mg.ARITH_EXACT, plan=plan, **opts) as s:
            s.set_fields_host(u0, v1, v2)
            o.form_rhs()
            r0 = s.form_rhs()
            f0 = s.level(0, "rhs")
            assert np.array_equal(f0[1:-1, 1:-1], o.rhs(0)[1:-1, 1:-1]), "level-0 rhs"
            assert_norm(r0, u0, f0, v1, v2, nu, dt, dx, "form_rhs")
            for c in range(ncyc):
                o.cycle()
                r = s.cycle()
                for l in range(maxlvl):
                    u = s.level(l, "u")
                    assert np.array_equal(u, o.u(l)), (c, l)
                    if l == 0:
                        assert np.array_equal(u[0, :], u0[0, :]) and np.array_equal(u[-1, :], u0[-1, :]), c
                        assert np.array_equal(u[:, 0], u0[:, 0]) and np.array_equal(u[:, -1], u0[:, -1]), c
                    else:
                        assert not (u[0, :].any() or u[-1, :].any() or u[:, 0].any() or u[:, -1].any()), (c, l)
                        assert np.array_equal(s.level(l, "rhs")[1:-1, 1:-1], o.rhs(l)[1:-1, 1:-1]), (c, l)
                assert_norm(r, s.level(0, "u"), f0, v1, v2, nu, dt, dx, ("cycle", c))
    finally:
        o.close()


# ---- B: the level matrix, EXACT, against the oracle ---------------------------------------------------------------
@pytest.mark.parametrize("regime", REGIMES, ids=regime_id)
@pytest.mark.parametrize("plan", PLANS)
@pytest.mark.parametrize("pair", PAIRS, ids=pair_id)
def test_level_matrix_exact(mg, pair, plan, regime):
    n, maxlvl = pair
    for shape in (1, 2):
        side_by_side(mg, n, maxlvl, *regime, shape, plan_id(mg, plan))


@pytest.mark.parametrize("plan", PLANS)
@pytest.mark.parametrize("pair", [(8, 2), (16, 3), (64, 5), (128, 2), (256, 7), (1024, 9)], ids=pair_id)
def test_level_matrix_exact_three_repetitions(mg, pair, plan):
    """shape = 3: the reference's `for sh` loop (multigrid.cpp:52) takes any count"""
    side_by_side(mg, *pair, 8.0, 0.1, 3, plan_id(mg, plan), ncyc=2)


# ---- C: FAST arithmetic -------------------------------------------------------------------------------------------
def run_levels(mg, n, maxlvl, D, dtfac, shape, plan, arith, ncyc=3, seed=0, **opts):
    u0, v1, v2, nu, dt, dx = problem(n, D, dtfac, seed)
    out = []
    with mg.Solver(n, nu, dt, dx, 1e-12, maxlvl=maxlvl, shape=shape, arith=arith, plan=plan, **opts) as s:
        s.set_fields_host(u0, v1, v2)
        norms = [s.form_rhs()]
        for _ in range(ncyc):
            norms.append(s.cycle())
            out.append([s.level(l, "u") for l in range(maxlvl)] + [s.level(l, "rhs")[1:-1, 1:-1] for l in range(1, maxlvl)])
    return out, norms


@pytest.mark.parametrize("regime", REGIMES[:3], ids=regime_id)
@pytest.mark.parametrize("pair", PAIRS, ids=pair_id)
def test_fast_fused_equals_unfused(mg, pair, regime):
    """injection under FAST: the streaming kernels and the one-operator kernels share Arith<FAST>, so the two plans give
    the same bits on every level after every cycle"""
    for shape in (1, 2):
        a, na = run_levels(mg, *pair, *regime, shape, mg.PLAN_UNFUSED, mg.ARITH_FAST)
        b, nb = run_levels(mg, *pair, *regime, shape, mg.PLAN_FUSED, mg.ARITH_FAST)
        for c, (x, y) in enumerate(zip(a, b)):
            for l, (p, q) in enumerate(zip(x, y)):
                assert np.array_equal(p, q), (shape, c, l)
        assert np.allclose(na, nb, rtol=1e-12, atol=0), (shape, na, nb)


# FAST against the EXACT oracle after one cycle from the same state, with the coarsest level solved directly (a fixed
# linear operator: an iterated coarse solve stops at an ABSOLUTE tolerance, and one iteration more or less there would
# dominate the comparison).  Measured on one B200 (1000 W power limit) over the pairs below, both plans, D = 1 and
# D = 8: the largest relative L2 gap of u on level 0 is 4.55e-16 (the test prints each gap).  The bar is 100 times that.
FAST_GAP_MEASURED = 4.55e-16
FAST_GAP_BAR = 100 * FAST_GAP_MEASURED


@pytest.mark.parametrize("plan", PLANS)
@pytest.mark.parametrize("pair", [(8, 1), (8, 2), (16, 3), (32, 2), (64, 1), (64, 5), (128, 2), (256, 3), (256, 7),
                                  (1024, 5), (1024, 9)], ids=pair_id)
def test_fast_against_exact_oracle(mg, pair, plan):
    n, maxlvl = pair
    for D in (1.0, 8.0):
        u0, v1, v2, nu, dt, dx = problem(n, D)
        o = OracleSolver(n, u0, v1, v2, nu, dt, dx, 1e-12, 1, maxlvl=maxlvl, coarse_exact=True)
        o.form_rhs(); o.cycle()
        want = o.u(0).copy()
        o.close()
        with mg.Solver(n, nu, dt, dx, 1e-12, maxlvl=maxlvl, arith=mg.ARITH_FAST, plan=plan_id(mg, plan), coarse_exact=1) as s:
            s.set_fields_host(u0, v1, v2)
            s.form_rhs(); s.cycle()
            got = s.level(0, "u")
        gap = np.linalg.norm(got - want) / np.linalg.norm(want)
        print(f"FAST_GAP n={n} maxlvl={maxlvl} plan={plan} D={D:g} rel_l2={gap:.3e}")
        assert gap <= FAST_GAP_BAR, (D, gap)
        assert not np.array_equal(got, want) or n <= 8, "FAST should not reproduce the EXACT rounding"


# ---- D: options at the edge levels --------------------------------------------------------------------------------
@pytest.mark.parametrize("plan", PLANS)
@pytest.mark.parametrize("pair", [(16, 3), (64, 5), (64, 4), (128, 2), (256, 3), (1024, 9)], ids=pair_id)
def test_full_weighting_at_the_edge_levels(mg, pair, plan):
    """restriction = 2 against the oracle's cycle with full weighting, coarsest n_c in {4, 8, 64}"""
    for D in (1.0, 8.0):
        side_by_side(mg, *pair, D, 0.1, 1, plan_id(mg, plan), oracle_cls=FwOracleSolver, restriction=mg.RESTRICT_FW)


@pytest.mark.parametrize("plan", PLANS)
@pytest.mark.parametrize("pair", [(4, 1), (64, 5), (64, 4), (64, 3), (64, 1), (256, 3), (1024, 5)], ids=pair_id)
def test_exact_coarse_solve_at_the_edge_levels(mg, pair, plan):
    """coarse_exact = 1 against the oracle's banded LU, n_c in {4, 8, 16, 64}; n_c = 64 fills 4032 of the 4096
    element slots of k_coarse_lu_factor per step"""
    for D in (1.0, 8.0):
        side_by_side(mg, *pair, D, 0.1, 1, plan_id(mg, plan), oracle_kw=dict(coarse_exact=True), coarse_exact=1)


@pytest.mark.parametrize("plan", PLANS)
@pytest.mark.parametrize("pair", [(16, 3), (64, 5), (256, 7), (1024, 9)], ids=pair_id)
def test_corrected_towers_at_the_deepest_hierarchy(mg, pair, plan):
    side_by_side(mg, *pair, 8.0, 0.1, 1, plan_id(mg, plan), oracle_kw=dict(correct_towers=True), correct_towers=1)


class NiterOracleSolver(FwOracleSolver):
    """the oracle's cycle (injection) composed from its C operators with `niter` smoothing iterations per leg"""

    def __init__(self, *a, niter=3, **kw):
        super().__init__(*a, **kw)
        self.niter = niter

    def cycle(self, l=0):
        o, L = self.o, self.o.lib
        nl = self.n >> l
        h = self.dx * float(1 << l)
        u, f, v1, v2 = self.u(l), self.rhs(l), self.v1(l), self.v2(l)
        if l == self.maxlvl - 1:
            return super().cycle(l)
        for _ in range(self.shape):
            for _ in range(self.niter):
                L.orc_gauss_seidel(_p(u), _p(f), nl, _p(v1), _p(v2), self.dt, self.nu, h)
            self.rhs(l + 1)[...] = o.restriction(o.residual(u, f, nl, v1, v2, self.dt, self.nu, h), nl)
            self.u(l + 1)[...] = 0.0
            self.cycle(l + 1)
            u += o.prolongation(self.u(l + 1), nl // 2)
            for _ in range(self.niter):
                L.orc_gauss_seidel(_p(u), _p(f), nl, _p(v1), _p(v2), self.dt, self.nu, h)


@pytest.mark.parametrize("plan", PLANS)
@pytest.mark.parametrize("niter", [1, 2, 4])
@pytest.mark.parametrize("pair", [(64, 5), (32, 3)], ids=pair_id)
def test_smoothing_counts_where_the_pass_runs_on_levels_8_and_16(mg, pair, niter, plan):
    """niter != 3 with passes on the levels n = 16 and n = 8: the fused plan cuts the sweeps into passes of at most
    three iterations (4 = 3 + 1); both plans equal the oracle's cycle with the same count bit for bit"""
    n, maxlvl = pair
    side_by_side(mg, n, maxlvl, 8.0, 0.1, 1, plan_id(mg, plan), oracle_cls=NiterOracleSolver,
                 oracle_kw=dict(niter=niter), niter=niter)


# ---- E: the reported norms of timestep() against the truth -------------------------------------------------------
@pytest.mark.parametrize("plan", PLANS)
@pytest.mark.parametrize("D", [1.0, 8.0])
@pytest.mark.parametrize("pair", PAIRS, ids=pair_id)
def test_timestep_norms_against_the_truth(mg, pair, D, plan):
    """res of each step is the true residual of the returned field; res0 is the true residual of the previous step's
    field under the new right-hand side B u_prev; converged agrees with res/res0 <= tol on the true values.  A
    partials count that does not match the launched plan fails here."""
    n, maxlvl = pair
    tol = 1e-7
    u0, v1, v2, nu, dt, dx = problem(n, D, seed=7)
    with mg.Solver(n, nu, dt, dx, tol, maxlvl=maxlvl, plan=plan_id(mg, plan)) as s:
        s.set_fields_host(u0, v1, v2)
        prev = u0
        for step in range(3):
            info = s.timestep(1)[0]
            u, f = s.get_u_host(), s.level(0, "rhs")
            bu, mag = true_rhs(prev, v1, v2, nu, dt, dx)
            assert np.all(abs(f[1:-1, 1:-1].astype(LD) - bu) <= 8 * EPS * mag), step
            r0, s0 = true_residual(prev, f, v1, v2, nu, dt, dx)
            r, sc = true_residual(u, f, v1, v2, nu, dt, dx)
            assert norm_ok(info.res0, r0, s0), (step, info.res0, r0, s0)
            assert norm_ok(info.res, r, sc), (step, info.res, r, sc)
            assert info.history()[0] == info.res0 and info.history()[-1] == info.res
            assert 1 <= info.cycles <= 50
            ratio = r / r0
            band = (1e-12 * r + C_NORM * EPS * sc) / r0 + ratio * (1e-12 * r0 + C_NORM * EPS * s0) / r0
            if abs(ratio - tol) > 2 * band:
                assert bool(info.converged) == (ratio <= tol), (step, info.cycles, ratio, band)
            prev = u


# ---- F: the drop-in entry points ----------------------------------------------------------------------------------
def drivers(mg):
    L = mg.lib()
    pp = C.POINTER(C.c_void_p)
    L.mgb200_mg_inner.argtypes = [pp, pp, pp, pp, C.c_void_p, C.c_double, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double,
                                  C.c_double, C.POINTER(mg.Options), C.c_void_p]
    L.mgb200_mg_outer.argtypes = [pp, pp, pp, pp, C.c_void_p, C.c_double, C.c_int, C.c_int, C.c_double, C.c_double,
                                  C.c_double, C.c_int, C.POINTER(mg.Options), C.c_void_p, C.POINTER(mg.SolveInfo)]
    return L


@pytest.mark.parametrize("n,maxlvl", [(96, 4), (160, 4), (200, 3), (100, 2), (64, 5), (256, 2)])
def test_mg_inner_and_mg_outer_at_other_sizes(mg, n, maxlvl):
    """mgb200_mg_inner / mgb200_mg_outer on towers the caller built the reference's way (every coarse level
    (n/2+1)^2 doubles, velocities by the never-halved restriction), at sizes that are even on every level above the
    coarsest but not powers of two, and with a coarsest level of 128 at (256, 2): bit for bit against the oracle"""
    L = drivers(mg)
    tol = 1e-6
    u0, v1, v2, nu, dt, dx = problem(n, 8.0, seed=3)
    o = OracleSolver(n, u0, v1, v2, nu, dt, dx, tol, 1, maxlvl=maxlvl)
    o.form_rhs()

    def tower(get):
        out = []
        for l in range(maxlvl):
            nl = n >> l
            a = torch.zeros((n + 1) ** 2 if l == 0 else (n // 2 + 1) ** 2, dtype=torch.float64, device="cuda")
            a[: (nl + 1) ** 2] = torch.from_numpy(np.ascontiguousarray(get(l))).reshape(-1).cuda()
            out.append(a)
        return out

    U, F, V1, V2 = tower(o.u), tower(o.rhs), tower(o.v1), tower(o.v2)
    tmp = torch.zeros((n + 1) ** 2, dtype=torch.float64, device="cuda")
    arr = lambda ts: (C.c_void_p * maxlvl)(*[t.data_ptr() for t in ts])
    opt = mg.default_options(arith=mg.ARITH_EXACT)
    lvl = lambda t, l: t[l][: ((n >> l) + 1) ** 2].cpu().numpy().reshape((n >> l) + 1, (n >> l) + 1)
    rc = L.mgb200_mg_inner(arr(U), arr(F), arr(V1), arr(V2), tmp.data_ptr(), dx, n, 0, maxlvl, 1, dt, nu, C.byref(opt), None)
    assert rc == 0, L.mgb200_last_error()
    o.cycle()
    for l in range(maxlvl):
        assert np.array_equal(lvl(U, l), o.u(l)), l
        if l > 0:
            assert np.array_equal(lvl(F, l)[1:-1, 1:-1], o.rhs(l)[1:-1, 1:-1]), l
    info = mg.SolveInfo()
    rc = L.mgb200_mg_outer(arr(U), arr(V1), arr(V2), arr(F), tmp.data_ptr(), nu, maxlvl, n, dt, dx, tol, 1, C.byref(opt), None,
                           C.byref(info))
    assert rc == 0, L.mgb200_last_error()
    it, hist = o.solve()
    assert info.cycles == it and bool(info.converged) == bool(hist[-1] / hist[0] <= tol)
    assert np.allclose(info.history(), hist, rtol=1e-12, atol=0)
    for l in range(maxlvl):
        assert np.array_equal(lvl(U, l), o.u(l)), l
    o.close()


def host_ops(mg):
    L = mg.lib()
    dp, l, d, i = C.POINTER(C.c_double), C.c_long, C.c_double, C.c_int
    L.mgb200_host_residual.argtypes = [dp, dp, dp, l, dp, dp, d, d, d, i]
    L.mgb200_host_compute_norm.argtypes = [dp, l, dp]
    L.mgb200_host_gauss_seidel.argtypes = [dp, dp, l, dp, dp, d, d, d, i, i]
    L.mgb200_host_compute_rhs.argtypes = [dp, dp, l, dp, dp, d, d, d, i]
    L.mgb200_host_prolongation.argtypes = [dp, dp, i]
    L.mgb200_host_restriction.argtypes = [dp, dp, i]
    return L


@pytest.mark.parametrize("n", [5, 100, 257])
def test_host_operators(mg, oracle, n):
    """the gs.h flavour (mgb200_host_*: host arrays through device copies) against the oracle, EXACT, bit for bit; the
    norm against the correctly rounded one.  Arrays are prefilled, so a kernel that writes outside the interior fails."""
    L = host_ops(mg)
    u, v1, v2, nu, dt, dx = problem(n, 8.0, seed=11)
    rng = np.random.default_rng(n)
    f = rng.uniform(-1.0, 1.0, (n + 1, n + 1))
    ex = mg.ARITH_EXACT
    # compute_rhs
    got = rng.uniform(-1.0, 1.0, (n + 1, n + 1)); want = got.copy()
    assert L.mgb200_host_compute_rhs(_p(got), _p(u), n, _p(v1), _p(v2), dt, nu, dx, ex) == 0, L.mgb200_last_error()
    oracle.compute_rhs(u, n, v1, v2, dt, nu, dx, rhs=want)
    assert np.array_equal(got, want)
    # residual
    got = rng.uniform(-1.0, 1.0, (n + 1, n + 1)); want = got.copy()
    assert L.mgb200_host_residual(_p(got), _p(u), _p(f), n, _p(v1), _p(v2), dt, nu, dx, ex) == 0, L.mgb200_last_error()
    oracle.residual(u, f, n, v1, v2, dt, nu, dx, res=want)
    assert np.array_equal(got, want)
    # compute_norm
    out = C.c_double(0.0)
    assert L.mgb200_host_compute_norm(_p(want), n, C.byref(out)) == 0, L.mgb200_last_error()
    true = fsum_norm(want[1:-1, 1:-1])
    assert abs(out.value - true) <= 1e-14 * true, (out.value, true)
    # gauss_seidel, one and three iterations
    for iters in (1, 3):
        got = u.copy(); want = u.copy()
        assert L.mgb200_host_gauss_seidel(_p(got), _p(f), n, _p(v1), _p(v2), dt, nu, dx, iters, ex) == 0, L.mgb200_last_error()
        oracle.gauss_seidel(want, f, n, v1, v2, dt, nu, dx, iters)
        assert np.array_equal(got, want), iters
    # prolongation (n = coarse n) and restriction (n = fine n, even)
    fine = np.full((2 * n + 1, 2 * n + 1), np.nan)
    assert L.mgb200_host_prolongation(_p(fine), _p(u), n) == 0, L.mgb200_last_error()
    assert np.array_equal(fine, oracle.prolongation(u, n))
    big = rng.uniform(-1.0, 1.0, (2 * n + 1, 2 * n + 1))
    coarse = np.full((n + 1, n + 1), np.nan)
    assert L.mgb200_host_restriction(_p(coarse), _p(big), 2 * n) == 0, L.mgb200_last_error()
    assert np.array_equal(coarse, oracle.restriction(big, 2 * n))


def test_timestepper_cache_is_keyed_on_maxlvl(mg):
    """the one-call driver keeps its handle between calls; maxlvl A, then B, then A again must each give what a fresh
    handle gives (and A and B differ, so reusing the wrong hierarchy would show)"""
    n, nsteps, tol = 64, 2, 1e-8
    u0, v1, v2, nu, dt, dx = problem(n, 8.0, seed=5)
    T = nsteps * dt
    assert int(T / dt) == nsteps

    def fresh(maxlvl):
        with mg.Solver(n, nu, dt, dx, tol, maxlvl=maxlvl, arith=mg.ARITH_EXACT) as s:
            s.set_fields_host(u0, v1, v2)
            s.timestep(nsteps)
            return s.get_u_host()

    want = {m: fresh(m) for m in (2, 5)}
    assert not np.array_equal(want[2], want[5])
    o = OracleSolver(n, u0, v1, v2, nu, dt, dx, tol, 1, maxlvl=5)
    o.advance(nsteps)
    assert np.array_equal(want[5], o.u(0))
    o.close()
    mg.release_cached()
    for m in (2, 5, 2):
        uT = np.zeros_like(u0)
        mg.timestepper_host(uT, u0, v1, v2, nu, m, n, dt, T, dx, tol, 1, arith=mg.ARITH_EXACT)
        assert np.array_equal(uT, want[m]), m
    mg.release_cached()


@pytest.mark.parametrize("n,maxlvl", [(256, 8), (256, 2), (256, 0), (64, 6), (4, 2), (96, 2), (100, 1), (2, 1)])
def test_rejected_level_counts_and_sizes(mg, n, maxlvl):
    """a coarsest level outside 4..64 or a size that is not a power of two >= 4 is refused by the handle and by the
    one-call driver, and a valid solve works afterwards"""
    dx = 1.0 / n; dt = dx / 10
    with pytest.raises(mg.MgError):
        mg.Solver(n, -4e-4, dt, dx, 1e-8, maxlvl=maxlvl)
    z = np.zeros((n + 1, n + 1))
    with pytest.raises(mg.MgError):
        mg.timestepper_host(z.copy(), z, z, z, -4e-4, maxlvl, n, dt, 2 * dt, dx, 1e-8, 1)
    u0, v1, v2, nu, dt, dx = problem(64, 1.0)
    uT = np.zeros_like(u0)
    info = mg.timestepper_host(uT, u0, v1, v2, nu, 3, 64, dt, 2 * dt, dx, 1e-8, 1, arith=mg.ARITH_EXACT)
    o = OracleSolver(64, u0, v1, v2, nu, dt, dx, 1e-8, 1, maxlvl=3)
    o.advance(2)
    assert info.converged and np.array_equal(uT, o.u(0))
    o.close()
    with mg.Solver(64, nu, dt, dx, 1e-8, maxlvl=3, arith=mg.ARITH_EXACT) as s:
        s.set_fields_host(u0, v1, v2)
        s.timestep(2)
        assert np.array_equal(s.get_u_host(), uT)
    mg.release_cached()


# ---- H: row slabs -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world", [2, 4])
def test_sharded_deep_and_shallow_hierarchies(world):
    """row slabs with a coarsest level of 4 and of 64, injection and full weighting, random nonzero boundaries: the
    same bits and cycle counts as the single-GPU solve"""
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr",
           "127.0.0.1", "--master-port", str(29600 + world), os.path.join(ROOT, "tests", "sharded_levels_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    line = [l for l in r.stdout.splitlines() if l.startswith("SHARDED_LEVELS_RESULT ")]
    assert r.returncode == 0 and line, r.stdout[-2000:] + r.stderr[-4000:]
    res = json.loads(line[0][len("SHARDED_LEVELS_RESULT "):])
    assert len(res) == 4
    for key, v in res.items():
        assert v["sharded_levels"] >= 1, (key, v)
        assert v["cycles"] == v["ref_cycles"], (key, v)
        assert v["bitwise"], (key, v)
