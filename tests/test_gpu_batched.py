"""Batched solver handles on the GPU: every member of a batch must give exactly what a handle of that problem alone
gives (u on every level, cycle counts, converged flags), each member stopping at its own convergence; a batch of one
member must equal a single-problem handle bit for bit, norms and histories included."""
import os

import numpy as np
import pytest

from oracle.oracle import OracleSolver

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

TOL = 1e-8


@pytest.fixture(scope="module")
def mg():
    import hpcclassmultigridproject_b200 as m
    m.lib()
    assert torch.cuda.is_available()
    return m


def member_fields(n, b, vscale=1.0):
    """a Gaussian bump placed by member index, a vortex scaled per member; zero boundary lines for u"""
    x = np.linspace(0.0, 1.0, n + 1)
    X, Y = np.meshgrid(x, x, indexing="ij")
    rng = np.random.default_rng(1000 + b)
    cx, cy = 0.3 + 0.4 * rng.random(), 0.3 + 0.4 * rng.random()
    u0 = np.exp(-((X - cx) ** 2 + (Y - cy) ** 2) / 0.01) + 0.05 * rng.standard_normal((n + 1, n + 1))
    u0[0, :] = u0[-1, :] = 0.0; u0[:, 0] = u0[:, -1] = 0.0
    s = vscale * (0.5 + rng.random())
    v1 = s * np.sin(np.pi * X) * np.cos(np.pi * Y)
    v2 = -s * np.cos(np.pi * X) * np.sin(np.pi * Y)
    return u0, v1, v2


def stack(fl):
    return [np.ascontiguousarray(np.stack([f[k] for f in fl])) for k in range(3)]


def params(n):
    dx = 1.0 / n
    return dict(nu=-4e-4, dt=dx / 10, dx=dx)


def solo_run(mg, n, fields, steps, tol=TOL, nu=None, **opts):
    """per step: (infos, u on every level) of a single-problem handle"""
    p = params(n)
    if nu is not None:
        p["nu"] = nu
    out = []
    with mg.Solver(n, p["nu"], p["dt"], p["dx"], tol, **opts) as s:
        s.set_fields_host(*fields)
        for _ in range(steps):
            info = s.timestep(1)[0]
            out.append((info, [s.level(l, "u") for l in range(s.maxlvl)]))
    return out


def check_member(got_info, got_levels, want, exact_norms=False):
    info, levels = want
    assert got_info.cycles == info.cycles
    assert got_info.converged == info.converged
    for l, (g, w) in enumerate(zip(got_levels, levels)):
        assert np.array_equal(g, w, equal_nan=True), f"level {l}"
    if exact_norms:
        assert got_info.history() == info.history()
        assert got_info.res0 == info.res0 and got_info.res == info.res


def batched_steps(mg, n, fl, steps, tol=TOL, nu=None, **opts):
    """per step: (B infos, per level the (B, n_l+1, n_l+1) u) of one batched handle"""
    p = params(n)
    if nu is not None:
        p["nu"] = nu
    out = []
    with mg.Solver(n, p["nu"], p["dt"], p["dx"], tol, batch=len(fl), **opts) as s:
        assert s.members == len(fl)
        s.set_fields_host(*stack(fl))
        for _ in range(steps):
            infos = s.timestep(1)[0]
            out.append((infos, [s.level(l, "u") for l in range(s.maxlvl)]))
    return out


def compare(mg, n, fl, steps, tol=TOL, nu=None, exact_norms=False, **opts):
    got = batched_steps(mg, n, fl, steps, tol=tol, nu=nu, **opts)
    for b, f in enumerate(fl):
        want = solo_run(mg, n, f, steps, tol=tol, nu=nu, **opts)
        for k in range(steps):
            infos, levels = got[k]
            check_member(infos[b], [lv[b] for lv in levels], want[k], exact_norms)
    return got


@pytest.mark.parametrize("n", [32, 256, 1024])
@pytest.mark.parametrize("shape", [1, 2])
@pytest.mark.parametrize("arith", ["fast", "exact"])
def test_batch_of_one_equals_single_handle(mg, n, shape, arith):
    a = mg.ARITH_EXACT if arith == "exact" else mg.ARITH_FAST
    compare(mg, n, [member_fields(n, 0)], 3, exact_norms=True, shape=shape, arith=a)


@pytest.mark.parametrize("n", [64, 256])
def test_exact_members_equal_oracle_every_cycle(mg, oracle, n):
    """EXACT arithmetic, three members: every level's u and coarse rhs after every cycle equal the oracle's"""
    p = params(n)
    fl = [member_fields(n, b) for b in range(3)]
    orcs = [OracleSolver(n, *f, p["nu"], p["dt"], p["dx"], 1e-12) for f in fl]
    with mg.Solver(n, p["nu"], p["dt"], p["dx"], 1e-12, batch=3, arith=mg.ARITH_EXACT) as s:
        s.set_fields_host(*stack(fl))
        for step in range(2):
            for o in orcs:
                o.form_rhs()
            r0 = s.form_rhs()
            for b, o in enumerate(orcs):
                assert np.array_equal(s.level(0, "rhs")[b][1:-1, 1:-1], o.rhs(0)[1:-1, 1:-1])
                assert abs(r0[b] - o.residual_norm()) <= 1e-12 * r0[b]
            for _ in range(2):
                for o in orcs:
                    o.cycle()
                r = s.cycle()
                for l in range(s.maxlvl):
                    us, rs = s.level(l, "u"), s.level(l, "rhs")
                    for b, o in enumerate(orcs):
                        assert np.array_equal(us[b], o.u(l)), (step, l, b)
                        if l > 0:
                            assert np.array_equal(rs[b][1:-1, 1:-1], o.rhs(l)[1:-1, 1:-1]), (step, l, b)
                for b, o in enumerate(orcs):
                    ro = o.residual_norm()
                    assert abs(r[b] - ro) <= 1e-9 * ro
    for o in orcs:
        o.close()


OPTION_CASES = [
    ("niter1", 64, dict(niter=1)),
    ("niter2", 64, dict(niter=2)),
    ("niter4", 128, dict(niter=4)),
    ("full_weighting", 128, dict(restriction=2)),
    ("coarse_exact", 128, dict(coarse_exact=1)),
    ("correct_towers", 128, dict(correct_towers=1)),
    ("coarsest4", 64, dict(maxlvl=5)),
    ("coarsest64", 256, dict(maxlvl=3)),
    ("one_level", 32, dict(maxlvl=1)),
    ("wcycle", 128, dict(shape=2)),
    ("no_graph", 128, dict(use_graph=0)),
]


@pytest.mark.parametrize("B", [3, 5])
@pytest.mark.parametrize("name,n,opts", OPTION_CASES, ids=[c[0] for c in OPTION_CASES])
def test_options_matrix(mg, B, name, n, opts):
    fl = [member_fields(n, b, vscale=1.0 + 2.0 * b) for b in range(B)]
    compare(mg, n, fl, 3, **opts)


@pytest.mark.parametrize("B", [3, 5])
def test_host_loop(mg, monkeypatch, B):
    """MGB200_DEVICE_LOOP=0: mg_outer's loop on the host, one flag per member per cycle"""
    monkeypatch.setenv("MGB200_DEVICE_LOOP", "0")
    n = 128
    compare(mg, n, [member_fields(n, b, vscale=1.0 + b) for b in range(B)], 3)


@pytest.mark.parametrize("loop", ["device", "host"])
def test_members_stop_at_their_own_convergence(mg, monkeypatch, loop):
    """one batch, members with different cycle counts per step: no advection (1 cycle per step at N = 256), strong
    advection (more cycles), u0 = 0 (res0 = 0: 0 cycles, the field stays zero) and a member with vscale 40; each equals
    its own handle after every one of five steps, and leaving the last member out changes none of the others"""
    if loop == "host":
        monkeypatch.setenv("MGB200_DEVICE_LOOP", "0")
    monkeypatch.setenv("MGB200_QUIET", "1")
    n = 256
    tol = 1e-10
    z = member_fields(n, 3)
    fl = [member_fields(n, 0, vscale=0.0), member_fields(n, 1, vscale=1.0), (np.zeros_like(z[0]), z[1], z[2]),
          member_fields(n, 2, vscale=10.0), member_fields(n, 4, vscale=40.0)]
    got = compare(mg, n, fl, 5, tol=tol)
    counts = [[i.cycles for i in infos] for infos, _ in got]
    print("cycles per step and member:", counts)
    assert all(c[2] == 0 for c in counts), counts
    assert np.array_equal(got[-1][1][0][2], np.zeros((n + 1, n + 1)))
    assert all(c[0] < c[3] for c in counts), counts                  # the members ran different cycle counts
    got4 = batched_steps(mg, n, fl[:4], 5, tol=tol)
    for k in range(5):
        for b in range(4):
            assert got4[k][0][b].cycles == got[k][0][b].cycles
            for l in range(len(got4[k][1])):
                assert np.array_equal(got4[k][1][l][b], got[k][1][l][b], equal_nan=True)


def test_forty_members_more_than_one_wave(mg):
    n = 256
    fl = [member_fields(n, b, vscale=0.5 + 0.1 * b) for b in range(40)]
    got = batched_steps(mg, n, fl, 2)
    for b in (0, 17, 39):
        want = solo_run(mg, n, fl[b], 2)
        for k in range(2):
            check_member(got[k][0][b], [lv[b] for lv in got[k][1]], want[k])


def test_handles_used_alternately(mg):
    """two batched handles of different sizes and a single-problem handle in one process, stepped in turn"""
    n = 128
    p = params(n)
    f3 = [member_fields(n, b) for b in range(3)]
    f2 = [member_fields(n, 10 + b) for b in range(2)]
    f1 = member_fields(n, 20)
    want3 = [solo_run(mg, n, f, 3) for f in f3]
    want2 = [solo_run(mg, n, f, 3) for f in f2]
    want1 = solo_run(mg, n, f1, 3)
    with mg.Solver(n, p["nu"], p["dt"], p["dx"], TOL, batch=3) as a, mg.Solver(n, p["nu"], p["dt"], p["dx"], TOL, batch=2) as b, \
            mg.Solver(n, p["nu"], p["dt"], p["dx"], TOL) as c:
        a.set_fields_host(*stack(f3)); b.set_fields_host(*stack(f2)); c.set_fields_host(*f1)
        assert c.members == 1
        for k in range(3):
            ia = a.timestep(1)[0]; ic = c.timestep(1)[0]; ib = b.timestep(1)[0]
            ua, ub, uc = a.get_u_host(), b.get_u_host(), c.get_u_host()
            for m in range(3):
                assert ia[m].cycles == want3[m][k][0].cycles and np.array_equal(ua[m], want3[m][k][1][0])
            for m in range(2):
                assert ib[m].cycles == want2[m][k][0].cycles and np.array_equal(ub[m], want2[m][k][1][0])
            assert ic.cycles == want1[k][0].cycles and np.array_equal(uc, want1[k][1][0])


def test_device_fields_and_multi_step(mg):
    """set_fields_device / get_u_device with (B, n+1, n+1) tensors; timestep(4) in one call equals 4 single steps"""
    n = 128
    p = params(n)
    fl = [member_fields(n, b) for b in range(3)]
    want = [solo_run(mg, n, f, 4) for f in fl]
    with mg.Solver(n, p["nu"], p["dt"], p["dx"], TOL, batch=3) as s:
        s.set_fields_device(*[torch.from_numpy(a).cuda() for a in stack(fl)])
        steps = s.timestep(4)
        out = torch.empty((3, n + 1, n + 1), dtype=torch.float64, device="cuda")
        s.get_u_device(out)
        u = out.cpu().numpy()
        for b in range(3):
            assert [steps[k][b].cycles for k in range(4)] == [want[b][k][0].cycles for k in range(4)]
            assert np.array_equal(u[b], want[b][3][1][0])
        assert s.cycle_bytes > 0


def test_refusals(mg):
    p = params(64)
    args = (64, p["nu"], p["dt"], p["dx"], TOL)
    with pytest.raises(mg.MgError, match="fused plan"):
        mg.Solver(*args, batch=2, plan=mg.PLAN_UNFUSED)
    with pytest.raises(mg.MgError, match="niter"):
        mg.Solver(*args, batch=2, niter=0)
    with pytest.raises(mg.MgError, match="batch"):
        mg.Solver(*args, batch=0)
    with pytest.raises(mg.MgError, match="65535"):
        mg.Solver(*args, batch=65536)
