"""options.restriction = 2: full-weighting restriction of the residual on either plan.  On the fused plan it is the
POST_FW flavour of the down-leg streaming pass; it must do exactly what the unfused plan does with restriction = 1
(one-operator kernels: residual, then k_restrict_fw), on one GPU and on row slabs over several."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from oracle_fw import FwOracleSolver

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def mg():
    import hpcclassmultigridproject_b200 as m
    m.lib()
    assert torch.cuda.is_available()
    return m


def rel_l2(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


def cycles(mg, n, plan, restriction, arith, shape, niter, ncyc=3):
    dx = 1.0 / n; dt = dx / 10
    with mg.Solver(n, -4e-4, dt, dx, 1e-12, shape=shape, arith=arith, plan=plan, niter=niter, restriction=restriction) as s:
        s.set_fields_reference_ic(2.0)
        norms = [s.form_rhs()]
        levels = []
        for _ in range(ncyc):
            norms.append(s.cycle())
            levels.append([s.level(l, "u") for l in range(s.maxlvl)] + [s.level(l, "rhs") for l in range(1, s.maxlvl)])
    return levels, norms


@pytest.mark.parametrize("n", [256, 1024, 4096])
@pytest.mark.parametrize("arith", ["fast", "exact"])
@pytest.mark.parametrize("shape", [1, 2])
@pytest.mark.parametrize("niter", [1, 3, 4])
def test_fused_equals_unfused(mg, n, arith, shape, niter):
    """u on every level (and the coarse right-hand sides) after every cycle, bit for bit; the residual norms are
    reduced in a different order by the two plans"""
    a = mg.ARITH_EXACT if arith == "exact" else mg.ARITH_FAST
    lu, nu_ = cycles(mg, n, mg.PLAN_UNFUSED, mg.RESTRICT_FW_UNFUSED, a, shape, niter)
    lf, nf = cycles(mg, n, mg.PLAN_FUSED, mg.RESTRICT_FW, a, shape, niter)
    for c, (x, y) in enumerate(zip(lu, lf)):
        for l, (p, q) in enumerate(zip(x, y)):
            if l >= len(x) // 2 + 1:                                   # coarse rhs: interior (the boundary is never read)
                p, q = p[1:-1, 1:-1], q[1:-1, 1:-1]
            assert np.array_equal(p, q), (c, l)
    assert np.allclose(nu_, nf, rtol=1e-9, atol=0)


def test_exact_equals_oracle(mg, oracle):
    n = 256; dx = 1.0 / n; dt = dx / 10; nu = -4e-4
    u0, v1, v2 = oracle.initial_conditions(n, 2.0)
    o = FwOracleSolver(n, u0, v1, v2, nu, dt, dx, 1e-12, 1)
    with mg.Solver(n, nu, dt, dx, 1e-12, arith=mg.ARITH_EXACT, restriction=mg.RESTRICT_FW) as s:
        s.set_fields_host(u0, v1, v2)
        o.form_rhs(); s.form_rhs()
        for c in range(3):
            o.cycle(); r = s.cycle()
            for l in range(s.maxlvl):
                assert np.array_equal(s.level(l, "u"), o.u(l)), (c, l)
                if l > 0:
                    assert np.array_equal(s.level(l, "rhs")[1:-1, 1:-1], o.rhs(l)[1:-1, 1:-1]), (c, l)
            ro = o.residual_norm()
            assert abs(r - ro) <= 1e-9 * ro
    o.close()


def test_device_loop_equals_host_loop(mg, monkeypatch):
    n = 1024; dx = 1.0 / n; dt = dx / 10
    out = []
    for loop in ("1", "0"):
        monkeypatch.setenv("MGB200_DEVICE_LOOP", loop)
        with mg.Solver(n, -4e-4, dt, dx, 1e-10, restriction=mg.RESTRICT_FW) as s:
            s.set_fields_reference_ic(2.0)
            infos = s.timestep(5)
            out.append((s.get_u_host(), [i.cycles for i in infos], [i.history() for i in infos]))
    assert np.array_equal(out[0][0], out[1][0])
    assert out[0][1] == out[1][1]
    assert out[0][2] == out[1][2]


def test_value_1_still_rejected_on_the_fused_plan(mg):
    n = 256; dx = 1.0 / n
    with pytest.raises(mg.MgError):
        mg.Solver(n, -4e-4, dx / 10, dx, 1e-10, plan=mg.PLAN_FUSED, restriction=mg.RESTRICT_FW_UNFUSED)
    with pytest.raises(mg.MgError):
        mg.Solver(n, -4e-4, dx / 10, dx, 1e-10, restriction=3)


def test_fewer_cycles_at_a_large_diffusion_number(mg):
    """N = 16384, nu = -1.6e-3 (|nu| N as at N = 65536, nu = -4e-4): full weighting needs fewer cycles to 1e-10 and
    reaches the same solution"""
    n = 16384; dx = 1.0 / n; dt = dx / 10; nu = -1.6e-3
    out = []
    for restriction in (mg.RESTRICT_INJECT, mg.RESTRICT_FW):
        with mg.Solver(n, nu, dt, dx, 1e-10, restriction=restriction) as s:
            s.set_fields_reference_ic(1.0)
            info = s.timestep(1)[0]
            assert info.converged
            out.append((s.get_u_host(), info.cycles))
    assert out[1][1] < out[0][1], (out[0][1], out[1][1])
    assert rel_l2(out[1][0], out[0][0]) <= 1e-8


@pytest.mark.parametrize("world", [2, 4, 8])
def test_sharded_equals_single_gpu(world):
    """row slabs (peer memory and the NCCL fallback), with and without an agglomerated coarse level: bit-identical
    to the single-GPU full-weighting solve"""
    if not torch.cuda.is_available() or torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    for p2p in ("1", "0"):
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr",
               "127.0.0.1", "--master-port", str(29500 + world), os.path.join(ROOT, "tests", "sharded_fw_worker.py")]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ, MGB200_P2P=p2p))
        line = [l for l in r.stdout.splitlines() if l.startswith("SHARDED_FW_RESULT ")]
        assert r.returncode == 0 and line, r.stdout[-2000:] + r.stderr[-4000:]
        for key, res in json.loads(line[0][len("SHARDED_FW_RESULT "):]).items():
            assert res["sharded_levels"] >= 1, (p2p, key, res)
            assert res["cycles"] == res["ref_cycles"], (p2p, key, res)
            assert res["bitwise"], (p2p, key, res)
