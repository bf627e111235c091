"""The oracle's cycle with full weighting (tests/oracle_fw.py) at N = 1024 with the diffusion number of the large
configurations (|nu| * N held fixed): injection converges at the GPU's measured rates, full weighting in about half
the cycles.  dt = dx/10, reference initial conditions with vscale = 1, the reference's flat velocity towers."""
import numpy as np
import pytest

from oracle.oracle import Oracle, OracleSolver
from oracle_fw import FwOracleSolver

N = 1024

# nu at N = 1024 analogous to: C3 (N = 16384), N = 32768, C5 (N = 65536);
# cycles to 1e-6 with injection, with full weighting; injection's per-cycle factor (last cycle)
CASES = [(-6.4e-3, 3, 2, 1.3e-8 / 6.8e-6), (-1.28e-2, 4, 3, 8.4e-7 / 3.0e-5), (-2.56e-2, 8, 4, 0.147)]


def solve(nu, fw):
    u0, v1, v2 = Oracle().initial_conditions(N, 1.0)
    dx = 1.0 / N; dt = dx / 10
    s = (FwOracleSolver if fw else OracleSolver)(N, u0, v1, v2, nu, dt, dx, 1e-6, 1)
    s.form_rhs()
    it, hist = s.solve()
    s.close()
    return it, hist / hist[0]


@pytest.mark.timeout(900)
@pytest.mark.parametrize("nu,inj_cycles,fw_cycles,inj_factor", CASES)
def test_full_weighting_halves_the_cycles(nu, inj_cycles, fw_cycles, inj_factor):
    it_i, h_i = solve(nu, False)
    it_f, h_f = solve(nu, True)
    assert it_i == inj_cycles, h_i
    assert it_f == fw_cycles, h_f
    assert abs(h_i[-1] / h_i[-2] - inj_factor) <= 0.05 * inj_factor, h_i
    assert np.all(h_f[1:] < h_i[1:it_f + 1])                       # every cycle reduces the residual further
