"""TEST INFRASTRUCTURE: the oracle's multigrid cycle with the full-weighting restriction of the residual.

The oracle's own cycle (orc_cycle, multigrid.cpp:17-92) restricts by injection, as the reference does.  This is the
same cycle composed in Python from the oracle's C operators -- gauss_seidel, residual, norm, prolongation and
restriction_fw (gs.cpp:277-280) -- called in the order and on the arrays orc_cycle uses, so that it gives the bits
orc_cycle would give with orc_restriction_fw in place of orc_restriction."""
import numpy as np

from oracle.oracle import OracleSolver, _p

NITER, COARSE_MAXIT, COARSE_TOL, MAX_CYCLE = 3, 1000, 1e-5, 50     # multigrid.cpp:41, :60, :94


class FwOracleSolver(OracleSolver):
    def __init__(self, n, u0, v1, v2, nu, dt, dx, tol, shape=1, maxlvl=None):
        super().__init__(n, u0, v1, v2, nu, dt, dx, tol, shape, maxlvl)
        self.nu, self.dt, self.dx, self.tol, self.shape = nu, dt, dx, tol, shape

    def cycle(self, l=0):
        o, L = self.o, self.o.lib
        nl = self.n >> l
        h = self.dx * float(1 << l)                                   # dx2 = 2*dx per level (multigrid.cpp:49)
        u, f, v1, v2 = self.u(l), self.rhs(l), self.v1(l), self.v2(l)
        gs = lambda: L.orc_gauss_seidel(_p(u), _p(f), nl, _p(v1), _p(v2), self.dt, self.nu, h)
        for _ in range(self.shape):                                   # :52
            if l == self.maxlvl - 1:                                  # coarsest: to an ABSOLUTE residual norm (:58-65)
                rn, it = 1.0, 0
                tmp = np.zeros((nl + 1, nl + 1))
                while it < COARSE_MAXIT and rn > COARSE_TOL:
                    gs()
                    L.orc_residual(_p(tmp), _p(u), _p(f), nl, _p(v1), _p(v2), self.dt, self.nu, h)
                    rn = L.orc_norm(_p(tmp), nl)
                    it += 1
                continue
            nc = nl // 2
            for _ in range(NITER):                                    # :69-72
                gs()
            res = o.residual(u, f, nl, v1, v2, self.dt, self.nu, h)   # :73
            self.rhs(l + 1)[...] = o.restriction_fw(res, nl)          # :75 with full weighting
            self.u(l + 1)[...] = 0.0                                  # :77
            self.cycle(l + 1)                                         # :79
            u += o.prolongation(self.u(l + 1), nc)                    # :81-83
            for _ in range(NITER):                                    # :85-88
                gs()

    def solve(self):
        """mg_outer (multigrid.cpp:97-120): (cycles, [res0, res1, ...])"""
        hist = [self.residual_norm()]
        while len(hist) - 1 < MAX_CYCLE and hist[-1] / hist[0] > self.tol:
            self.cycle(0)
            hist.append(self.residual_norm())
        return len(hist) - 1, np.array(hist)
