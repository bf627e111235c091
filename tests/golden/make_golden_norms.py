#!/usr/bin/env python
"""Generate tests/golden/solve_norms.json: ||uT||_2 of the golden runs that keep no field (make_golden.py,
keep_u=False) as test_oracle_golden.exact_norm computes it, which gives the same bits on every host.

Their npz files hold norm_uT as np.linalg.norm returned it where the reference ran, and that value depends on the
BLAS's summation order (its kernel and thread count).  This script recomputes each field with the oracle, requires
that it reproduces the reference's cycle counts, residual histories, mid value and stored norm_uT bit for bit, and only
then stores the exact norm of the same field.  Run it where np.linalg.norm reproduces the stored norm_uT:
    python tests/golden/make_golden_norms.py
"""
import json
import os
import sys

import numpy as np

OUT = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(OUT))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle.oracle import Oracle, OracleSolver  # noqa: E402
from test_oracle_golden import SOLVES, exact_norm  # noqa: E402

if __name__ == "__main__":
    oracle = Oracle()
    norms = {}
    for tag in SOLVES:
        g = np.load(os.path.join(OUT, tag + ".npz"))
        if "uT" in g:
            continue
        n, steps = int(g["n"]), int(g["steps"])
        u0, v1, v2 = oracle.initial_conditions(n, float(g["vscale"]))
        s = OracleSolver(n, u0, v1, v2, float(g["nu"]), float(g["dt"]), float(g["dx"]), float(g["tol"]), int(g["shape"]))
        for k in range(steps):
            s.form_rhs()
            it, hist = s.solve()
            assert it == int(g["cycles"][k]) and np.array_equal(hist, g["hist"][k][: it + 1]), tag
        uT = s.u(0)
        assert uT[n // 2, n // 2] == float(g["mid"]), tag
        assert float(np.linalg.norm(uT)) == float(g["norm_uT"]), f"{tag}: this BLAS does not reproduce the stored norm"
        norms[tag] = exact_norm(uT)
        s.close()
    with open(os.path.join(OUT, "solve_norms.json"), "w") as f:
        json.dump(norms, f, indent=1)
        f.write("\n")
    print(norms)
