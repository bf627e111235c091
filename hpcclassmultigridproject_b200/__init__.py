"""hpcclassmultigridproject_b200 -- B200-native geometric multigrid for the implicit 2-D
advection-diffusion step (one hot path of soniareilly/HPCClassMultigridProject).

The product is the C-ABI shared library ``libmgb200.so`` (CUDA kernels for sm_100a + the C++
V-cycle driver, sources under ``csrc/``, interface in ``include/mgb200.h``).  This package only
binds that ABI with ctypes so tests and bench.py can drive it from Python; there is no Python
or CPU implementation of the path, and importing the binding fails loudly when the library is
missing.
"""
from .api import (  # noqa: F401
    comm_unique_id, default_options, slab_plan, ARITH_EXACT, ARITH_FAST, PLAN_FUSED, PLAN_UNFUSED, RESTRICT_INJECT,
    RESTRICT_FW_UNFUSED, RESTRICT_FW, MgError, Options, SolveInfo, Solver, lib, maxlvl_for, ops,
    release_cached, timestepper_device, timestepper_host,
)
