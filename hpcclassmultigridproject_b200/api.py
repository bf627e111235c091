"""ctypes binding of include/mgb200.h.  Device arrays are passed as raw pointers; helpers accept
torch CUDA tensors (float64) and take ``tensor.data_ptr()``."""
from __future__ import annotations

import ctypes as C
import math
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MGB200_LIB") or os.path.join(HERE, "libmgb200.so")   # MGB200_LIB: a tuning variant of the library

ARITH_FAST, ARITH_EXACT = 0, 1
PLAN_FUSED, PLAN_UNFUSED = 0, 1
# Options.restriction: injection (the reference), full weighting on the UNFUSED plan only, full weighting on either plan
RESTRICT_INJECT, RESTRICT_FW_UNFUSED, RESTRICT_FW = 0, 1, 2


class MgError(RuntimeError):
    pass


class Options(C.Structure):
    _fields_ = [("struct_size", C.c_int), ("shape", C.c_int), ("niter", C.c_int), ("coarse_maxit", C.c_int),
                ("coarse_tol", C.c_double), ("max_cycle", C.c_int), ("arith", C.c_int), ("plan", C.c_int),
                ("correct_towers", C.c_int), ("use_graph", C.c_int), ("device", C.c_int), ("restriction", C.c_int),
                ("coarse_exact", C.c_int), ("reserved", C.c_int * 6)]


class SolveInfo(C.Structure):
    _fields_ = [("cycles", C.c_int), ("converged", C.c_int), ("res0", C.c_double), ("res", C.c_double),
                ("hist", C.c_double * 52)]

    def history(self):
        return [self.hist[k] for k in range(self.cycles + 1)]


_lib = None
_vp, _d, _l, _i = C.c_void_p, C.c_double, C.c_long, C.c_int


def lib():
    """Load libmgb200.so (never builds, never falls back)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MgError(f"{LIB_PATH} is missing: build it with `python -m hpcclassmultigridproject_b200._build` "
                      "(nvcc, sm_100a).  There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    L.mgb200_last_error.restype = C.c_char_p
    L.mgb200_version.restype = _i
    L.mgb200_gauss_seidel.argtypes = [_vp, _vp, _l, _l, _vp, _vp, _d, _d, _d, _i, _i, _vp]
    L.mgb200_residual.argtypes = [_vp, _vp, _vp, _l, _l, _vp, _vp, _d, _d, _d, _i, _vp]
    L.mgb200_compute_norm.argtypes = [_vp, _l, _l, C.POINTER(_d), _vp]
    L.mgb200_norm2_async.argtypes = [_vp, _l, _l, _vp, _vp]
    L.mgb200_residual_norm2_async.argtypes = [_vp, _vp, _vp, _l, _l, _vp, _vp, _d, _d, _d, _i, _vp, _vp]
    L.mgb200_compute_rhs.argtypes = [_vp, _vp, _l, _l, _vp, _vp, _d, _d, _d, _i, _vp]
    L.mgb200_restriction.argtypes = [_vp, _l, _vp, _l, _l, _vp]
    L.mgb200_prolongation.argtypes = [_vp, _l, _vp, _l, _l, _vp]
    L.mgb200_prolong_correct.argtypes = [_vp, _l, _vp, _l, _l, _vp]
    L.mgb200_vecadd.argtypes = [_vp, _vp, _vp, _l, _l, _vp]
    L.mgb200_restriction_fw.argtypes = L.mgb200_restriction.argtypes
    L.mgb200_initial_conditions.argtypes = [_vp, _vp, _vp, _l, _l, _d, _vp]
    L.mgb200_initial_conditions_rows.argtypes = [_vp, _vp, _vp, _l, _l, _d, _l, _l, _vp]
    L.mgb200_default_options.argtypes = [C.POINTER(Options)]
    L.mgb200_default_options.restype = None
    L.mgb200_create.argtypes = [C.POINTER(_vp), _l, _i, _d, _d, _d, _d, C.POINTER(Options)]
    L.mgb200_create_batched.argtypes = [C.POINTER(_vp), _l, _i, _i, _d, _d, _d, _d, C.POINTER(Options)]
    L.mgb200_batch_size.argtypes = [_vp]; L.mgb200_batch_size.restype = _i
    L.mgb200_comm_unique_id.argtypes = [C.c_char_p]
    L.mgb200_create_sharded.argtypes = [C.POINTER(_vp), _l, _i, _d, _d, _d, _d, C.POINTER(Options), _i, _i, C.c_char_p, _l]
    L.mgb200_slab.argtypes = [_vp, _i, C.POINTER(_l * 6)]
    L.mgb200_slab_plan.argtypes = [_l, _i, _i, _i, _l, _i, C.POINTER(_l * 6)]
    L.mgb200_destroy.argtypes = [_vp]
    L.mgb200_set_fields_device.argtypes = [_vp, _vp, _vp, _vp, _l]
    L.mgb200_set_fields_host.argtypes = [_vp, _vp, _vp, _vp]
    L.mgb200_set_fields_reference_ic.argtypes = [_vp, _d]
    L.mgb200_form_rhs.argtypes = [_vp, C.POINTER(_d)]
    L.mgb200_cycle.argtypes = [_vp, C.POINTER(_d)]
    L.mgb200_cycle_async.argtypes = [_vp]
    L.mgb200_last_norm.argtypes = [_vp, C.POINTER(_d)]
    L.mgb200_solve.argtypes = [_vp, C.POINTER(SolveInfo)]
    L.mgb200_timestep.argtypes = [_vp, _i, C.POINTER(SolveInfo)]
    L.mgb200_get_u_device.argtypes = [_vp, _vp, _l]
    L.mgb200_get_u_host.argtypes = [_vp, _vp]
    L.mgb200_get_level_host.argtypes = [_vp, _i, _i, _vp]
    L.mgb200_synchronize.argtypes = [_vp]
    L.mgb200_stream.argtypes = [_vp]; L.mgb200_stream.restype = _vp
    L.mgb200_kernel_launches.argtypes = [_vp]; L.mgb200_kernel_launches.restype = _l
    L.mgb200_cycle_bytes.argtypes = [_vp]; L.mgb200_cycle_bytes.restype = _d
    L.mgb200_profile_level0.argtypes = [_vp, _i, C.POINTER(_d), C.POINTER(_d), C.POINTER(_d), C.POINTER(_d)]
    L.mgb200_timestepper_host.argtypes = [_vp, _vp, _vp, _vp, _d, _i, _i, _d, _d, _d, _d, _i, C.POINTER(Options),
                                          C.POINTER(SolveInfo)]
    L.mgb200_timestepper_device.argtypes = L.mgb200_timestepper_host.argtypes
    L.mgb200_release_cached.argtypes = []
    _lib = L
    return L


def _ck(rc):
    if rc != 0:
        raise MgError(f"mgb200 error {rc}: {lib().mgb200_last_error().decode()}")


def _ptr(t):
    """raw address of a torch tensor / numpy array / int"""
    if t is None:
        return None
    if isinstance(t, int):
        return t
    if hasattr(t, "data_ptr"):
        return t.data_ptr()
    return t.ctypes.data


def maxlvl_for(n: int) -> int:
    """multigrid.cpp:193"""
    return int(math.log2(n)) - 4


def default_options(**kw) -> Options:
    o = Options()
    lib().mgb200_default_options(C.byref(o))
    for k, v in kw.items():
        setattr(o, k, v)
    return o


def comm_unique_id() -> bytes:
    """128-byte NCCL unique id (rank 0 creates it, the host program broadcasts it)"""
    buf = C.create_string_buffer(128)
    _ck(lib().mgb200_comm_unique_id(buf))
    return buf.raw


def slab_plan(n, maxlvl, nranks, rank, lvl, shard_min_rows=0):
    """row window of `rank` at level `lvl` (pure arithmetic, needs no GPU):
    dict(sharded, present, own_lo, own_hi, mem_lo, mem_hi)"""
    out = (_l * 6)()
    _ck(lib().mgb200_slab_plan(n, maxlvl, nranks, rank, shard_min_rows, lvl, C.byref(out)))
    return dict(zip(("sharded", "present", "own_lo", "own_hi", "mem_lo", "mem_hi"), [int(x) for x in out]))


class _Ops:
    """The gs.h / gscu.h operators on torch CUDA tensors (float64, row stride = tensor.stride(0))."""

    @staticmethod
    def _ld(t):
        assert t.is_cuda and t.dtype.is_floating_point and t.element_size() == 8 and t.stride(1) == 1
        return t.stride(0)

    def gauss_seidel(self, u, rhs, n, v1, v2, dt, nu, dx, iters=1, arith=ARITH_EXACT, stream=None):
        _ck(lib().mgb200_gauss_seidel(_ptr(u), _ptr(rhs), n, self._ld(u), _ptr(v1), _ptr(v2), dt, nu, dx, iters, arith, stream))
        return u

    def residual(self, res, u, rhs, n, v1, v2, dt, nu, dx, arith=ARITH_EXACT, stream=None):
        _ck(lib().mgb200_residual(_ptr(res), _ptr(u), _ptr(rhs), n, self._ld(u), _ptr(v1), _ptr(v2), dt, nu, dx, arith, stream))
        return res

    def compute_norm(self, a, n, stream=None) -> float:
        out = _d(0.0)
        _ck(lib().mgb200_compute_norm(_ptr(a), n, self._ld(a), C.byref(out), stream))
        return out.value

    def residual_norm2(self, res, u, rhs, n, v1, v2, dt, nu, dx, out_dev, arith=ARITH_EXACT, stream=None):
        _ck(lib().mgb200_residual_norm2_async(_ptr(res), _ptr(u), _ptr(rhs), n, self._ld(u), _ptr(v1), _ptr(v2), dt, nu,
                                              dx, arith, _ptr(out_dev), stream))

    def compute_rhs(self, rhs, u, n, v1, v2, dt, nu, dx, arith=ARITH_EXACT, stream=None):
        _ck(lib().mgb200_compute_rhs(_ptr(rhs), _ptr(u), n, self._ld(u), _ptr(v1), _ptr(v2), dt, nu, dx, arith, stream))
        return rhs

    def restriction(self, coarse, fine, nf, stream=None):
        _ck(lib().mgb200_restriction(_ptr(coarse), self._ld(coarse), _ptr(fine), self._ld(fine), nf, stream))
        return coarse

    def restriction_fw(self, coarse, fine, nf, stream=None):
        """opt-in full weighting (gs.cpp:277-280, commented out in the reference)"""
        _ck(lib().mgb200_restriction_fw(_ptr(coarse), self._ld(coarse), _ptr(fine), self._ld(fine), nf, stream))
        return coarse

    def prolongation(self, fine, coarse, nc, stream=None):
        _ck(lib().mgb200_prolongation(_ptr(fine), self._ld(fine), _ptr(coarse), self._ld(coarse), nc, stream))
        return fine

    def prolong_correct(self, u_fine, coarse, nc, stream=None):
        _ck(lib().mgb200_prolong_correct(_ptr(u_fine), self._ld(u_fine), _ptr(coarse), self._ld(coarse), nc, stream))
        return u_fine

    def vecadd(self, c, a, b, n, stream=None):
        _ck(lib().mgb200_vecadd(_ptr(c), _ptr(a), _ptr(b), n, self._ld(a), stream))
        return c

    def initial_conditions(self, u0, v1, v2, n, vscale=1.0, stream=None):
        _ck(lib().mgb200_initial_conditions(_ptr(u0), _ptr(v1), _ptr(v2), n, self._ld(u0), vscale, stream))

    def initial_conditions_rows(self, u0, v1, v2, n, vscale, row_lo, row_hi, stream=None):
        """rows row_lo..row_hi only; the tensors hold just those rows"""
        _ck(lib().mgb200_initial_conditions_rows(_ptr(u0), _ptr(v1), _ptr(v2), n, self._ld(u0), vscale, row_lo, row_hi, stream))


ops = _Ops()


class Solver:
    """mgb200_solver handle: the V/W-cycle driver (mg_inner / mg_outer / timestepper).

    batch=B: a batched handle of B independent problems of this size (mgb200_create_batched).  Fields are then
    (B, n+1, n+1) arrays; form_rhs / cycle / last_norm return B norms, solve B infos, timestep a list of nsteps lists
    of B infos, get_u_host / level (B, n+1, n+1) arrays."""

    def __init__(self, n, nu, dt, dx, tol, maxlvl=None, rank=0, nranks=1, unique_id=None, shard_min_rows=0, batch=None, **opts):
        """nranks > 1: row-slab sharded handle (one process per GPU); unique_id = comm_unique_id() of rank 0"""
        self.n = n
        self.maxlvl = maxlvl_for(n) if maxlvl is None else maxlvl
        self.opt = default_options(**opts)
        self.rank, self.nranks = rank, nranks
        self.batch = batch
        self.h = _vp()
        if batch is not None:
            assert nranks == 1, "batched handles run on one GPU"
            _ck(lib().mgb200_create_batched(C.byref(self.h), n, self.maxlvl, batch, nu, dt, dx, tol, C.byref(self.opt)))
        elif nranks == 1:
            _ck(lib().mgb200_create(C.byref(self.h), n, self.maxlvl, nu, dt, dx, tol, C.byref(self.opt)))
        else:
            assert unique_id is not None and len(unique_id) == 128
            _ck(lib().mgb200_create_sharded(C.byref(self.h), n, self.maxlvl, nu, dt, dx, tol, C.byref(self.opt), rank, nranks,
                                            unique_id, shard_min_rows))

    def slab(self, lvl=0):
        out = (_l * 6)()
        _ck(lib().mgb200_slab(self.h, lvl, C.byref(out)))
        return dict(zip(("sharded", "present", "own_lo", "own_hi", "mem_lo", "mem_hi"), [int(x) for x in out]))

    def close(self):
        if getattr(self, "h", None):
            lib().mgb200_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def members(self) -> int:
        """problems the handle holds (1 unless batched)"""
        return lib().mgb200_batch_size(self.h)

    def _shape(self, nl):
        return (nl + 1, nl + 1) if self.batch is None else (self.batch, nl + 1, nl + 1)

    def _norms(self, fn):
        r = (_d * self.members)()
        _ck(fn(self.h, r))
        return r[0] if self.batch is None else list(r)

    def set_fields_device(self, u0, v1, v2):
        if self.batch is not None:
            for a in (u0, v1, v2):
                assert tuple(a.shape) == self._shape(self.n) and a.stride(0) == (self.n + 1) * a.stride(1), "members (n+1) rows apart"
            _ck(lib().mgb200_set_fields_device(self.h, _ptr(u0), _ptr(v1), _ptr(v2), u0.stride(1)))
            return
        _ck(lib().mgb200_set_fields_device(self.h, _ptr(u0), _ptr(v1), _ptr(v2), u0.stride(0)))

    def set_fields_host(self, u0, v1, v2):
        """numpy arrays or pinned torch CPU tensors, dense (n+1)^2 (batched: dense (B, n+1, n+1))"""
        if self.batch is not None:
            for a in (u0, v1, v2):
                assert tuple(a.shape) == self._shape(self.n), (tuple(a.shape), self._shape(self.n))
                assert a.flags["C_CONTIGUOUS"] if hasattr(a, "flags") else a.is_contiguous()
        _ck(lib().mgb200_set_fields_host(self.h, _ptr(u0), _ptr(v1), _ptr(v2)))

    def set_fields_reference_ic(self, vscale=1.0):
        _ck(lib().mgb200_set_fields_reference_ic(self.h, vscale))

    def form_rhs(self):
        return self._norms(lib().mgb200_form_rhs)

    def cycle(self):
        return self._norms(lib().mgb200_cycle)

    def cycle_async(self):
        _ck(lib().mgb200_cycle_async(self.h))

    def last_norm(self):
        return self._norms(lib().mgb200_last_norm)

    def solve(self):
        """SolveInfo (batched: a list of B)"""
        infos = (SolveInfo * self.members)()
        _ck(lib().mgb200_solve(self.h, infos))
        return infos[0] if self.batch is None else list(infos)

    def timestep(self, nsteps):
        """nsteps SolveInfos (batched: nsteps lists of B)"""
        B = self.members
        infos = (SolveInfo * (nsteps * B))()
        _ck(lib().mgb200_timestep(self.h, nsteps, infos))
        if self.batch is None:
            return list(infos)
        return [list(infos[k * B:(k + 1) * B]) for k in range(nsteps)]

    def get_u_host(self, out=None):
        import numpy as np
        if out is None:
            out = np.full(self._shape(self.n), np.nan) if self.nranks > 1 else np.empty(self._shape(self.n))
        assert out.shape == self._shape(self.n) and out.flags["C_CONTIGUOUS"]
        _ck(lib().mgb200_get_u_host(self.h, _ptr(out)))
        return out

    def set_fields_host_window(self, u0w, v1w, v2w):
        """sharded handle: the arrays hold ONLY this rank's window, rows slab(0)['mem_lo'] .. ['mem_hi'] of the dense
        (n+1)-wide fields (numpy or pinned torch CPU tensors).  mgb200_set_fields_host reads nothing outside the
        window, so it is handed the address the full array WOULD start at."""
        w = self.slab(0)
        rows = w["mem_hi"] - w["mem_lo"] + 1
        off = w["mem_lo"] * (self.n + 1) * 8
        for a in (u0w, v1w, v2w):
            assert tuple(a.shape) == (rows, self.n + 1), (tuple(a.shape), rows)
        _ck(lib().mgb200_set_fields_host(self.h, _ptr(u0w) - off, _ptr(v1w) - off, _ptr(v2w) - off))

    def get_u_host_rows(self, out=None):
        """the rows this rank OWNS as an (own_hi - own_lo + 1) x (n+1) array (no full-size host array needed)"""
        import numpy as np
        w = self.slab(0)
        lo, hi = (w["own_lo"], w["own_hi"]) if self.nranks > 1 else (0, self.n)
        if out is None:
            out = np.empty((hi - lo + 1, self.n + 1))
        assert tuple(out.shape) == (hi - lo + 1, self.n + 1)
        _ck(lib().mgb200_get_u_host(self.h, _ptr(out) - lo * (self.n + 1) * 8))
        return lo, hi, out

    def get_u_device(self, out):
        if self.batch is not None:
            assert tuple(out.shape) == self._shape(self.n) and out.stride(0) == (self.n + 1) * out.stride(1)
            _ck(lib().mgb200_get_u_device(self.h, _ptr(out), out.stride(1)))
            return out
        _ck(lib().mgb200_get_u_device(self.h, _ptr(out), out.stride(0)))
        return out

    def level(self, lvl, which="u"):
        """dense copy of a level array; a slab rank fills only the rows it holds (the rest is NaN)"""
        import numpy as np
        nl = self.n >> lvl
        out = np.full(self._shape(nl), np.nan)
        _ck(lib().mgb200_get_level_host(self.h, lvl, {"u": 0, "rhs": 1, "v1": 2, "v2": 3}[which], _ptr(out)))
        return out

    def synchronize(self):
        _ck(lib().mgb200_synchronize(self.h))

    def profile_level0(self, reps=5):
        """[(avg ms, algorithmic bytes)] of one launch of the two level-0 kernels of the plan"""
        v = [_d(0.0) for _ in range(4)]
        _ck(lib().mgb200_profile_level0(self.h, reps, *[C.byref(x) for x in v]))
        return [(v[0].value, v[1].value), (v[2].value, v[3].value)]

    @property
    def stream(self):
        return lib().mgb200_stream(self.h)

    @property
    def kernel_launches(self) -> int:
        return lib().mgb200_kernel_launches(self.h)

    @property
    def cycle_bytes(self) -> float:
        return lib().mgb200_cycle_bytes(self.h)


def release_cached():
    """free the handle the one-call drivers keep between calls"""
    _ck(lib().mgb200_release_cached())


def timestepper_device(uT, u0, v1, v2, nu, maxlvl, n, dt, T, dx, tol, shape=1, **opts):
    """timestepper(...) of multigrid.cu:130 on DEVICE arrays (ld = n+1)."""
    o = default_options(**opts)
    info = SolveInfo()
    _ck(lib().mgb200_timestepper_device(_ptr(uT), _ptr(u0), _ptr(v1), _ptr(v2), nu, maxlvl, n, dt, T, dx, tol, shape,
                                        C.byref(o), C.byref(info)))
    return info


def timestepper_host(uT, u0, v1, v2, nu, maxlvl, n, dt, T, dx, tol, shape=1, **opts):
    """timestepper(uT,u0,v1,v2,nu,maxlvl,n,dt,T,dx,tol,shape) of multigrid.cpp:124 on HOST arrays."""
    o = default_options(**opts)
    info = SolveInfo()
    _ck(lib().mgb200_timestepper_host(_ptr(uT), _ptr(u0), _ptr(v1), _ptr(v2), nu, maxlvl, n, dt, T, dx, tol, shape,
                                      C.byref(o), C.byref(info)))
    return info
