#!/usr/bin/env python
"""bench.py -- BASELINE.json metric: V-cycle ms & HBM GB/s (fraction of peak) at N=16384^2.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Own arm.  Workload = BASELINE.json configs[2] (SURVEY.md 8d "C3"): N=16384, nu=-4e-4, vscale=1,
tol=1e-6, V-cycle, reference initial conditions generated on the device (synthetic, resident in
HBM before the timed region).  One STEP = one implicit Crank-Nicolson time step = compute_rhs +
mg_outer (V-cycles until ||r||/||r0|| <= tol; multigrid.cpp:165-169).  `value` = timed ms divided
by the V-cycles executed in the timed region, i.e. ms per V-cycle INCLUDING its convergence check
and the amortised compute_rhs of its time step.  Fields are 2.1 GB each (>> 126 MB L2), so no
L2 flush is needed between iterations.

`e2e` = the same metric through the reference-facing entry point mgb200_timestepper_host
(timestepper(uT,u0,v1,v2,...) of multigrid.cpp:124 with HOST arrays, pinned): H2D of u0,v1,v2,
tower construction, one time step, D2H of uT, all inside the timed region, every step (the level
towers' HBM allocation is reused between calls of the same shape; the first call is the warm-up).

`--impl reference` times the reference's own CPU implementation (oracle/_ref/libmgref_O3.so: the
unmodified gs.cpp + multigrid.cpp, run inside an OpenMP team as multigrid.cpp:252-258 does) on a
bounded sample of the same workload.

`--dump-outputs DIR` writes the field and the residual history the last timed step left (dump_outputs).  The inputs
depend only on the arguments, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark writes nothing into the tree it runs from, bytecode caches included

N_FULL = 16384
NU, VSCALE, TOL = -4e-4, 1.0, 1e-6
W_REF_BYTES_PER_NODE = 475.0          # SURVEY.md 8d: reference pass structure, one pass per operator


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock + throttle reasons during the timed region (pynvml, 100 ms period)."""

    def __init__(self, index=0):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        if self.nv:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._t:
            self._t.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": []}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


# ---------------------------------------------------------------------------------------------
# CPU baseline: the compiled reference (or the oracle port) on a bounded sample
def cpu_vcycle_ms(n_target, steps, warmup, threads=None, budget_s=240.0):
    """ms per V-cycle (+ convergence check) of the reference CPU implementation at n_target.  The reference's
    towers take ~145 B per fine node (39 GB at N=16384; multigrid.cpp:138-162): the true size is run when the
    host has the memory (BASELINE.md section 4), otherwise the largest size that fits, scaled by the node-count
    ratio and FLAGGED as such.  Returns (ms, kind, threads, sample text, extra dict)."""
    import numpy as np
    import psutil
    from oracle.oracle import Oracle, OracleSolver, Towers, ref_available
    threads = threads or os.cpu_count() or 1
    free_gb = psutil.virtual_memory().available / 2**30
    n = n_target
    while n > 256 and (145.0 * (n + 1) ** 2 / 2**30 > 0.8 * free_gb or n > 32768):      # the reference's int indices stop at 32768
        n //= 2
    scale = (n_target + 1) ** 2 / float((n + 1) ** 2)
    dx = 1.0 / n; dt = dx / 10
    o = Oracle()
    u0, v1, v2 = o.initial_conditions(n, VSCALE)
    times = []
    t_start = time.perf_counter()
    if ref_available("O3"):
        kind = "reference"
        tw = Towers(Oracle("O3"), n, u0, v1, v2, NU, dt, dx, TOL, 1)
        del u0, v1, v2
        tw.form_rhs()
        for k in range(warmup + steps):
            t = time.perf_counter()
            tw.cycle_and_norm(threads)
            if k >= warmup:
                times.append(time.perf_counter() - t)
            if len(times) >= 2 and time.perf_counter() - t_start > budget_s:           # bounded sample
                break
    else:
        kind, threads = "port", 1
        s = OracleSolver(n, u0, v1, v2, NU, dt, dx, TOL, 1)
        s.form_rhs()
        for k in range(warmup + steps):
            t = time.perf_counter()
            s.cycle(); s.residual_norm()
            if k >= warmup:
                times.append(time.perf_counter() - t)
            if len(times) >= 2 and time.perf_counter() - t_start > budget_s:
                break
    ms = 1e3 * float(np.mean(times)) * scale
    impl = "gs.cpp+multigrid.cpp -O3, OpenMP tasks" if kind == "reference" else "oracle/mg_oracle.c -O2, serial"
    sample = (f"{len(times)} V-cycle(s)+check at N={n} after {warmup} warm-up"
              + (f", mean x{scale:.3f} (node count ratio to N={n_target}: host RAM {free_gb:.0f} GB < 145 B/node)" if n != n_target else "")
              + f"; {impl}")
    extra = {"measured_N": n, "scaled": n != n_target, "scale_factor": scale, "cycles_timed": len(times)}
    return ms, kind, threads, sample, extra


def run_reference(args, rank):
    if rank != 0:
        return
    n = args.n
    ms, kind, cores, sample, extra = cpu_vcycle_ms(n, max(1, args.steps), max(0, min(args.warmup, 2)))
    line = {
        "impl": "reference", "metric": metric_name(n), "value": ms, "unit": "ms", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": False, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic (reference initial conditions, multigrid.cpp:206-233)",
        "config": workload_config(n, args.gpus),
        "cpu_baseline": dict({"value": ms, "unit": "ms", "cores": cores, "kind": kind, "sample": sample}, **extra),
        "e2e": {"value": ms, "unit": "ms", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "effective_GBps_Wref": W_REF_BYTES_PER_NODE * (n + 1) ** 2 / (ms * 1e-3) / 1e9,
    }
    print(json.dumps(line), flush=True)


def metric_name(n):
    return f"V-cycle ms at N={n}^2 (fine-grid V-cycle incl. convergence check)"


def workload_config(n, gpus):
    """the same dict for both arms (own and reference): BASELINE.json configs[2] ("C3") at the default size,
    configs[4] ("C5") at N=65536, otherwise just the size"""
    tag = {16384: "C3: ", 65536: "C5: "}.get(n, "")
    field_gb = (n + 1) ** 2 * 8 / 1e9
    return {"workload": f"{tag}N={n}^2 advection-diffusion Crank-Nicolson step, nu={NU}, vscale={VSCALE}, "
                        f"tol={TOL}, V-cycle (3 pre + 3 post RB-GS), {gpus} GPU(s)",
            "N": n, "nu": NU, "vscale": VSCALE, "tol": TOL, "shape": 1, "levels": int(math.log2(n)) - 4,
            "l2_policy": (f"inputs ({field_gb:.2g} GB per field) exceed the 126 MB L2; no flush needed" if field_gb > 0.3 else
                          f"inputs ({field_gb:.2g} GB per field) are comparable to the 126 MB L2: a 256 MB buffer is "
                          "rewritten between timed steps")}


# ---------------------------------------------------------------------------------------------
def parity_block(mg, s, n, rank, world, dist, arith_name):
    """Parity evidence for the configuration that was just timed: from FRESH reference initial conditions run one
    implicit time step to tol and describe the result -- cycle count, ||uT||_2, uT[N/2,N/2], a 129 x 129 strided
    sample, and the rank-count-independent field digest (hpcclassmultigridproject_b200/digest.py) -- then compare it
    with the fixture the compiled reference produced for this configuration (tests/golden/make_golden_large.py).
    Sharded ranks describe their own rows; rank 0 stitches.  Returns (dict, ok)."""
    import numpy as np
    from hpcclassmultigridproject_b200 import digest
    s.set_fields_reference_ic(VSCALE)
    info = s.timestep(1)[0]
    lo, hi, u = s.get_u_host_rows()                     # the rows this rank owns (all rows on one GPU)
    st = max(1, n // 128)
    rows = [i for i in range(0, n + 1, st) if lo <= i <= hi]
    mine = {
        "digests": digest.slab_digests(u, n, lo, hi, base_row=lo) if n % digest.NSLAB == 0 else {},
        "sumsq": float(np.einsum("ij,ij->", u, u)),
        "mid": float(u[n // 2 - lo, n // 2]) if lo <= n // 2 <= hi else None,
        "sample_rows": rows, "sample": u[[i - lo for i in rows], ::st].copy(),
    }
    del u
    parts = [mine]
    if world > 1:
        parts = [None] * world if rank == 0 else None
        dist.gather_object(mine, parts, dst=0)
    if rank != 0:
        return None, True
    dig = {}
    for q in parts:
        dig.update(q["digests"])
    sample = np.concatenate([q["sample"] for q in parts], axis=0)
    assert [i for q in parts for i in q["sample_rows"]] == list(range(0, n + 1, st))
    norm = math.sqrt(math.fsum(q["sumsq"] for q in parts))
    mid = [q["mid"] for q in parts if q["mid"] is not None][0]
    out = {"cycles": int(info.cycles), "converged": bool(info.converged), "res_history": [float(x) for x in info.history()],
           "norm_uT": norm, "mid": mid, "arith": arith_name,
           "u_sha256": digest.combine(dig) if len(dig) == digest.NSLAB else None,
           "digest": "sha256 over the sha256 of 8 fixed row slabs (same value for any rank count)"}
    ok = True
    fx = os.path.join(ROOT, "tests", "golden", f"large_c3_n{n}_tol1e-6.npz")
    if os.path.exists(fx) and (NU, VSCALE, TOL) == (-4e-4, 1.0, 1e-6):
        g = np.load(fx)
        rel = float(np.linalg.norm(sample - g["sample"]) / np.linalg.norm(g["sample"]))
        ref = {"fixture": os.path.relpath(fx, ROOT), "cycles": int(g["cycles"]), "norm_uT": float(g["norm_uT"]), "mid": float(g["mid"]),
               "u_sha256_reference": str(g["u_sha256"]), "sample_rel_l2": rel,
               "norm_rel_err": abs(norm - float(g["norm_uT"])) / float(g["norm_uT"]),
               "mid_rel_err": abs(mid - float(g["mid"])) / abs(float(g["mid"])), "bar": 1e-10}
        ok = (out["cycles"] == ref["cycles"] and rel <= 1e-10 and ref["norm_rel_err"] <= 1e-10 and ref["mid_rel_err"] <= 1e-10)
        ref["ok"] = ok
        out["reference"] = ref
    else:
        out["reference"] = None         # no compiled-reference fixture for this size (the reference stops at N=32768)
    return out, ok


DUMP_U_BYTES = 32 << 20


def dump_outputs(out_dir, s, infos, n, rank, world, dist):
    """--dump-outputs: what the timed steps hand back to a caller, after the last of them, as <out_dir>/<name>.npy
    (float64), so that two builds run with the same arguments can be compared output for output.
      u.npy                 the field uT: every row when the field fits in DUMP_U_BYTES, otherwise that many bytes of
                            whole rows drawn by a fixed seed (the same rows for every run at this N), in row order
      residual_history.npy  ||r0|| and the residual norm after each V-cycle of the last time step"""
    import numpy as np
    nrows = min(n + 1, DUMP_U_BYTES // ((n + 1) * 8))
    rows = np.arange(n + 1) if nrows == n + 1 else np.sort(np.random.default_rng(0).choice(n + 1, nrows, replace=False))
    lo, hi, u = s.get_u_host_rows()                     # the rows this rank owns (all rows on one GPU)
    parts = [u[rows[(rows >= lo) & (rows <= hi)] - lo]]
    del u
    if world > 1:
        mine = parts[0]
        parts = [None] * world if rank == 0 else None
        dist.gather_object(mine, parts, dst=0)          # rank r owns the r-th slab of rows: rank order is row order
    if rank != 0:
        return
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "u.npy"), np.concatenate(parts, axis=0))
    np.save(os.path.join(out_dir, "residual_history.npy"), np.array(infos[-1].history(), dtype=np.float64))


# ---------------------------------------------------------------------------------------------
def run_own(args, rank, world):
    import torch
    import hpcclassmultigridproject_b200 as mg

    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    # host buffers of the e2e leg next to this rank's GPU (undone before the CPU leg, which uses every core)
    from hpcclassmultigridproject_b200.affinity import bind_near_gpu
    all_cpus = os.sched_getaffinity(0)
    affinity = None if os.environ.get("MGB200_BENCH_NO_AFFINITY") else bind_near_gpu(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    plan = mg.PLAN_UNFUSED if args.plan == "unfused" else mg.PLAN_FUSED
    arith = mg.ARITH_EXACT if args.arith == "exact" else mg.ARITH_FAST
    n = args.n
    dx = 1.0 / n; dt = dx / 10
    hbm_peak, peak_src = peaks()

    def barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
            torch.cuda.synchronize()

    uid = None
    if world > 1:
        box = [mg.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        uid = box[0]
    s = mg.Solver(n, NU, dt, dx, TOL, plan=plan, arith=arith, device=local, rank=rank, nranks=world, unique_id=uid)
    s.set_fields_reference_ic(VSCALE)
    s.synchronize()
    for _ in range(args.warmup):
        s.timestep(1)
    barrier()
    l0 = s.kernel_launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ext = torch.cuda.ExternalStream(s.stream)
    with ClockSampler(local) as clk:
        ev0.record(ext)
        infos = s.timestep(args.steps)
        ev1.record(ext)
        ev1.synchronize()
    barrier()
    if args.dump_outputs:                               # before the measurements below move the field on
        dump_outputs(args.dump_outputs, s, infos, n, rank, world, dist)
    ms_total = ev0.elapsed_time(ev1)
    if dist:
        t = torch.tensor([ms_total], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    cycles = sum(i.cycles for i in infos)
    launches = s.kernel_launches - l0
    ms_cycle = ms_total / max(1, cycles)
    m0 = float(n + 1) ** 2

    # the V-cycle alone (cycle + residual norm, no compute_rhs, no host round trip): K more cycles
    # on the same system enqueued back to back (the work of a cycle does not depend on the data),
    # CUDA events on the solver's stream
    ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.cycle()
    barrier()
    ev2.record(ext)
    for _ in range(max(3, args.steps)):
        s.cycle_async()
    ev3.record(ext)
    ev3.synchronize()
    vc = ev2.elapsed_time(ev3) / max(3, args.steps)
    if dist:
        t = torch.tensor([vc], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        vc = float(t.item())

    # dominant kernel: the level-0 streaming pass (fused) / colour half-sweep (unfused)
    prof = s.profile_level0(reps=5)
    (ms_a, by_a), (ms_b, by_b) = prof
    dom_ms, dom_bytes = (ms_a + ms_b) / 2, (by_a + by_b) / 2
    achieved = dom_bytes / (dom_ms * 1e-3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp) and n == N_FULL and world == 1:
        try:
            traffic = json.load(open(tp)).get(f"{args.plan}_level0_bytes_per_launch")   # from the committed ncu capture (see "source" there)
        except Exception:
            traffic = None
    cycle_bytes = s.cycle_bytes
    slab = s.slab(0)
    parity, parity_ok = (None, True) if args.no_parity else parity_block(mg, s, n, rank, world, dist, args.arith)
    if world == 1:
        s.close()

    # ---- e2e through the reference-facing entry point, host buffers, copies timed ----------
    e2e = None
    if not args.no_e2e and world == 1:
        d = [torch.empty(n + 1, n + 1, dtype=torch.float64, device="cuda") for _ in range(3)]
        mg.ops.initial_conditions(*d, n, VSCALE)
        host = [torch.empty(n + 1, n + 1, dtype=torch.float64).pin_memory() for _ in range(4)]
        for h, t in zip(host, d):
            h.copy_(t)
        del d
        torch.cuda.synchronize(); torch.cuda.empty_cache()
        reps, tt, cyc = max(1, min(args.steps, 3)), [], 0
        for k in range(1 + reps):
            t0 = time.perf_counter()
            info = mg.timestepper_host(host[3], host[0], host[1], host[2], NU, mg.maxlvl_for(n), n, dt, dt, dx, TOL, 1,
                                       plan=plan, arith=arith, device=local)
            el = time.perf_counter() - t0
            if k >= 1:
                tt.append(el); cyc += info.cycles
        e2e = {"value": 1e3 * sum(tt) / max(1, cyc), "unit": "ms", "h2d_bytes_per_step": int(3 * m0 * 8),
               "d2h_bytes_per_step": int(m0 * 8), "call": "mgb200_timestepper_host (timestepper, multigrid.cpp:124), T=dt",
               "ms_per_call": 1e3 * sum(tt) / len(tt), "cycles_per_call": cyc / len(tt),
               "host_link_GBps": 4 * m0 * 8 / (sum(tt) / len(tt)) / 1e9,
               "note": "copy-bound: (H2D + D2H bytes) / call time = host_link_GBps, per GPU"}
        mg.release_cached()
        del host
    elif not args.no_e2e:
        # sharded: the same sequence through the handle API, every rank moving its own row slab:
        # pinned host slab (+halo, + the rows the coarse-velocity towers read) -> device, one time
        # step, owned rows of the result -> pinned host
        own_rows = slab["own_hi"] - slab["own_lo"] + 1
        win_rows = slab["mem_hi"] - slab["mem_lo"] + 1
        # each rank keeps ONLY its window of the inputs and its own rows of the result in (pinned) host memory
        d = [torch.empty(win_rows, n + 1, dtype=torch.float64, device="cuda") for _ in range(3)]
        mg.ops.initial_conditions_rows(*d, n, VSCALE, slab["mem_lo"], slab["mem_hi"])
        host = [torch.empty(win_rows, n + 1, dtype=torch.float64).pin_memory() for _ in range(3)]
        for h, t in zip(host, d):
            h.copy_(t)
        del d
        out_rows = torch.empty(own_rows, n + 1, dtype=torch.float64).pin_memory()
        torch.cuda.synchronize(); torch.cuda.empty_cache()
        reps, tt, cyc = max(1, min(args.steps, 3)), [], 0
        for k in range(1 + reps):
            barrier()
            t0 = time.perf_counter()
            s.set_fields_host_window(host[0], host[1], host[2])
            info = s.timestep(1)[0]
            s.get_u_host_rows(out_rows)
            barrier()
            el = time.perf_counter() - t0
            if k >= 1:
                tt.append(el); cyc += info.cycles
        t = torch.tensor([sum(tt)], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e = {"value": 1e3 * float(t.item()) / max(1, cyc), "unit": "ms",
               "h2d_bytes_per_step": int(world * 3 * win_rows * (n + 1) * 8),
               "d2h_bytes_per_step": int(m0 * 8),
               "call": "mgb200_set_fields_host + mgb200_timestep(1) + mgb200_get_u_host on every rank's slab",
               "ms_per_call": 1e3 * float(t.item()) / len(tt), "cycles_per_call": cyc / len(tt),
               "host_link_GBps": (3 * win_rows + own_rows) * (n + 1) * 8 / (float(t.item()) / len(tt)) / 1e9,
               "note": "every rank moves its own slab over its own host link; the rows the coarse-velocity towers need "
                       "travel once (owner -> peers over NVLink); host_link_GBps is per GPU"}
        del host, out_rows
    if world > 1:
        s.close()

    os.sched_setaffinity(0, all_cpus)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        ms, kind, cores, sample, extra = cpu_vcycle_ms(n, 2, 1, budget_s=60.0)
        cpu = dict({"value": ms, "unit": "ms", "cores": cores, "kind": kind, "sample": sample}, **extra)

    if rank == 0:
        line = {
            "metric": metric_name(n), "value": ms_cycle, "unit": "ms", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic (reference initial conditions, multigrid.cpp:206-233, generated on device)",
            "config": workload_config(n, world),
            "impl_config": {"plan": args.plan, "arith": args.arith,
                            "step": "one implicit time step = compute_rhs + V-cycles to tol; value = ms / V-cycles"},
            "parity": parity,
            "cycles_per_step": cycles / args.steps, "vcycles_timed": cycles, "vcycle_only_ms": vc,
            "effective_GBps_Wref": W_REF_BYTES_PER_NODE * m0 / (ms_cycle * 1e-3) / 1e9,
            "plan_GBps": cycle_bytes / (ms_cycle * 1e-3) / 1e9, "plan_bytes_per_cycle": cycle_bytes,
            "plan_frac_of_hbm_peak": cycle_bytes / (ms_cycle * 1e-3) / 1e9 / hbm_peak,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                         "traffic": traffic, "peak_source": peak_src,
                         "kernel": ("level-0 streaming pass (3 RB-GS iterations fused with residual+injection / "
                                    "prolong+correct+norm)") if args.plan == "fused" else "level-0 colour half-sweep + residual",
                         "launch_ms": [ms_a, ms_b], "launch_bytes": [by_a, by_b]},
            "clocks": clk.summary(), "gpu_launches": int(launches), "e2e": e2e, "host_affinity": affinity, "cpu_baseline": cpu,
        }
        print(json.dumps(line), flush=True)
    if dist:
        dist.destroy_process_group()
    if rank == 0 and not parity_ok:
        print("bench.py: PARITY MISMATCH against " + str(parity["reference"]), file=sys.stderr, flush=True)
        sys.exit(3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--size", "--n", dest="n", type=int, default=N_FULL, help="finest grid N (default: the BASELINE config)")
    ap.add_argument("--plan", default="fused", choices=["fused", "unfused"])
    ap.add_argument("--arith", default="fast", choices=["fast", "exact"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the field and residual history of the last timed step "
                    "to DIR/*.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "own":
        ap.error("--dump-outputs needs --impl own")
    args.warmup = max(args.warmup, 3) if args.impl == "own" else args.warmup
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference(args, rank)
    else:
        run_own(args, rank, world)


if __name__ == "__main__":
    main()
