"""Throughput of batched solver handles against single-problem handles stepped one after another.

For each N and batch size B: B problems with seeded fields (a Gaussian bump and a vortex per member), advanced by
`--steps` time steps (compute_rhs + V-cycles to tol) of ONE batched handle, and by B single-problem handles stepped
one after another on the same inputs.  Both are timed with the host clock around calls that end in a device
synchronisation (timestep() synchronises), after `--warmup` untimed steps of every handle.  At the largest sizes at
most --max-solo single-problem handles are timed and their time per member-step stands for all B.  One JSON line per
configuration; the card's name, power limit and maximum SM clock come first (read-only nvidia-smi query).

    python tools/batch_throughput.py [--sizes 64,256,1024,2048] [--batches 1,8,64,256] [--steps 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def member_fields(n, b):
    x = np.linspace(0.0, 1.0, n + 1)
    X, Y = np.meshgrid(x, x, indexing="ij")
    rng = np.random.default_rng(1000 + b)
    cx, cy = 0.3 + 0.4 * rng.random(), 0.3 + 0.4 * rng.random()
    u0 = np.exp(-((X - cx) ** 2 + (Y - cy) ** 2) / 0.01)
    u0[0, :] = u0[-1, :] = 0.0; u0[:, 0] = u0[:, -1] = 0.0
    s = 0.5 + rng.random()
    return u0, s * np.sin(np.pi * X) * np.cos(np.pi * Y), -s * np.cos(np.pi * X) * np.sin(np.pi * Y)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="64,256,1024,2048")
    ap.add_argument("--batches", default="1,8,64,256")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--max-solo", type=int, default=64)
    ap.add_argument("--mem-gb", type=float, default=120.0, help="skip a batch whose level arrays would exceed this")
    a = ap.parse_args()
    import torch
    import hpcclassmultigridproject_b200 as mg
    assert torch.cuda.is_available(), "batch_throughput needs a CUDA device"
    print(json.dumps({"card": card()}), flush=True)
    for n in [int(x) for x in a.sizes.split(",")]:
        dx = 1.0 / n; dt = dx / 10; nu = -4e-4; tol = 1e-8
        for B in [int(x) for x in a.batches.split(",")]:
            gb = 5 * 2 * (n + 1) * (n + 1) * 8 * 4 / 3 * B / 1e9        # 5 arrays, split-layout slack, all levels
            if gb > a.mem_gb:
                print(json.dumps({"n": n, "batch": B, "status": "not measured (memory)"}), flush=True)
                continue
            fl = [member_fields(n, b) for b in range(B)]
            U = [np.ascontiguousarray(np.stack([f[k] for f in fl])) for k in range(3)]
            with mg.Solver(n, nu, dt, dx, tol, batch=B) as s:
                s.set_fields_host(*U)
                s.timestep(a.warmup)
                t0 = time.perf_counter()
                infos = s.timestep(a.steps)
                t_batch = time.perf_counter() - t0
                cycles = sum(i.cycles for step in infos for i in step)
                bytes_per_cycle = s.cycle_bytes
            nsolo = min(B, a.max_solo)
            solos = [mg.Solver(n, nu, dt, dx, tol) for _ in range(nsolo)]
            try:
                for b, h in enumerate(solos):
                    h.set_fields_host(*fl[b])
                    h.timestep(a.warmup)
                t0 = time.perf_counter()
                solo_cycles = 0
                for h in solos:
                    solo_cycles += sum(i.cycles for i in h.timestep(a.steps))
                t_solo = (time.perf_counter() - t0) * B / nsolo
            finally:
                for h in solos:
                    h.close()
            ms = t_batch * 1e3 / (B * a.steps)
            print(json.dumps({
                "n": n, "batch": B, "steps": a.steps,
                "member_steps_per_s": B * a.steps / t_batch,
                "ms_per_member_step": ms,
                "solo_ms_per_member_step": t_solo * 1e3 / (B * a.steps),
                "speedup_over_solo": t_solo / t_batch,
                "cycles_per_member_step": cycles / (B * a.steps),
                "solo_cycles_per_member_step": solo_cycles / (nsolo * a.steps),
                "plan_GBps": bytes_per_cycle / B * cycles / t_batch / 1e9,      # cycle_bytes counts all B members
                "solo_handles_timed": nsolo,
            }), flush=True)


if __name__ == "__main__":
    main()
