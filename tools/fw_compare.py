"""Injection (options.restriction = 0, the reference) against full weighting (= 2) on the fused plan: cycles per time
step, time per cycle and per step (time to solution), the level-0 down-leg pass time (profile_level0) and the
relative L2 difference of the two solutions.  Both arms are built and warmed up first, then timed in alternation.

    python tools/fw_compare.py [--n 16384] [--nus -4e-4,-8e-4,-1.6e-3] [--steps 3] [--repeats 3] [--out fw.json]
    python tools/fw_compare.py --gpus 8 --n 65536 --nus -4e-4        # row slabs, one process per GPU (torchrun)

The card's name and power limit are read in the same run and stored with the numbers."""
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
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=16384)
    ap.add_argument("--nus", default="-4e-4,-8e-4,-1.6e-3")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--tol", type=float, default=1e-6)
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--out", default="fw_compare.json")
    a = ap.parse_args()
    if a.gpus > 1 and "RANK" not in os.environ:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={a.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29611", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))

    import torch
    import hpcclassmultigridproject_b200 as mg
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n = a.n; dx = 1.0 / n; dt = dx / 10
    result = dict(card=card(), n=n, gpus=world, tol=a.tol, steps=a.steps, repeats=a.repeats, arms={})

    def make(nu, restriction):
        kw = dict(restriction=restriction, device=local)
        if world > 1:
            box = [mg.comm_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(box, src=0)
            kw.update(rank=rank, nranks=world, unique_id=box[0])
        return mg.Solver(n, nu, dt, dx, a.tol, **kw)

    for nu in [float(x) for x in a.nus.split(",")]:
        solvers = {r: make(nu, r) for r in (mg.RESTRICT_INJECT, mg.RESTRICT_FW)}
        rec = {r: dict(ms_step=[], cycles=[]) for r in solvers}
        for s in solvers.values():                               # warm-up: graph capture, tile plans, first launches
            s.set_fields_reference_ic(1.0)
            s.timestep(1)
        for _ in range(a.repeats):
            for r, s in solvers.items():
                s.set_fields_reference_ic(1.0)
                s.synchronize()
                if dist: dist.barrier()
                t0 = time.perf_counter()
                infos = s.timestep(a.steps)                      # ends in a device synchronise
                el = (time.perf_counter() - t0) * 1e3
                rec[r]["ms_step"].append(el / a.steps)
                rec[r]["cycles"].append(float(np.mean([i.cycles for i in infos])))
        sols = {r: s.get_u_host() for r, s in solvers.items()}
        down = {r: s.profile_level0(20)[0][0] for r, s in solvers.items()}
        for s in solvers.values():
            s.close()
        if rank == 0:
            if world > 1:
                rel = None                                        # each rank holds its own rows only
            else:
                rel = float(np.linalg.norm(sols[2] - sols[0]) / np.linalg.norm(sols[0]))
            arms = {}
            for r, name in ((0, "injection"), (2, "full_weighting")):
                ms = float(np.median(rec[r]["ms_step"])); cyc = float(np.median(rec[r]["cycles"]))
                arms[name] = dict(cycles_per_step=cyc, ms_per_step=ms, ms_per_cycle=ms / cyc,
                                  ms_per_step_all=rec[r]["ms_step"], down_leg_pass_ms=down[r])
            arms["rel_l2_fw_vs_injection"] = rel
            result["arms"][str(nu)] = arms
            print(json.dumps({str(nu): arms}), flush=True)
    if rank == 0:
        with open(a.out, "w") as f:
            json.dump(result, f, indent=1)
        print("card:", result["card"])
    if dist:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
