"""Worker of tests/test_gpu_levels.py: one process per GPU (torchrun).  Row-slab solves of a deep hierarchy
(maxlvl = log2(n) - 2, coarsest level 4) and a shallow one (coarsest level 64), with injection and with full
weighting, on seeded random fields whose boundary lines are nonzero and at diffusion number 8; checked on rank 0
against the single-GPU solve of the same build."""
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import hpcclassmultigridproject_b200 as mg  # noqa: E402


def fields(n, seed):
    rng = np.random.default_rng(seed)
    u0 = rng.uniform(0.25, 1.25, (n + 1, n + 1)) * rng.choice([-1.0, 1.0], (n + 1, n + 1))
    return u0, rng.uniform(-1.0, 1.0, (n + 1, n + 1)), rng.uniform(-1.0, 1.0, (n + 1, n + 1))


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n = 1024; dx = 1.0 / n; dt = dx / 10; tol = 1e-9
    nu = -8.0 * dx * dx / (2.0 * dt)
    u0, v1, v2 = fields(n, 2024)
    out = {}
    for maxlvl in (int(np.log2(n)) - 2, int(np.log2(n)) - 5):
        for restriction in (mg.RESTRICT_INJECT, mg.RESTRICT_FW):
            box = [mg.comm_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(box, src=0)
            with mg.Solver(n, nu, dt, dx, tol, maxlvl=maxlvl, arith=mg.ARITH_EXACT, device=local, rank=rank, nranks=world,
                           unique_id=box[0], restriction=restriction) as s:
                w = s.slab(0)
                s.set_fields_host_window(*(np.ascontiguousarray(a[w["mem_lo"]:w["mem_hi"] + 1]) for a in (u0, v1, v2)))
                infos = s.timestep(2)
                lo, hi, rows = s.get_u_host_rows()
                nshard = sum(1 for l in range(s.maxlvl) if s.slab(l)["sharded"])
            mine = np.zeros((n + 1, n + 1))
            mine[lo:hi + 1] = rows
            full = torch.from_numpy(mine).cuda()
            dist.reduce(full, dst=0, op=dist.ReduceOp.SUM)       # the owned row ranges partition 0..n
            if rank == 0:
                got = full.cpu().numpy()
                with mg.Solver(n, nu, dt, dx, tol, maxlvl=maxlvl, arith=mg.ARITH_EXACT, device=local,
                               restriction=restriction) as ref:
                    ref.set_fields_host(u0, v1, v2)
                    rinfos = ref.timestep(2)
                    want = ref.get_u_host()
                out[f"maxlvl{maxlvl}/restriction{restriction}"] = dict(
                    bitwise=bool(np.array_equal(got, want)), cycles=[i.cycles for i in infos],
                    ref_cycles=[i.cycles for i in rinfos], sharded_levels=nshard)
    if rank == 0:
        print("SHARDED_LEVELS_RESULT " + json.dumps(out), flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
