"""Worker of tests/test_gpu_full_weighting.py: one process per GPU (torchrun), sharded full-weighting solves checked
on rank 0 against the single-GPU full-weighting solve of the same build.  shard_min_rows = 32 shards every level
the slab arithmetic allows; 1024 leaves the N = 2048 problem one sharded level and an agglomerated child."""
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import hpcclassmultigridproject_b200 as mg  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    out = {}
    for n, shard_min in ((1024, 32), (2048, 1024 // world)):
        dx = 1.0 / n; dt = dx / 10; nu = -1e-3; tol = 1e-10
        box = [mg.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        with mg.Solver(n, nu, dt, dx, tol, arith=mg.ARITH_EXACT, device=local, rank=rank, nranks=world, unique_id=box[0],
                       shard_min_rows=shard_min, restriction=mg.RESTRICT_FW) as s:
            s.set_fields_reference_ic(2.0)
            infos = s.timestep(2)
            mine = s.get_u_host()
            nshard = sum(1 for l in range(s.maxlvl) if s.slab(l)["sharded"])
        rows = torch.from_numpy(np.nan_to_num(mine, nan=0.0)).cuda()
        dist.reduce(rows, dst=0, op=dist.ReduceOp.SUM)
        if rank == 0:
            got = rows.cpu().numpy()
            with mg.Solver(n, nu, dt, dx, tol, arith=mg.ARITH_EXACT, device=local, restriction=mg.RESTRICT_FW) as ref:
                ref.set_fields_reference_ic(2.0)
                rinfos = ref.timestep(2)
                want = ref.get_u_host()
            out[f"{n}/{shard_min}"] = dict(bitwise=bool(np.array_equal(got, want)), cycles=[i.cycles for i in infos],
                                           ref_cycles=[i.cycles for i in rinfos], sharded_levels=nshard)
    if rank == 0:
        print("SHARDED_FW_RESULT " + json.dumps(out), flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
