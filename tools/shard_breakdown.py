"""Per-step device times of the sharded four-index transform (torchrun, one rank per GPU)."""
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from quantum_systems_b200 import sharded  # noqa: E402


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 148
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
    ctx = sharded.ProcessContext()
    u = sharded.ShardedTwoBody.empty(ctx, n, torch.float64)
    u.local().normal_()
    C = torch.from_numpy(np.linalg.qr(np.random.default_rng(0).standard_normal((n, n)))[0]).cuda()
    w = sharded._RankTransform(ctx, rank, n, n, torch.float64, torch.float64)
    w.prepare(C, C)
    recv = ctx.shared_cached("recv", [w.recv_numel(r) for r in range(world)], torch.float64)
    out = u.spare
    names = ["step1", "step2_scatter", "barrier", "step3", "step4_scatter", "barrier2"]
    acc = {k: [] for k in names}
    for it in range(4):
        ctx.barrier()
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(names) + 1)]
        ev[0].record()
        w.step1(u.buffers[rank][rank]); ev[1].record()
        w.step2_scatter(recv[rank]); ev[2].record()
        ctx.barrier(); ev[3].record()
        w.step3(recv[rank][rank]); ev[4].record()
        w.step4_scatter(out[rank]); ev[5].record()
        ctx.barrier(); ev[6].record()
        torch.cuda.synchronize()
        if it:
            for i, k in enumerate(names):
                acc[k].append(ev[i].elapsed_time(ev[i + 1]))
    res = {k: round(min(v), 3) for k, v in acc.items()}
    res["total"] = round(sum(res.values()), 3)
    flops_step = 2.0 * n**5 / world
    res["tflops_per_gpu"] = {k: round(flops_step / res[k] * 1e-9, 2) for k in names if k.startswith("step")}
    shard_gb = 8 * n**4 / world / 1e9
    res["scatter_gbs_out"] = {k: round(shard_gb * (world - 1) / world / res[k] * 1e3, 1) for k in ("step2_scatter", "step4_scatter")}
    gathered = [None] * world
    dist.all_gather_object(gathered, res)
    if rank == 0:
        table = {k: [g[k] for g in gathered] for k in names + ["total"]}
        print(json.dumps({"n": n, "world": world, "per_rank_ms": table, "rank0": gathered[0], "rank_last": gathered[-1]}))
    ctx.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
