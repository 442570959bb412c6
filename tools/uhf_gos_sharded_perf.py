"""The sharded UHF spin-orbital system (hartree_fock.general_orbital_system_sharded) next to the spin-doubling route
(ShardedBasisSet.from_spatial_planes + change_basis(spin_orbital_coefficients(state)[0])), one rank per GPU:

    torchrun --nproc-per-node=8 tools/uhf_gos_sharded_perf.py --l 200 --out profiles/r08_uhf_gos_sharded_b200.jsonl
    python tools/uhf_gos_sharded_perf.py --l 100 --out ...     (one process: a world of one GPU)

The spatial planes come from odqd_spatial_planes (ODQD(l, 20, 2001, DW(1, 5)), every rank builds its own planes);
the state is an open-shell UHF ground state from ground_state_unrestricted_sharded.  One JSON line per record, written
by rank 0.  The device record holds every rank's GPU name, power limit and SM clocks (read-only nvidia-smi query)
and the per-GPU streaming-copy and FP64 tensor-pipe probes (ops.probe_copy_gbs, ops.probe_dmma_tflops) of this run.
The two routes alternate, after one warm-up call of each.  Per call and rank, CUDA events split the new route into
the four block transforms (images, quarter steps, exchanges and barriers up to the first assembly launch) and the
assembly; the block share is 4 x 8 l^5 real flops (x 4 for complex blocks) over the slowest rank's block time and W
times the DMMA probe.  Call times are host clocks around calls that end in a device synchronise on every rank.
Peak memory: torch's peak above the start of the call, and the device memory in use after it (cudaMemGetInfo,
which also counts the IPC buffers torch does not see).  Parity: the first and last local plane of both results.

Both routes write their (2l)^4 result into ONE sharded tensor allocated up front (``into=``; the spin-doubling route
builds its input there and transforms into its spare set), so repeated calls allocate no peer memory: at l = 200 on 8
GPUs one result set with its spare is 51.2 GB per rank in float64 (``--out-dtype``, the default here) and 102.4 GB in
complex128, next to the recv and scratch buffers of the spin-doubled transform.
"""

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from quantum_systems_b200 import hartree_fock, ops, sharded  # noqa: E402
from quantum_systems_b200.odqd import grid_orbitals  # noqa: E402
from quantum_systems_b200.potentials import DWPotential  # noqa: E402


class TimedEngine(sharded.CudaEngine):
    """Records a CUDA event before and after every assembly launch."""

    events = []

    def spin_orbital_planes(self, *args):
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        super().spin_orbital_planes(*args)
        stop.record()
        self.events.append((start, stop))


def device_record():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()),
                        "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock, max_clock = (x.strip() for x in q.stdout.splitlines()[0].split(","))
    return {"gpu": name, "power_limit": power, "sm_clock": clock, "max_sm_clock": max_clock,
            "copy_gbs": round(ops.probe_copy_gbs(), 1), "dmma_tflops": round(ops.probe_dmma_tflops(), 2)}


def used_bytes():
    free, total = torch.cuda.mem_get_info()
    return total - free


def call(fn, ctx):
    torch.cuda.synchronize()
    ctx.barrier()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    ctx.barrier()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0, torch.cuda.max_memory_allocated() - base


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--l", type=int, default=200)
    ap.add_argument("--n-alpha", type=int, default=11)
    ap.add_argument("--n-beta", type=int, default=10)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out-dtype", choices=("float64", "complex128"), default="float64")
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("uhf_gos_sharded_perf.py measures on CUDA devices; none is visible")
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if not dist.is_initialized():
        if "RANK" not in os.environ:  # one process without torchrun: a world of one
            os.environ.update(RANK="0", WORLD_SIZE="1", MASTER_ADDR="127.0.0.1", MASTER_PORT="29561")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    engine = TimedEngine()
    ctx = sharded.ProcessContext(engine=engine)
    rank, world, l = ctx.rank, ctx.world, args.l
    out_dtype = getattr(torch, args.out_dtype)
    records = []
    try:
        devices = [None] * world
        dist.all_gather_object(devices, device_record())
        records.append({"record": "device", "world": world, "ranks": devices})

        grid, eps, Cg = grid_orbitals(l, 20.0, 2001, DWPotential(1.0, 5.0))
        planes = sharded.odqd_spatial_planes(Cg, grid[1:-1])
        h, s = np.diag(eps), np.eye(l)
        basis = sharded.ShardedBasisSet.from_slabs(ctx, l, h, s, planes)
        t0 = time.perf_counter()
        state = hartree_fock.ground_state_unrestricted_sharded(basis, args.n_alpha, args.n_beta)
        uhf_s = time.perf_counter() - t0
        C, _ = hartree_fock.spin_orbital_coefficients(state)
        target = sharded.ShardedTwoBody.empty(ctx, 2 * l, out_dtype)  # both routes' result, with its spare set

        def new_route():
            engine.events.clear()
            start = torch.cuda.Event(enable_timing=True)
            start.record()
            out = hartree_fock.general_orbital_system_sharded(state, basis, out_dtype=out_dtype, into=target)
            return out, start

        def spin_doubling_route():
            doubled = sharded.ShardedBasisSet.from_spatial_planes(ctx, h, s, l, planes, out_dtype=out_dtype,
                                                                  into=target)
            doubled.change_basis(C)  # into the spare set of target
            return doubled

        times = {"new": [], "spin_doubling": []}
        blocks_ms, assembly_ms, peaks, used = [], [], {}, {}
        parity = None
        for it in range(args.reps + 1):  # the first round is the warm-up
            (out, start), seconds, peak = call(new_route, ctx)
            first_stop = engine.events[0][0]
            b_ms = start.elapsed_time(first_stop)
            a_ms = sum(a.elapsed_time(b) for a, b in engine.events)
            used_new = used_bytes()
            sample = None
            p0, p1 = out.u.planes(rank)
            if it == 0 and p1 > p0:
                sample = out.u.local()[[0, p1 - p0 - 1]].clone()
            del out
            ref, seconds_ref, peak_ref = call(spin_doubling_route, ctx)
            used_ref = used_bytes()
            if it == 0:
                if sample is not None:
                    want = ref.u.local()[[0, p1 - p0 - 1]]
                    parity = float((sample - want).abs().max() / want.abs().max())
                peaks = {"new": peak, "spin_doubling": peak_ref}
                used = {"new": used_new, "spin_doubling": used_ref}
            else:
                times["new"].append(seconds)
                times["spin_doubling"].append(seconds_ref)
                blocks_ms.append(b_ms)
                assembly_ms.append(a_ms)
            del ref, sample
            torch.cuda.empty_cache()
        p0, p1 = sharded.block_partition(2 * l, world)[1][rank : rank + 2]
        mine = {"rank": rank, "planes": [p0, p1], "blocks_ms": [round(x, 3) for x in blocks_ms],
                "assembly_ms": [round(x, 3) for x in assembly_ms], "seconds": {k: [round(t, 4) for t in v]
                                                                                for k, v in times.items()},
                "torch_peak_bytes": peaks, "device_used_bytes_after_call": used, "parity_planes_max_rel": parity}
        ranks = [None] * world
        dist.all_gather_object(ranks, mine)
        if rank == 0:
            complex_blocks = basis.u.dtype == torch.complex128 or state.C_alpha.is_complex()
            flops = 4 * 8.0 * l**5 * (4 if complex_blocks else 1)
            dmma = sum(d["dmma_tflops"] for d in devices)
            blocks = np.median([max(r["blocks_ms"][i] for r in ranks) for i in range(args.reps)])
            assembly = np.median([max(r["assembly_ms"][i] for r in ranks) for i in range(args.reps)])
            block_size = 16 if complex_blocks else 8
            out_size = 16 if out_dtype == torch.complex128 else 8
            nbytes = 4 * l**4 * block_size + 16 * l**4 * out_size  # the blocks read once, every output element written
            copy = sum(d["copy_gbs"] for d in devices)
            med = {k: float(np.median([np.median(r["seconds"][k]) for r in ranks])) for k in times}
            records.append({"record": "uhf", "l": l, "n_alpha": args.n_alpha, "n_beta": args.n_beta,
                            "converged": state.converged, "iterations": state.iterations, "seconds": round(uhf_s, 3)})
            records.append({
                "record": "summary", "l": l, "world": world, "reps": args.reps, "out_dtype": args.out_dtype,
                "block_transforms_ms": round(float(blocks), 3),
                "block_transforms_tflops": round(flops / blocks / 1e9, 1),
                "block_transforms_fraction_of_aggregate_dmma_probe": round(flops / blocks / 1e9 / dmma, 3),
                "assembly_ms": round(float(assembly), 3),
                "assembly_gbs": round(nbytes / assembly / 1e6, 1),
                "assembly_fraction_of_aggregate_copy_probe": round(nbytes / assembly / 1e6 / copy, 3),
                "call_median_s": {k: round(v, 4) for k, v in med.items()},
                "new_over_spin_doubling": round(med["new"] / med["spin_doubling"], 3),
            })
            records.extend({"record": "rank", **r} for r in ranks)
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                for rec in records:
                    f.write(json.dumps(rec) + "\n")
                    print(json.dumps(rec), flush=True)
    finally:
        torch.cuda.synchronize()
        ctx.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
