"""torchrun worker of tests/test_gpu_unrestricted_hf.py::test_sharded_processes_agree (one rank per GPU): a sharded UHF
ground state ends with the same coefficients and iteration count on every rank and matches the one-GPU solver."""

import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from quantum_systems_b200 import hartree_fock, sharded  # noqa: E402
from quantum_systems_b200.odqd import ODQD  # noqa: E402


def main():
    rank = int(os.environ["RANK"])
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
    ctx = sharded.ProcessContext()
    try:
        od = ODQD(8, 8, 201, potential=ODQD.HOPotential(0.25), np=np)
        basis = sharded.ShardedBasisSet.from_global(ctx, od.h, od.s, od.u)
        state = hartree_fock.ground_state_unrestricted_sharded(basis, 2, 1)
        assert state.converged
        for C in (state.C_alpha.contiguous(), state.C_beta.contiguous()):
            gathered = [torch.empty_like(C) for _ in range(ctx.world)]
            dist.all_gather(gathered, C)
            assert all(torch.equal(g, gathered[0]) for g in gathered), "ranks hold different C"
        iterations = [None] * ctx.world
        dist.all_gather_object(iterations, state.iterations)
        assert len(set(iterations)) == 1, f"ranks took different iteration counts: {iterations}"
        # a different initial guess on every rank: rank 0's is used everywhere
        n = basis.h.shape[0]
        guess = torch.linalg.qr(torch.eye(n, dtype=torch.float64, device="cuda")
                                + 0.05 * rank * torch.ones((n, n), dtype=torch.float64, device="cuda"))[0]
        seeded = hartree_fock.ground_state_unrestricted_sharded(basis, 2, 1, C=(guess, guess.clone()))
        Ca = seeded.C_alpha.contiguous()
        gathered = [torch.empty_like(Ca) for _ in range(ctx.world)]
        dist.all_gather(gathered, Ca)
        assert all(torch.equal(g, gathered[0]) for g in gathered), "ranks hold different C from different guesses"
        single = hartree_fock.ground_state_unrestricted(ODQD(8, 8, 201, potential=ODQD.HOPotential(0.25)), 2, 1)
        assert abs(state.energy - single.energy) <= 1e-12 * abs(single.energy)
        torch.cuda.synchronize()
        if rank == 0:
            print("MULTI_GPU_UHF_OK", flush=True)
    finally:
        ctx.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
