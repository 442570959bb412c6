"""torchrun worker of the two ``test_sharded_processes_agree`` tests (one rank per GPU), run as
``_multi_gpu_hf_worker.py ghf`` (tests/test_gpu_hartree_fock.py) or ``... uhf`` (tests/test_gpu_unrestricted_hf.py):
a sharded GHF or UHF ground state ends with the same coefficients and iteration count on every rank and matches the
one-GPU solver."""

import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from quantum_systems_b200 import GeneralOrbitalSystem, hartree_fock, sharded  # noqa: E402
from quantum_systems_b200.odqd import ODQD  # noqa: E402


def gather_equal(ctx, C):
    """True when every rank holds the same ``C``."""
    C = C.contiguous()
    gathered = [torch.empty_like(C) for _ in range(ctx.world)]
    dist.all_gather(gathered, C)
    return all(torch.equal(g, gathered[0]) for g in gathered)


def main(mode):
    rank = int(os.environ["RANK"])
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
    ctx = sharded.ProcessContext()
    try:
        od = ODQD(8, 8, 201, potential=ODQD.HOPotential(0.25), np=np)
        if mode == "ghf":
            basis = sharded.ShardedBasisSet.from_spatial(ctx, od.h, od.s, od.u, anti_symmetrize=True)
            state = hartree_fock.ground_state_sharded(basis, 4)
            coefficients = (state.C,)
        else:
            basis = sharded.ShardedBasisSet.from_global(ctx, od.h, od.s, od.u)
            state = hartree_fock.ground_state_unrestricted_sharded(basis, 2, 1)
            coefficients = (state.C_alpha, state.C_beta)
        assert state.converged
        for C in coefficients:
            assert gather_equal(ctx, C), "ranks hold different C"
        iterations = [None] * ctx.world
        dist.all_gather_object(iterations, state.iterations)
        assert len(set(iterations)) == 1, f"ranks took different iteration counts: {iterations}"
        # a different initial guess on every rank: rank 0's is used everywhere
        n = basis.h.shape[0]
        guess = torch.linalg.qr(torch.eye(n, dtype=torch.float64, device="cuda")
                                + 0.05 * rank * torch.ones((n, n), dtype=torch.float64, device="cuda"))[0]
        if mode == "ghf":
            seeded = hartree_fock.ground_state_sharded(basis, 4, C=guess)
            assert gather_equal(ctx, seeded.C), "ranks hold different C from different guesses"
            assert abs(seeded.energy - state.energy) <= 1e-10 * abs(state.energy)
            single = hartree_fock.ground_state(GeneralOrbitalSystem(4, ODQD(8, 8, 201,
                                                                           potential=ODQD.HOPotential(0.25))))
        else:
            seeded = hartree_fock.ground_state_unrestricted_sharded(basis, 2, 1, C=(guess, guess.clone()))
            assert gather_equal(ctx, seeded.C_alpha), "ranks hold different C from different guesses"
            single = hartree_fock.ground_state_unrestricted(ODQD(8, 8, 201, potential=ODQD.HOPotential(0.25)), 2, 1)
        assert abs(state.energy - single.energy) <= 1e-12 * abs(single.energy)
        torch.cuda.synchronize()
        if rank == 0:
            print({"ghf": "MULTI_GPU_HF_OK", "uhf": "MULTI_GPU_UHF_OK"}[mode], flush=True)
    finally:
        ctx.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    main(sys.argv[1])
