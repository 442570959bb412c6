"""torchrun worker of ``test_sharded_processes_agree`` in tests/test_gpu_uhf_gos_sharded.py (one rank per GPU): the
sharded spin-orbital system of a UHF state, in the peer and in the collective schedule, holds on every rank the
planes of the single-GPU ``hartree_fock.general_orbital_system``."""

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
    try:
        for l, n_alpha, n_beta in [(11, 3, 2), (20, 4, 0), (16, 5, 5)]:
            od = ODQD(l, 8.0, 401, potential=ODQD.HOPotential(0.25), np=np)
            for exchange in ("peer", "collective"):
                ctx = sharded.ProcessContext(exchange=exchange)
                basis = sharded.ShardedBasisSet.from_global(ctx, od.h, od.s, od.u)
                state = hartree_fock.ground_state_unrestricted_sharded(basis, n_alpha, n_beta)
                assert state.converged
                # the single-GPU system of this very state: the comparison does not depend on two SCF runs agreeing
                U = torch.as_tensor(hartree_fock.general_orbital_system(state, od).u).cuda()
                new = None
                for _ in range(2):  # the second call runs on the cached staging buffers and into the first result
                    new = hartree_fock.general_orbital_system_sharded(state, basis, into=new.u if new else None)
                    p0, p1 = new.u.planes(rank)
                    err = float((new.u.local() - U[p0:p1]).abs().max()) if p1 > p0 else 0.0
                    assert err <= 1e-13 * float(U.abs().max()), f"{exchange} l={l}: rank {rank} differs by {err}"
                    slab = new.u.local()
                    assert torch.equal(slab, -slab.transpose(2, 3))
                    e = new.compute_reference_energy(n_alpha + n_beta)
                    assert abs(e - state.energy) <= 1e-10 * abs(state.energy), (e, state.energy)
                torch.cuda.synchronize()
                ctx.close()
        dist.barrier()
        if rank == 0:
            print("MULTI_GPU_UHF_GOS_OK", flush=True)
    finally:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
