"""Linear-response TDHF measurements: the batched Coulomb-exchange kernel (ops.coulomb_exchange) at n = 128 and 200
for k = 1 ... 16 densities per launch beside k separate ops.fock_from_density builds, and hartree_fock.excited_states
for the l = 100 double well (RHF singlet RPA and UHF 11 alpha + 10 beta RPA, 10 roots) with the numpy oracle's dense
solve on the host cores beside it.

    python tools/lr_perf.py --out profiles/r10_lr_b200.jsonl

One JSON line per record.  The first record holds the GPU name, its power limit, its maximum SM clock, the
streaming-copy bandwidth (read + write bytes) and the FP64 DMMA probe measured in the same run.  Kernel times are CUDA
events around >= 20 launches after warm-up; every u is larger than the 126 MB L2.  The kernel's bound is the larger
of (bytes of u) / (copy probe) and 4 k n^4 / (DMMA probe).
"""

import argparse
import json
import os
import sys
import time


def time_calls(fn, launches):
    import torch

    for _ in range(3):
        fn()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    for _ in range(launches):
        fn()
    stop.record()
    torch.cuda.synchronize()
    return start.elapsed_time(stop) / launches


TARGETS_MS = {(128, 8): 0.55, (128, 16): 0.75}


def kernel_records(dev, launches):
    import torch

    from quantum_systems_b200 import ops

    gen = torch.Generator(device="cuda").manual_seed(7)
    out = []
    for n in (128, 200):
        u = torch.randn((n,) * 4, dtype=torch.float64, device="cuda", generator=gen)
        rho_all = torch.randn((16, n, n), dtype=torch.float64, device="cuda", generator=gen)
        h = torch.zeros((n, n), dtype=torch.float64, device="cuda")
        f = torch.empty((n, n), dtype=torch.float64, device="cuda")
        fock_ms = time_calls(lambda: ops.fock_from_density(h, u, rho_all[0], 1.0, -0.5, f=f), launches)
        u_bytes = u.numel() * 8
        for k in (1, 2, 4, 8, 16):
            rho = rho_all[:k].contiguous()
            J, K = torch.empty_like(rho), torch.empty_like(rho)
            ms = time_calls(lambda: ops.coulomb_exchange(u, rho, J=J, K=K), launches)
            hbm_ms = u_bytes / (dev["copy_gbs"] * 1e6)
            dmma_ms = 4 * k * n ** 4 / (dev["dmma_tflops"] * 1e9)
            bound = max(hbm_ms, dmma_ms)
            rec = {"record": "coulomb_exchange", "n": n, "k": k, "ms": round(ms, 4),
                   "bound_ms": round(bound, 4), "bound": "HBM" if hbm_ms >= dmma_ms else "DMMA",
                   "share_of_bound": round(bound / ms, 3), "k_fock_from_density_ms": round(k * fock_ms, 4),
                   "fock_from_density_ms": round(fock_ms, 4), "speedup_over_k_fock": round(k * fock_ms / ms, 2)}
            if (n, k) in TARGETS_MS:
                rec["target_ms"] = TARGETS_MS[(n, k)]
                rec["target_met"] = ms <= TARGETS_MS[(n, k)]
            out.append(rec)
        del u
        torch.cuda.empty_cache()
    return out


def solver_record(label, system, state, oracle_case):
    """Wall time of excited_states (RPA, 10 roots), its iterations and densities, the share of the kernel (timed in a
    second run with every ops.coulomb_exchange call bracketed by CUDA events) and the oracle's dense solve."""
    import numpy as np
    import torch

    import lr_oracle
    from quantum_systems_b200 import hartree_fock, ops

    def solve():
        return hartree_fock.excited_states(system, state, n_states=10, tol=1e-6)

    solve()  # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    try:
        res = solve()
    except ValueError as err:
        return {"record": "excited_states", "case": label, "refused": str(err)}
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0

    kernel_ms = [0.0]
    original = ops.coulomb_exchange

    def timed(*a, **kw):
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        r = original(*a, **kw)
        stop.record()
        torch.cuda.synchronize()
        kernel_ms[0] += start.elapsed_time(stop)
        return r

    ops.coulomb_exchange = timed
    try:
        solve()
    finally:
        ops.coulomb_exchange = original

    host = lambda a: a.cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)  # noqa: E731
    h, u = host(system.h).real, host(system.u).real
    t0 = time.perf_counter()
    kind, C, occ = oracle_case(host)
    omega = lr_oracle.spectrum(*lr_oracle.matrices(kind, h, u, C, occ))[0]
    oracle_s = time.perf_counter() - t0
    return {"record": "excited_states", "case": label, "wall_ms": round(wall * 1e3, 1), "iterations": res.iterations,
            "densities_built": res.densities_built, "converged": res.converged,
            "kernel_ms": round(kernel_ms[0], 2), "kernel_share": round(kernel_ms[0] / (wall * 1e3), 3),
            "oracle_s": round(oracle_s, 2), "host_cpus": os.cpu_count(),
            "max_abs_diff_to_oracle": float(np.abs(host(res.energies) - omega[:10]).max()),
            "energies": [round(float(x), 10) for x in host(res.energies)]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--launches", type=int, default=20)
    args = ap.parse_args()
    here = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for sub in ("tests", "tools", ""):
        sys.path.insert(0, os.path.join(here, sub))

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("lr_perf.py measures on a CUDA device; none is visible")
    from hf_perf import emit, gpu_record
    from quantum_systems_b200 import ODQD, SpatialOrbitalSystem, hartree_fock, ops

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as out:
        dev = gpu_record()
        dev["dmma_tflops"] = round(ops.probe_dmma_tflops(), 2)
        emit(out, dev)
        for rec in kernel_records(dev, args.launches):
            emit(out, rec)

        def dw():
            return ODQD(100, 20, 2001, potential=ODQD.DWPotential(1.0, 5.0))

        system = SpatialOrbitalSystem(20, dw())
        state = hartree_fock.ground_state(system)
        emit(out, solver_record("RHF singlet RPA, SpatialOrbitalSystem(20, ODQD(100, 20, 2001, DW(1, 5)))", system,
                                state, lambda host: ("rhf", host(state.C), 10)))
        system = SpatialOrbitalSystem(20, dw())
        ustate = hartree_fock.ground_state_unrestricted(system, 11, 10)
        emit(out, solver_record("UHF RPA, 11 alpha + 10 beta on ODQD(100, 20, 2001, DW(1, 5))", system, ustate,
                                lambda host: ("uhf", (host(ustate.C_alpha), host(ustate.C_beta)), (11, 10))))


if __name__ == "__main__":
    main()
