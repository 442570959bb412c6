"""Hartree-Fock measurements: the qs_fock_density kernel alone and full SCF runs, next to the numpy oracle.

    python tools/hf_perf.py --out profiles/r04_hf_b200.jsonl

One JSON line per record.  The first record holds the GPU name, its power limit and the streaming-copy bandwidth
measured in the same run (ops.probe_copy_gbs, read + write bytes); the kernel's bandwidth is quoted as a fraction of
that.  Kernel times are CUDA events around >= 20 launches after warm-up; every u is larger than the 126 MB L2.
"""

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import hf_oracle  # noqa: E402  (host baseline)
from quantum_systems_b200 import ODQD, GeneralOrbitalSystem, SpatialOrbitalSystem, hartree_fock, ops  # noqa: E402


def emit(out, rec):
    line = json.dumps(rec)
    print(line, flush=True)
    out.write(line + "\n")
    out.flush()


def gpu_record():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = (x.strip() for x in q.stdout.splitlines()[0].split(","))
    return {"record": "device", "gpu": name, "power_limit": power, "max_sm_clock": clock,
            "copy_gbs": round(ops.probe_copy_gbs(), 1)}


def time_kernel(h, u, rho, scales, launches):
    f = torch.empty((h.shape[0],) * 2, dtype=ops._result_dtype(h, u, rho), device="cuda")
    for _ in range(5):
        ops.fock_from_density(h, u, rho, *scales, f=f)
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    for _ in range(launches):
        ops.fock_from_density(h, u, rho, *scales, f=f)
    stop.record()
    torch.cuda.synchronize()
    return start.elapsed_time(stop) / launches


def kernel_case(label, u, scales, copy_gbs, launches):
    n = u.shape[0]
    gen = torch.Generator(device="cuda").manual_seed(0)
    rho = torch.randn((n, n), dtype=torch.float64, device="cuda", generator=gen)
    rho = rho + rho.T
    h = torch.randn((n, n), dtype=torch.float64, device="cuda", generator=gen)
    ms = time_kernel(h, u, rho, scales, launches)
    out_bytes = n * n * (16 if u.is_complex() else 8)
    algorithmic = u.numel() * u.element_size() + rho.numel() * 8 + h.numel() * 8 + out_bytes
    gbs = algorithmic / ms / 1e6
    return {"record": "kernel", "case": label, "n": n, "u_dtype": str(u.dtype).replace("torch.", ""),
            "scales": list(scales), "launches": launches, "ms": round(ms, 4), "algorithmic_bytes": algorithmic,
            "gbs": round(gbs, 1), "fraction_of_copy_bw": round(gbs / copy_gbs, 3)}


def scf_case(label, make, restricted, anti):
    """Wall time of a whole ground_state call (warmed up by one call on the same system), with the Fock-kernel
    share from CUDA events around every ops.fock_from_density the solver makes."""
    system = make()
    hartree_fock.ground_state(system)
    events = []
    plain = ops.fock_from_density

    def timed(*args, **kwargs):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = plain(*args, **kwargs)
        b.record()
        events.append((a, b))
        return out

    ops.fock_from_density = timed
    try:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        state = hartree_fock.ground_state(system)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
    finally:
        ops.fock_from_density = plain
    fock_ms = sum(a.elapsed_time(b) for a, b in events)
    it = state.iterations
    h, u = system.h.cpu().numpy(), system.u.cpu().numpy()
    s = system.s.cpu().numpy() if system.s is not None else None
    t0 = time.perf_counter()
    ref = hf_oracle.ground_state(h, u, system.n, restricted, anti, s=s, e_nuc=system.nuclear_repulsion_energy)
    host_s = time.perf_counter() - t0
    return {"record": "scf", "case": label, "l": system.l, "n_occ": system.n, "converged": state.converged,
            "iterations": it, "energy": state.energy, "oracle_energy": ref["energy"],
            "oracle_iterations": ref["iterations"], "wall_s": round(wall, 5),
            "per_iteration_ms": round(1e3 * wall / it, 4), "fock_kernel_per_iteration_ms": round(fock_ms / it, 4),
            "other_per_iteration_ms": round((1e3 * wall - fock_ms) / it, 4), "oracle_host_s": round(host_s, 4),
            "host_cores": os.cpu_count()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--launches", type=int, default=30)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("hf_perf.py measures on a CUDA device; none is visible")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as out:
        dev = gpu_record()
        emit(out, dev)
        bw = dev["copy_gbs"]
        gen = torch.Generator(device="cuda").manual_seed(1)
        u = torch.randn((128,) * 4, dtype=torch.float64, device="cuda", generator=gen)
        emit(out, kernel_case("n=128 real, random u", u, (1.0, -0.5), bw, args.launches))
        del u
        gos = GeneralOrbitalSystem(64, ODQD(64, 10, 401, potential=ODQD.HOPotential(0.25)))
        emit(out, kernel_case("n=128 complex128, GOS of ODQD(64, 10, 401)", gos.u, (1.0, 0.0), bw, args.launches))
        del gos
        u = torch.complex(*(torch.randn((256,) * 4, dtype=torch.float64, device="cuda", generator=gen) for _ in "ri"))
        emit(out, kernel_case("n=256 complex128, random u", u, (1.0, 0.0), bw, args.launches))
        del u
        torch.cuda.empty_cache()
        emit(out, scf_case(
            "configs[2]: SpatialOrbitalSystem(20, ODQD(100, 20, 2001, DW(1, 5))), RHF",
            lambda: SpatialOrbitalSystem(20, ODQD(100, 20, 2001, potential=ODQD.DWPotential(1.0, 5.0))), True, False,
        ))
        emit(out, scf_case(
            "configs[0]: GeneralOrbitalSystem(2, ODQD(20, 10, 201, HO 0.25)), GHF",
            lambda: GeneralOrbitalSystem(2, ODQD(20, 10, 201, potential=ODQD.HOPotential(0.25))), False, True,
        ))
        emit(out, {"record": "scf_sharded", "case": "configs[4] basis, 8 GPUs, GHF l = 200, n_occ = 20",
                   "per_iteration_ms": "not measured"})


if __name__ == "__main__":
    main()
