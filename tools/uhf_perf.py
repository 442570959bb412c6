"""Unrestricted Hartree-Fock measurements: the qs_fock_density_unrestricted kernel next to one single-density
qs_fock_density build and the three-build baseline J[rho_a + rho_b], K[rho_a], K[rho_b], and a full UHF next to
the numpy oracle.

    python tools/uhf_perf.py --out profiles/r05_uhf_b200.jsonl

One JSON line per record.  The first record holds the GPU name, its power limit, its maximum SM clock and the
streaming-copy bandwidth measured in the same run (ops.probe_copy_gbs, read + write bytes).  Kernel times are CUDA
events around >= 20 launches after warm-up; every u is larger than the 126 MB L2, so each build reads u from HBM.
"""

import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from hf_perf import emit, gpu_record  # noqa: E402
from quantum_systems_b200 import ODQD, hartree_fock, ops  # noqa: E402
from uhf_oracle import uhf_ground_state  # noqa: E402  (host baseline)


def time_calls(fn, launches):
    for _ in range(5):
        fn()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    for _ in range(launches):
        fn()
    stop.record()
    torch.cuda.synchronize()
    return start.elapsed_time(stop) / launches


def hermitian(n, dtype, gen):
    x = torch.randn((n, n), dtype=torch.float64, device="cuda", generator=gen)
    if dtype == torch.complex128:
        x = torch.complex(x, torch.randn((n, n), dtype=torch.float64, device="cuda", generator=gen))
    return (x + x.mH).contiguous()


def kernel_case(label, u, rho_dtype, copy_gbs, launches):
    n = u.shape[0]
    gen = torch.Generator(device="cuda").manual_seed(0)
    rho_a, rho_b, h = hermitian(n, rho_dtype, gen), hermitian(n, rho_dtype, gen), hermitian(n, torch.float64, gen)
    dt = ops._result_dtype(h, u, rho_a)
    fa, fb, f = (torch.empty((n, n), dtype=dt, device="cuda") for _ in range(3))
    zero = torch.zeros_like(h)
    rho_t = rho_a + rho_b

    def unrestricted():
        ops.fock_from_density_unrestricted(h, u, rho_a, rho_b, f_alpha=fa, f_beta=fb)

    def single():
        ops.fock_from_density(h, u, rho_a, 1.0, -1.0, f=f)

    def three():
        ops.fock_from_density(h, u, rho_t, 1.0, 0.0, f=f)
        ops.fock_from_density(zero, u, rho_a, 0.0, -1.0, f=fa)
        ops.fock_from_density(zero, u, rho_b, 0.0, -1.0, f=fb)

    ms = {name: time_calls(fn, launches) for name, fn in
          (("unrestricted", unrestricted), ("single_density", single), ("three_call_baseline", three))}
    u_bytes = u.numel() * u.element_size()
    reads = 1 if (not u.is_complex() and rho_dtype == torch.float64) else 2
    gbs = reads * u_bytes / ms["unrestricted"] / 1e6
    return {"record": "kernel", "case": label, "n": n, "u_dtype": str(u.dtype).replace("torch.", ""),
            "rho_dtype": str(rho_dtype).replace("torch.", ""), "launches": launches,
            "ms": {k: round(v, 4) for k, v in ms.items()},
            "unrestricted_over_single": round(ms["unrestricted"] / ms["single_density"], 3),
            "unrestricted_over_three_call": round(ms["unrestricted"] / ms["three_call_baseline"], 3),
            "u_reads_per_unrestricted_build": reads, "u_gbs": round(gbs, 1),
            "fraction_of_copy_bw": round(gbs / copy_gbs, 3)}


def scf_case(label, make, n_alpha, n_beta):
    """Wall time of a whole ground_state_unrestricted call (warmed up by one call on the same basis), with the
    Fock-kernel share from CUDA events around every build the solver makes, next to the numpy oracle."""
    basis = make()
    hartree_fock.ground_state_unrestricted(basis, n_alpha, n_beta)
    events = []
    plain = ops.fock_from_density_unrestricted

    def timed(*args, **kwargs):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = plain(*args, **kwargs)
        b.record()
        events.append((a, b))
        return out

    ops.fock_from_density_unrestricted = timed
    try:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        state = hartree_fock.ground_state_unrestricted(basis, n_alpha, n_beta)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
    finally:
        ops.fock_from_density_unrestricted = plain
    fock_ms = sum(a.elapsed_time(b) for a, b in events)
    it = state.iterations
    h, u = basis.h.cpu().numpy(), basis.u.cpu().numpy()
    s = basis.s.cpu().numpy() if basis.s is not None else None
    t0 = time.perf_counter()
    ref = uhf_ground_state(h, u, n_alpha, n_beta, s=s, e_nuc=basis.nuclear_repulsion_energy)
    host_s = time.perf_counter() - t0
    return {"record": "scf", "case": label, "l": basis.l, "n_alpha": n_alpha, "n_beta": n_beta,
            "converged": state.converged, "iterations": it, "energy": state.energy,
            "spin_squared": state.spin_squared, "oracle_energy": ref["energy"],
            "oracle_iterations": ref["iterations"], "oracle_converged": bool(ref["converged"]),
            "wall_s": round(wall, 5), "per_iteration_ms": round(1e3 * wall / it, 4),
            "fock_kernel_per_iteration_ms": round(fock_ms / it, 4), "oracle_host_s": round(host_s, 4),
            "host_cores": os.cpu_count()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--launches", type=int, default=30)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("uhf_perf.py measures on a CUDA device; none is visible")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as out:
        dev = gpu_record()
        emit(out, dev)
        bw = dev["copy_gbs"]
        gen = torch.Generator(device="cuda").manual_seed(1)
        u = torch.randn((128,) * 4, dtype=torch.float64, device="cuda", generator=gen)
        emit(out, kernel_case("n=128 real u, real densities", u, torch.float64, bw, args.launches))
        u = torch.complex(*(torch.randn((128,) * 4, dtype=torch.float64, device="cuda", generator=gen) for _ in "ri"))
        emit(out, kernel_case("n=128 complex128 u, complex densities", u, torch.complex128, bw, args.launches))
        del u
        torch.cuda.empty_cache()
        u = torch.randn((200,) * 4, dtype=torch.float64, device="cuda", generator=gen)
        emit(out, kernel_case("n=200 real u, real densities", u, torch.float64, bw, args.launches))
        del u
        torch.cuda.empty_cache()
        emit(out, scf_case("ODQD(100, 20, 2001, DW(1, 5)), UHF n_alpha = 11, n_beta = 10",
                           lambda: ODQD(100, 20, 2001, potential=ODQD.DWPotential(1.0, 5.0)), 11, 10))


if __name__ == "__main__":
    main()
