"""Time-dependent Hartree-Fock measurements: the RK4 step of hartree_fock.propagate for RHF, UHF and GHF with the
share of its Fock kernels and the numpy oracle's step beside it, and the one-read unrestricted Fock pass for complex
densities on a real u against the two-read route it replaced.

    python tools/tdhf_perf.py --out profiles/r09_tdhf_b200.jsonl [--compare-with OTHER_TREE]

One JSON line per record.  The first record holds the GPU name, its power limit, its maximum SM clock and the
streaming-copy bandwidth measured in the same run (ops.probe_copy_gbs, read + write bytes).  ``--compare-with``
times the unrestricted Fock pass of this tree and of another checkout's package (e.g. the parent commit, built) in
alternating subprocesses, three rounds each.  Kernel times are CUDA events around >= 20 launches after warm-up;
every u of the kernel records is larger than the 126 MB L2.
"""

import argparse
import json
import os
import subprocess
import sys
import time


def fock_records(launches):
    """The unrestricted Fock pass, real u and complex densities, at l = 128 and 200 (the package on sys.path)."""
    import torch

    from quantum_systems_b200 import ops

    gen = torch.Generator(device="cuda").manual_seed(1)
    out = []
    for n in (128, 200):
        u = torch.randn((n,) * 4, dtype=torch.float64, device="cuda", generator=gen)
        rho = []
        for _ in range(2):
            x = torch.randn((n, n), dtype=torch.complex128, device="cuda", generator=gen)
            rho.append((x + x.mH).contiguous())
        h = torch.randn((n, n), dtype=torch.float64, device="cuda", generator=gen)
        fa, fb = (torch.empty((n, n), dtype=torch.complex128, device="cuda") for _ in range(2))

        def build():
            ops.fock_from_density_unrestricted(h, u, *rho, f_alpha=fa, f_beta=fb)

        ms = time_calls(build, launches)
        u_bytes = u.numel() * 8
        out.append({"record": "fock_unrestricted_complex", "n": n, "ms": round(ms, 4),
                    "u_gb": round(u_bytes / 1e9, 3), "u_bytes_per_build_over_time_gbs": round(u_bytes / ms / 1e6, 1)})
        del u
        torch.cuda.empty_cache()
    return out


def time_calls(fn, launches):
    import torch

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


def pulse(t):
    import math

    return 0.05 * math.sin(0.5 * t)


def step_record(label, system, state, kind, steps, dt):
    """Per-step time of ``propagate`` (host clock around a synchronised call, after a warm-up call), the Fock
    kernels' share (CUDA events around every build of a second call) and the numpy oracle's step."""
    import numpy as np
    import torch

    import tdhf_oracle
    from oracle import hf_oracle
    from quantum_systems_b200 import hartree_fock, ops
    from quantum_systems_b200.time_evolution_operators import DipoleFieldInteraction

    system.set_time_evolution_operator(DipoleFieldInteraction(pulse))
    hartree_fock.propagate(system, state, 2 * dt, dt)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    run = hartree_fock.propagate(system, state, steps * dt, dt)
    torch.cuda.synchronize()
    step_ms = 1e3 * (time.perf_counter() - t0) / steps

    events = []
    names = ("fock_from_density", "fock_from_density_unrestricted")
    plain = {name: getattr(ops, name) for name in names}

    def timed(fn):
        def call(*args, **kwargs):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            result = fn(*args, **kwargs)
            b.record()
            events.append((a, b))
            return result

        return call

    for name in names:
        setattr(ops, name, timed(plain[name]))
    try:
        hartree_fock.propagate(system, state, steps * dt, dt)
        torch.cuda.synchronize()
    finally:
        for name in names:
            setattr(ops, name, plain[name])
    fock_ms = sum(a.elapsed_time(b) for a, b in events) / steps

    h0 = system.h.cpu().numpy()
    u = system.u.cpu().numpy()
    d = system.dipole_moment.cpu().numpy()
    if kind == "uhf":
        C_occ, scales = (state.C_alpha[:, :state.n_alpha].cpu().numpy(),
                         state.C_beta[:, :state.n_beta].cpu().numpy()), None
    else:
        C_occ = (state.C[:, :system.n].cpu().numpy(),)
        scales = hf_oracle.scales(kind == "rhf", system._basis_set.anti_symmetrized_u)
    s = system.s.cpu().numpy() if system.s is not None else None
    oracle_steps = 2
    t0 = time.perf_counter()
    tdhf_oracle.propagate(kind, tdhf_oracle.dipole_field(h0, d, pulse), lambda t: u, C_occ, 0.0, oracle_steps, dt,
                          s=s, dipole=d, scales=scales)
    oracle_ms = 1e3 * (time.perf_counter() - t0) / oracle_steps
    return {"record": "tdhf_step", "case": label, "l": system.l, "steps": steps, "dt": dt,
            "step_ms": round(step_ms, 4), "fock_kernels_ms_per_step": round(fock_ms, 4),
            "fock_share": round(fock_ms / step_ms, 3), "oracle_step_ms": round(oracle_ms, 2),
            "oracle_over_gpu": round(oracle_ms / step_ms, 1), "host_cores": os.cpu_count(),
            "energy_drift": float(np.ptp(run.energy.cpu().numpy()))}


def compare(other, launches, out, emit):
    """The Fock records of this tree and of ``other`` in alternating subprocesses."""
    here = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for round_ in range(3):
        for tree in (other, here):
            proc = subprocess.run([sys.executable, os.path.abspath(__file__), "--fock-only", "--package-root", tree,
                                   "--launches", str(launches)], capture_output=True, text=True, check=True)
            for line in proc.stdout.splitlines():
                rec = json.loads(line)
                rec.update(round=round_, tree="other" if tree == other else "this")
                emit(out, rec)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--launches", type=int, default=30)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--compare-with", help="root of another checkout whose built package is timed alternately")
    ap.add_argument("--fock-only", action="store_true", help="print the Fock records of --package-root and exit")
    ap.add_argument("--package-root")
    args = ap.parse_args()
    here = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, os.path.join(here, "tests"))
    sys.path.insert(0, os.path.join(here, "tools"))
    sys.path.insert(0, here)
    if args.package_root:
        sys.path.insert(0, os.path.abspath(args.package_root))

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("tdhf_perf.py measures on a CUDA device; none is visible")
    if args.fock_only:
        for rec in fock_records(args.launches):
            print(json.dumps(rec), flush=True)
        return

    from hf_perf import emit, gpu_record
    from quantum_systems_b200 import ODQD, GeneralOrbitalSystem, SpatialOrbitalSystem, hartree_fock

    if not args.out:
        raise SystemExit("--out is required")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as out:
        dev = gpu_record()
        emit(out, dev)
        if args.compare_with:
            compare(args.compare_with, args.launches, out, emit)

        def dw():
            return ODQD(100, 20, 2001, potential=ODQD.DWPotential(1.0, 5.0))

        system = SpatialOrbitalSystem(20, dw())
        emit(out, step_record("RHF SpatialOrbitalSystem(20, ODQD(100, 20, 2001, DW(1, 5)))", system,
                              hartree_fock.ground_state(system), "rhf", args.steps, 1e-2))
        system = SpatialOrbitalSystem(20, dw())
        emit(out, step_record("UHF 11 alpha + 10 beta on ODQD(100, 20, 2001, DW(1, 5))", system,
                              hartree_fock.ground_state_unrestricted(system, 11, 10), "uhf", args.steps, 1e-2))
        system = GeneralOrbitalSystem(2, ODQD(20, 10, 201, potential=ODQD.HOPotential(0.25)))
        emit(out, step_record("GHF GeneralOrbitalSystem(2, ODQD(20, 10, 201, HO 0.25))", system,
                              hartree_fock.ground_state(system), "ghf", args.steps, 1e-2))


if __name__ == "__main__":
    main()
