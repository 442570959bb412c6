"""The UHF spin-orbital system from spin blocks (hartree_fock.general_orbital_system) on one GPU: the assembly kernel
next to the streaming-copy probe, the four-coefficient transform next to the plain one, and the whole call next to
the spin-doubling route GeneralOrbitalSystem(n, basis.copy_basis()).change_basis(C).

    python tools/uhf_gos_perf.py --out profiles/r06_uhf_gos_b200.jsonl

One JSON line per record.  The first record holds the GPU name, power limit, current and maximum SM clock (read-only
nvidia-smi query), the streaming-copy bandwidth (ops.probe_copy_gbs, read + write bytes) and the FP64 tensor-pipe
peak (ops.probe_dmma_tflops) measured in the same run.  Kernel times are CUDA events around >= 10 launches after
warm-up; every tensor involved is larger than the 126 MB L2.  End-to-end times are host clocks around calls that end
in a device synchronise, after one warm-up call of each route; peak memory is torch.cuda.max_memory_allocated above
what was allocated before the call.
"""

import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from hf_perf import emit  # noqa: E402
from quantum_systems_b200 import ODQD, GeneralOrbitalSystem, _native, hartree_fock, ops  # noqa: E402


def device_record():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock, max_clock = (x.strip() for x in q.stdout.splitlines()[0].split(","))
    return {"record": "device", "gpu": name, "power_limit": power, "sm_clock": clock, "max_sm_clock": max_clock,
            "copy_gbs": round(ops.probe_copy_gbs(), 1), "dmma_tflops": round(ops.probe_dmma_tflops(), 2)}


def event_ms(fn, launches):
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


def assembly_case(l, copy_gbs, launches):
    """qs_spin_orbital_two_body on float64 blocks into the complex128 result (the default cast), UHF order of
    11 alpha + 10 beta electrons, b_ba derived and given."""
    gen = torch.Generator(device="cuda").manual_seed(l)
    blocks = [torch.randn((l,) * 4, dtype=torch.float64, device="cuda", generator=gen) for _ in range(4)]
    orbital, spin = (torch.from_numpy(t.astype(np.int32)).cuda() for t in hartree_fock.spin_orbital_order(11, 10, l))
    out = torch.empty((2 * l,) * 4, dtype=torch.complex128, device="cuda")
    stream = ops._stream()
    recs = []
    for derived in (True, False):
        ba = None if derived else blocks[2]

        def launch():
            _native.call("qs_spin_orbital_two_body", *(ops._ptr(b) for b in (blocks[0], blocks[1], ba, blocks[3])),
                         ops.QS_F64, l, ops._ptr(orbital), ops._ptr(spin), ops._ptr(out), ops.QS_C128, 0, 2 * l,
                         stream)

        ms = event_ms(launch, launches)
        nbytes = 4 * l**4 * 8 + 16 * l**4 * 16
        gbs = nbytes / ms / 1e6
        recs.append({"record": "assembly", "l": l, "in": "float64", "out": "complex128", "b_ba": "derived" if derived
                     else "given", "launches": launches, "ms": round(ms, 4), "algorithmic_bytes": nbytes,
                     "gbs": round(gbs, 1), "fraction_of_copy_probe": round(gbs / copy_gbs, 3)})
    return recs


def transform_case(n, dmma_tflops, launches):
    """The four-coefficient transform (two real matrices) next to the plain four full steps at the same n."""
    gen = torch.Generator(device="cuda").manual_seed(n)
    u = torch.randn((n,) * 4, dtype=torch.float64, device="cuda", generator=gen)
    Ca, Cb = (torch.randn((n, n), dtype=torch.float64, device="cuda", generator=gen) for _ in range(2))
    plain = event_ms(lambda: ops.transform_two_body(u, Ca, symmetry=0), launches)
    mixed = event_ms(lambda: ops.transform_two_body_mixed(u, Ca, Cb), launches)
    flops = 8.0 * n**5
    share = {k: flops / ms / 1e9 / dmma_tflops for k, ms in (("plain", plain), ("mixed", mixed))}
    return {"record": "transform", "n": n, "dtype": "float64", "launches": launches,
            "ms": {"plain": round(plain, 4), "mixed": round(mixed, 4)},
            "fraction_of_dmma_probe": {k: round(v, 4) for k, v in share.items()},
            "mixed_over_plain": round(mixed / plain, 4)}


def timed(fn):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0, torch.cuda.max_memory_allocated() - base


def end_to_end_case(label, basis, n_alpha, n_beta, slow, reps):
    state = hartree_fock.ground_state_unrestricted(basis, n_alpha, n_beta)
    n = n_alpha + n_beta

    def new_route():
        return hartree_fock.general_orbital_system(state, basis)

    def slow_route():
        C, _ = hartree_fock.spin_orbital_coefficients(state)
        system = GeneralOrbitalSystem(n, basis.copy_basis())
        system.change_basis(C)
        return system

    rec = {"record": "end_to_end", "case": label, "l": basis.l, "n_alpha": n_alpha, "n_beta": n_beta,
           "uhf_converged": state.converged, "cast_to_complex": basis.cast_to_complex_on_spin_doubling}
    routes = [("new", new_route)] + ([("slow", slow_route)] if slow else [])
    times = {name: [] for name, _ in routes}
    peaks = {}
    results = {}
    for name, fn in routes:  # warm-up, with the peak memory of one call
        out, _, peaks[name] = timed(fn)
        results[name] = out.u[:2].clone()  # two leading planes: the whole results would not fit next to each other
        if name == "new":
            rec["u_dtype"] = str(out.u.dtype).replace("torch.", "")
        del out
    if slow:
        a, b = results["new"], results["slow"]
        rec["planes_0_1_max_abs_diff_over_max"] = float((a - b).abs().max() / b.abs().max())
    results.clear()
    torch.cuda.empty_cache()
    for _ in range(reps):  # alternating
        for name, fn in routes:
            out, seconds, _ = timed(fn)
            times[name].append(seconds)
            del out
            torch.cuda.empty_cache()
    rec["seconds"] = {k: [round(t, 5) for t in v] for k, v in times.items()}
    rec["median_s"] = {k: round(float(np.median(v)), 5) for k, v in times.items()}
    rec["peak_bytes"] = peaks
    if slow:
        rec["speedup"] = round(rec["median_s"]["slow"] / rec["median_s"]["new"], 2)
    l = basis.l
    s_out = 16 if rec["u_dtype"] == "complex128" else 8
    rec["spin_doubling_route_computed_bytes"] = 4 * (2 * l) ** 4 * s_out  # input, output, two workspace buffers
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--launches", type=int, default=10)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("uhf_gos_perf.py measures on a CUDA device; none is visible")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as out:
        dev = device_record()
        emit(out, dev)
        for l in (100, 128):
            for rec in assembly_case(l, dev["copy_gbs"], args.launches):
                emit(out, rec)
            torch.cuda.empty_cache()
        for n in (100, 128):
            emit(out, transform_case(n, dev["dmma_tflops"], args.launches))
            torch.cuda.empty_cache()
        dw = ODQD.DWPotential(1.0, 5.0)
        emit(out, end_to_end_case("ODQD(100, 20, 2001, DW(1, 5)), complex default", ODQD(100, 20, 2001, potential=dw),
                                  11, 10, True, args.reps))
        basis = ODQD(128, 20, 2001, potential=dw)
        basis.cast_to_complex_on_spin_doubling = False
        emit(out, end_to_end_case("ODQD(128, 20, 2001, DW(1, 5)), cast_to_complex_on_spin_doubling=False", basis,
                                  11, 10, True, args.reps))
        del basis
        torch.cuda.empty_cache()
        emit(out, end_to_end_case("ODQD(128, 20, 2001, DW(1, 5)), complex default, new route only",
                                  ODQD(128, 20, 2001, potential=dw), 11, 10, False, args.reps))


if __name__ == "__main__":
    main()
