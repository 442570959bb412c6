"""Quick device-side timings of the hot-path operators (development aid, not the bench contract)."""
import sys, os, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from quantum_systems_b200 import ops


def timed(fn, reps=5, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    best = 1e30
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); e1.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return best


def main():
    peak = ops.probe_dmma_tflops()
    print(json.dumps({"dmma_peak_tflops": peak}))
    for n, cplx in [(40, True), (64, False), (96, False), (128, False), (128, True), (160, False), (100, False)]:
        dt = torch.complex128 if cplx else torch.float64
        u = torch.randn((n,) * 4, dtype=dt, device="cuda")
        C = torch.linalg.qr(torch.randn((n, n), dtype=dt, device="cuda"))[0].contiguous()
        ms = timed(lambda: ops.transform_two_body(u, C))
        flops = 8.0 * n**5 * (4 if cplx else 1)
        print(json.dumps({"op": "transform_two_body", "n": n, "complex": cplx, "ms": round(ms, 3),
                          "tflops": round(flops / ms * 1e-9, 2), "frac_of_dmma_peak": round(flops / ms * 1e-9 / peak, 3)}))
        del u
    # symmetry-aware path: exactly antisymmetric / particle-exchange-symmetric input vs the plain four full steps
    for n, cplx in ((128, False), (128, True), (160, False)):
        dt = torch.complex128 if cplx else torch.float64
        base = torch.randn((n,) * 4, dtype=dt, device="cuda")
        C = torch.linalg.qr(torch.randn((n, n), dtype=torch.float64, device="cuda"))[0].contiguous()
        for kind in ("exchange", "antisym"):
            u = (0.5 * (base + base.permute(1, 0, 3, 2))).contiguous() if kind == "exchange" else (base - base.permute(0, 1, 3, 2)).contiguous()
            full = timed(lambda: ops.transform_two_body(u, C, symmetry=0))
            auto = timed(lambda: ops.transform_two_body(u, C))
            detect = timed(lambda: ops.two_body_symmetry(u))
            flops = 8.0 * n**5 * (2 if cplx else 1)
            print(json.dumps({"op": "transform_two_body (symmetry-aware)", "n": n, "complex_u": cplx, "symmetry": kind,
                              "plain_ms": round(full, 3), "auto_ms": round(auto, 3), "detection_ms": round(detect, 3),
                              "speedup": round(full / auto, 3), "effective_tflops": round(flops / auto * 1e-9, 2)}))
            del u
        del base
    # complex u with REAL coefficients: the split (2M) quarter GEMM; 16 n^5 real flops are necessary
    for n in (40, 96, 128):
        u = torch.randn((n,) * 4, dtype=torch.complex128, device="cuda")
        C = torch.linalg.qr(torch.randn((n, n), dtype=torch.float64, device="cuda"))[0].contiguous()
        for label, coeff in (("real C", C), ("complex-typed real C", C.to(torch.complex128))):
            ms = timed(lambda: ops.transform_two_body(u, coeff))
            print(json.dumps({"op": "transform_two_body", "n": n, "u": "complex128", "C": label, "ms": round(ms, 3),
                              "tflops_2M": round(16.0 * n**5 / ms * 1e-9, 2),
                              "frac_of_dmma_peak_2M": round(16.0 * n**5 / ms * 1e-9 / peak, 3)}))
        del u
    for l in [64, 100]:
        u = torch.randn((l,) * 4, dtype=torch.float64, device="cuda")
        for od in (torch.float64, torch.complex128):
            ms = timed(lambda: ops.add_spin_two_body(u, anti_symmetrize=True, out_dtype=od))
            byt = 8 * l**4 + 16 * l**4 * (16 if od == torch.complex128 else 8)
            print(json.dumps({"op": "add_spin+antisym", "l": l, "out": str(od), "ms": round(ms, 3), "gbs": round(byt / ms * 1e-6, 1)}))
        del u
    n = 128
    u = torch.randn((n,) * 4, dtype=torch.float64, device="cuda")
    ms = timed(lambda: ops.anti_symmetrize(u))
    print(json.dumps({"op": "antisym", "n": n, "ms": round(ms, 3), "gbs": round(16 * n**4 / ms * 1e-6, 1)}))
    h = torch.randn((n, n), dtype=torch.float64, device="cuda")
    ms = timed(lambda: ops.fock_general(h, u, 10))
    print(json.dumps({"op": "fock_general", "n": n, "n_occ": 10, "ms": round(ms, 4)}))
    del u
    import numpy as np
    for l, G in [(20, 201), (100, 2001)]:
        C = torch.randn((G - 2, l), dtype=torch.float64, device="cuda")
        grid = torch.linspace(-10, 10, G, dtype=torch.float64, device="cuda")[1:-1].contiguous()
        ms = timed(lambda: ops.odqd_coulomb(C, grid, 1.0, 0.25), reps=3, warm=1)
        Gp = G - 2
        flops = 2.0 * l**2 * Gp**2 + 2.0 * l**4 * Gp
        print(json.dumps({"op": "odqd_coulomb", "l": l, "G": G, "ms": round(ms, 3), "tflops": round(flops / ms * 1e-9, 2)}))


if __name__ == "__main__":
    main()
