"""Every FP64 contraction kernel against an extended-precision reference, element by element, under the rounding-
error bound of its documented algorithm (tests/precise.py, DESIGN §2).  The 1e-12 max-scaled parity tests leave three
to four orders of magnitude of slack and never look at elements below 1e-12 of the largest; these cases would fail a
kernel that computes in ~46 bits, drops one term or skips one k-chunk.

Input families: (a) N(0, 1); (b) graded, ``u`` scaled by ``g_a g_b g_c g_d`` with ``g = logspace(0, -4, n)`` and a
near-identity ``C`` so the output keeps its dynamic range; (c) cancellation, a round trip through ``C`` and
``C⁻¹`` with cond(C) = 1e3; (d) physical, the ODQD grid Coulomb elements.  Dense longdouble references are used up
to n = 48 (and for small ``n`` with large ``m``); above that ``u = A ⊗ B`` (``u[a,b,c,d] = A[a,c] B[b,d]``, minus the
``(c, d)`` swap for the anti-symmetric cases) with dyadic ``A``, ``B`` is an exact FP64 tensor whose transform has
an O(n³)-per-plane reference, and whole planes are compared at the leading indices where the kernels switch: 0, the
64 and 128 boundaries, n - 1 and two random ones.

Past n = 128 the same exact inputs reach the schedules whose machinery is idle at small n: the sharded peer schedule
and the sharded anti-symmetric pair schedule on emulated ranks (tests/sharded_bounds.py: whole planes plus a sweep of
every element of every rank), the single-GPU symmetry-aware path, the mixed four-matrix transform and the consumers of
a sharded tensor.  Their buffers, outputs and workspaces start as NaN, so an element that was never written or was
computed from memory nobody wrote fails the check; each case asserts the property it is there for.

The module prints, per kernel family, the largest criterion-A ratio (|error| / bound) and the largest ratio of the
kernel's RMS error to plain numpy FP64's (criterion B), and its wall time (``pytest -s``)."""

import collections
import ctypes
import functools
import itertools
import time
import types

import numpy as np
import pytest

import precise as P

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import sharded_bounds as SB  # noqa: E402  (needs torch)

_STATS = collections.defaultdict(list)
_SWEEP = collections.defaultdict(list)  # family -> largest |got - X̂ Ŷ| / bound of each whole-tensor sweep


@pytest.fixture(scope="module", autouse=True)
def report():
    t0 = time.perf_counter()
    yield
    lines = [f"rounding bounds: {time.perf_counter() - t0:.1f} s wall for the module"]
    for family, rows in sorted(_STATS.items()):
        a = max(r["a"] for r in rows)
        b = max(r["rms"] / max(r["rms_fp64"], 1e-300) for r in rows)
        lines.append(f"  {family:34s} {len(rows):3d} checks  max A ratio {a:.3g}  max RMS(GPU)/RMS(FP64) {b:.3g}")
    for family, ratios in sorted(_SWEEP.items()):
        lines.append(f"  {family + ' (sweep)':34s} {len(ratios):3d} tensors max |error| / bound {max(ratios):.3g}")
    lines.append(f"  peak device memory {torch.cuda.max_memory_allocated() / 2**30:.1f} GiB")
    print("\n" + "\n".join(lines))


def check(family, got, ref, absval, k, fp64, what):
    _STATS[family].append(P.assert_rounding_bound(got, ref, absval, k, fp64, what))


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def host(t):
    return t.cpu().numpy()


def rand(rng, shape, complex_=False):
    return rng.standard_normal(shape) + (1j * rng.standard_normal(shape) if complex_ else 0)


plane_indices = SB.plane_indices


_PoisonedTorch = SB.PoisonedTorch


@pytest.fixture
def poisoned_ops(monkeypatch):
    """``ops`` with NaN-filled outputs and workspaces: an element that no kernel writes, or one computed from
    workspace that nobody wrote, is non-finite."""
    from quantum_systems_b200 import ops

    monkeypatch.setattr(ops, "torch", _PoisonedTorch())
    return ops


# ------------------------------------------------------------------------------------------- four-index transform

# (label, n, m, u complex, C complex, bi-orthogonal C~): dense references.  Real K' = n, complex K' = 2n; the quarter
# GEMM's k-chunk is 16 and a last chunk of 1..8 real columns runs as one half (DESIGN §4.1).
DENSE = [
    ("K'=13 odd pitch", 13, 13, False, False, False),
    ("K'=16", 16, 16, False, False, True),
    ("K'=20", 20, 20, False, False, False),
    ("K'=33", 33, 33, False, False, False),
    ("K'=16 complex", 8, 8, True, True, False),
    ("K'=24 complex", 12, 12, True, True, True),
    ("K'=26 complex", 13, 13, True, True, False),
    ("split K=20", 20, 20, True, False, False),
    ("split K=25", 25, 25, True, False, True),
    ("real u complex C", 15, 15, False, True, False),
] + [(f"W'={m}", 5, m, False, False, False) for m in (5, 12, 20, 28, 36, 44, 52, 60, 65, 70)] + [
    ("complex W'=66", 4, 33, True, True, False),
    ("split W'=33", 4, 33, True, False, False),
]

# (label, n, u complex, C complex): A ⊗ B inputs, whole planes.  K = 127, 128, 129 and 144 (K > 128 chunk loop).
KRON = [(f"n={n} {kind}", n, kind in ("complex", "split"), kind == "complex")
        for n in (127, 128, 129, 144) for kind in ("real", "complex", "split")] + [
    ("m=130 rectangular", 6, False, False), ("complex m=100 rectangular", 5, True, True)]


@pytest.mark.parametrize("case", DENSE, ids=[c[0] for c in DENSE])
def test_transform_dense(case):
    from quantum_systems_b200 import ops

    label, n, m, u_c, c_c, biorth = case
    rng = np.random.default_rng(n * 131 + m)
    u, C = rand(rng, (n,) * 4, u_c), rand(rng, (n, m), c_c)
    Ct = rand(rng, (m, n), c_c) if biorth else C.conj().T
    ref, absval, fp64 = P.companions(P.quarter_steps, u, C, Ct)
    got = host(ops.transform_two_body(dev(u), dev(C), dev(Ct) if biorth else None, symmetry=0))
    check("quarter GEMM (dense)", got, ref, absval, P.k_transform([n] * 4, [u_c or c_c] * 4), fp64, label)


def kron_case(n, u_c, c_c, anti=False, same=False, m=None, seed=0):
    rng = np.random.default_rng(seed * 1000 + n)
    m = n if m is None else m
    A = P.dyadic(rng, (n, n), u_c)
    B = A if same else P.dyadic(rng, (n, n), u_c)
    C = rand(rng, (n, m), c_c)
    Ct = C.conj().T
    Ad, Bd = dev(A), dev(B)
    u = Ad[:, None, :, None] * Bd[None, :, None, :]
    if anti:
        u = u - Ad[:, None, None, :] * Bd[None, :, :, None]
    return rng, A, B, C, Ct, u.contiguous()


def check_kron_planes(family, label, out, A, B, C, Ct, planes, anti, cplx):
    n = C.shape[0]
    ref, absval, fp64 = P.companions(P.kron_transform_planes, A, B, C, Ct, planes=planes, anti=anti)
    got = host(out[planes])
    check(family, got, ref, absval, P.k_transform([n] * 4, [cplx] * 4), fp64, f"{label}, planes {planes}")


@pytest.mark.parametrize("case", KRON, ids=[c[0] for c in KRON])
def test_transform_large_k_planes(case):
    from quantum_systems_b200 import ops

    label, n, u_c, c_c = case
    m = {"m=130 rectangular": 130, "complex m=100 rectangular": 100}.get(label, n)
    rng, A, B, C, Ct, u = kron_case(n, u_c, c_c, m=m)
    out = ops.transform_two_body(u, dev(C), symmetry=0)
    del u
    check_kron_planes("quarter GEMM (planes)", label, out, A, B, C, Ct, plane_indices(m, rng), False, u_c or c_c)


# (id, n, m, u complex, C complex, bi-orthogonal C~, kind): kind 1 anti-symmetric in the last pair, 2 particle-exchange
# symmetric (B = A), 3 both (anti-symmetric with B = A: the library picks 1).  Complex dyadic products and their
# differences are exact (<= 46 bits), so every symmetry holds exactly.
SYMMETRY = [(f"{name}-{n}", n, n, False, False, False, kind) for name, kind in (("antisymmetric", 1), ("exchange", 2))
            for n in (128, 130)] + [
    ("both-144", 144, 144, False, False, False, 3),
    ("antisymmetric-129-unpaired", 129, 129, False, False, False, 1),
    ("exchange-144", 144, 144, False, False, False, 2),
    ("antisymmetric-complex-biorth-129", 129, 129, True, True, True, 1),
    ("exchange-complex-biorth-144", 144, 144, True, True, True, 2),
    ("both-complex-130", 130, 130, True, True, False, 3),
    ("antisymmetric-split-144", 144, 144, True, False, False, 1),
    ("exchange-split-129", 129, 129, True, False, False, 2),
    ("antisymmetric-real-u-complex-C-144", 144, 144, False, True, False, 1),
    ("exchange-real-u-complex-C-129", 129, 129, False, True, False, 2),
    ("antisymmetric-144-to-129", 144, 129, False, False, False, 1),
    ("exchange-129-to-144", 129, 144, False, False, False, 2),
]


@pytest.mark.parametrize("case", SYMMETRY, ids=[c[0] for c in SYMMETRY])
def test_symmetry_aware_default_path(case, poisoned_ops):
    """The single-GPU symmetry-aware transform (``two_body_steps`` with symmetry 1/2: masked step 2, packed pair
    steps 3-4, mirror fill) with NaN-filled output and workspace."""
    ops = poisoned_ops
    label, n, m, u_c, c_c, biorth, kind = case
    anti = kind != ops.PARTICLE_EXCHANGE
    rng, A, B, C, Ct, u = kron_case(n, u_c, c_c, anti=anti, same=kind != ops.ANTISYMMETRIC_LAST_PAIR, m=m,
                                    seed=kind)
    if biorth:
        Ct = rand(rng, (m, n), c_c)
    if kind == 3:
        assert ops.two_body_symmetry(u) == ops.ANTISYMMETRIC_LAST_PAIR | ops.PARTICLE_EXCHANGE
    want = ops.ANTISYMMETRIC_LAST_PAIR if anti else ops.PARTICLE_EXCHANGE
    out = ops.transform_two_body(u, dev(C), dev(Ct) if biorth else None)
    assert ops.proven_symmetry(out) == want, "the symmetry-aware path did not run"
    # step 2 skips tiles: column tiles r right of every s of a row tile (r < s, or r <= s)
    t_dtype = torch.complex128 if (u_c or c_c) else torch.float64
    c_dtype = torch.complex128 if c_c else torch.float64
    X = m * n * n
    kept = SB.planned_tiles(X, n, m, t_dtype, c_dtype, n, 1, int(anti), 1, 1, n * n, m)
    assert kept < SB.planned_tiles(X, n, m, t_dtype, c_dtype, n), "the step-2 mask keeps every tile"
    del u
    check_kron_planes("symmetry-aware transform", f"{label} symmetry {want}", out, A, B, C, Ct,
                      plane_indices(m, rng), anti, u_c or c_c)


# (label, n, m, u complex, C complex, explicit bras): four different matrices, so step 4 rebuilds its bra image in the
# slot step 3 read.  A ⊗ B inputs, whole planes, K > 128.
MIXED = [
    ("n=129 real", 129, 129, False, False, False),
    ("n=144 real explicit bras", 144, 144, False, False, True),
    ("n=144 complex", 144, 144, True, True, False),
    ("n=129 complex explicit bras", 129, 129, True, True, True),
    ("n=144 split explicit bras", 144, 144, True, False, True),
    ("n=129 real u complex C", 129, 129, False, True, False),
    ("144 -> 130 rectangular", 144, 130, False, False, False),
    ("144 -> 130 complex rectangular explicit bras", 144, 130, True, True, True),
]


@pytest.mark.parametrize("case", MIXED, ids=[c[0] for c in MIXED])
def test_mixed_transform_large_k_planes(case, poisoned_ops):
    ops = poisoned_ops
    label, n, m, u_c, c_c, explicit = case
    assert n > 128  # the K > 128 chunk loop
    rng, A, B, C_r, _, u = kron_case(n, u_c, c_c, m=m, seed=7)
    C_s = rand(rng, (n, m), c_c)
    Ct_p = rand(rng, (m, n), c_c) if explicit else C_r.conj().T
    Ct_q = rand(rng, (m, n), c_c) if explicit else C_s.conj().T
    out = ops.transform_two_body_mixed(u, dev(C_r), dev(C_s), *((dev(Ct_p), dev(Ct_q)) if explicit else ()))
    del u
    planes = plane_indices(m, rng)
    ref, absval, fp64 = P.companions(P.kron_transform_planes, A, B, C_r, Ct_p, C_s, Ct_q, planes=planes)
    check("mixed transform (planes)", host(out[planes]), ref, absval, P.k_transform([n] * 4, [u_c or c_c] * 4), fp64,
          f"{label}, planes {planes}")


@functools.lru_cache(maxsize=None)
def graded_case():
    """Family (b) at n = 48 in full, with its reference (shared by the plain, default, streamed and sharded paths)."""
    n = 48
    rng = np.random.default_rng(48)
    u, C = P.graded_two_body(rng, n), P.near_identity(rng, n)
    return u, C, P.companions(P.quarter_steps, u, C, C.T)


def test_transform_graded_full_every_path(monkeypatch):
    from quantum_systems_b200 import ops, sharded, streamed

    u, C, (ref, absval, fp64) = graded_case()
    n = u.shape[0]
    k = P.k_transform([n] * 4, [False] * 4)
    for symmetry in (0, None):
        got = host(ops.transform_two_body(dev(u), dev(C), symmetry=symmetry))
        check("quarter GEMM (graded, n=48)", got, ref, absval, k, fp64, f"ops, symmetry={symmetry}")
    monkeypatch.setattr(streamed, "MIN_BYTES", 0)
    assert streamed.applicable(u, dev(C))
    check("streamed transform", np.asarray(streamed.transform_two_body(u, dev(C))), ref, absval, k, fp64, "streamed")
    ctx = sharded.EmulatedContext(3)
    basis = sharded.ShardedBasisSet.from_global(ctx, np.eye(n), np.eye(n), u)
    out = sharded.transform_two_body_sharded(basis.u, dev(C), dev(C.T))
    check("sharded transform", host(out.gather()), ref, absval, k, fp64, "EmulatedContext(3)")


def test_transform_round_trip_cancellation():
    from quantum_systems_b200 import ops

    n = 48
    rng = np.random.default_rng(4848)
    u = rng.standard_normal((n,) * 4)
    C, Ci = P.conditioned(rng, n)

    def round_trip(u, C, Ci, dt, absolute=False):
        return P.quarter_steps(P.quarter_steps(u, C, Ci, dt), Ci, C, dt)

    ref, absval, fp64 = P.companions(round_trip, u, C, Ci)
    mid = ops.transform_two_body(dev(u), dev(C), dev(Ci), symmetry=0)
    got = host(ops.transform_two_body(mid, dev(Ci), dev(C), symmetry=0))
    check("quarter GEMM (round trip)", got, ref, absval, P.k_transform([n] * 8, [False] * 8), fp64, "C then C^-1")


@pytest.mark.parametrize("n,m", [(13, 13), (33, 20), (129, 129), (144, 150)])
@pytest.mark.parametrize("h_c,c_c,biorth", [(False, False, False), (True, True, True), (True, False, False),
                                             (False, True, True)], ids=["real", "complex-biorth", "split", "realh"])
def test_one_body_and_functions(n, m, h_c, c_c, biorth):
    from quantum_systems_b200 import ops

    rng = np.random.default_rng(n + m)
    h, C = rand(rng, (n, n), h_c), rand(rng, (n, m), c_c)
    Ct = rand(rng, (m, n), c_c) if biorth else C.conj().T
    ref, absval, fp64 = P.companions(P.one_body, h, C, Ct)
    got = host(ops.transform_one_body(dev(h), dev(C), dev(Ct) if biorth else None))
    check("one-body transform", got, ref, absval, P.k_transform([n, n], [h_c or c_c] * 2), fp64, "h")
    spf = rand(rng, (n, 7, 5), h_c) * P.graded(n)[:, None, None]
    for bra, M in ((False, C), (True, Ct)):
        def fn(spf, M, dt, absolute=False):
            flat = spf.reshape(n, -1)
            return ((M @ flat) if bra else (M.T @ flat)).reshape((-1,) + spf.shape[1:])

        ref, absval, fp64 = P.companions(fn, spf, M)
        got = host(ops.transform_functions(dev(spf), dev(M), bra))
        check("transform_functions", got, ref, absval, P.k_transform([n], [h_c or c_c]), fp64, f"bra={bra}")


# ---------------------------------------------------------------------------- sharded transform on emulated ranks
# EmulatedContext(W) runs every rank's kernels on this GPU, with the same scattering stores as one process per GPU;
# only the destination pointers differ.  The input is an exact A ⊗ B tensor built slab by slab, every buffer the
# schedule allocates starts as NaN, and tests/sharded_bounds.py checks whole planes under criteria A and B and every
# element of every rank under criterion A.


nan_engine = SB.nan_engine


# (label, n, m, W, u complex, C complex, bi-orthogonal C~, graded family, chain, what the case reaches)
SHARDED_FULL = [
    ("128 W=8", 128, 128, 8, False, False, False, False, False, {"even", "K=128"}),
    ("129 W=2 odd pitch", 129, 129, 2, False, False, False, False, False, {"uneven", "odd pitch"}),
    ("129 W=3 complex biorth", 129, 129, 3, True, True, True, False, False, {"even", "A=43"}),
    ("144 W=5 split", 144, 144, 5, True, False, False, False, False, {"uneven"}),
    ("144 W=8 real u complex C", 144, 144, 8, False, True, False, False, False, {"even", "A=18", "own output"}),
    ("144 W=3 graded", 144, 144, 3, False, False, False, True, False, {"even"}),
    ("130 -> 144 W=4", 130, 144, 4, False, False, False, False, False, {"uneven"}),
    ("144 -> 129 W=3 complex biorth", 144, 129, 3, True, True, True, False, False, {"even"}),
    ("144 -> 5 W=8", 144, 5, 8, False, False, False, False, False, {"idle ranks"}),
    ("129 W=3 twice", 129, 129, 3, False, False, False, False, True, {"even", "recycled"}),
]
SHARDED_PAIRS = [
    ("130 W=2 couples", 130, 130, 2, False, False, False, False, False, {"even", "couples"}),
    ("129 W=3 unpaired", 129, 129, 3, False, False, False, False, False, {"even", "unpaired"}),
    ("144 W=5 complex biorth", 144, 144, 5, True, True, True, False, False, {"uneven"}),
    ("144 W=8 split", 144, 144, 8, True, False, False, False, False, {"even"}),
    ("144 -> 131 W=3", 144, 131, 3, False, False, False, False, False, {"even", "unpaired"}),
    ("144 W=4 graded", 144, 144, 4, False, False, False, True, False, {"even", "couples"}),
    ("130 W=2 twice", 130, 130, 2, False, False, False, False, True, {"even", "couples", "recycled"}),
]


def exact_case(n, m, u_c, c_c, biorth, graded, seed):
    """Dyadic ``A``, ``B`` (family a), or scaled by power-of-two ``g_a g_c`` with a near-identity ``C`` (family b)."""
    rng = np.random.default_rng(seed)
    A, B = P.dyadic(rng, (n, n), u_c), P.dyadic(rng, (n, n), u_c)
    if graded:
        g = np.outer(P.pow2_graded(n), P.pow2_graded(n))
        A, B, C = A * g, B * g, P.near_identity(rng, n, m, c_c)
    else:
        C = rand(rng, (n, m), c_c)
    Ct = rand(rng, (m, n), c_c) if biorth else C.conj().T
    return rng, A, B, C, Ct


def assert_reaches(reach, out, n, m, W, u_dtype, t_dtype):
    """The property each case is there for, so that a change of defaults cannot turn it into a duplicate."""
    from quantum_systems_b200 import ops, sharded

    _, off = sharded.block_partition(n, W)
    sizes = {b - a for a, b in zip(off, off[1:])}
    if "even" in reach:
        assert len(sizes) == 1, f"sources {sizes} are not even"
    if "uneven" in reach:
        assert len(sizes) > 1, "every source holds equally many planes"
    for A in (43, 18):
        if f"A={A}" in reach:
            assert sharded.block_partition(n, W)[0] == A
    if "K=128" in reach:
        assert n == 128 and t_dtype == torch.float64
    if "odd pitch" in reach:
        assert sharded.padded_pitch(n, u_dtype) != n
    if "own output" in reach:
        assert u_dtype != t_dtype and out.spare is None, "the output is the input's spare"
    if "idle ranks" in reach:
        assert m < W and any(out.planes(r)[0] == out.planes(r)[1] for r in range(W))
    if "couples" in reach:
        assert t_dtype == torch.float64 and m % 2 == 0
    if "unpaired" in reach:
        assert t_dtype == torch.float64 and m % 2 == 1
    if W > 1 and m >= 16:
        assert ops.scatter_deal(m) > 1, "step 4 deals no columns"
    assert n > 128 or "K=128" in reach


def run_sharded_case(case, pairs):
    from quantum_systems_b200 import sharded

    label, n, m, W, u_c, c_c, biorth, graded, chain, reach = case
    family = "sharded pair schedule" if pairs else "sharded full steps"
    rng, A, B, C, Ct = exact_case(n, m, u_c, c_c, biorth, graded, seed=n * 10 + W)
    u_dtype = torch.complex128 if u_c else torch.float64
    t_dtype = torch.complex128 if (u_c or c_c) else torch.float64
    engine = nan_engine()()
    ctx = sharded.EmulatedContext(W, engine=engine)
    u = SB.exact_sharded(ctx, A, B, pairs, u_dtype, "cuda")
    symmetry = None if pairs else 0
    out = sharded.transform_two_body_sharded(u, dev(C), dev(Ct) if biorth else None, symmetry=symmetry)
    assert out.proven_antisymmetric == pairs, "the case did not take the schedule it is there for"
    if pairs:
        assert engine.symmetry_tests > 0, "the anti-symmetry of the input was not tested on the device"
        kept = SB.pair_step2_tiles(ctx, n, m, t_dtype, torch.complex128 if c_c else torch.float64)
        assert any(k < planned for k, planned in kept), f"step 2 skipped no tile: {kept}"
    assert_reaches(reach, out, n, m, W, u_dtype, t_dtype)
    arrays, factors = (A, B, C, Ct), P.kron_factors
    k = P.k_transform([n] * 4, [u_c or c_c] * 4)
    if chain:
        C2 = rand(rng, (m, m), c_c)
        tests = engine.symmetry_tests
        out = sharded.transform_two_body_sharded(out, dev(C2), symmetry=symmetry)
        with pytest.raises(RuntimeError, match="recycled"):
            u.buffers  # the second result went into the first input's buffers (ping-pong)
        if pairs:
            assert out.proven_antisymmetric and engine.symmetry_tests == tests, "the proof was not trusted"
        arrays, factors = (A, B, C, Ct, C2, C2.conj().T), SB.chain_factors
        k = P.k_transform([n] * 8, [u_c or c_c] * 8)
    del u
    ratio = SB.check_sharded(functools.partial(check, family), out, factors, arrays, k, pairs, rng, label)
    _SWEEP[family].append(ratio)


@pytest.mark.parametrize("case", SHARDED_FULL, ids=[c[0] for c in SHARDED_FULL])
def test_sharded_full_steps(case):
    run_sharded_case(case, pairs=False)


@pytest.mark.parametrize("case", SHARDED_PAIRS, ids=[c[0] for c in SHARDED_PAIRS])
def test_sharded_pair_schedule(case):
    run_sharded_case(case, pairs=True)


# ------------------------------------------------------------------------------------------ structured transforms


@pytest.mark.parametrize("n,m,biorth", [(33, 20, False), (64, 48, True)])
@pytest.mark.parametrize("anti", [False, True])
def test_diagonal_transform(n, m, biorth, anti):
    from quantum_systems_b200 import ops

    rng = np.random.default_rng(n * m)
    g = P.graded(n)
    W = rng.standard_normal((n, n)) * np.outer(g, g)
    C = rand(rng, (n, m), True)
    Ct = rand(rng, (m, n), True) if biorth else C.conj().T
    ref, absval, fp64 = P.companions(P.diagonal_rows, W, C, Ct, anti=anti)
    got = host(ops.transform_two_body_diagonal(dev(W), dev(C), dev(Ct) if biorth else None, anti_symmetrize=anti))
    check("diagonal transform", got, ref, absval, P.k_diagonal(n, True, anti=anti), fp64, f"anti={anti}")


@pytest.mark.parametrize("l,G,length,planes", [(20, 201, 6.0, None), (10, 1001, 10.0, None),
                                               (100, 2001, 10.0, (37, 45))])
def test_odqd_coulomb(l, G, length, planes):
    from quantum_systems_b200 import ops
    from quantum_systems_b200.odqd import grid_orbitals
    from quantum_systems_b200.potentials import HOPotential

    grid, _, C = grid_orbitals(l, length, G, HOPotential(0.25))
    inner = grid[1:-1]
    out = host(ops.odqd_coulomb(dev(C), dev(inner), 1.0, 0.25, planes=planes))
    k = P.k_diagonal(G - 2, False, generated_w=True)
    if planes is None:
        ref, absval, fp64 = P.companions(P.odqd_rows, C, grid=inner, alpha=1.0, a=0.25)
        check("ODQD Coulomb", out, ref, absval, k, fp64, f"l={l} G={G}")
        return
    rng = np.random.default_rng(l)
    rows = [(a, int(c)) for a in (planes[0], planes[1] - 1) for c in rng.integers(0, l, 3)]
    ref, absval, fp64 = P.companions(P.odqd_rows, C, grid=inner, alpha=1.0, a=0.25, rows=rows)
    got = np.stack([out[a - planes[0], :, c, :] for a, c in rows])
    check("ODQD Coulomb", got, ref, absval, k, fp64, f"l={l} G={G} pairs {rows}")


# ----------------------------------------------------------------------------------------------------- Fock kernels


@pytest.mark.parametrize("u_c", [False, True], ids=["real", "complex"])
def test_fock_occupied_kernels(u_c):
    from quantum_systems_b200 import GeneralOrbitalSystem, SpatialOrbitalSystem, _native, ops

    n = 40
    rng = np.random.default_rng(40 + u_c)
    u, h = P.graded_two_body(rng, n, complex_=u_c), rand(rng, (n, n), u_c) * 1e-8
    ud, hd = dev(u), dev(h)
    for n_occ in (0, 1, 31, 32, 33, n):
        for spatial in (False, True):
            ref, absval, fp64 = P.companions(P.fock_occupied, h, u, n_occ=n_occ, spatial=spatial)
            k = (2 if spatial else 1) * n_occ + 1
            what = f"n_occ={n_occ} spatial={spatial}"
            got = host((ops.fock_spatial if spatial else ops.fock_general)(hd, ud, n_occ))
            check("fock_general / fock_spatial", got, ref, absval, k, fp64, what)
            system = SpatialOrbitalSystem if spatial else GeneralOrbitalSystem
            got = system.construct_fock_matrix(types.SimpleNamespace(n=n_occ), h, u)  # host u: qs_fock_gathered
            check("fock_gathered", np.asarray(got), ref, absval, k, fp64, what)
        ref, absval, fp64 = P.companions(P.fock_occupied, h, u, n_occ=n_occ, spatial=False)
        for q0, q1 in ((n // 2, n // 2), (n // 2, n // 2 + 1), (0, n)):
            f = torch.full((n, n), 7.0, dtype=hd.dtype, device="cuda")
            u_cols = ud[:, :, q0:q1, :].contiguous()
            code = ops._code(ud)
            _native.call("qs_fock_general_cols", ops._ptr(hd), code, ops._ptr(u_cols), code, n, n_occ, ops._ptr(f),
                         q0, q1, ops._stream())
            got = host(f)
            check("qs_fock_general_cols", got[:, q0:q1], ref[:, q0:q1], absval[:, q0:q1], n_occ + 1, fp64[:, q0:q1],
                  f"n_occ={n_occ} columns [{q0}, {q1})")
            outside = np.ones(n, dtype=bool)
            outside[q0:q1] = False
            assert np.all(got[:, outside] == 7.0), f"columns outside [{q0}, {q1}) were written"


def graded_density(rng, n, complex_, scale=1.0):
    g = P.graded(n)
    return scale * rand(rng, (n, n), complex_) * np.outer(g, g)


def k_density(n, u_c, rho_c, terms):
    """``terms n² + 1`` (``2 n² + 1`` restricted, ``3 n² + 1`` unrestricted), doubled for complex products."""
    return terms * n * n * (2 if u_c and rho_c else 1) + 1


@pytest.mark.parametrize("n", [1, 64, 65])
@pytest.mark.parametrize("u_c,rho_c,h_c", list(itertools.product([False, True], repeat=3)),
                         ids=lambda c: "c" if c else "r")
def test_fock_density_dense(n, u_c, rho_c, h_c):
    from quantum_systems_b200 import ops

    rng = np.random.default_rng(n)
    u, rho, h = P.graded_two_body(rng, n, u_c), graded_density(rng, n, rho_c), rand(rng, (n, n), h_c) * 1e-6
    ref, absval, fp64 = P.companions(P.fock_density, h, u, rho, a_d=1.0, a_x=-0.5)
    got = host(ops.fock_from_density(dev(h), dev(u), dev(rho), 1.0, -0.5))
    check("fock_from_density", got, ref, absval, k_density(n, u_c, rho_c, 2), fp64, f"n={n}")


@pytest.mark.parametrize("n", [129, 130])
@pytest.mark.parametrize("u_c,rho_c,h_c", list(itertools.product([False, True], repeat=3)),
                         ids=lambda c: "c" if c else "r")
def test_fock_density_kron(n, u_c, rho_c, h_c):
    from quantum_systems_b200 import ops

    rng = np.random.default_rng(n)
    g = P.pow2_graded(n)
    A = P.dyadic(rng, (n, n), u_c) * np.outer(g, g)
    B = P.dyadic(rng, (n, n), u_c) * np.outer(g, g)
    rho, h = graded_density(rng, n, rho_c), rand(rng, (n, n), h_c) * 1e-6
    Ad, Bd = dev(A), dev(B)
    u = (Ad[:, None, :, None] * Bd[None, :, None, :]).contiguous()  # u[p,r,q,s] = A[p,q] B[r,s]
    ref, absval, fp64 = P.companions(P.kron_fock_density, h, A, B, rho, a_d=1.0, a_x=-0.5)
    got = host(ops.fock_from_density(dev(h), u, dev(rho), 1.0, -0.5))
    check("fock_from_density", got, ref, absval, k_density(n, u_c, rho_c, 2), fp64, f"n={n} A⊗B")


def test_fock_density_unaligned_u_takes_8_byte_pieces():
    """Even n with real ``u`` 8 bytes off a 16-byte boundary: the 8-byte piece path of an even row length."""
    from quantum_systems_b200 import ops

    n = 64
    rng = np.random.default_rng(64064)
    u, rho, h = P.graded_two_body(rng, n), graded_density(rng, n, False), rand(rng, (n, n)) * 1e-6
    buf = torch.empty(n**4 + 1, dtype=torch.float64, device="cuda")
    ud = buf[1:].view(n, n, n, n)
    ud.copy_(dev(u))
    assert ud.data_ptr() % 16 == 8
    ref, absval, fp64 = P.companions(P.fock_density, h, u, rho, a_d=1.0, a_x=-0.5)
    got = host(ops.fock_from_density(dev(h), ud, dev(rho), 1.0, -0.5))
    check("fock_from_density", got, ref, absval, k_density(n, False, False, 2), fp64, "unaligned u")
    ref, absval, fp64 = P.companions(P.fock_unrestricted, h, u, rho, 1e-6 * rho[::-1].copy())
    got = np.stack([host(f) for f in ops.fock_from_density_unrestricted(dev(h), ud, dev(rho),
                                                                         dev(1e-6 * rho[::-1].copy()))])
    check("fock_from_density_unrestricted", got, ref, absval, k_density(n, False, False, 3), fp64, "unaligned u")


@pytest.mark.parametrize("n", [64, 65])
@pytest.mark.parametrize("u_c,rho_c", [(False, False), (False, True), (True, False), (True, True)],
                         ids=["packed", "complex-rho", "complex-u", "complex"])
def test_fock_density_unrestricted(n, u_c, rho_c):
    from quantum_systems_b200 import ops

    rng = np.random.default_rng(n + 7)
    u, h = P.graded_two_body(rng, n, u_c), rand(rng, (n, n), u_c) * 1e-6
    ra, rb = graded_density(rng, n, rho_c), graded_density(rng, n, rho_c, scale=1e-6)
    ref, absval, fp64 = P.companions(P.fock_unrestricted, h, u, ra, rb)
    got = np.stack([host(f) for f in ops.fock_from_density_unrestricted(dev(h), dev(u), dev(ra), dev(rb))])
    check("fock_from_density_unrestricted", got, ref, absval, k_density(n, u_c, rho_c, 3), fp64, f"n={n}")


# (n, W, complex): consumers of a sharded tensor at n > 128, each rank reading its own planes
CONSUMERS = [(129, 3, False), (129, 5, True), (144, 3, True), (144, 5, False)]


@pytest.mark.parametrize("n,W,cplx", CONSUMERS, ids=[f"n={n} W={W} {'complex' if c else 'real'}" for n, W, c in CONSUMERS])
def test_sharded_consumers(n, W, cplx):
    from quantum_systems_b200 import sharded

    rng, A, B, _, _ = exact_case(n, n, cplx, False, False, True, seed=n + W)
    dtype = torch.complex128 if cplx else torch.float64
    ctx = sharded.EmulatedContext(W, engine=nan_engine()())
    h = rand(rng, (n, n), cplx) * 1e-6
    hd = dev(h)
    _, off = sharded.block_partition(n, W)
    assert off[1] < n - 1
    for anti in (False, True):
        u = SB.exact_sharded(ctx, A, B, anti, dtype, "cuda")
        basis = sharded.ShardedBasisSet(ctx, n, hd, None, u)
        for n_occ in (1, 33, off[1] - 1, off[1] + 1, n):
            f = torch.full((n, n), float("nan"), dtype=dtype, device="cuda")
            got = host(basis.construct_fock_matrix(hd, u, n_occ, f=f))  # qs_fock_general on rows p0..p1 per rank
            ref, absval, fp64 = P.companions(P.kron_fock_occupied, h, A, B, n_occ=n_occ, anti=anti)
            check("sharded consumers", got, ref, absval, n_occ + 1, fp64, f"construct_fock_matrix n_occ={n_occ}")
        if anti:
            break
        for n_occ in (1, off[1] + 1, n):
            traces = np.array(u.occupied_traces(hd, n_occ))
            ref, absval, fp64 = P.companions(P.kron_occupied_traces, h, A, B, n_occ=n_occ)
            check("sharded consumers", traces if cplx else traces.real, ref, absval, n_occ * n_occ, fp64,
                  f"occupied_traces n_occ={n_occ}")
            tr_h, direct, exchange = u.occupied_traces(hd, n_occ)
            energy = 2 * tr_h + 2 * direct - exchange
            assert basis.compute_reference_energy(n_occ) == (energy if cplx else energy.real)
        rho, rho_b = graded_density(rng, n, cplx), graded_density(rng, n, cplx, scale=1e-6)
        got = host(basis.fock_from_density(hd, dev(rho), 1.0, -0.5))
        ref, absval, fp64 = P.companions(P.kron_fock_density, h, A, B, rho, a_d=1.0, a_x=-0.5)
        check("sharded consumers", got, ref, absval, k_density(n, cplx, cplx, 2), fp64, "fock_from_density")
        got = np.stack([host(f) for f in basis.fock_from_density_unrestricted(hd, dev(rho), dev(rho_b))])
        ref, absval, fp64 = P.companions(P.kron_fock_unrestricted, h, A, B, rho, rho_b)
        check("sharded consumers", got, ref, absval, k_density(n, cplx, cplx, 3), fp64,
              "fock_from_density_unrestricted")
        del u, basis


# ---------------------------------------------------------------------------------------------- S² and the traces


@pytest.mark.parametrize("n,planes", [(2, None), (64, None), (520, (517, 518))])
@pytest.mark.parametrize("anti", [False, True])
def test_spin_squared_two_body(n, planes, anti):
    from quantum_systems_b200 import ops

    rng = np.random.default_rng(n)
    S = rand(rng, (3, n, n), True)
    out = ops.spin_squared_two_body(*(dev(s) for s in S), anti_symmetrize=anti, planes=planes)
    k = (12 if anti else 6) + 1
    if planes is None:
        ref, absval, fp64 = P.companions(P.spin_2_tb, S, anti=anti)
        check("spin_squared_two_body", host(out), ref, absval, k, fp64, f"n={n}")
        return
    # n = 520: 6 n 16 bytes of shared memory, past the 48 KiB default; one plane, three rows of it
    q = [0, 255, n - 1]
    ref, absval, fp64 = P.companions(P.spin_2_tb, S, p=[planes[0]], q=q, anti=anti)
    check("spin_squared_two_body", host(out[:, q]), ref, absval, k, fp64, f"n={n} plane {planes[0]} rows {q}")


@pytest.mark.parametrize("u_c", [False, True], ids=["real", "complex"])
def test_occupied_traces(u_c):
    from quantum_systems_b200 import ops

    n, n_occ = 40, 17
    rng = np.random.default_rng(17)
    u, h = P.graded_two_body(rng, n, u_c), rand(rng, (n, n), u_c) * P.graded(n)
    ref, absval, fp64 = P.companions(P.occupied_traces, h, u, n_occ=n_occ)
    got = host(ops.occupied_traces(dev(h), dev(u), n_occ))
    if not u_c:
        assert np.all(got.imag == 0)
        got = got.real
    check("occupied_traces", got, ref, absval, n_occ * n_occ, fp64, "graded")
