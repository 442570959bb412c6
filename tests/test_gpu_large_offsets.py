"""Every kernel on single tensors past 2**31 and 2**32 elements, the sizes the large workloads run at (the l = 128
UHF spin-orbital system, a configs[5] shard, the single-GPU transform at n >= 216).  A 32-bit element offset wraps
there; each case is built at the smallest extent whose largest offset crosses the boundary it is listed under in
tests/large_offsets.py (``CASES``), and asserts that claim.

* Data movement (add-spin, anti-symmetrise, spin-orbital assembly, cyclic fill, extract_block, scale_add): hash-coded
  inputs, an exact expectation from the index formula alone, ``torch.equal`` chunk by chunk, NaN-filled outputs.
* Contractions (the four-index transform, the symmetry-aware path, the sharded transform on one rank): ``u = A ⊗ B``
  with dyadic factors, whole planes on both sides of the boundary under criteria A and B (tests/precise.py), then every
  element under criterion A on the device (``sharded_bounds.sweep_slabs``).  The Fock builds, the traces and the
  diagonal / ODQD transforms against their kron or row references on the planes past the boundary.
* Symmetry detection: an exactly (anti-)symmetric tensor is detected, one changed element in the last plane makes it
  not so, and so does the control in plane 0.

Each case allocates inside itself, skips with the numbers when its planned peak exceeds the budget or the free device
memory, and frees everything before the next one.  ``pytest -s`` prints the wall time and peak memory of each case."""

import ctypes
import gc
import time

import numpy as np
import pytest

import large_offsets as LO
import precise as P

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import sharded_bounds as SB  # noqa: E402  (needs torch)

F64, C128 = torch.float64, torch.complex128
_REPORT = {}  # case -> (planned bytes, peak bytes, seconds)
_CURRENT = []


@pytest.fixture(scope="module", autouse=True)
def report():
    t0 = time.perf_counter()
    yield
    props = torch.cuda.get_device_properties(0)
    lines = [f"large offsets: {time.perf_counter() - t0:.1f} s wall for the module on {props.name}"]
    for name, (planned, peak, secs) in _REPORT.items():
        lines.append(f"  {name:32s} planned {planned / 1e9:6.1f} GB  peak {peak / 1e9:6.1f} GB  {secs:6.1f} s")
    print("\n" + "\n".join(lines))


@pytest.fixture(autouse=True)
def one_case_at_a_time():
    """Runs after the test function has returned (its tensors are gone): empty the cache, record the peak above what
    was allocated when the case began."""
    gc.collect()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    start = torch.cuda.memory_allocated()
    t0 = time.perf_counter()
    yield
    torch.cuda.synchronize()
    if _CURRENT:
        name = _CURRENT.pop()
        _REPORT[name] = (LO.planned_bytes(name), torch.cuda.max_memory_allocated() - start, time.perf_counter() - t0)
    gc.collect()
    torch.cuda.empty_cache()


def large(name):
    """The case ``name``: its claim asserted, skipped with the numbers when it does not fit."""
    case = LO.CASES[name]
    assert case.offset(case.extent) >= case.boundary, f"{name} does not cross {case.boundary}"
    planned = LO.planned_bytes(name)
    free, total = torch.cuda.mem_get_info()
    if planned > LO.BUDGET or planned > free:
        pytest.skip(f"{name}: planned peak {planned / 1e9:.1f} GB; budget {LO.BUDGET / 1e9:.0f} GB, "
                    f"free {free / 1e9:.1f} of {total / 1e9:.1f} GB")
    _CURRENT.append(name)
    return case


@pytest.fixture
def poisoned_ops(monkeypatch):
    from quantum_systems_b200 import ops

    monkeypatch.setattr(ops, "torch", SB.PoisonedTorch())
    return ops


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def rand(rng, shape, complex_=False):
    return rng.standard_normal(shape) + (1j * rng.standard_normal(shape) if complex_ else 0)


def check(got, ref, absval, k, fp64, what):
    P.assert_rounding_bound(got, ref, absval, k, fp64, what)


def boundary_planes(n, boundary, extra=()):
    """Planes 0, n - 1 and those on both sides of the plane that holds element offset ``boundary``."""
    pb = boundary // n**3
    return sorted({0, n - 1, pb - 1, pb, min(pb + 1, n - 1)} | set(extra))


def kron_tensor(A, B, anti, dtype):
    """``u = A ⊗ B`` (minus the (c, d) swap when ``anti``) built chunk by chunk on the device."""
    n = A.shape[0]
    Ad, Bd = dev(A).to(dtype), dev(B).to(dtype)

    def planes(p0, p1, device):
        t = Ad[p0:p1, None, :, None] * Bd[None, :, None, :]
        return t - Ad[p0:p1, None, None, :] * Bd[None, :, :, None] if anti else t

    return LO.fill(torch.empty((n,) * 4, dtype=dtype, device="cuda"), planes)


def check_kron_result(out, arrays, k, anti, boundary, what):
    """Whole planes on both sides of the boundary under criteria A and B, then every element under criterion A."""
    m = out.shape[0]
    SB.check_planes(check, out, P.kron_factors, arrays, boundary_planes(m, boundary), k, anti, what, batch=2)
    SB.sweep_slabs([("whole tensor", 0, out)], P.kron_factors, arrays, k, anti, what, boundary=boundary)


# ------------------------------------------------------------------------------------------ four-index transform


# (case, complex, orbitals n of u; None: the case's extent, a square transform).  The rectangular 160 -> 257 case is
# the one whose stores cross 2**32 on one B200: only its last quarter step writes past 2**32 elements (the square
# n = 257 transform does not fit).
TRANSFORM = [("transform-216-real", False, None), ("transform-216-complex", True, None),
             ("transform-217-real-odd-pitch", False, None), ("transform-257-real", False, None),
             ("transform-160-257-real", False, LO.RECT_N)]


@pytest.mark.parametrize("name,cplx,n", TRANSFORM, ids=[c[0] for c in TRANSFORM])
def test_transform_full_steps(name, cplx, n, poisoned_ops):
    from quantum_systems_b200 import sharded

    ops = poisoned_ops
    case = large(name)
    m = case.extent
    n = m if n is None else n
    dtype = C128 if cplx else F64
    if "odd-pitch" in name:
        assert sharded.padded_pitch(n, dtype) != n, "the odd extent takes no padded pitch"
    if n != m:
        assert (n * m**3 - 1 < case.boundary <= m**4 - 1), "only the last step's stores should cross the boundary"
    rng = np.random.default_rng(n * 1000 + m)
    A, B, C = P.dyadic(rng, (n, n), cplx), P.dyadic(rng, (n, n), cplx), rand(rng, (n, m), cplx)
    u = kron_tensor(A, B, False, dtype)
    out = ops.transform_two_body(u, dev(C), symmetry=0)
    del u
    assert tuple(out.shape) == (m,) * 4
    check_kron_result(out, (A, B, C, C.conj().T), P.k_transform([n] * 4, [cplx] * 4), False, case.boundary, name)


@pytest.mark.parametrize("name", ["symmetric-216-antisymmetric", "symmetric-216-exchange"])
def test_symmetry_aware_path(name, poisoned_ops):
    """Detection, masked steps 2-4 and the mirror fill on a result past 2**31."""
    ops = poisoned_ops
    case = large(name)
    n = case.extent
    anti = name.endswith("antisymmetric")
    kind = ops.ANTISYMMETRIC_LAST_PAIR if anti else ops.PARTICLE_EXCHANGE
    rng = np.random.default_rng(n + kind)
    A = P.dyadic(rng, (n, n))
    B = P.dyadic(rng, (n, n)) if anti else A  # B = A: u[a,b,c,d] = u[b,a,d,c] exactly
    C = rand(rng, (n, n))
    u = kron_tensor(A, B, anti, F64)
    out = ops.transform_two_body(u, dev(C))
    assert ops.proven_symmetry(out) == kind, "the symmetry-aware path did not run"
    del u
    check_kron_result(out, (A, B, C, C.T), P.k_transform([n] * 4, [False] * 4), anti, case.boundary, name)


# --------------------------------------------------------------------------------------------- symmetry detection


def is_antisymmetric_last_pair(u):
    from quantum_systems_b200 import _native, ops

    flag = ctypes.c_int(1)
    scratch = torch.empty(2, dtype=torch.int32, device="cuda")
    _native.call("qs_is_antisymmetric_last_pair", ops._ptr(u), ops._code(u), u.shape[0], u.shape[0],
                 ctypes.byref(flag), ops._ptr(scratch), ops._stream())
    return bool(flag.value)


def exchange_symmetrized(n, dtype):
    """``u = h(pqrs) + h(qpsr)``: exactly particle-exchange symmetric."""
    def planes(p0, p1, device):
        p, q, r, s = LO.axes(p0, p1, n, device)
        return LO.coded(LO.lin4(p, q, r, s, n), dtype) + LO.coded(LO.lin4(q, p, s, r, n), dtype)

    return planes


@pytest.mark.parametrize("name,dtype", [("detect-216-real", F64), ("detect-216-complex", C128),
                                        ("detect-257-real", F64)])
def test_symmetry_detection_sees_the_last_plane(name, dtype):
    from quantum_systems_b200 import ops

    case = large(name)
    n = case.extent
    u = torch.empty((n,) * 4, dtype=dtype, device="cuda")
    bump = 1j if dtype == C128 else 1.0
    for kind, planes, last, first in (
            (ops.ANTISYMMETRIC_LAST_PAIR, LO.antisymmetrized(n, dtype), (n - 1, n - 1, n - 1, n - 2), (0, 0, 1, 2)),
            (ops.PARTICLE_EXCHANGE, exchange_symmetrized(n, dtype), (n - 1, n - 2, n - 1, n - 3), (0, 1, 2, 3))):
        assert int(np.ravel_multi_index(last, (n,) * 4)) >= case.boundary
        LO.fill(u, planes)
        assert ops.two_body_symmetry(u) & kind, f"{name}: symmetry {kind} not detected"
        if kind == ops.ANTISYMMETRIC_LAST_PAIR:
            assert is_antisymmetric_last_pair(u)
        for where in (last, first):
            u[where] += bump
            assert not ops.two_body_symmetry(u) & kind, f"{name}: element {where} changed, symmetry {kind} still found"
            if kind == ops.ANTISYMMETRIC_LAST_PAIR:
                assert not is_antisymmetric_last_pair(u), f"{name}: element {where} changed, slab still anti-symmetric"
            u[where] -= bump


# ------------------------------------------------------------------------------------------------ data movement


def test_cyclic_antisymmetric_fill():
    from quantum_systems_b200 import _native, ops

    case = large("cyclic-fill-216")
    m = case.extent
    lib = _native.load()
    wanted = torch.tensor([[bool(lib.qs_cyclic_pair_wanted(r, s, m)) for s in range(m)] for r in range(m)],
                          device="cuda")
    assert 0 < int(wanted.sum()) < m * m

    def computed(p0, p1, device):
        p, q, r, s = LO.axes(p0, p1, m, device)
        return torch.where(wanted, LO.coded(LO.lin4(p, q, r, s, m), F64), float("nan"))

    def filled(p0, p1, device):
        p, q, r, s = LO.axes(p0, p1, m, device)
        mirror = torch.where(r == s, 0.0, -LO.coded(LO.lin4(p, q, s, r, m), F64))
        return torch.where(wanted, LO.coded(LO.lin4(p, q, r, s, m), F64), mirror)

    out = LO.fill(torch.empty((m,) * 4, dtype=F64, device="cuda"), computed)
    _native.call("qs_cyclic_antisymmetric_fill", ops._ptr(out), ops._code(out), m, m, ops._stream())
    LO.assert_exact(out, filled, "cyclic fill", case.boundary)


def add_spin_expected(l, anti):
    n = 2 * l

    def planes(p0, p1, device):
        P_, Q, R, S = LO.axes(p0, p1, n, device)
        p, q, r, s = P_ >> 1, Q >> 1, R >> 1, S >> 1
        s1, s2, s3, s4 = P_ & 1, Q & 1, R & 1, S & 1
        out = LO.coded(LO.lin4(p, q, r, s, l), F64) * ((s1 == s3) & (s2 == s4))
        if anti:
            out = out - LO.coded(LO.lin4(p, q, s, r, l), F64) * ((s1 == s4) & (s2 == s3))
        return out

    return planes


@pytest.mark.parametrize("name,out_dtypes", [("add-spin-108", (F64, C128)), ("add-spin-129-real", (F64,))])
def test_add_spin_two_body(name, out_dtypes, poisoned_ops):
    ops = poisoned_ops
    case = large(name)
    l = case.extent
    u = LO.fill(torch.empty((l,) * 4, dtype=F64, device="cuda"),
                lambda p0, p1, device: LO.coded(LO.lin4(*LO.axes(p0, p1, l, device), l), F64))
    for out_dtype in out_dtypes:
        for anti in (False, True):
            out = ops.add_spin_two_body(u, anti_symmetrize=anti, out_dtype=out_dtype)
            LO.assert_exact(out, add_spin_expected(l, anti), f"{name} anti={anti} out {out_dtype}", case.boundary)
            del out
            torch.cuda.empty_cache()


@pytest.mark.parametrize("name,dtype", [("antisymmetrize-216-real", F64), ("antisymmetrize-216-complex", C128),
                                        ("antisymmetrize-257-real", F64)])
def test_anti_symmetrize(name, dtype, poisoned_ops):
    ops = poisoned_ops
    case = large(name)
    n = case.extent
    u = LO.fill(torch.empty((n,) * 4, dtype=dtype, device="cuda"),
                lambda p0, p1, device: LO.coded(LO.lin4(*LO.axes(p0, p1, n, device), n), dtype))
    out = ops.anti_symmetrize(u)
    del u
    LO.assert_exact(out, LO.antisymmetrized(n, dtype), name, case.boundary)


def spin_orbital_tables(l):
    """Spin-orbital ``I`` is orbital ``I // 2``; the spins of every third orbital are swapped, so the tables are
    not the plain interleaved order."""
    orbital = np.arange(2 * l) // 2
    spin = (np.arange(2 * l) % 2) ^ (orbital % 3 == 0)
    return orbital.astype(np.int64), spin.astype(np.int64)


def spin_orbital_expected(l, dtype, orbital, spin, derived):
    """``U[I,J,K,L] = [sI=sK][sJ=sL] b_{sI sJ}[oI,oJ,oK,oL] - [sI=sL][sJ=sK] b_{sI sJ}[oI,oJ,oL,oK]`` for the blocks
    hash-coded with salt ``2 sI + sJ``; a derived ``b_ba[i,j,k,l]`` is ``b_ab[j,i,l,k]``."""
    n = 2 * l

    def planes(p0, p1, device):
        orb, spn = (torch.from_numpy(t).to(device) for t in (orbital, spin))
        I, J, K, L = LO.axes(p0, p1, n, device)
        oI, oJ, oK, oL = orb[I], orb[J], orb[K], orb[L]
        sI, sJ, sK, sL = spn[I], spn[J], spn[K], spn[L]
        block = 2 * sI + sJ
        from_ab = (block == 2) & derived

        def value(a, b, c, d):
            lin = torch.where(from_ab, LO.lin4(b, a, d, c, l), LO.lin4(a, b, c, d, l))
            return LO.coded(lin, dtype, torch.where(from_ab, 1, block))

        zero = torch.zeros((), dtype=dtype, device=device)
        direct = torch.where((sI == sK) & (sJ == sL), value(oI, oJ, oK, oL), zero)
        return direct - torch.where((sI == sL) & (sJ == sK), value(oI, oJ, oL, oK), zero)

    return planes


@pytest.mark.parametrize("name,dtype", [("spin-orbital-108-real", F64), ("spin-orbital-128-complex", C128)])
def test_spin_orbital_two_body(name, dtype, poisoned_ops):
    """The DESIGN §4.12 assembly; at l = 128 complex128 its (2l)^4 result is 2**32 elements."""
    ops = poisoned_ops
    case = large(name)
    l = case.extent
    blocks = [LO.fill(torch.empty((l,) * 4, dtype=dtype, device="cuda"),
                      lambda p0, p1, device, salt=salt: LO.coded(LO.lin4(*LO.axes(p0, p1, l, device), l), dtype, salt))
              for salt in range(4)]
    orbital, spin = spin_orbital_tables(l)
    for derived in (False, True):
        out = ops.spin_orbital_two_body(blocks[0], blocks[1], None if derived else blocks[2], blocks[3], orbital, spin)
        assert ops.proven_symmetry(out) == ops.ANTISYMMETRIC_LAST_PAIR
        LO.assert_exact(out, spin_orbital_expected(l, dtype, orbital, spin, derived), f"{name} derived={derived}",
                        case.boundary, chunk_elems=2**25)
        del out
        torch.cuda.empty_cache()


def test_extract_block_from_the_last_planes():
    from quantum_systems_b200 import ops

    case = large("extract-block-216")
    n = case.extent
    u = LO.fill(torch.empty((n,) * 4, dtype=C128, device="cuda"),
                lambda p0, p1, device: LO.coded(LO.lin4(*LO.axes(p0, p1, n, device), n), C128))
    a, b, c, d = (n - 3, n), (0, n), (5, n), (1, n - 1)
    first = int(np.ravel_multi_index([lo for lo, _ in (a, b, c, d)], (n,) * 4))
    last = int(np.ravel_multi_index([hi - 1 for _, hi in (a, b, c, d)], (n,) * 4))
    assert first < case.boundary <= last, "the block does not span element offset 2**31"
    got = ops.extract_block(u, a, b, c, d)

    def want(p0, p1, device):
        p = torch.arange(a[0] + p0, a[0] + p1, device=device).view(-1, 1, 1, 1)
        q, r, s = (torch.arange(*rng_, device=device).view(shape)
                   for rng_, shape in ((b, (1, -1, 1, 1)), (c, (1, 1, -1, 1)), (d, (1, 1, 1, -1))))
        return LO.coded(LO.lin4(p, q, r, s, n), C128)

    assert tuple(got.shape) == (3, n, n - 5, n - 2)
    LO.assert_exact(got, want, "extract_block u[n-3:, :, 5:, 1:n-1]", None)


@pytest.mark.parametrize("name,dtype,alpha,beta,in_place", [
    ("scale-add-complex", C128, 0.5 - 0.25j, -1.5 + 0.75j, False),
    ("scale-add-real-odd", F64, -0.75, 0.5, True),
    ("scale-add-real-s32", F64, 0.5, -1.25, True),
])
def test_scale_add(name, dtype, alpha, beta, in_place, poisoned_ops):
    """``alpha x + beta y`` over more than 2**31 (2**32) elements with dyadic factors: exact for hash-coded x, y; an
    odd real count also runs the kernel's tail element."""
    ops = poisoned_ops
    case = large(name)
    count = case.extent
    assert count % 2 == 1

    def coded(salt):
        return lambda p0, p1, device: LO.coded(torch.arange(p0, p1, device=device), dtype, salt)

    x = LO.fill(torch.empty(count, dtype=dtype, device="cuda"), coded(0))
    y = LO.fill(torch.empty(count, dtype=dtype, device="cuda"), coded(1))
    out = ops.scale_add(x, alpha, y, beta, out=x if in_place else None)
    assert (out is x) == in_place
    del y
    LO.assert_exact(out, lambda p0, p1, device: alpha * coded(0)(p0, p1, device) + beta * coded(1)(p0, p1, device),
                    name, case.boundary)


# ------------------------------------------------------------------------------------------ Fock builds and traces


def kron_u(n, cplx, seed):
    rng = np.random.default_rng(seed)
    g = P.pow2_graded(n)
    A = P.dyadic(rng, (n, n), cplx) * np.outer(g, g)
    B = P.dyadic(rng, (n, n), cplx) * np.outer(g, g)
    return rng, A, B, kron_tensor(A, B, False, C128 if cplx else F64)  # u[p,r,q,s] = A[p,q] B[r,s]


@pytest.mark.parametrize("name,cplx", [("fock-density-216-real", False), ("fock-density-216-complex", True)])
def test_fock_from_density(name, cplx, poisoned_ops):
    ops = poisoned_ops
    case = large(name)
    n = case.extent
    rng, A, B, u = kron_u(n, cplx, n + cplx)
    h, rho, rho_b = rand(rng, (n, n), cplx) * 1e-6, rand(rng, (n, n), cplx), rand(rng, (n, n), cplx) * 1e-3
    k2, k3 = (t * n * n * (2 if cplx else 1) + 1 for t in (2, 3))
    got = ops.fock_from_density(dev(h), u, dev(rho), 1.0, -0.5).cpu().numpy()
    ref, absval, fp64 = P.companions(P.kron_fock_density, h, A, B, rho, a_d=1.0, a_x=-0.5)
    check(got, ref, absval, k2, fp64, f"{name} fock_from_density")
    got = np.stack([f.cpu().numpy() for f in ops.fock_from_density_unrestricted(dev(h), u, dev(rho), dev(rho_b))])
    ref, absval, fp64 = P.companions(P.kron_fock_unrestricted, h, A, B, rho, rho_b)
    check(got, ref, absval, k3, fp64, f"{name} fock_from_density_unrestricted")


def test_fock_occupied_and_traces():
    from quantum_systems_b200 import ops

    case = large("fock-occupied-216")
    n = case.extent
    rng, A, B, u = kron_u(n, False, 2160)
    h = rand(rng, (n, n)) * 1e-6
    hd = dev(h)
    for n_occ in (n - 1, n):  # plane p = n - 1 and i = n - 1 read past the boundary
        for spatial in (False, True):
            got = (ops.fock_spatial if spatial else ops.fock_general)(hd, u, n_occ).cpu().numpy()
            ref, absval, fp64 = P.companions(P.kron_fock_occupied, h, A, B, n_occ=n_occ, spatial=spatial)
            check(got, ref, absval, (2 if spatial else 1) * n_occ + 1, fp64, f"n_occ={n_occ} spatial={spatial}")
        got = ops.occupied_traces(hd, u, n_occ).cpu().numpy()
        assert np.all(got.imag == 0)
        ref, absval, fp64 = P.companions(P.kron_occupied_traces, h, A, B, n_occ=n_occ)
        check(got.real, ref, absval, n_occ * n_occ, fp64, f"occupied_traces n_occ={n_occ}")


# ------------------------------------------------------------------------------------------ structured transforms


def assert_written(out, what):
    """No element of the NaN-filled ``out`` is left NaN, checked plane chunk by plane chunk (``torch.isfinite`` of the
    whole tensor would hold a full-size temporary)."""
    step = max(1, LO.CHUNK_ELEMS // out[0].numel())
    for p0 in range(0, out.shape[0], step):
        assert not bool(out[p0 : p0 + step].isnan().any()), f"{what}: unwritten in planes [{p0}, {p0 + step})"


@pytest.mark.parametrize("anti", [False, True])
def test_diagonal_transform(anti, poisoned_ops):
    ops = poisoned_ops
    case = large("diagonal-216")
    n, m = LO.DIAGONAL_GRID, case.extent
    rng = np.random.default_rng(m + anti)
    W, C = rand(rng, (n, n)), rand(rng, (n, m))
    out = ops.transform_two_body_diagonal(dev(W), dev(C), anti_symmetrize=anti)
    assert_written(out, f"diagonal anti={anti}")
    k = P.k_diagonal(n, False, anti=anti)
    for p in (case.boundary // m**3, m - 1):
        ref, absval, fp64 = P.companions(P.diagonal_plane, W, C, C.T, p=p, anti=anti)
        check(out[p].cpu().numpy(), ref, absval, k, fp64, f"diagonal anti={anti} plane {p}")


def test_odqd_coulomb(poisoned_ops):
    from quantum_systems_b200.odqd import grid_orbitals
    from quantum_systems_b200.potentials import HOPotential

    case = large("odqd-216")
    l = case.extent
    grid, _, C = grid_orbitals(l, 10.0, LO.ODQD_GRID, HOPotential(0.25))
    inner = grid[1:-1]
    out = poisoned_ops.odqd_coulomb(dev(C), dev(inner), 1.0, 0.25)
    assert_written(out, "ODQD")
    rng = np.random.default_rng(l)
    rows = [(a, int(c)) for a in (case.boundary // l**3, l - 1) for c in (*rng.integers(0, l, 2), l - 1)]
    ref, absval, fp64 = P.companions(P.odqd_rows, C, grid=inner, alpha=1.0, a=0.25, rows=rows)
    got = np.stack([out[a, :, c, :].cpu().numpy() for a, c in rows])
    check(got, ref, absval, P.k_diagonal(LO.ODQD_GRID - 2, False, generated_w=True), fp64, f"ODQD rows {rows}")


# ------------------------------------------------------------------------------------------------- sharded, W = 1


def test_sharded_transform_and_consumers_on_one_rank():
    """``EmulatedContext(1)``: the single shard is the whole tensor, so the sharded schedule's addressing runs past
    2**31 on one GPU; every buffer the schedule allocates starts as NaN."""
    from quantum_systems_b200 import sharded

    case = large("sharded-216-one-rank")
    n = case.extent
    rng = np.random.default_rng(216216)
    A, B, C = P.dyadic(rng, (n, n)), P.dyadic(rng, (n, n)), rand(rng, (n, n))
    ctx = sharded.EmulatedContext(1, engine=SB.nan_engine()())
    u = SB.exact_sharded(ctx, A, B, False, F64, "cuda")
    assert u.local(0).numel() > case.boundary
    h = rand(rng, (n, n)) * 1e-6
    hd = dev(h)
    basis = sharded.ShardedBasisSet(ctx, n, hd, None, u)
    f = torch.full((n, n), float("nan"), dtype=F64, device="cuda")
    got = basis.construct_fock_matrix(hd, u, n, f=f).cpu().numpy()
    ref, absval, fp64 = P.companions(P.kron_fock_occupied, h, A, B, n_occ=n)
    check(got, ref, absval, n + 1, fp64, "sharded construct_fock_matrix")
    traces = np.array(u.occupied_traces(hd, n))
    ref, absval, fp64 = P.companions(P.kron_occupied_traces, h, A, B, n_occ=n)
    check(traces.real, ref, absval, n * n, fp64, "sharded occupied_traces")
    rho = rand(rng, (n, n))
    got = basis.fock_from_density(hd, dev(rho), 1.0, -0.5).cpu().numpy()
    ref, absval, fp64 = P.companions(P.kron_fock_density, h, A, B, rho, a_d=1.0, a_x=-0.5)
    check(got, ref, absval, 2 * n * n + 1, fp64, "sharded fock_from_density")
    del basis
    out = sharded.transform_two_body_sharded(u, dev(C), symmetry=0)
    del u
    arrays, k = (A, B, C, C.T), P.k_transform([n] * 4, [False] * 4)
    SB.check_planes(check, out, P.kron_factors, arrays, boundary_planes(n, case.boundary), k, False,
                    "sharded W=1", batch=2)
    SB.sweep_slabs([("rank 0", 0, out.local(0))], P.kron_factors, arrays, k, False, "sharded W=1",
                   boundary=case.boundary)
