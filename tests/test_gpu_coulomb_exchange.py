"""The batched Coulomb-exchange kernel (ops.coulomb_exchange, qs_coulomb_exchange_batch) against extended-precision
references under the rounding-error bound, its bit-identity properties (batch composition, position and width; uneven
shards), ragged n, poisoned buffers, refusals and a u past 2^31 elements."""

import ctypes

import numpy as np
import pytest

import precise as P

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import large_offsets as LO  # noqa: E402  (needs torch)

def inputs(n, k, seed=0, device="cuda"):
    g = torch.Generator(device="cpu").manual_seed(seed)
    u = torch.randn((n, n, n, n), generator=g, dtype=torch.float64)
    rho = torch.randn((k, n, n), generator=g, dtype=torch.float64)
    return u.to(device), rho.to(device)


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


# The contractions of the kernel in the calling convention of tests/precise.py (P.companions evaluates each in
# longdouble, as the FP64 absolute-value companion and in plain FP64).  Both return [J, K], shape (2, k, n, n).


def coulomb_exchange(u, rho, dt, absolute=False):
    """``J[d,p,q] = sum_rs u[p,r,q,s] rho[d,s,r]``, ``K[d,p,q] = sum_rs u[p,r,s,q] rho[d,s,r]``."""
    return np.stack([np.einsum("prqs,dsr->dpq", u, rho), np.einsum("prsq,dsr->dpq", u, rho)])


def kron_coulomb_exchange(A, B, rho, dt, absolute=False):
    """``coulomb_exchange`` of ``u[p,r,q,s] = A[p,q] B[r,s]``: ``J_d = A sum_rs B[r,s] rho_d[s,r]`` and
    ``K_d = A rho_d B``.  Products of non-negative inputs stay so: the absolute-value companion of this form is the
    exact ``|terms|`` of the dense sum."""
    J = A[None] * np.einsum("rs,dsr->d", B, rho)[:, None, None]
    return np.stack([J, np.matmul(np.matmul(A, rho), B)])


def k_eff(n):
    """Each element is a sum of ``n^2`` rounded products.  The kernel adds them in a tree (DMMA steps over s, the r of
    a chunk, the even and odd J halves, the chunk partials of pass 2), so no path holds more than ``n^2 - 1``
    additions: ``n^2 + 1`` rounded operations bound it, the count of the density Fock kernel."""
    return n * n + 1


def check(got, fn, arrays, n, what):
    ref, absval, fp64 = P.companions(fn, *arrays)
    got = np.stack([got[0].cpu().numpy(), got[1].cpu().numpy()])
    P.assert_rounding_bound(got, ref, absval, k_eff(n), fp64, what)


def graded_densities(rng, n, k):
    g = P.graded(n)
    return rng.standard_normal((k, n, n)) * np.outer(g, g)


def with_zero_terms(u, rho):
    """Plane 3 of ``u`` (when there is one) and the last density of a batch of two or more set to zero: every term of
    those J and K elements is zero, so they must come out exactly zero, whatever their neighbours hold."""
    if u.shape[0] > 3:
        u[3] = 0.0
    if rho.shape[0] > 1:
        rho[-1] = 0.0
    return u, rho


@pytest.mark.parametrize("family,n,k", [
    ("normal", 1, 1), ("normal", 7, 3), ("normal", 16, 16),
    ("graded", 7, 17), ("graded", 33, 16), ("graded", 48, 5),
    ("cancellation", 33, 4), ("cancellation", 40, 9),
])
def test_against_extended_precision(family, n, k):
    """Families (a) N(0, 1), (b) graded ``u`` (``P.graded_two_body``) and graded densities, (c) cancellation:
    ``u[p,r,q,s] = A[p,q] C^-1[r,s]`` and ``rho_0 = C`` with cond(C) = 1e3, so ``K_0 = A C C^-1`` and
    ``J_0 = A tr(C^-1 C)`` are sums whose terms are about cond(C) times the result."""
    from quantum_systems_b200 import ops

    rng = np.random.default_rng(1000 * n + k)
    if family == "normal":
        u, rho = rng.standard_normal((n,) * 4), rng.standard_normal((k, n, n))
    elif family == "graded":
        u, rho = with_zero_terms(P.graded_two_body(rng, n), graded_densities(rng, n, k))
    else:
        C, C_inv = P.conditioned(rng, n, 1e3)
        A = rng.standard_normal((n, n))
        u = np.einsum("pq,rs->prqs", A, C_inv)  # rounded in FP64; the reference contracts this very tensor
        rho = np.stack([C] + [C * rng.standard_normal(n) for _ in range(k - 1)])
    got = ops.coulomb_exchange(dev(u), dev(rho))
    check(got, coulomb_exchange, (u, rho), n, f"{family} n={n} k={k}")


@pytest.mark.parametrize("k", [1, 16, 17])
@pytest.mark.parametrize("n", [129, 130])
def test_structured_kron_input_at_n_over_48(n, k):
    """``u = A (x) B`` with dyadic, power-of-two graded factors (an exact FP64 tensor) past n = 48, whose reference is
    O(k n^3): k = 1, the widest launch and one past it (two launches), odd and even n (8- and 16-byte copies)."""
    from quantum_systems_b200 import ops

    rng = np.random.default_rng(n * 100 + k)
    g = P.pow2_graded(n)
    A = P.dyadic(rng, (n, n)) * np.outer(g, g)
    B = P.dyadic(rng, (n, n)) * np.outer(g, g)
    A[3] = 0.0  # row 3 of every J and K has only zero terms
    rho = graded_densities(rng, n, k)
    if k > 1:
        rho[-1] = 0.0
    Ad, Bd = dev(A), dev(B)
    u = (Ad[:, None, :, None] * Bd[None, :, None, :]).contiguous()  # u[p,r,q,s] = A[p,q] B[r,s], exact
    got = ops.coulomb_exchange(u, dev(rho))
    check(got, kron_coulomb_exchange, (A, B, rho), n, f"A(x)B n={n} k={k}")


def test_unaligned_even_n_takes_8_byte_copies():
    """Even n with ``u`` 8 bytes off a 16-byte boundary: the 8-byte copy path of an even row length, held to the
    bound and bit-identical to the 16-byte path (the copies move data; the arithmetic is the same)."""
    from quantum_systems_b200 import ops

    n, k = 64, 9
    rng = np.random.default_rng(64064)
    u, rho = with_zero_terms(P.graded_two_body(rng, n), graded_densities(rng, n, k))
    buf = torch.empty(n**4 + 1, dtype=torch.float64, device="cuda")
    ud = buf[1:].view(n, n, n, n)
    ud.copy_(dev(u))
    assert ud.data_ptr() % 16 == 8
    got = ops.coulomb_exchange(ud, dev(rho))
    check(got, coulomb_exchange, (u, rho), n, "unaligned u")
    aligned = ops.coulomb_exchange(dev(u), dev(rho))
    assert torch.equal(got[0], aligned[0]) and torch.equal(got[1], aligned[1])


def test_batch_composition_position_and_width_are_bit_identical():
    from quantum_systems_b200 import ops

    n = 40
    u, rho = inputs(n, 33, seed=3)
    J1, K1 = ops.coulomb_exchange(u, rho[5:6])
    for batch, pos in [(rho, 5), (rho[5:13], 0), (rho[:16], 5), (torch.flip(rho, [0]).contiguous(), 27),
                       (torch.cat([rho[7:9], rho[5:6]]).contiguous(), 2)]:
        J, K = ops.coulomb_exchange(u, batch)
        assert torch.equal(J[pos], J1[0]) and torch.equal(K[pos], K1[0])


@pytest.mark.parametrize("shards", [2, 3, 7])
def test_uneven_shards_are_bit_identical(shards):
    from quantum_systems_b200 import ops

    n, k = 45, 9
    u, rho = inputs(n, k, seed=shards)
    J, K = ops.coulomb_exchange(u, rho)
    cuts = np.unique(np.round(np.sqrt(np.linspace(0, 1, shards + 1)) * n).astype(int))
    Js = torch.full_like(J, float("nan"))
    Ks = torch.full_like(K, float("nan"))
    for p0, p1 in zip(cuts[:-1], cuts[1:]):
        ops.coulomb_exchange(u[p0:p1].contiguous(), rho, planes=(p0, p1), J=Js, K=Ks)
    assert torch.equal(Js, J) and torch.equal(Ks, K)


def test_new_outputs_are_zero_outside_the_planes_and_given_ones_untouched():
    from quantum_systems_b200 import ops

    n, k = 20, 4
    u, rho = inputs(n, k, seed=9)
    J, K = ops.coulomb_exchange(u, rho)
    Jp, Kp = ops.coulomb_exchange(u[3:11].contiguous(), rho, planes=(3, 11))
    assert torch.equal(Jp[:, 3:11], J[:, 3:11]) and torch.equal(Kp[:, 3:11], K[:, 3:11])
    assert not Jp[:, :3].any() and not Kp[:, 11:].any()
    Jn = torch.full_like(J, float("nan"))
    Kn = torch.full_like(K, float("nan"))
    ops.coulomb_exchange(u[3:11].contiguous(), rho, planes=(3, 11), J=Jn, K=Kn)
    assert torch.isnan(Jn[:, :3]).all() and torch.isnan(Kn[:, 11:]).all()
    assert torch.equal(Jn[:, 3:11], J[:, 3:11])


def test_poisoned_workspace_and_outputs():
    from quantum_systems_b200 import _native, ops

    n, k = 33, 16
    u, rho = inputs(n, k, seed=11)
    J, K = ops.coulomb_exchange(u, rho)
    nbytes = ctypes.c_int64(0)
    _native.call("qs_coulomb_exchange_batch_workspace_bytes", n, k, 0, n, 0, 0, ctypes.byref(nbytes))
    ws = torch.full((nbytes.value // 8,), float("nan"), dtype=torch.float64, device="cuda")
    Jn = torch.full_like(J, float("nan"))
    Kn = torch.full_like(K, float("nan"))
    _native.call("qs_coulomb_exchange_batch", ctypes.c_void_p(u.data_ptr()), 0, ctypes.c_void_p(rho.data_ptr()), 0,
                 n, k, ctypes.c_void_p(Jn.data_ptr()), ctypes.c_void_p(Kn.data_ptr()), 0, n,
                 ctypes.c_void_p(ws.data_ptr()), nbytes.value, ops._stream())
    assert torch.equal(Jn, J) and torch.equal(Kn, K)


def test_workspace_stays_below_a_tenth_of_u():
    from quantum_systems_b200 import _native

    for n in (100, 128, 200, 257, 380):
        nbytes = ctypes.c_int64(0)
        _native.call("qs_coulomb_exchange_batch_workspace_bytes", n, 16, 0, n, 0, 0, ctypes.byref(nbytes))
        assert 2 * nbytes.value < 0.1 * 8 * n ** 4  # written once, read once


def test_refusals():
    from quantum_systems_b200 import _native, ops

    n = 6
    u, rho = inputs(n, 2)
    with pytest.raises(RuntimeError, match="complex u or densities"):
        ops.coulomb_exchange(u.to(torch.complex128), rho)
    with pytest.raises(RuntimeError, match="complex u or densities"):
        ops.coulomb_exchange(u, rho.to(torch.complex128))
    with pytest.raises(ValueError):
        ops.coulomb_exchange(u, rho[0])
    with pytest.raises(ValueError):
        ops.coulomb_exchange(u[:3].contiguous(), rho)
    with pytest.raises(ValueError):
        ops.coulomb_exchange(u, rho, planes=(2, 9))
    with pytest.raises(ValueError):
        ops.coulomb_exchange(u, rho, J=torch.empty((1, n, n), dtype=torch.float64, device="cuda"))
    J = torch.empty((17, n, n), dtype=torch.float64, device="cuda")
    big = torch.zeros((17, n, n), dtype=torch.float64, device="cuda")
    ws = torch.empty(1 << 20, dtype=torch.uint8, device="cuda")
    p = ctypes.c_void_p
    with pytest.raises(RuntimeError, match="at most 16"):
        _native.call("qs_coulomb_exchange_batch", p(u.data_ptr()), 0, p(big.data_ptr()), 0, n, 17, p(J.data_ptr()),
                     p(J.data_ptr()), 0, n, p(ws.data_ptr()), 1 << 20, ops._stream())
    with pytest.raises(RuntimeError, match="workspace too small"):
        _native.call("qs_coulomb_exchange_batch", p(u.data_ptr()), 0, p(big.data_ptr()), 0, n, 2, p(J.data_ptr()),
                     p(J.data_ptr()), 0, n, p(ws.data_ptr()), 8, ops._stream())
    with pytest.raises(RuntimeError, match="exceeds 384"):
        _native.call("qs_coulomb_exchange_batch", p(u.data_ptr()), 0, p(big.data_ptr()), 0, 385, 2, p(J.data_ptr()),
                     p(J.data_ptr()), 0, 385, p(ws.data_ptr()), 1 << 20, ops._stream())


def test_u_past_two_to_the_31_elements():
    """``LARGE``: n = 216, the smallest extent whose u passes 2^31 elements (17.4 GB), built exactly as A (x) B and
    skipped with its numbers when the plan does not fit.  Every element of J and K, including the rows of the planes
    past the boundary, is held to the rounding bound; the last two planes computed as a shard are bit-identical."""
    from quantum_systems_b200 import ops

    n = large_case()
    rng = np.random.default_rng(216)
    g = P.pow2_graded(n)
    A = P.dyadic(rng, (n, n)) * np.outer(g, g)
    B = P.dyadic(rng, (n, n)) * np.outer(g, g)
    rho = graded_densities(rng, n, LARGE_K)
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    Ad, Bd = dev(A), dev(B)
    u = (Ad[:, None, :, None] * Bd[None, :, None, :]).contiguous()
    assert u.numel() > LO.S31
    rho_d = dev(rho)
    got = ops.coulomb_exchange(u, rho_d)
    check(got, kron_coulomb_exchange, (A, B, rho), n, "n=216 past 2^31")
    J, K = ops.coulomb_exchange(u[n - 2:], rho_d, planes=(n - 2, n))
    assert torch.equal(J[:, n - 2:], got[0][:, n - 2:]) and torch.equal(K[:, n - 2:], got[1][:, n - 2:])
    peak = torch.cuda.max_memory_allocated() - base
    del u
    torch.cuda.empty_cache()
    assert peak <= LARGE.nbytes(n), f"peak {peak / 1e9:.1f} GB above the plan {LARGE.nbytes(n) / 1e9:.1f} GB"


LARGE_K = 3
# the case in the form of tests/large_offsets.py: boundary, extent, largest element offset, planned peak bytes
LARGE = LO.Case(LO.S31, 216, lambda n: n**4 - 1, lambda n: n**4 * 8 + LO._bytes(
    "qs_coulomb_exchange_batch_workspace_bytes", n, LARGE_K, 0, n, 0, 0) + 1024 + LO.SCRATCH, True)


def large_case():
    """The extent of ``LARGE``, its claim asserted; skipped with the numbers when the plan does not fit."""
    assert LARGE.offset(LARGE.extent) >= LARGE.boundary
    planned = LARGE.nbytes(LARGE.extent)
    free, total = torch.cuda.mem_get_info()
    if planned > LO.BUDGET or planned > free:
        pytest.skip(f"coulomb-exchange-216: planned peak {planned / 1e9:.1f} GB; budget {LO.BUDGET / 1e9:.0f} GB, "
                    f"free {free / 1e9:.1f} of {total / 1e9:.1f} GB")
    return LARGE.extent
