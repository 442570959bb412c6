"""The rounding-error check of tests/precise.py checks itself: its extended-precision references against exact
rational arithmetic, a correct FP64 evaluation in another order passes it on every input family the GPU file uses,
and kernels that are subtly wrong fail it -- including two that the 1e-12 max-scaled check accepts."""

import itertools
from fractions import Fraction

import numpy as np
import pytest
import scipy.linalg

import precise as P
from conftest import assert_close_scaled


def exact(x):
    return np.vectorize(Fraction, otypes=[object])(np.asarray(x, dtype=np.float64))


def assert_pinned(ref, exact_value, absval, k):
    """The longdouble reference is within a few longdouble roundings of the exact value (and so far below the
    FP64 bound): ``|ref - exact| <= gamma_ld(k) |terms|``."""
    eps_ld = Fraction(2) ** -(np.finfo(np.longdouble).nmant + 1)
    for idx in itertools.product(*(range(s) for s in ref.shape)):
        err = abs(Fraction(*np.longdouble(ref[idx]).as_integer_ratio()) - exact_value[idx])
        assert err <= 2 * k * eps_ld * Fraction(float(absval[idx])) * (1 + Fraction(1, 10**6)), idx


@pytest.mark.parametrize("n", [2, 3])
def test_transform_reference_is_exact_to_longdouble(n):
    rng = np.random.default_rng(n)
    u, C, Ct = rng.standard_normal((n,) * 4), rng.standard_normal((n, n)), rng.standard_normal((n, n))
    ref, absval, _ = P.companions(P.quarter_steps, u, C, Ct)
    eu, eC, eCt = exact(u), exact(C), exact(Ct)
    want = np.empty((n,) * 4, dtype=object)
    for p, q, r, s in itertools.product(range(n), repeat=4):
        want[p, q, r, s] = sum(eCt[p, a] * eCt[q, b] * eu[a, b, c, d] * eC[c, r] * eC[d, s]
                               for a, b, c, d in itertools.product(range(n), repeat=4))
    assert_pinned(ref, want, absval, P.k_transform([n] * 4, [False] * 4))


@pytest.mark.parametrize("n", [2, 3])
def test_fock_density_reference_is_exact_to_longdouble(n):
    rng = np.random.default_rng(10 + n)
    h, u, rho = rng.standard_normal((n, n)), rng.standard_normal((n,) * 4), rng.standard_normal((n, n))
    ref, absval, _ = P.companions(P.fock_density, h, u, rho, a_d=1.0, a_x=-0.5)
    eh, eu, er = exact(h), exact(u), exact(rho)
    want = np.empty((n, n), dtype=object)
    for p, q in itertools.product(range(n), repeat=2):
        want[p, q] = eh[p, q] + sum(eu[p, r, q, s] * er[s, r] - Fraction(1, 2) * eu[p, r, s, q] * er[s, r]
                                    for r, s in itertools.product(range(n), repeat=2))
    assert_pinned(ref, want, absval, 2 * n * n + 1)


@pytest.mark.parametrize("n,m", [(3, 2), (2, 3)])
def test_diagonal_reference_is_exact_to_longdouble(n, m):
    rng = np.random.default_rng(20 + n)
    W, C, Ct = rng.standard_normal((n, n)), rng.standard_normal((n, m)), rng.standard_normal((m, n))
    ref, absval, _ = P.companions(P.diagonal_rows, W, C, Ct)
    eW, eC, eCt = exact(W), exact(C), exact(Ct)
    want = np.empty((m,) * 4, dtype=object)
    for p, q, r, s in itertools.product(range(m), repeat=4):
        want[p, q, r, s] = sum(eCt[p, a] * eC[a, r] * eCt[q, b] * eC[b, s] * eW[a, b]
                               for a, b in itertools.product(range(n), repeat=2))
    assert_pinned(ref, want, absval, P.k_diagonal(n, False))
    # the ODQD form is the same contraction with C~ = C^T and the generated W
    grid = np.linspace(-2.0, 2.0, n)
    got = P.odqd_rows(P.cast(C, P.LD), P.LD, grid=grid, alpha=1.0, a=0.25)
    W_ld = P.shielded_coulomb(grid, 1.0, 0.25, P.LD)
    np.testing.assert_array_equal(got, P.diagonal_rows(W_ld, P.cast(C, P.LD), P.cast(C, P.LD).T, P.LD))
    # one plane at a time, plain and anti-symmetrised, with its absolute-value companion
    for anti in (False, True):
        whole, whole_abs, _ = P.companions(P.diagonal_rows, W, C, Ct, anti=anti)
        for p in range(m):
            plane, plane_abs, _ = P.companions(P.diagonal_plane, W, C, Ct, p=p, anti=anti)
            np.testing.assert_array_equal(plane, whole[p])
            np.testing.assert_array_equal(plane_abs, whole_abs[p])


def test_kron_forms_match_the_dense_contractions():
    rng = np.random.default_rng(5)
    n, m = 5, 4
    A, B = P.dyadic(rng, (n, n), True), P.dyadic(rng, (n, n))
    C, Ct = rng.standard_normal((n, m)), rng.standard_normal((m, n)) + 1j * rng.standard_normal((m, n))
    for anti in (False, True):
        u = P.kron_two_body(A, B, anti)
        dense, dense_abs, _ = P.companions(P.quarter_steps, u, C, Ct)
        planes = [0, m - 1]
        ref, absval, _ = P.companions(P.kron_transform_planes, A, B, C, Ct, planes=planes, anti=anti)
        assert np.max(np.abs(ref - dense[planes])) <= 1e-17 * np.max(dense_abs)
        if anti:
            assert np.all(absval >= dense_abs[planes] * (1 - 1e-12))
        else:
            np.testing.assert_allclose(absval, dense_abs[planes], rtol=1e-13)
    h, rho = rng.standard_normal((n, n)), rng.standard_normal((n, n))
    A = P.dyadic(rng, (n, n))
    u = np.einsum("pq,rs->prqs", A, B)
    n_occ = 3
    for anti in (False, True):
        dense, dense_abs, _ = P.companions(P.fock_occupied, h, P.kron_two_body(A, B, anti), n_occ=n_occ, spatial=False)
        ref, absval, _ = P.companions(P.kron_fock_occupied, h, A, B, n_occ=n_occ, anti=anti)
        assert np.max(np.abs(ref - dense)) <= 1e-17 * np.max(dense_abs)
        assert np.all(absval >= dense_abs * (1 - 1e-12))
    dense, dense_abs, _ = P.companions(P.fock_occupied, h, P.kron_two_body(A, B), n_occ=n_occ, spatial=True)
    ref, absval, _ = P.companions(P.kron_fock_occupied, h, A, B, n_occ=n_occ, spatial=True)
    assert np.max(np.abs(ref - dense)) <= 1e-17 * np.max(dense_abs)
    assert np.all(absval >= dense_abs * (1 - 1e-12))
    dense, dense_abs, _ = P.companions(P.occupied_traces, h, P.kron_two_body(A, B), n_occ=n_occ)
    ref, absval, _ = P.companions(P.kron_occupied_traces, h, A, B, n_occ=n_occ)
    assert np.max(np.abs(ref - dense)) <= 1e-17 * np.max(dense_abs)
    np.testing.assert_allclose(absval, dense_abs, rtol=1e-13)
    rb = rng.standard_normal((n, n))
    dense, dense_abs, _ = P.companions(P.fock_unrestricted, h, u, rho, rb)
    ref, absval, _ = P.companions(P.kron_fock_unrestricted, h, A, B, rho, rb)
    assert np.max(np.abs(ref - dense)) <= 1e-17 * np.max(dense_abs)
    np.testing.assert_allclose(absval, dense_abs, rtol=1e-13)
    dense, dense_abs, _ = P.companions(P.fock_density, h, u, rho, a_d=1.0, a_x=-0.5)
    ref, absval, _ = P.companions(P.kron_fock_density, h, A, B, rho, a_d=1.0, a_x=-0.5)
    assert np.max(np.abs(ref - dense)) <= 1e-17 * np.max(dense_abs)
    np.testing.assert_allclose(absval, dense_abs, rtol=1e-13)


def test_kron_forms_with_one_matrix_per_index_and_chained_match_the_dense_contractions():
    from sharded_bounds import chain_factors, kron_planes_of

    rng = np.random.default_rng(6)
    n, m = 5, 4
    A, B = P.dyadic(rng, (n, n), True), P.dyadic(rng, (n, n))
    C_r, C_s = rng.standard_normal((n, m)), rng.standard_normal((n, m)) + 1j * rng.standard_normal((n, m))
    Ct_p, Ct_q = rng.standard_normal((m, n)) + 1j * rng.standard_normal((m, n)), rng.standard_normal((m, n))
    planes = [0, m - 1]
    for anti in (False, True):
        dense, dense_abs, _ = P.companions(P.mixed_steps, P.kron_two_body(A, B, anti), C_r, C_s, Ct_p, Ct_q)
        ref, absval, _ = P.companions(P.kron_transform_planes, A, B, C_r, Ct_p, C_s, Ct_q, planes=planes, anti=anti)
        assert np.max(np.abs(ref - dense[planes])) <= 1e-17 * np.max(dense_abs)
        if anti:
            assert np.all(absval >= dense_abs[planes] * (1 - 1e-12))
        else:
            np.testing.assert_allclose(absval, dense_abs[planes], rtol=1e-13)
    # with the defaults it is the one-matrix form
    one = P.companions(P.kron_transform_planes, A, B, C_r, Ct_p, planes=planes, anti=True)
    both = P.companions(P.kron_transform_planes, A, B, C_r, Ct_p, C_r, Ct_p, planes=planes, anti=True)
    for x, y in zip(one, both):
        np.testing.assert_array_equal(x, y)
    # two transforms in a row: the eight-step composite, its absolute-value companion built from |C1| and |C2|
    C1, Ct1 = rng.standard_normal((n, n)), rng.standard_normal((n, n))
    C2 = rng.standard_normal((n, m)) + 1j * rng.standard_normal((n, m))
    Ct2 = C2.conj().T

    def eight_steps(u, C1, Ct1, C2, Ct2, dt, absolute=False):
        return P.quarter_steps(P.quarter_steps(u, C1, Ct1, dt), C2, Ct2, dt)

    for anti in (False, True):
        dense, dense_abs, _ = P.companions(eight_steps, P.kron_two_body(A, B, anti), C1, Ct1, C2, Ct2)
        ref, absval, _ = P.companions(kron_planes_of(chain_factors), A, B, C1, Ct1, C2, Ct2, planes=planes, anti=anti)
        assert np.max(np.abs(ref - dense[planes])) <= 1e-16 * np.max(dense_abs)
        if anti:
            assert np.all(absval >= dense_abs[planes] * (1 - 1e-12))
        else:
            np.testing.assert_allclose(absval, dense_abs[planes], rtol=1e-13)


# ------------------------------------------------------------------ a correct FP64 evaluation passes on every family


def einsum_transform(u, C, Ct):
    """The four-index transform in FP64 through BLAS in numpy's own order -- not the kernels' order."""
    return np.einsum("pa,qb,abcd,cr,ds->pqrs", Ct, Ct, u, C, C, optimize=True)


def transform_families(n):
    rng = np.random.default_rng(n)
    a = rng.standard_normal((n,) * 4)
    Q = np.linalg.qr(rng.standard_normal((n, n)))[0]
    yield "a, real", a, Q, Q.T, False
    ac = a + 1j * rng.standard_normal((n,) * 4)
    Cc = rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n))
    yield "a, complex", ac, Cc, Cc.conj().T, True
    Cn = P.near_identity(rng, n)
    yield "b, near-identity C", P.graded_two_body(rng, n), Cn, Cn.T, False
    C, Ci = P.conditioned(rng, n)
    yield "c, bi-orthogonal", a, C, Ci, False


@pytest.mark.parametrize("n", [7, 16])
def test_fp64_in_another_order_passes_on_every_transform_family(n):
    for name, u, C, Ct, cplx in transform_families(n):
        ref, absval, fp64 = P.companions(P.quarter_steps, u, C, Ct)
        P.assert_rounding_bound(einsum_transform(u, C, Ct), ref, absval, P.k_transform([n] * 4, [cplx] * 4),
                                fp64, name)


def test_fp64_passes_the_round_trip_and_the_other_families():
    rng = np.random.default_rng(3)
    n = 10
    u = P.graded_two_body(rng, n)
    C, Ci = P.conditioned(rng, n)

    def round_trip(u, C, Ci, Ci2, C2, dt, absolute=False):
        return P.quarter_steps(P.quarter_steps(u, C, Ci, dt), Ci2, C2, dt)

    ref, absval, fp64 = P.companions(round_trip, u, C, Ci, Ci, C)
    got = einsum_transform(einsum_transform(u, C, Ci), Ci, C)
    P.assert_rounding_bound(got, ref, absval, P.k_transform([n] * 8, [False] * 8), fp64, "round trip")
    assert np.max(np.abs(got - u)) > 1e-14 * np.max(np.abs(u))  # the round trip does cancel: cond(C) = 1e3

    # (d) ODQD grid elements
    l, G = 6, 101
    grid = np.linspace(-6.0, 6.0, G)
    inner = grid[1:-1]
    dx = grid[1] - grid[0]
    _, Cg = scipy.linalg.eigh_tridiagonal(1.0 / dx**2 + 0.5 * inner**2, -np.ones(G - 3) / (2 * dx**2),
                                          select="i", select_range=(0, l - 1))
    ref, absval, fp64 = P.companions(P.odqd_rows, Cg, grid=inner, alpha=1.0, a=0.25)
    W = 1.0 / np.sqrt((inner[:, None] - inner[None, :]) ** 2 + 0.25**2)
    got = np.einsum("pa,qb,pc,qd,pq->abcd", Cg, Cg, Cg, Cg, W, optimize=True)
    P.assert_rounding_bound(got, ref, absval, P.k_diagonal(G - 2, False, generated_w=True), fp64, "ODQD")

    # density Fock, restricted and unrestricted, on graded densities
    n = 9
    g = P.graded(n)
    h, u = rng.standard_normal((n, n)), P.graded_two_body(rng, n, complex_=True)
    ra, rb = np.outer(g, g) * rng.standard_normal((n, n)), 1e-6 * np.outer(g, g) * rng.standard_normal((n, n))
    ref, absval, fp64 = P.companions(P.fock_density, h, u, ra, a_d=1.0, a_x=-0.5)
    got = h + np.einsum("prqs,rs->pq", u, ra.T) - 0.5 * np.einsum("prsq,sr->pq", u, ra)
    P.assert_rounding_bound(got, ref, absval, 2 * n * n + 1, fp64, "density Fock")
    ref, absval, fp64 = P.companions(P.fock_unrestricted, h, u, ra, rb)
    j = np.einsum("prqs,sr->pq", u, ra + rb)
    got = np.stack([h + j - np.einsum("prsq,sr->pq", u, r) for r in (ra, rb)])
    P.assert_rounding_bound(got, ref, absval, 3 * n * n + 1, fp64, "unrestricted Fock")


# ------------------------------------------------------------------------------------------- mutants are rejected


def steps_dropping_last_chunk(u, C, Ct, rows=128, chunk=16):
    """FP64 quarter steps in which step 1 skips the last k-chunk of the first row tile (a stale or skipped stage)."""
    n = u.shape[0]
    A = u.reshape(-1, n).copy()
    A[:rows, chunk * ((n - 1) // chunk):] = 0.0
    t = np.ascontiguousarray(np.moveaxis((A @ C).reshape(n, n, n, -1), 3, 0))
    for M in (C, Ct.T, Ct.T):
        t = np.ascontiguousarray(np.moveaxis(np.tensordot(t, M, ([3], [0])), 3, 0))
    return t


def rejected(got, ref, absval, k, fp64):
    with pytest.raises(AssertionError, match="criterion"):
        P.assert_rounding_bound(got, ref, absval, k, fp64, "mutant")


def test_mutants_fail_the_check_and_the_first_two_pass_the_scaled_one():
    rng = np.random.default_rng(24)
    n = 24
    u = P.graded_two_body(rng, n, lo=-3.0)
    C = P.near_identity(rng, n)
    ref, absval, fp64 = P.companions(P.quarter_steps, u, C, C.T)
    k = P.k_transform([n] * 4, [False] * 4)
    P.assert_rounding_bound(fp64, ref, absval, k, fp64, "FP64 itself")
    want = np.asarray(ref, dtype=np.float64)

    # 1. operands rounded to 46-bit mantissas
    m46 = P.quarter_steps(P.chop(u, 46), P.chop(C, 46), P.chop(C.T, 46), np.float64)
    assert_close_scaled(m46, want)
    rejected(m46, ref, absval, k, fp64)
    # 2. one input term dropped
    u2 = u.copy()
    u2[n - 1, n - 1, n - 1, n - 1] = 0.0
    dropped = P.quarter_steps(u2, C, C.T, np.float64)
    assert_close_scaled(dropped, want)
    rejected(dropped, ref, absval, k, fp64)
    # 3. the last k-chunk of one row tile skipped in step 1 (K = 24: chunk [16, 24) of rows 0..127)
    rejected(steps_dropping_last_chunk(u, C, C.T), ref, absval, k, fp64)
    # 4. two tail elements of the graded output swapped
    swapped = fp64.copy()
    swapped[n - 1, n - 1, n - 2, n - 1], swapped[n - 1, n - 1, n - 1, n - 2] = (
        fp64[n - 1, n - 1, n - 1, n - 2], fp64[n - 1, n - 1, n - 2, n - 1])
    rejected(swapped, ref, absval, k, fp64)

    # 5. one sign flip in an anti-symmetric pair of the anti-symmetrised diagonal transform
    m = 12
    W = np.outer(P.graded(m), P.graded(m)) * rng.standard_normal((m, m))
    Cd = P.near_identity(rng, m, complex_=True)
    ref, absval, fp64 = P.companions(P.diagonal_rows, W, Cd, Cd.conj().T, anti=True)
    flipped = fp64.copy()
    flipped[m - 1, m - 2, m - 3, m - 1] = -flipped[m - 1, m - 2, m - 3, m - 1]
    rejected(flipped, ref, absval, P.k_diagonal(m, True, anti=True), fp64)

    # 6. one exchange term of the density Fock matrix evaluated in float32
    n = 12
    h, uf, rho = rng.standard_normal((n, n)), P.graded_two_body(rng, n), rng.standard_normal((n, n))
    ref, absval, fp64 = P.companions(P.fock_density, h, uf, rho, a_d=1.0, a_x=-0.5)
    bad = fp64.copy()
    p, q = 0, 1  # a leading element: the float32 error is far above the FP64 rounding of its terms
    x32 = np.einsum("rs,sr->", uf[p, :, :, q].astype(np.float32), rho.astype(np.float32)).astype(np.float64)
    bad[p, q] = h[p, q] + np.einsum("rs,sr->", uf[p, :, q, :], rho) - 0.5 * x32
    rejected(bad, ref, absval, 2 * n * n + 1, fp64)


def test_zero_terms_must_give_exact_zeros_and_the_message_names_the_worst_element():
    ref = np.zeros((2, 3), dtype=np.longdouble)
    absval = np.zeros((2, 3))
    absval[0] = 1.0
    got = np.zeros((2, 3))
    got[1, 2] = 1e-300
    with pytest.raises(AssertionError, match=r"element \(1, 2\).*exactly zero"):
        P.assert_rounding_bound(got, ref, absval, 4, got * 0)
    got = np.zeros((2, 3))
    got[0, 1] = 1e-10
    with pytest.raises(AssertionError, match=r"criterion A.*worst element \(0, 1\)"):
        P.assert_rounding_bound(got, ref, absval, 4, got * 0)
