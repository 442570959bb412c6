"""Extended-precision references of the library's FP64 contractions, and the rounding-error bound a kernel's result
is held to (DESIGN §2, "rounding-error bound").  Plain numpy, no torch.

Every contraction below is written once and evaluated three ways by ``companions``:

* in ``np.longdouble`` (64-bit mantissa on x86, 113 on aarch64): the reference, 2^-11 of FP64's rounding error or
  better, so what remains of ``got - ref`` is the kernel's own error;
* in FP64 on the absolute values of the inputs (complex moduli, every subtraction turned into an addition): the
  "absolute-value companion" ``|terms|``, the scale of the rounding error of each element.  It has no cancellation,
  so FP64 is accurate enough for it;
* in plain FP64 on the inputs: what a correct FP64 evaluation of the same sums achieves, which calibrates criterion B.

``assert_rounding_bound`` then checks each element against the classical bound of a floating-point sum of products
(criterion A) and the mean error against the plain FP64 evaluation (criterion B).
"""

import numpy as np
import pytest

if np.finfo(np.longdouble).nmant < 63:
    pytest.skip(
        f"np.longdouble has a {np.finfo(np.longdouble).nmant}-bit mantissa on this platform; the extended-precision "
        "references need at least 63 bits (x86 extended or IEEE quad)",
        allow_module_level=True,
    )

LD = np.longdouble
F64 = np.float64
U = 2.0**-53  # unit roundoff of FP64


def gamma(k):
    """``k u / (1 - k u)``: relative error bound of a sum of ``k`` rounded operations (Higham, Lemma 3.1)."""
    return k * U / (1.0 - k * U)


def cast(x, dt):
    """``x`` in precision ``dt`` (``np.longdouble`` or ``np.float64``), complex staying complex."""
    x = np.asarray(x)
    if np.iscomplexobj(x):
        return x.astype(np.clongdouble if dt is LD else np.complex128)
    return x.astype(dt)


def _sub(a, b, absolute):
    return a + b if absolute else a - b


# ----------------------------------------------------------------------------------------------- the contractions
# Each takes its inputs already in precision `dt` and `absolute` (True: the absolute-value companion).


def quarter_steps(u, C, Ct, dt, absolute=False):
    """Four-index transform in the kernels' order (DESIGN §4.1): contract s, r with ``C``, then q, p with ``C̃ᵀ``;
    every step puts the new index first, ``u[a,b,c,d] -> T1[s,a,b,c] -> T2[r,s,a,b] -> T3[q,r,s,a] -> u'[p,q,r,s]``.
    ``u`` may be a slab of leading planes only when ``Ct`` is cut to the matching columns."""
    t = u
    for M in (C, C, Ct.T, Ct.T):
        t = np.ascontiguousarray(np.moveaxis(np.tensordot(t, M, ([3], [0])), 3, 0))
    return t


def one_body(h, C, Ct, dt, absolute=False):
    """``C̃ (h C)``: two steps."""
    return Ct @ (h @ C)


def mixed_steps(u, C_r, C_s, Ct_p, Ct_q, dt, absolute=False):
    """The kernels' order with one matrix per step: s with ``C_s``, r with ``C_r``, q with ``Ct_qᵀ``, p with
    ``Ct_pᵀ``, the new index first every time."""
    t = u
    for M in (C_s, C_r, Ct_q.T, Ct_p.T):
        t = np.ascontiguousarray(np.moveaxis(np.tensordot(t, M, ([3], [0])), 3, 0))
    return t


def kron_factors(A, B, C, Ct, C_s=None, Ct_q=None, dt=None, absolute=False):
    """The two-index factors of the transform of ``u[a,b,c,d] = A[a,c] B[b,d]`` with one matrix per index, in the
    convention of ``mixed_steps`` (``C`` is ``C_r``, ``Ct`` is ``Ct_p``; ``C_s`` and ``Ct_q`` default to them):
    ``X = C̃_p A C_r``, ``Y = C̃_q B C_s`` and, for the exchanged term of the anti-symmetric tensor,
    ``X' = C̃_p A C_s``, ``Y' = C̃_q B C_r``.  Products of non-negative inputs stay so: the same form gives the
    factors of the absolute-value companion."""
    C_s = C if C_s is None else C_s
    Ct_q = Ct if Ct_q is None else Ct_q
    return Ct @ (A @ C), Ct_q @ (B @ C_s), Ct @ (A @ C_s), Ct_q @ (B @ C)


def kron_planes(factors, planes, anti=False, absolute=False):
    """Planes ``u'[p] = X[p,r] Y[q,s] (- X'[p,s] Y'[q,r])`` from the ``kron_factors`` ``(X, Y, X', Y')``."""
    X, Y, Xx, Yx = factors
    planes = list(planes)
    out = X[planes][:, None, :, None] * Y[None, :, None, :]
    if anti:
        out = _sub(out, Xx[planes][:, None, None, :] * Yx[None, :, :, None], absolute)
    return out


def kron_transform_planes(A, B, C, Ct, C_s=None, Ct_q=None, planes=(), dt=None, anti=False, absolute=False):
    """Planes ``u'[p]`` (``p`` in ``planes``) of the four-index transform of ``u[a,b,c,d] = A[a,c] B[b,d]``
    (minus ``A[a,d] B[b,c]`` when ``anti``): ``u'[p,q,r,s] = X[p,r] Y[q,s] (- X'[p,s] Y'[q,r])`` with the
    ``kron_factors`` ``X = C̃ A C``, ``Y = C̃ B C`` (``C̃_q B C_s`` with one matrix per index).  O(n³) per plane;
    the absolute-value companion of this form is the exact ``|terms|`` of the dense transform when ``anti`` is
    off and an upper bound of it when on."""
    return kron_planes(kron_factors(A, B, C, Ct, C_s, Ct_q), planes, anti, absolute)


def diagonal_rows(W, C, Ct, dt, rows=None, anti=False, absolute=False):
    """Two-GEMM transform of a diagonal two-body operator (DESIGN §4.4): ``D[(p,r),a] = C̃[p,a] C[a,r]``,
    ``T = D W``, ``u'[p,q,r,s] = sum_b T[(p,r),b] D[(q,s),b]``.  ``rows=None``: the whole ``(m,m,m,m)`` result
    ``u'[p,q,r,s]``; else a list of ``(p, r)`` pairs and the result ``[k, q, s] = u'[p_k, q, r_k, s]``."""
    n, m = C.shape
    D = (Ct[:, None, :] * C.T[None, :, :]).reshape(m * m, n)  # [(p, r), a]
    sel = np.arange(m * m) if rows is None else np.array([p * m + r for p, r in rows])
    out = ((D[sel] @ W) @ D.T).reshape(len(sel), m, m)  # [(p, r), q, s]
    if rows is None:
        out = out.reshape(m, m, m, m).transpose(0, 2, 1, 3)  # [p, r, q, s] -> [p, q, r, s]
        if anti:
            out = _sub(out, out.transpose(0, 1, 3, 2), absolute)
    elif anti:
        raise ValueError("the anti-symmetrised form needs the whole result")
    return np.ascontiguousarray(out)


def diagonal_plane(W, C, Ct, dt, p, anti=False, absolute=False):
    """Plane ``u'[p]`` of ``diagonal_rows`` (minus its ``r <-> s`` exchange when ``anti``) from the ``m`` rows
    ``(p, r)``: O(m n² + m³) instead of the whole result."""
    m = C.shape[1]
    R = diagonal_rows(W, C, Ct, dt, rows=[(p, r) for r in range(m)])  # [r, q, s] = u'[p, q, r, s]
    plane = R.transpose(1, 0, 2)
    return _sub(plane, R.transpose(1, 2, 0), absolute) if anti else np.ascontiguousarray(plane)


def shielded_coulomb(grid, alpha, a, dt):
    """``W[p,q] = alpha / sqrt((x_p - x_q)^2 + a^2)`` (reference one_dim_qd.py:29-32) in precision ``dt``."""
    grid = cast(grid, dt)
    dx = grid[:, None] - grid[None, :]
    return dt(alpha) / np.sqrt(dx * dx + dt(a) * dt(a))


def odqd_rows(C, dt, grid, alpha, a, rows=None, absolute=False):
    """ODQD grid Coulomb elements ``u[a,b,c,d] = sum_pq C_pa C_qb C_pc C_qd W_pq``: the diagonal transform with
    ``C̃ = Cᵀ`` and the generated ``W`` (positive, so the same in the absolute-value companion); ``rows`` as in
    ``diagonal_rows`` (pairs ``(a, c)``)."""
    return diagonal_rows(shielded_coulomb(grid, alpha, a, dt), C, C.T, dt, rows=rows)


def fock_density(h, u, rho, a_d, a_x, dt, absolute=False):
    """``h + a_d sum_rs u[p,r,q,s] rho[s,r] + a_x sum_rs u[p,r,s,q] rho[s,r]`` (the scales are exact)."""
    a_d, a_x = (abs(a_d), abs(a_x)) if absolute else (a_d, a_x)
    return h + a_d * np.einsum("prqs,sr->pq", u, rho) + a_x * np.einsum("prsq,sr->pq", u, rho)


def fock_unrestricted(h, u, rho_a, rho_b, dt, absolute=False):
    """Both UHF Fock matrices ``h + J[rho_a + rho_b] - K[rho_s]``, the direct term formed from both densities'
    separate sums (DESIGN §4.11).  Returns an array ``[2, n, n]``."""
    j = np.einsum("prqs,sr->pq", u, rho_a) + np.einsum("prqs,sr->pq", u, rho_b)
    return np.stack([_sub(h + j, np.einsum("prsq,sr->pq", u, r), absolute) for r in (rho_a, rho_b)])


def kron_fock_density(h, A, B, rho, a_d, a_x, dt, absolute=False):
    """``fock_density`` of ``u[p,r,q,s] = A[p,q] B[r,s]``: ``h + a_d A tr(B rho) + a_x A rho B``.  The
    absolute-value companion of this form is the exact ``|terms|`` of the dense sum."""
    a_d, a_x = (abs(a_d), abs(a_x)) if absolute else (a_d, a_x)
    return h + a_d * A * np.sum(B * rho.T) + a_x * (A @ rho @ B)


def kron_fock_unrestricted(h, A, B, rho_a, rho_b, dt, absolute=False):
    """``fock_unrestricted`` of ``u[p,r,q,s] = A[p,q] B[r,s]``: ``h + A tr(B rho_a) + A tr(B rho_b) - A rho_s B``,
    the direct term from both densities' separate sums.  The absolute-value companion is the exact ``|terms|``."""
    j = A * np.sum(B * rho_a.T) + A * np.sum(B * rho_b.T)
    return np.stack([_sub(h + j, A @ r @ B, absolute) for r in (rho_a, rho_b)])


def kron_fock_occupied(h, A, B, n_occ, dt, anti=False, spatial=False, absolute=False):
    """``fock_occupied`` (general form) of ``u[a,b,c,d] = A[a,c] B[b,d]`` (minus ``A[a,d] B[b,c]``):
    ``h + A sum_i B[i,i] (- sum_i A[p,i] B[i,q])`` over ``i < n_occ``.  ``spatial``: the spatial form of the plain
    ``A ⊗ B``, ``h + 2 A sum_i B[i,i] - sum_i A[p,i] B[i,q]``.  The absolute-value companion is the exact ``|terms|``
    of the general form without ``anti`` and an upper bound of it otherwise."""
    o = slice(0, n_occ)
    f = h + (2 if spatial else 1) * A * np.sum(np.diagonal(B)[o])
    return _sub(f, A[:, o] @ B[o, :], absolute) if anti or spatial else f


def fock_occupied(h, u, n_occ, spatial, dt, absolute=False):
    """``h + sum_i u[p,i,q,i]`` over ``i < n_occ``, or ``h + 2 sum_i u[p,i,q,i] - sum_i u[p,i,i,q]`` (spatial)."""
    i = np.arange(n_occ)
    direct = u[:, i, :, i].sum(axis=0)
    if not spatial:
        return h + direct
    return _sub(h + 2 * direct, u[:, i, i, :].sum(axis=1), absolute)


def spin_2_tb(S, dt, p=None, q=None, anti=False, absolute=False):
    """``out[p,q,r,s] = sum_i S_i[p,r] S_i[q,s]`` (minus ``S_i[p,s] S_i[q,r]`` when ``anti``) for the stacked
    spin matrices ``S`` (3, n, n); ``p`` / ``q`` select index lists of the two leading axes."""
    Sp = S if p is None else S[:, p]
    Sq = S if q is None else S[:, q]
    out = np.einsum("ipr,iqs->pqrs", Sp, Sq)
    if anti:
        out = _sub(out, np.einsum("ips,iqr->pqrs", Sp, Sq), absolute)
    return out


def kron_occupied_traces(h, A, B, n_occ, dt, absolute=False):
    """``occupied_traces`` of ``u[a,b,c,d] = A[a,c] B[b,d]``: ``u[i,j,i,j] = A[i,i] B[j,j]`` and
    ``u[i,j,j,i] = A[i,j] B[j,i]``, summed as the ``n_occ²`` products of the dense form."""
    o = np.arange(n_occ)
    return np.array([h[o, o].sum(), np.sum(np.outer(A[o, o], B[o, o])), np.sum(A[:n_occ, :n_occ] * B[:n_occ, :n_occ].T)])


def occupied_traces(h, u, n_occ, dt, absolute=False):
    """``(tr h[o,o], sum_ij u[i,j,i,j], sum_ij u[i,j,j,i])`` over ``i, j < n_occ``."""
    o = np.arange(n_occ)
    uo = u[:n_occ, :n_occ, :n_occ, :n_occ]
    return np.array([h[o, o].sum(), np.einsum("ijij->", uo), np.einsum("ijji->", uo)])


# ------------------------------------------------------------------------------------------- reference and bound


def chop(x, bits):
    """``x`` rounded to ``bits`` mantissa bits (a kernel that computes in fewer bits than FP64)."""
    def one(v):
        m, e = np.frexp(v)
        return np.ldexp(np.round(m * 2.0**bits) / 2.0**bits, e)

    return one(x.real) + 1j * one(x.imag) if np.iscomplexobj(x) else one(x)


def companions(fn, *arrays, **kw):
    """``(ref, absval, fp64)`` of ``fn`` over the positional ``arrays`` (keyword arguments pass through): the
    ``np.longdouble`` reference, the FP64 absolute-value companion and the plain FP64 evaluation."""
    ref = fn(*(cast(x, LD) for x in arrays), dt=LD, **kw)
    absval = fn(*(np.abs(np.asarray(x)).astype(F64) for x in arrays), dt=F64, absolute=True, **kw)
    fp64 = fn(*(cast(x, F64) for x in arrays), dt=F64, **kw)
    return ref, np.real(absval).astype(F64), fp64


def rounding_ratios(got, ref, absval):
    """Per element ``|got - ref| / (u |terms|)`` where ``|terms| > 0``, and the elements with ``|terms| == 0``
    whose value is not exactly zero."""
    got = np.asarray(got)
    err = np.abs(cast(got, LD) - ref).astype(F64)
    live = absval > 0
    ratio = np.zeros_like(err)
    ratio[live] = err[live] / (U * absval[live])
    stray = (~live) & (got != 0)
    return ratio, stray


def assert_rounding_bound(got, ref, absval, k_eff, fp64, what=""):
    """Hold ``got`` to the rounding error of an FP64 evaluation of ``ref``'s sums, ``k_eff`` rounded operations
    deep (DESIGN §2):

    A, per element: ``|got - ref| <= 2 gamma(k_eff) |terms|`` (times sqrt 2 for complex values), and exactly zero
    where ``|terms| == 0``.  Rigorous for any evaluation order of the documented algorithm.
    B, aggregate: ``RMS(|got - ref| / (u |terms|)) <= max(4 RMS of the same ratio for fp64, 1)``, ``fp64`` being a
    plain numpy FP64 evaluation of the same sums.  Catches a uniformly less precise kernel that A's worst-case
    slack lets through.

    Returns ``{"a": largest |got - ref| / bound, "rms": RMS ratio of got, "rms_fp64": that of fp64}``."""
    got, ref, absval = np.asarray(got), np.asarray(ref), np.asarray(absval)
    assert got.shape == ref.shape == absval.shape, f"{what}: shapes {got.shape}, {ref.shape}, {absval.shape}"
    assert np.all(np.isfinite(got)), f"{what}: non-finite elements"
    if got.size == 0:
        return {"a": 0.0, "rms": 0.0, "rms_fp64": 0.0}
    ratio, stray = rounding_ratios(got, ref, absval)
    if stray.any():
        idx = tuple(int(i) for i in np.argwhere(stray)[0])
        raise AssertionError(f"{what}: element {idx} is {got[idx]!r} where every term is exactly zero "
                             f"({int(stray.sum())} such elements)")
    limit = 2.0 * gamma(k_eff) / U * (np.sqrt(2.0) if np.iscomplexobj(got) or np.iscomplexobj(ref) else 1.0)
    worst = np.unravel_index(int(np.argmax(ratio)), ratio.shape)
    a = float(ratio[worst]) / limit
    live = absval > 0
    rms = float(np.sqrt(np.mean(ratio[live] ** 2))) if live.any() else 0.0
    rms_fp64 = float(np.sqrt(np.mean(rounding_ratios(fp64, ref, absval)[0][live] ** 2))) if live.any() else 0.0
    rms_limit = max(4.0 * rms_fp64, 1.0)
    detail = (f"worst element {tuple(int(i) for i in worst)}: |got - ref| = {ratio[worst]:.3g} u|terms|, "
              f"{a:.3g} of the bound 2 gamma({k_eff}); RMS ratio {rms:.3g} (FP64 numpy {rms_fp64:.3g}, limit "
              f"{rms_limit:.3g})")
    assert a <= 1.0, f"{what}: criterion A (per element) fails -- {detail}"
    assert rms <= rms_limit, f"{what}: criterion B (aggregate) fails -- {detail}"
    return {"a": a, "rms": rms, "rms_fp64": rms_fp64}


def k_transform(Ks, complex_operands):
    """``k_eff`` of a chain of quarter steps of lengths ``Ks``: ``sum (K' + 1)``, ``K' = 2K`` for steps with a
    complex operand (a complex product is two real products per output component)."""
    return sum((2 * K if c else K) + 1 for K, c in zip(Ks, complex_operands))


def k_diagonal(n, complex_, generated_w=False, anti=False):
    """``k_eff`` of the two-GEMM diagonal transform over ``n`` original orbitals: the pair product ``C̃[p,a] C[a,r]``
    (two terms when complex), two GEMMs of length ``K'``, five roundings of a generated ``W`` (difference, square,
    sum, correctly rounded sqrt and division) and the anti-symmetrising subtraction."""
    return (2 if complex_ else 1) + k_transform([n, n], [complex_] * 2) + (5 if generated_w else 0) + int(anti)


# ------------------------------------------------------------------------------------------------ input families


def graded(n, lo=-4.0):
    """``logspace(0, lo, n)``: orbital weights whose products keep a ``10^(4 lo)`` dynamic range in ``u``."""
    return np.logspace(0.0, lo, n)


def pow2_graded(n):
    """``graded(n)`` rounded to powers of two, so that dyadic values scaled by it stay exact in products."""
    return 2.0 ** np.round(np.log2(graded(n)))


def graded_two_body(rng, n, complex_=False, lo=-4.0):
    """Family (b): ``u[a,b,c,d] = z_abcd g_a g_b g_c g_d`` with ``z`` standard normal."""
    g = graded(n, lo)
    u = rng.standard_normal((n,) * 4) + (1j * rng.standard_normal((n,) * 4) if complex_ else 0)
    return u * np.einsum("a,b,c,d->abcd", g, g, g, g)


def near_identity(rng, n, m=None, complex_=False, eps=1e-2):
    """``I + eps Z``: a basis change that keeps the graded output graded."""
    m = n if m is None else m
    z = rng.standard_normal((n, m)) + (1j * rng.standard_normal((n, m)) if complex_ else 0)
    return np.eye(n, m) + eps * z


def conditioned(rng, n, cond=1e3, complex_=False):
    """Family (c): ``Q1 diag(logspace(0, -log10 cond)) Q2`` and its FP64 inverse, the bi-orthogonal pair whose
    round trip cancels to the input."""
    def orth():
        z = rng.standard_normal((n, n)) + (1j * rng.standard_normal((n, n)) if complex_ else 0)
        return np.linalg.qr(z)[0]

    C = orth() @ np.diag(np.logspace(0.0, -np.log10(cond), n)) @ orth()
    return C, np.linalg.inv(C)


def dyadic(rng, shape, complex_=False, bits=20):
    """Standard normal values rounded to ``bits`` fractional bits (scaled to unit size): products of two and
    differences of such products are exact in FP64, so ``A ⊗ B`` is an exact FP64 tensor."""
    def part():
        return np.round(np.clip(rng.standard_normal(shape), -4, 4) * 2.0 ** (bits - 2)) / 2.0 ** (bits - 2)

    return part() + (1j * part() if complex_ else 0)


def kron_two_body(A, B, anti=False):
    """The dense tensor ``u[a,b,c,d] = A[a,c] B[b,d]`` (minus ``A[a,d] B[b,c]``), exact for ``dyadic`` factors."""
    u = np.einsum("ac,bd->abcd", A, B)
    if anti:
        u = u - np.einsum("ad,bc->abcd", A, B)
    return u
