"""The rounding-error check of tests/precise.py applied to a sharded four-index transform, on any engine
(``sharded.CudaEngine`` on the device, the numpy stand-in of tests/_numpy_engine.py on the host).

The input is the exact tensor ``u = A ⊗ B`` (``u[a,b,c,d] = A[a,c] B[b,d]``, minus the ``(c, d)`` swap when
anti-symmetric) with dyadic ``A``, ``B``, built slab by slab on the ranks' own device: no rank ever holds the
whole tensor.  Its transform is ``u'[p,q,r,s] = X[p,r] Y[q,s] (- X'[p,s] Y'[q,r])`` (``precise.kron_factors``),
and the result is held to the bound in two ways:

(a) whole planes under criteria A and B (``precise.assert_rounding_bound``): the first and last plane of every rank
    that owns any, the planes where the kernels switch (0, 63, 64, 127, 128, m - 1) and two random ones, compared in
    batches of a few planes so that the longdouble references stay small;
(b) every element of every rank under criterion A, on the device of the ranks (``sweep``).  This finds a plane
    stored under the wrong p, a column dealt to the wrong place or an element never written anywhere in the
    tensor, where (a) only samples.

Run with an engine whose ``empty`` returns NaN-filled memory, an element computed from a tile that was skipped,
a row nobody wrote or an output element never stored is non-finite, and both checks reject it."""

import bisect
import ctypes
import functools

import numpy as np
import torch

import precise as P

# (b)'s extra slack in units of u, beyond the kernel's own 2 gamma(k) |terms| (sqrt 2 larger for complex values):
# the device compares with fl(X̂ Ŷ) - fl(X̂' Ŷ') instead of the exact value.  X̂ = fl64(X_ld) is off by at most
# u |X| for the rounding to FP64 plus the longdouble error of X_ld, gamma_ld(4n) |X|abs <= 4n 2^-64 |X|abs, at most
# 0.5 u for n <= 256 even for complex factors (x86 extended; far less in IEEE quad): 1.5 u for each of the two
# factors.  The FP64 product adds u (real) or sqrt 2 gamma(2) < 2.9 u (complex), the subtraction of the anti-symmetric
# form u: 2 x 1.5 + 2.9 + 1 = 6.9 u of (|X||Y| + |X'||Y'|).  The bound itself is evaluated in FP64 from the rounded
# |X|, |Y|, which costs a relative few u of 2 gamma(k), far less than the remaining 1.1 u.  ``n`` is the contraction
# length of the factors (the extent of ``A``); ``sweep_slabs`` refuses a larger one.
SWEEP_SLACK = 8.0
SWEEP_MAX_N = 256


def plane_indices(m, rng, extra=()):
    """The planes where the kernels switch (0, the 64 and 128 boundaries, m - 1), ``extra`` and two random ones."""
    fixed = {i for i in (0, 63, 64, 127, 128, m - 1) if i < m} | {int(i) for i in extra}
    return sorted(fixed | {int(i) for i in rng.integers(0, m, 2)})


def rank_planes(u, rng):
    """``plane_indices`` plus the first and last plane of every rank that owns any."""
    ends = [p for r in range(u.ctx.world) for p in (u.planes(r)[0], u.planes(r)[1] - 1) if u.planes(r)[1] > u.planes(r)[0]]
    return plane_indices(u.n, rng, ends)


def exact_sharded(ctx, A, B, anti, dtype, device):
    """``u = A ⊗ B`` (anti-symmetrised when ``anti``) as a ``ShardedTwoBody``, every rank building its own planes
    ``A[p0:p1, None, :, None] * B[None, :, None, :]`` on ``device``; exact for dyadic ``A``, ``B``."""
    from quantum_systems_b200 import sharded

    n = A.shape[0]
    Ad, Bd = (torch.from_numpy(np.ascontiguousarray(x)).to(device) for x in (A, B))

    def slab(p0, p1):
        t = Ad[p0:p1, None, :, None] * Bd[None, :, None, :]
        if anti:
            t = t - Ad[p0:p1, None, None, :] * Bd[None, :, :, None]
        return t

    return sharded.ShardedBasisSet.from_slabs(ctx, n, np.eye(n), np.eye(n), slab, dtype).u


def planes_of(u, planes):
    """Planes ``u[p]`` of a sharded tensor or of a plain torch tensor, copied to the host (only these planes, not
    the whole tensor)."""
    if isinstance(u, torch.Tensor):
        return u[list(planes)].cpu().numpy()
    rows = []
    for p in planes:
        r = bisect.bisect_right(u.offsets, p) - 1
        rows.append(u.local(r)[p - u.offsets[r]])
    return torch.stack(rows).cpu().numpy()


def kron_planes_of(factors_fn):
    """``precise.kron_planes`` over the factors ``factors_fn(*arrays)`` in the form ``precise.companions`` takes."""
    def planes_fn(*arrays, planes, dt, anti=False, absolute=False):
        return P.kron_planes(factors_fn(*arrays, dt=dt, absolute=absolute), planes, anti, absolute)

    return planes_fn


def chain_factors(A, B, C1, Ct1, C2, Ct2, dt=None, absolute=False):
    """``kron_factors`` of two transforms in a row, formed step by step, ``X = C̃2 (C̃1 A C1) C2``, so that the
    absolute-value companion is built from ``|C1|`` and ``|C2|`` (the eight-step composite's ``|terms|``)."""
    return P.kron_factors(Ct1 @ (A @ C1), Ct1 @ (B @ C1), C2, Ct2)


def check_planes(check, u, factors_fn, arrays, planes, k, anti, what, batch=4):
    """(a): criteria A and B on ``planes``, ``batch`` planes per reference.  ``check(got, ref, absval, k, fp64,
    what)`` records or asserts.  An anti-symmetric result must be so exactly on every checked plane."""
    planes_fn = kron_planes_of(factors_fn)
    for i in range(0, len(planes), batch):
        chunk = planes[i : i + batch]
        got = planes_of(u, chunk)
        ref, absval, fp64 = P.companions(planes_fn, *arrays, planes=chunk, anti=anti)
        check(got, ref, absval, k, fp64, f"{what}, planes {chunk}")
        if anti:
            assert np.array_equal(got, -got.transpose(0, 1, 3, 2)), f"{what}: planes {chunk} not exactly anti-symmetric"
            assert np.all(np.diagonal(got, axis1=2, axis2=3) == 0), f"{what}: planes {chunk} with a non-zero diagonal"


def sweep(u, factors_fn, arrays, k, anti, what, chunk=8):
    """(b): every element of every rank against ``fl(X̂ Ŷ) (- fl(X̂' Ŷ'))`` under criterion A plus ``SWEEP_SLACK``
    (criterion A only: the aggregate B needs the longdouble reference), rank by rank (``sweep_slabs``).  Returns
    the largest ``|got - X̂ Ŷ| / bound``."""
    slabs = [(f"rank {r}", u.planes(r)[0], u.local(r)) for r in u.ctx.local_ranks]
    return sweep_slabs(slabs, factors_fn, arrays, k, anti, what, chunk)


def sweep_slabs(slabs, factors_fn, arrays, k, anti, what, chunk=8, boundary=None):
    """(b) over ``slabs``, a list of ``(label, first plane, tensor of leading planes)`` of one dtype on one device
    (a rank's shard, or a whole single-GPU result as ``("", 0, out)``), streamed in chunks of ``chunk`` planes on
    that device.  ``boundary``: an element offset the sweep must reach within one slab (2**31 for the checks of
    64-bit addressing); a violation reports where it lies relative to it.  Returns the largest
    ``|got - X̂ Ŷ| / bound``."""
    assert np.shape(arrays[0])[0] <= SWEEP_MAX_N, f"{what}: SWEEP_SLACK is derived for n <= {SWEEP_MAX_N}"
    dev = slabs[0][2].device
    out_dtype = slabs[0][2].dtype
    if boundary is not None:
        assert max(s.numel() for _, _, s in slabs) > boundary, f"{what}: no slab reaches element offset {boundary}"

    def to_dev(x):
        x = np.asarray(x)
        if out_dtype == torch.float64:
            assert not np.iscomplexobj(x) or not np.any(x.imag), "complex factors of a real result"
            x = np.real(x)
        return torch.from_numpy(np.ascontiguousarray(P.cast(x, P.F64))).to(device=dev, dtype=out_dtype)

    fac = [to_dev(x) for x in factors_fn(*(P.cast(x, P.LD) for x in arrays), dt=P.LD)]
    absf = factors_fn(*(np.abs(np.asarray(x)).astype(P.LD) for x in arrays), dt=P.LD, absolute=True)
    absf = [torch.from_numpy(np.asarray(x, dtype=P.F64)).to(dev) for x in absf]
    cplx = out_dtype == torch.complex128
    coef = 2.0 * P.gamma(k) * (np.sqrt(2.0) if cplx else 1.0) + SWEEP_SLACK * P.U
    worst = 0.0
    for label, p0, slab in slabs:
        p1 = p0 + slab.shape[0]
        plane = slab[0].numel() if slab.shape[0] else 0
        for c0 in range(p0, p1, chunk):
            c1 = min(c0 + chunk, p1)
            X, Y, Xx, Yx = fac
            Xa, Ya, Xxa, Yxa = absf
            want = X[c0:c1, None, :, None] * Y[None, :, None, :]
            bound = Xa[c0:c1, None, :, None] * Ya[None, :, None, :]
            if anti:
                want = want - Xx[c0:c1, None, None, :] * Yx[None, :, :, None]
                bound = bound + Xxa[c0:c1, None, None, :] * Yxa[None, :, :, None]
            got = slab[c0 - p0 : c1 - p0]
            err = (got - want).abs()
            bound = coef * bound
            bad = ~(err <= bound)  # NaN compares false: non-finite elements are violations
            if bool(bad.any()):
                idx = tuple(int(i) for i in torch.nonzero(bad)[0])
                g = (c0 + idx[0],) + idx[1:]
                offset = (c0 - p0 + idx[0]) * plane + int(np.ravel_multi_index(idx[1:], tuple(got.shape[1:])))
                where = "" if boundary is None else f", element offset {offset} ({offset / boundary:.3f} x {boundary})"
                raise AssertionError(
                    f"{what}: sweep (criterion A) fails at element {g} ({label}{where}): got {complex(got[idx])!r}, "
                    f"X Y = {complex(want[idx])!r}, |error| {float(err[idx]):.3g} > bound {float(bound[idx]):.3g}; "
                    f"{int(bad.sum())} such elements in planes [{c0}, {c1})")
            live = bound > 0
            if bool(live.any()):
                worst = max(worst, float((err[live] / bound[live]).max()))
    return worst


def check_sharded(check, u, factors_fn, arrays, k, anti, rng, what, batch=4):
    """(a) on ``rank_planes`` and (b) on the whole tensor; returns (b)'s largest ratio."""
    check_planes(check, u, factors_fn, arrays, rank_planes(u, rng), k, anti, what, batch)
    return sweep(u, factors_fn, arrays, k, anti, what)


# -------------------------------------------------------------------------------------------- poisoned memory


class PoisonedTorch:
    """Stands in for ``torch`` inside ``ops``: every floating-point ``empty`` / ``empty_like`` (outputs, workspaces)
    comes back filled with NaN, 0xFF bytes for the byte workspaces (NaN doubles); everything else is torch itself."""

    def __getattr__(self, name):
        return getattr(torch, name)

    @staticmethod
    def empty(*args, **kwargs):
        return PoisonedTorch.poison(torch.empty(*args, **kwargs))

    @staticmethod
    def empty_like(*args, **kwargs):
        return PoisonedTorch.poison(torch.empty_like(*args, **kwargs))

    @staticmethod
    def poison(t):
        if t.dtype == torch.uint8:
            t.fill_(0xFF)
        elif t.is_floating_point() or t.is_complex():
            t.fill_(float("nan") if not t.is_complex() else complex(float("nan"), float("nan")))
        return t


@functools.lru_cache(maxsize=None)
def nan_engine():
    """``sharded.CudaEngine`` whose ``empty`` returns NaN-filled memory (NaN + NaN j), so that slabs, spare, recv,
    per-rank scratch, padded copies and outputs are poisoned; it counts the device-side anti-symmetry tests."""
    from quantum_systems_b200 import sharded

    class NaNEngine(sharded.CudaEngine):
        symmetry_tests = 0

        def empty(self, numel, dtype):
            buf = super().empty(numel, dtype)
            buf.tensor.fill_(complex(float("nan"), float("nan")) if dtype == torch.complex128 else float("nan"))
            return buf

        def is_antisymmetric(self, buf, n, planes):
            self.symmetry_tests += 1
            return super().is_antisymmetric(buf, n, planes)

    return NaNEngine


# ------------------------------------------------------------------------------------- what a case reaches


def planned_tiles(X, K, W, a_dtype, m_dtype, x_inner, kind=0, strict=0, dh=1, mh=1, dl=1, ml=1):
    """Number of CTA tiles a quarter launch plans (``qs_quarter_plan_tiles``, host only).  ``kind`` 0: the unmasked
    launch, planned as a row table that keeps every row."""
    from quantum_systems_b200 import _native

    code = {torch.float64: 0, torch.complex128: 1}
    keep_all = np.zeros(-(-X // x_inner), dtype=np.int64) if kind == 0 else None
    table = ctypes.c_void_p(keep_all.ctypes.data) if kind == 0 else ctypes.c_void_p(0)
    count = ctypes.c_int64(0)
    rc = _native.load().qs_quarter_plan_tiles(X, K, W, code[a_dtype], code[m_dtype], x_inner, kind, strict, dh, mh,
                                              dl, ml, table, ctypes.c_void_p(0), 0, ctypes.byref(count))
    assert rc == 0
    return count.value


def pair_step2_tiles(ctx, n, m, t_dtype, c_dtype):
    """``[(kept, planned without a mask)]`` per rank for step 2 of the sharded pair schedule: the mask of
    ``qs_quarter_transform_scatter_pairs`` (kind 3, strict unless the pair lists are padded to couples)."""
    from quantum_systems_b200 import sharded

    _, off = sharded.block_partition(n, ctx.world)
    padded = t_dtype == torch.float64 and m % 2 == 0
    counts = []
    for r in range(ctx.world):
        A = off[r + 1] - off[r]
        if A > 0:
            X = m * A * n
            counts.append((planned_tiles(X, n, m, t_dtype, c_dtype, n, 3, 0 if padded else 1, 1, 1, A * n, m),
                           planned_tiles(X, n, m, t_dtype, c_dtype, n)))
    return counts
