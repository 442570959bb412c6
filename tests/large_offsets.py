"""The cases of tests/test_gpu_large_offsets.py, their memory plan, and the exact checker of the data-movement
kernels on tensors past 2**31 and 2**32 elements (DESIGN §2, "64-bit offsets").

Every case is built at an extent whose largest element offset crosses the boundary it is listed under; ``CASES``
holds that claim and the planned peak bytes, read by the GPU module (to assert the claim and to skip a case that does
not fit the device) and by tests/test_large_offsets_cpu.py (to check the claims and the plan without a GPU).

Hash-coded inputs: element ``lin`` (its int64 linear index) holds ``hash_code(lin)``, an integer below 2**40, made
on the device with torch int64 operations.  Every value is exact in FP64 and so is every difference or dyadic
multiple the kernels form, so a kernel result is compared with ``torch.equal`` against an expectation built from the
index formula alone.  The code is ``(lin M) mod 2**40`` followed by two xor-shift-multiply rounds: a difference of
the plain product, ``(a - b) M mod 2**40``, would depend only on ``a - b`` (up to one carry), and ``lin`` itself
makes ``u[p,q,r,s] - u[p,q,s,r] = (r - s)(n - 1)`` the same in every plane, so a plane read through a wrapped
offset would still match."""

import collections
import ctypes

import numpy as np
import torch

S31, S32 = 2**31, 2**32
BUDGET = 150 * 10**9  # planned peak device bytes of one case
MASK = 2**40 - 1
# odd multipliers; an int64 product that wraps modulo 2**64 is still right modulo 2**40, all the mask keeps
_M1, _M2, _M3, _SALT = 0x2545F491, 0x5BD1E9, 0x3C6EF3, 0x5851F42D
CHUNK_ELEMS = 2**26  # elements per chunk of the exact comparison
SCRATCH = 8 * 10**9  # device bytes of the checks' temporaries (hash chunks, sweep chunks of 8 planes at n <= 257)


def hash_code(lin, salt=0):
    """Integer code below 2**40 of the int64 indices ``lin``, ``salt`` selecting an independent code."""
    h = ((lin + salt * _SALT) * _M1) & MASK
    h = ((h ^ (h >> 19)) * _M2) & MASK
    return (((h ^ (h >> 17)) * _M3) & MASK) ^ (h >> 23)


def coded(lin, dtype, salt=0):
    """The values of a hash-coded tensor at ``lin``: ``hash_code(lin, 2 salt)`` (+ ``1j hash_code(lin, 2 salt + 1)``
    for complex128)."""
    re = hash_code(lin, 2 * salt).to(torch.float64)
    if dtype == torch.complex128:
        return torch.complex(re, hash_code(lin, 2 * salt + 1).to(torch.float64))
    return re


def lin_coded(lin, dtype, salt=0):
    """The plain ``lin`` code the hash replaces (tests/test_large_offsets_cpu.py shows why)."""
    return lin.to(dtype)


def axes(p0, p1, n, device):
    """Broadcastable int64 indices ``p, q, r, s`` of planes ``[p0, p1)`` of an ``(.., n, n, n)`` tensor."""
    p = torch.arange(p0, p1, device=device, dtype=torch.int64).view(-1, 1, 1, 1)
    q, r, s = (torch.arange(n, device=device, dtype=torch.int64).view(shape)
               for shape in ((1, -1, 1, 1), (1, 1, -1, 1), (1, 1, 1, -1)))
    return p, q, r, s


def lin4(p, q, r, s, n):
    return ((p * n + q) * n + r) * n + s


def antisymmetrized(n, dtype, code=coded, salt=0):
    """Planes ``[p0, p1)`` of ``u - u.transpose(0, 1, 3, 2)`` for the ``code``-coded ``u`` of extent ``n``."""
    def planes(p0, p1, device):
        p, q, r, s = axes(p0, p1, n, device)
        return code(lin4(p, q, r, s, n), dtype, salt) - code(lin4(p, q, s, r, n), dtype, salt)

    return planes


def fill(t, planes_fn, chunk_elems=CHUNK_ELEMS):
    """``t[p0:p1] = planes_fn(p0, p1, device)`` chunk by chunk."""
    plane = t[0].numel() if t.dim() > 1 else 1
    step = max(1, chunk_elems // plane)
    for p0 in range(0, t.shape[0], step):
        p1 = min(p0 + step, t.shape[0])
        t[p0:p1] = planes_fn(p0, p1, t.device)
    return t


def assert_exact(got, planes_fn, what, boundary, chunk_elems=CHUNK_ELEMS):
    """``torch.equal`` of ``got`` with ``planes_fn(p0, p1, device)``, plane chunk by plane chunk (NaN never equals:
    an element nobody wrote into a NaN-filled output fails).  ``got`` must reach element offset ``boundary``; a
    mismatch is reported with its offset relative to it (``boundary=None``: a tensor that is not itself large, such
    as a block cut from one)."""
    if boundary is not None:
        assert got.numel() > boundary, f"{what}: {got.numel()} elements do not reach offset {boundary}"
    plane = got[0].numel() if got.dim() > 1 else 1
    step = max(1, chunk_elems // plane)
    for p0 in range(0, got.shape[0], step):
        p1 = min(p0 + step, got.shape[0])
        want = planes_fn(p0, p1, got.device).to(got.dtype)
        part = got[p0:p1]
        if not torch.equal(part, want.expand_as(part)):
            bad = ~(part == want)
            idx = tuple(int(i) for i in torch.nonzero(bad)[0])
            offset = p0 * plane + int(np.ravel_multi_index(idx, tuple(part.shape)))
            where = "" if boundary is None else f" ({offset / boundary:.4f} x {boundary})"
            raise AssertionError(
                f"{what}: element {(p0 + idx[0],) + idx[1:]} at offset {offset}{where} "
                f"is {complex(part[idx])!r}, expected {complex(want.expand_as(part)[idx])!r}; {int(bad.sum())} such "
                f"elements in planes [{p0}, {p1})")


# ------------------------------------------------------------------------------------------------ the memory plan


def _bytes(entry, *args):
    from quantum_systems_b200 import _native

    nbytes = ctypes.c_int64(0)
    _native.call(entry, *args, ctypes.byref(nbytes))
    return nbytes.value


def transform_ws(n, m, u_c, c_c):
    return _bytes("qs_transform_two_body_workspace_bytes", n, m, int(u_c), int(c_c)) + 1024


def esize(complex_):
    return 16 if complex_ else 8


# name -> boundary, extent, largest element offset at an extent, planned peak bytes at an extent, and whether the
# extent is the smallest that crosses the boundary (the headline l = 128 spin-orbital system is not: it is the size
# DESIGN §4.12 runs)
Case = collections.namedtuple("Case", "boundary extent offset nbytes minimal")


def _q4(n):
    return n**4 - 1


def _spin(l):
    return (2 * l) ** 4 - 1


def _transform(c):
    return lambda n: 2 * n**4 * esize(c) + transform_ws(n, n, c, c) + SCRATCH


def _rect_transform(n):
    """``u`` (n^4), the (m^4) result and the workspace of an ``n -> m`` transform."""
    return lambda m: (n**4 + m**4) * 8 + transform_ws(n, m, False, False) + SCRATCH


def sharded_bytes(n, world, complex_):
    """Peak of the square sharded peer schedule (four full steps) with all ``world`` ranks on one device, from the
    sizes the schedule itself uses (``sharded._RankTransform``).  Every rank holds its slab and the slab's spare (the
    result's buffers, ping-pong), its recv buffer and its step scratch, and one step-1 padded copy is alive at a time.
    Before any of the transform's buffers exists, ``sharded_bounds.exact_sharded`` builds one rank's slab whole."""
    from quantum_systems_b200 import sharded

    dtype = torch.complex128 if complex_ else torch.float64
    ctx = sharded.EmulatedContext(world)
    work = [sharded._RankTransform(ctx, r, n, n, dtype, dtype) for r in range(world)]
    slabs = [w.A * n**3 for w in work]
    steps = sum(w.recv_numel(r) + w.scratch_numel() for r, w in enumerate(work))
    pad = max(w.A * n * n * w.Pu if w.Pu != n else 0 for w in work)
    return (2 * sum(slabs) + max(max(slabs), steps + pad)) * esize(complex_) + SCRATCH


def _sharded(world):
    return lambda n: sharded_bytes(n, world, False)


def _largest_shard(world):
    """Largest element offset within one rank's slab of the block partition."""
    return lambda n: -(-n // world) * n**3 - 1


def _two(c):
    return lambda n: 2 * n**4 * esize(c) + SCRATCH


def _one(c):
    return lambda n: n**4 * esize(c) + SCRATCH


def _add_spin(c):
    return lambda l: l**4 * 8 + (2 * l) ** 4 * esize(c) + SCRATCH


def _spin_orbital(c):
    return lambda l: 4 * l**4 * esize(c) + (2 * l) ** 4 * esize(c) + SCRATCH


def _fock_density(c):
    return lambda n: n**4 * esize(c) + _bytes("qs_fock_density_unrestricted_workspace_bytes", n, 0, n, int(c),
                                              int(c)) + SCRATCH


RECT_N = 160  # orbitals of the rectangular n -> m = 257 transform, whose last step alone stores past 2**32
DIAGONAL_GRID = 64  # grid points of the diagonal transform's W
ODQD_GRID = 401  # grid points of the ODQD build (399 interior)

CASES = {
    "transform-216-real": Case(S31, 216, _q4, _transform(False), True),
    "transform-216-complex": Case(S31, 216, _q4, _transform(True), True),
    "transform-217-real-odd-pitch": Case(S31, 217, _q4, _transform(False), False),
    "transform-257-real": Case(S32, 257, _q4, _transform(False), True),
    "transform-160-257-real": Case(S32, 257, _q4, _rect_transform(RECT_N), True),
    "symmetric-216-antisymmetric": Case(S31, 216, _q4, _transform(False), True),
    "symmetric-216-exchange": Case(S31, 216, _q4, _transform(False), True),
    "detect-216-real": Case(S31, 216, _q4, _one(False), True),
    "detect-216-complex": Case(S31, 216, _q4, _one(True), True),
    "detect-257-real": Case(S32, 257, _q4, _one(False), True),
    "cyclic-fill-216": Case(S31, 216, _q4, _one(False), True),
    "add-spin-108": Case(S31, 108, _spin, _add_spin(True), True),
    "add-spin-129-real": Case(S32, 129, _spin, _add_spin(False), True),
    "antisymmetrize-216-real": Case(S31, 216, _q4, _two(False), True),
    "antisymmetrize-216-complex": Case(S31, 216, _q4, _two(True), True),
    "antisymmetrize-257-real": Case(S32, 257, _q4, _two(False), True),
    "spin-orbital-108-real": Case(S31, 108, _spin, _spin_orbital(False), True),
    "spin-orbital-128-complex": Case(S31, 128, _spin, _spin_orbital(True), False),
    "fock-density-216-real": Case(S31, 216, _q4, _fock_density(False), True),
    "fock-density-216-complex": Case(S31, 216, _q4, _fock_density(True), True),
    "fock-occupied-216": Case(S31, 216, _q4, _one(False), True),
    "extract-block-216": Case(S31, 216, _q4, _one(True), True),
    "scale-add-complex": Case(S31, S31 + 1, lambda c: c - 1, lambda c: 3 * c * 16 + SCRATCH, True),
    "scale-add-real-odd": Case(S31, S31 + 1, lambda c: c - 1, lambda c: 2 * c * 8 + SCRATCH, True),
    "scale-add-real-s32": Case(S32, S32 + 1, lambda c: c - 1, lambda c: 2 * c * 8 + SCRATCH, True),
    "diagonal-216": Case(S31, 216, _q4, lambda m: m**4 * 8 + _bytes(
        "qs_transform_two_body_diagonal_workspace_bytes", DIAGONAL_GRID, m, 0, 0, 1) + 1024 + SCRATCH, True),
    "odqd-216": Case(S31, 216, _q4, lambda l: l**4 * 8 + _bytes(
        "qs_odqd_coulomb_workspace_bytes", l, ODQD_GRID - 2) + 1024 + SCRATCH, True),
    "sharded-216-one-rank": Case(S31, 216, _q4, _sharded(1), True),
    "sharded-257-two-ranks": Case(S31, 257, _largest_shard(2), _sharded(2), True),
}


def planned_bytes(name):
    case = CASES[name]
    return case.nbytes(case.extent)
