"""Tensor-level operators of the hot path: torch CUDA tensors in, torch CUDA tensors out.

Each function validates shapes/dtypes on the host, allocates the result and the scratch through
torch's caching allocator, and enqueues hand-written sm_100a kernels from ``libqsb200.so`` on the
current CUDA stream through the C ABI (``include/qsb200.h``).  torch performs no arithmetic here.
There is no CPU path: a CPU tensor, a missing library or a failing kernel raises.
"""

import ctypes

import torch

from . import _native
from ._native import QS_C128, QS_F64

_DTYPES = {torch.float64: QS_F64, torch.complex128: QS_C128}


def _code(t):
    try:
        return _DTYPES[t.dtype]
    except KeyError:
        raise TypeError(f"quantum_systems_b200 computes in float64/complex128 only, got {t.dtype}") from None


def _device_tensor(t, name):
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor on a CUDA device, got {type(t).__name__}")
    if not t.is_cuda:
        raise RuntimeError(f"{name} lives on {t.device}: quantum_systems_b200 has no CPU fallback")
    _code(t)
    return t if t.is_contiguous() else t.contiguous()


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _workspace(nbytes, device):
    """Scratch from the caching allocator, aligned to 1 KiB.  Returns (owner tensor, pointer)."""
    buf = torch.empty(int(nbytes) + 1024, dtype=torch.uint8, device=device)
    base = buf.data_ptr()
    aligned = (base + 1023) & ~1023
    return buf, ctypes.c_void_p(aligned)


def _result_dtype(*tensors):
    return torch.complex128 if any(t.dtype == torch.complex128 for t in tensors) else torch.float64


def _coefficients(C, C_tilde, tensor=_device_tensor):
    """Bring C (n, n_new) and the optional C_tilde (n_new, n) to one dtype (``tensor`` checks and converts each)."""
    C = tensor(C, "C")
    if C.dim() != 2:
        raise ValueError("C must be a matrix (n, n_new)")
    if C_tilde is not None:
        C_tilde = tensor(C_tilde, "C_tilde")
        if tuple(C_tilde.shape) != (C.shape[1], C.shape[0]):
            raise ValueError(f"C_tilde must have shape {(C.shape[1], C.shape[0])}, got {tuple(C_tilde.shape)}")
        dt = _result_dtype(C, C_tilde)
        C, C_tilde = C.to(dt), C_tilde.to(dt)
    return C, C_tilde


def real_coefficients_if_exact(u_is_complex, C, C_tilde):
    """Complex ``u`` with coefficients of complex dtype whose imaginary parts are all exactly zero (the usual
    case downstream: every array of a ``GeneralOrbitalSystem`` is complex128, basis_set.py:632-634, while
    Hartree-Fock coefficients of a real Hamiltonian are real-valued): hand the kernels the real parts, which
    selects the split "2M" quarter GEMM -- half the tensor-core work of the 4M product, same result (the
    skipped products are exact zeros).  Only when ``u`` is complex, so the result dtype does not change."""
    if not (u_is_complex and C.is_complex()):
        return C, C_tilde
    if _has_imaginary_part(C) or (C_tilde is not None and _has_imaginary_part(C_tilde)):
        return C, C_tilde
    return C.real.contiguous(), (C_tilde.real.contiguous() if C_tilde is not None else None)


def _has_imaginary_part(M):
    """``any(M.imag != 0)`` -- a device reduction read back by the host, i.e. a stream synchronisation.  The answer
    is remembered on the tensor object together with torch's in-place version counter, so a chain of basis changes
    with the same coefficient tensor synchronises once."""
    tag = getattr(M, "_qs_has_imag", None)
    if tag is not None and tag[1] == M._version:
        return tag[0]
    answer = bool(torch.any(M.imag != 0))
    M._qs_has_imag = (answer, M._version)
    return answer


# below this extent the symmetry test costs more than the tiles it saves
SYMMETRY_MIN_N = 48
# False: `transform_two_body(symmetry=None)` never tests for symmetries and always runs the four full quarter steps
EXPLOIT_SYMMETRY = True
ANTISYMMETRIC_LAST_PAIR = 1  # u[p,q,r,s] = -u[p,q,s,r]
PARTICLE_EXCHANGE = 2        # u[p,q,r,s] =  u[q,p,s,r]


def _mark_written(t):
    """A kernel of this library has written into ``t``, a tensor the caller supplied: bump torch's in-place version
    counter (shared by ``t``, its base and every other view of it) so that what the library remembers about the old
    contents -- the symmetry tag, the imaginary-part cache -- is void, exactly as after an in-place torch op."""
    torch.autograd.graph.increment_version(t)
    return t


def _tag_symmetry(t, kind):
    """Remember on the tensor object that the library itself has just made ``t`` EXACTLY (anti-)symmetric (mirror
    fill, fused anti-symmetrisation).  The tag carries torch's in-place version counter: any later in-place
    modification through torch or through this library (``_mark_written``) bumps ``t._version`` and voids it, and a
    new tensor (copy, host round trip, the ``u`` setter of a host array) never has it -- then the device-side test
    runs again."""
    t._qs_symmetry = (int(kind), t._version)
    return t


def proven_symmetry(t):
    """The symmetry kind the library has proven for this very tensor object, or 0.  Writes that bypass torch's
    version counter are not seen: ``t.data``, DLPack or ``__cuda_array_interface__`` consumers writing into the
    memory of ``t`` leave a stale proof behind."""
    tag = getattr(t, "_qs_symmetry", None)
    return tag[0] if tag is not None and tag[1] == t._version else 0


def two_body_symmetry(u, first_match=False):
    """Exact device-side test of the two symmetries the transform can exploit; returns a bit mask of
    ``ANTISYMMETRIC_LAST_PAIR`` and ``PARTICLE_EXCHANGE``.  Reads ``u`` once per test, stops at the first
    counter-example, synchronises the stream.  ``first_match`` skips the second test when the first holds."""
    u = _device_tensor(u, "u")
    n = u.shape[0]
    if tuple(u.shape) != (n, n, n, n):
        raise ValueError(f"u must be (n,n,n,n), got {tuple(u.shape)}")
    flags = ctypes.c_int(0)
    scratch = torch.empty(2, dtype=torch.int32, device=u.device)
    _native.call(
        "qs_two_body_symmetry", _ptr(u), _code(u), n, int(bool(first_match)), ctypes.byref(flags), _ptr(scratch),
        _stream(),
    )
    return flags.value


def transform_two_body(u, C, C_tilde=None, symmetry=None):
    """``u'_pqrs = sum C~[p,a] C~[q,b] u[a,b,c,d] C[c,r] C[d,s]`` (reference basis_set.py:336-350).

    ``symmetry=None`` (default) tests ``u`` for exact anti-symmetry in its last pair and for particle-exchange
    symmetry (``two_body_symmetry``) and, if one holds, skips the tiles of quarter steps 2-4 that only hold mirror
    images (``qs_transform_two_body_symmetric``); ``symmetry=0`` forces the plain four full steps."""
    u = _device_tensor(u, "u")
    C, C_tilde = _coefficients(C, C_tilde)
    C, C_tilde = real_coefficients_if_exact(u.is_complex(), C, C_tilde)
    n, m = C.shape
    if tuple(u.shape) != (n, n, n, n):
        raise ValueError(f"u must have shape {(n,) * 4} to be contracted with C {tuple(C.shape)}, got {tuple(u.shape)}")
    if symmetry is None:
        symmetry = 0
        if EXPLOIT_SYMMETRY and min(n, m) >= SYMMETRY_MIN_N:
            # a tensor this library has itself made exactly (anti-)symmetric is not tested again: no pass over u,
            # no host synchronisation in a chain of basis changes
            symmetry = proven_symmetry(u)
            if not symmetry:
                flags = two_body_symmetry(u, first_match=True)
                symmetry = (
                    ANTISYMMETRIC_LAST_PAIR if flags & ANTISYMMETRIC_LAST_PAIR
                    else PARTICLE_EXCHANGE if flags & PARTICLE_EXCHANGE else 0
                )
    out = torch.empty((m, m, m, m), dtype=_result_dtype(u, C), device=u.device)
    nbytes = ctypes.c_int64(0)
    _native.call("qs_transform_two_body_workspace_bytes", n, m, _code(u), _code(C), ctypes.byref(nbytes))
    owner, ws = _workspace(nbytes.value, u.device)
    _native.call(
        "qs_transform_two_body_symmetric", _ptr(u), _code(u), _ptr(C), _ptr(C_tilde), _code(C), n, m, int(symmetry),
        _ptr(out), ws, nbytes.value, _stream(),
    )
    owner.record_stream(torch.cuda.current_stream())
    if symmetry:
        _tag_symmetry(out, symmetry)  # the mirror fill has made the result exactly (anti-)symmetric
    return out


def transform_two_body_mixed(u, C_r, C_s, Ct_p=None, Ct_q=None):
    """``u'_pqrs = sum Ct_p[p,a] Ct_q[q,b] u[a,b,c,d] C_r[c,r] C_s[d,s]`` (``qs_transform_two_body_mixed``): the
    four-index transform with one coefficient matrix per index, ``Ct_p`` defaulting to ``C_r^dagger`` and ``Ct_q``
    to ``C_s^dagger``.  The mixed-spin blocks of an unrestricted basis change; no symmetry of ``u`` is used.  The
    matrices are brought to one dtype, and complex-typed ones without imaginary part are handed over as real ones
    for a complex ``u`` (``real_coefficients_if_exact``)."""
    u = _device_tensor(u, "u")
    C_r, C_s, Ct_p, Ct_q = mixed_coefficients(u.is_complex(), C_r, C_s, Ct_p, Ct_q)
    n, m = C_r.shape
    if tuple(u.shape) != (n, n, n, n):
        raise ValueError(f"u must have shape {(n,) * 4} to be contracted with C {tuple(C_r.shape)}, got {tuple(u.shape)}")
    out = torch.empty((m, m, m, m), dtype=_result_dtype(u, C_r), device=u.device)
    nbytes = ctypes.c_int64(0)
    _native.call("qs_transform_two_body_workspace_bytes", n, m, _code(u), _code(C_r), ctypes.byref(nbytes))
    owner, ws = _workspace(nbytes.value, u.device)
    _native.call(
        "qs_transform_two_body_mixed", _ptr(u), _code(u), _ptr(C_r), _ptr(C_s), _ptr(Ct_p), _ptr(Ct_q), _code(C_r),
        n, m, _ptr(out), ws, nbytes.value, _stream(),
    )
    owner.record_stream(torch.cuda.current_stream())
    return out


def mixed_coefficients(u_is_complex, C_r, C_s, Ct_p, Ct_q, tensor=_device_tensor):
    """The four matrices of a mixed transform in one dtype (``tensor`` checks and converts each: device tensors by
    default); for a complex ``u`` complex-typed ones without imaginary part become real ones
    (``real_coefficients_if_exact``), all four or none."""
    C_r, Ct_p = _coefficients(C_r, Ct_p, tensor)
    C_s, Ct_q = _coefficients(C_s, Ct_q, tensor)
    if C_r.shape != C_s.shape:
        raise ValueError(f"C_r and C_s must have one shape, got {tuple(C_r.shape)} and {tuple(C_s.shape)}")
    mats = [M for M in (C_r, C_s, Ct_p, Ct_q) if M is not None]
    dt = _result_dtype(*mats)
    C_r, C_s, Ct_p, Ct_q = (M.to(dt) if M is not None else None for M in (C_r, C_s, Ct_p, Ct_q))
    # all four real or none: one exact test over every matrix, so that the kernels see a single dtype
    if u_is_complex and dt == torch.complex128 and not any(_has_imaginary_part(M) for M in mats):
        C_r, C_s, Ct_p, Ct_q = (M.real.contiguous() if M is not None else None for M in (C_r, C_s, Ct_p, Ct_q))
    return C_r, C_s, Ct_p, Ct_q


def transform_one_body(h, C, C_tilde=None):
    """``C~ (h C)`` (reference basis_set.py:329-334)."""
    h = _device_tensor(h, "h")
    C, C_tilde = _coefficients(C, C_tilde)
    n, m = C.shape
    if tuple(h.shape) != (n, n):
        raise ValueError(f"h must have shape {(n, n)}, got {tuple(h.shape)}")
    out = torch.empty((m, m), dtype=_result_dtype(h, C), device=h.device)
    nbytes = ctypes.c_int64(0)
    _native.call("qs_transform_one_body_workspace_bytes", n, m, _code(h), _code(C), ctypes.byref(nbytes))
    owner, ws = _workspace(nbytes.value, h.device)
    _native.call(
        "qs_transform_one_body", _ptr(h), _code(h), _ptr(C), _ptr(C_tilde), _code(C), n, m, _ptr(out), ws, _stream()
    )
    owner.record_stream(torch.cuda.current_stream())
    return out


def scatter_deal(W):
    """Multiplier of the column dealing of a scattering quarter transform with ``W`` output columns
    (``qs_scatter_deal``): column j of the tile order is physical column ``(j * deal) % W``."""
    deal = ctypes.c_int64(1)
    _native.call("qs_scatter_deal", int(W), ctypes.byref(deal))
    return deal.value


def coeff_image(M, K, W, a_dtype, stride_k, stride_w, conj=False, deal=1):
    """Fragment-ordered image of ``M[k, w] = M.flat[k*stride_k + w*stride_w]`` for quarter_transform
    (``deal`` > 1: columns dealt for a scattering launch, see ``scatter_deal``)."""
    M = _device_tensor(M, "M")
    a_code = _DTYPES[a_dtype]
    nbytes = ctypes.c_int64(0)
    _native.call("qs_coeff_image_bytes", K, W, a_code, _code(M), ctypes.byref(nbytes))
    image = torch.empty(nbytes.value // 8, dtype=torch.float64, device=M.device)
    _native.call(
        "qs_build_coeff_image_dealt", _ptr(M), _code(M), stride_k, stride_w, int(bool(conj)), K, W, a_code, int(deal),
        _ptr(image), _stream(),
    )
    return image


def quarter_transform(A, X, K, lda, image, m_dtype, W, out, x_inner, sx0, sx1, w_inner, sw0, sw1):
    """One contraction ``sum_k A[x,k] M[k,w]`` with the 2-level strided store (see include/qsb200.h)."""
    A = _device_tensor(A, "A")
    _native.call(
        "qs_quarter_transform", _ptr(A), _code(A), X, K, lda, _ptr(image), _DTYPES[m_dtype], W, _ptr(out), x_inner,
        sx0, sx1, w_inner, sw0, sw1, _stream(),
    )
    return _mark_written(out)


def add_spin_two_body(u, anti_symmetrize=False, out_dtype=None, planes=None, out=None, first_spatial_plane=0):
    """Spin-double ``u`` (l,l,l,l) -> (2l,2l,2l,2l), optionally fused with the anti-symmetrisation
    and the widening cast (reference basis_set.py:772-778, :298-319).  ``planes=(P0, P1)`` restricts
    the leading spin-orbital index (multi-GPU shard); the result then has ``P1 - P0`` leading planes.
    A rank that holds only the spatial planes it needs passes that slab ``u[first_spatial_plane : ...]``
    (shape ``(planes, l, l, l)``) with ``first_spatial_plane``; it must cover ``P0 // 2 .. (P1 - 1) // 2``."""
    u = _device_tensor(u, "u")
    l = u.shape[-1]
    if u.dim() != 4 or tuple(u.shape[1:]) != (l, l, l):
        raise ValueError(f"u must be (planes,l,l,l), got {tuple(u.shape)}")
    out_dtype = u.dtype if out_dtype is None else out_dtype
    p0, p1 = (0, 2 * l) if planes is None else planes
    if p1 > p0 and not (first_spatial_plane <= p0 // 2 and (p1 - 1) // 2 < first_spatial_plane + u.shape[0]):
        raise ValueError(
            f"spin planes [{p0}, {p1}) need spatial planes [{p0 // 2}, {(p1 - 1) // 2 + 1}), the slab holds "
            f"[{first_spatial_plane}, {first_spatial_plane + u.shape[0]})"
        )
    if out is None:
        out = torch.empty((p1 - p0, 2 * l, 2 * l, 2 * l), dtype=out_dtype, device=u.device)
    else:
        _mark_written(out)
    # the kernel addresses spatial plane p at base + p * l^3: hand it the (virtual) base of the whole tensor
    base = ctypes.c_void_p(u.data_ptr() - first_spatial_plane * l**3 * u.element_size())
    _native.call(
        "qs_add_spin_two_body", base, _code(u), l, _ptr(out), _DTYPES[out_dtype], int(bool(anti_symmetrize)), p0,
        p1, _stream(),
    )
    if anti_symmetrize and planes is None:
        _tag_symmetry(out, ANTISYMMETRIC_LAST_PAIR)  # a - b and b - a are exact negatives
    return out


def anti_symmetrize(u):
    """``u - u.transpose(0,1,3,2)`` (reference basis_set.py:776-778); returns a new tensor."""
    u = _device_tensor(u, "u")
    n = u.shape[-1]
    if u.dim() != 4 or tuple(u.shape[1:]) != (n, n, n):
        raise ValueError(f"u must be (planes,n,n,n), got {tuple(u.shape)}")
    out = torch.empty_like(u)
    # `u` may be a leading-index shard: planes [0, u.shape[0]) of the local block
    _native.call("qs_anti_symmetrize", _ptr(u), _code(u), n, _ptr(out), 0, u.shape[0], _stream())
    if u.shape[0] == n:
        _tag_symmetry(out, ANTISYMMETRIC_LAST_PAIR)
    return out


def add_spin_one_body(h, out_dtype=None):
    """``kron(h, I_2)`` (reference basis_set.py:768-770)."""
    h = _device_tensor(h, "h")
    l = h.shape[0]
    if tuple(h.shape) != (l, l):
        raise ValueError(f"h must be square, got {tuple(h.shape)}")
    out_dtype = h.dtype if out_dtype is None else out_dtype
    out = torch.empty((2 * l, 2 * l), dtype=out_dtype, device=h.device)
    _native.call("qs_add_spin_one_body", _ptr(h), _code(h), l, _ptr(out), _DTYPES[out_dtype], _stream())
    return out


def spin_orbital_two_body(b_aa, b_ab, b_ba, b_bb, orbital, spin, out_dtype=None, planes=None):
    """The anti-symmetrised spin-orbital tensor of an unrestricted basis from the spin blocks ``b_st`` (l,l,l,l) of
    the spatial tensor (``qs_spin_orbital_two_body``)::

        U[I,J,K,L] = [sI=sK][sJ=sL] b_{sI sJ}[oI,oJ,oK,oL] - [sI=sL][sJ=sK] b_{sI sJ}[oI,oJ,oL,oK]

    Spin-orbital ``I`` is spatial orbital ``orbital[I]`` with spin ``spin[I]`` (0 = alpha, 1 = beta): host integer
    sequences of length ``2l`` that must pair every orbital below ``l`` with both spins exactly once.  ``b_ba=None``
    derives that block from ``b_ab`` by particle exchange, ``b_ba[i,j,k,l] = b_ab[j,i,l,k]``.  ``out_dtype`` (default:
    the blocks' dtype) may widen float64 to complex128.  ``planes=(P0, P1)`` writes only the leading planes
    ``[P0, P1)``; the whole result is tagged anti-symmetric in its last pair, which it is exactly."""
    import numpy as _numpy

    blocks = [_device_tensor(b, name) if b is not None else None
              for b, name in ((b_aa, "b_aa"), (b_ab, "b_ab"), (b_ba, "b_ba"), (b_bb, "b_bb"))]
    if blocks[0] is None or blocks[1] is None or blocks[3] is None:
        raise ValueError("b_aa, b_ab and b_bb are required; only b_ba may be derived")
    given = [b for b in blocks if b is not None]
    l = given[0].shape[0]
    for b in given:
        if tuple(b.shape) != (l,) * 4 or b.dtype != given[0].dtype or b.device != given[0].device:
            raise ValueError("the spin blocks must all be (l,l,l,l) of one dtype on one device")
    orbital = _numpy.asarray(orbital.cpu() if isinstance(orbital, torch.Tensor) else orbital)
    spin = _numpy.asarray(spin.cpu() if isinstance(spin, torch.Tensor) else spin)
    if orbital.shape != (2 * l,) or spin.shape != (2 * l,):
        raise ValueError(f"orbital and spin must be 1-d of length 2l = {2 * l}")
    if not (_numpy.issubdtype(orbital.dtype, _numpy.integer) and _numpy.issubdtype(spin.dtype, _numpy.integer)):
        raise TypeError("orbital and spin must be integer tables")
    if ((orbital < 0) | (orbital >= l)).any() or ((spin != 0) & (spin != 1)).any():
        raise ValueError(f"orbital must lie in [0, {l}) and spin in {{0, 1}}")
    if _numpy.unique(spin.astype(_numpy.int64) * l + orbital).size != 2 * l:
        raise ValueError("orbital and spin must pair every orbital with both spins exactly once")
    device = given[0].device
    orbital_d = torch.from_numpy(orbital.astype(_numpy.int32)).to(device)
    spin_d = torch.from_numpy(spin.astype(_numpy.int32)).to(device)
    out_dtype = given[0].dtype if out_dtype is None else out_dtype
    p0, p1 = (0, 2 * l) if planes is None else (int(planes[0]), int(planes[1]))
    if not 0 <= p0 <= p1 <= 2 * l:
        raise ValueError(f"planes {planes} out of range for 2l = {2 * l}")
    out = torch.empty((p1 - p0, 2 * l, 2 * l, 2 * l), dtype=out_dtype, device=device)
    _native.call(
        "qs_spin_orbital_two_body", *(_ptr(b) for b in blocks), _code(given[0]), l, _ptr(orbital_d), _ptr(spin_d),
        _ptr(out), _DTYPES[out_dtype], p0, p1, _stream(),
    )
    if planes is None:
        _tag_symmetry(out, ANTISYMMETRIC_LAST_PAIR)  # a - b and b - a are exact negatives
    return out


def _fock(name, h, u, n_occ, f):
    h = _device_tensor(h, "h")
    u = _device_tensor(u, "u")
    n = h.shape[0]
    if tuple(h.shape) != (n, n) or tuple(u.shape) != (n, n, n, n):
        raise ValueError(f"h must be (n,n) and u (n,n,n,n), got {tuple(h.shape)} and {tuple(u.shape)}")
    if f is None:
        f = torch.empty_like(h)
    else:
        if not (isinstance(f, torch.Tensor) and f.is_cuda and f.is_contiguous()):
            raise RuntimeError("f must be a contiguous CUDA tensor to be filled in place")
        if f.shape != h.shape or f.dtype != h.dtype:
            raise ValueError("f must have the shape and dtype of h")
        _mark_written(f)
    _native.call(name, _ptr(h), _code(h), _ptr(u), _code(u), n, int(n_occ), _ptr(f), 0, n, _stream())
    return f


def fock_general(h, u, n_occ, f=None):
    """``f = h + sum_i u[p,i,q,i]`` (reference general_orbital_system.py:119-159); ``f`` filled in place."""
    return _fock("qs_fock_general", h, u, n_occ, f)


def fock_spatial(h, u, n_occ, f=None):
    """``f = h + 2 u[p,i,q,i] - u[p,i,i,q]`` (reference spatial_orbital_system.py:150-190)."""
    return _fock("qs_fock_spatial", h, u, n_occ, f)


def fock_from_density(h, u, rho, scale_direct, scale_exchange, f=None, planes=None):
    """``f[p,q] = h[p,q] + a_d sum_rs u[p,r,q,s] rho[s,r] + a_x sum_rs u[p,r,s,q] rho[s,r]`` for a general density
    matrix ``rho`` (``qs_fock_density``): one read of ``u``, deterministic.  ``(1, 0)`` with an anti-symmetrised
    ``u`` is the GHF Fock matrix, ``(1, -1/2)`` with ``rho = 2 C_o C_o^dagger`` the RHF one.  ``planes=(p0, p1)``:
    ``u`` is the leading-index shard ``(p1 - p0, n, n, n)`` and only rows ``[p0, p1)`` of ``f`` are written (a new
    ``f`` is zero elsewhere).  ``f`` is complex128 when any input is; a given ``f`` is filled in place."""
    (f,) = _fock_density(
        "qs_fock_density", h, u, {"rho": rho}, {"f": f}, (float(scale_direct), float(scale_exchange)), planes
    )
    return f


def fock_from_density_unrestricted(h, u, rho_alpha, rho_beta, f_alpha=None, f_beta=None, planes=None):
    """Both unrestricted Fock matrices ``f_s[p,q] = h[p,q] + sum_rs u[p,r,q,s] (rho_a + rho_b)[s,r]
    - sum_rs u[p,r,s,q] rho_s[s,r]`` of the spin densities ``rho_alpha`` and ``rho_beta`` on a spatial ``u``
    (``qs_fock_density_unrestricted``).  Real ``u``: ``u`` is read once for both spins, with real or complex
    densities; complex ``u``: twice.  ``planes``, the in-place ``f_alpha`` / ``f_beta`` and the result dtype
    follow ``fock_from_density``; a real density is promoted to complex when the other one is complex.
    Returns ``(f_alpha, f_beta)``."""
    return _fock_density(
        "qs_fock_density_unrestricted", h, u, {"rho_alpha": rho_alpha, "rho_beta": rho_beta},
        {"f_alpha": f_alpha, "f_beta": f_beta}, (), planes,
    )


def _fock_density(entry, h, u, densities, fs, scales, planes):
    """The front end of the density Fock builds: checks ``h``, ``u`` and the ``densities`` (name -> tensor, a real
    one promoted when the other is complex), allocates or validates the outputs ``fs`` (name -> tensor or None) and
    calls ``entry`` with its workspace.  The C arguments are h, u, the densities, n, ``scales``, the outputs, the row
    range, the workspace and the stream.  Returns the tuple of outputs."""
    h = _device_tensor(h, "h")
    u = _device_tensor(u, "u")
    rhos = [_device_tensor(rho, name) for name, rho in densities.items()]
    if len(rhos) > 1 and rhos[0].dtype != rhos[1].dtype:
        rhos = [rho.to(torch.complex128) for rho in rhos]
    n = h.shape[0]
    p0, p1 = (0, n) if planes is None else (int(planes[0]), int(planes[1]))
    if not 0 <= p0 <= p1 <= n:
        raise ValueError(f"planes {planes} out of range for n = {n}")
    if (tuple(h.shape) != (n, n) or tuple(u.shape) != (p1 - p0, n, n, n)
            or [rho.shape for rho in rhos] != [h.shape] * len(rhos)):
        names = list(densities)
        shapes = ", ".join(str(tuple(t.shape)) for t in (h, *rhos, u))
        raise ValueError(f"{', '.join(['h'] + names[:-1])} and {names[-1]} must be (n,n) and u (planes,n,n,n), "
                         f"got {shapes}")
    dtype = _result_dtype(h, u, *rhos)
    outs = [_plane_output(name, f, (n, n), dtype, h.device, (p0, p1) == (0, n)) for name, f in fs.items()]
    if len(outs) > 1 and outs[0].dtype != outs[1].dtype:
        raise ValueError(f"{' and '.join(fs)} must have one dtype, got {outs[0].dtype} and {outs[1].dtype}")
    owner, ws, nbytes = _entry_workspace(entry, h.device, n, p0, p1, _code(u), _code(rhos[0]))
    _native.call(
        entry, _ptr(h), _code(h), _ptr(u), _code(u), *[_ptr(r) for r in rhos], _code(rhos[0]), n, *scales,
        *[_ptr(f) for f in outs], _code(outs[0]), p0, p1, ws, nbytes, _stream(),
    )
    owner.record_stream(torch.cuda.current_stream())
    return tuple(outs)


def _plane_output(name, out, shape, dtype, device, whole):
    """An output of a plane-range front end: a new tensor (``torch.empty`` when the call writes it ``whole``, else
    zeros, so rows outside the plane range read zero), or the caller's ``out``, checked and marked written."""
    if out is None:
        return (torch.empty if whole else torch.zeros)(shape, dtype=dtype, device=device)
    if not (isinstance(out, torch.Tensor) and out.is_cuda and out.is_contiguous()):
        raise RuntimeError(f"{name} must be a contiguous CUDA tensor to be filled in place")
    if tuple(out.shape) != shape:
        raise ValueError(f"{name} must be {shape}, got {tuple(out.shape)}")
    _code(out)
    return _mark_written(out)


def _entry_workspace(entry, device, *args):
    """The scratch ``entry + "_workspace_bytes"`` asks for with ``args``: ``(owner, pointer, bytes)``."""
    nbytes = ctypes.c_int64(0)
    _native.call(entry + "_workspace_bytes", *args, ctypes.byref(nbytes))
    owner, ws = _workspace(nbytes.value, device)
    return owner, ws, nbytes.value


# densities per launch of qs_coulomb_exchange_batch (QS_COULOMB_EXCHANGE_MAX_BATCH in include/qsb200.h)
COULOMB_EXCHANGE_MAX_BATCH = 16


def coulomb_exchange(u, rho, planes=None, J=None, K=None):
    """Coulomb and exchange matrices ``J[d,p,q] = sum_rs u[p,r,q,s] rho[d,s,r]`` and ``K[d,p,q] = sum_rs u[p,r,s,q]
    rho[d,s,r]`` of a batch of real densities ``rho`` (k, n, n) on a real ``u`` (``qs_coulomb_exchange_batch``, on the
    FP64 tensor pipe).  Each launch reads ``u`` once for up to ``COULOMB_EXCHANGE_MAX_BATCH`` densities; a larger
    batch takes ``ceil(k / COULOMB_EXCHANGE_MAX_BATCH)`` launches.  A density's ``J`` and ``K`` are bit-identical
    whatever else is in the batch.  ``planes``, the in-place ``J`` / ``K`` and the zero rows of new outputs outside
    the plane range follow ``fock_from_density``.  Complex ``u`` or densities are refused.  Returns ``(J, K)``."""
    u = _device_tensor(u, "u")
    rho = _device_tensor(rho, "rho")
    if rho.dim() != 3 or rho.shape[0] < 1 or rho.shape[1] != rho.shape[2]:
        raise ValueError(f"rho must be a batch (k, n, n) of k >= 1 densities, got {tuple(rho.shape)}")
    k, n = rho.shape[0], rho.shape[1]
    p0, p1 = (0, n) if planes is None else (int(planes[0]), int(planes[1]))
    if not 0 <= p0 <= p1 <= n:
        raise ValueError(f"planes {planes} out of range for n = {n}")
    if tuple(u.shape) != (p1 - p0, n, n, n):
        raise ValueError(f"u must be (planes, n, n, n) = {(p1 - p0, n, n, n)}, got {tuple(u.shape)}")
    for name, t in (("rho", rho), ("J", J), ("K", K)):
        if t is not None and isinstance(t, torch.Tensor) and t.device != u.device:
            raise ValueError(f"{name} lives on {t.device}, u on {u.device}")
    whole = (p0, p1) == (0, n)
    J, K = (_plane_output(name, out, (k, n, n), torch.float64, u.device, whole) for name, out in (("J", J), ("K", K)))
    if J.dtype != torch.float64 or K.dtype != torch.float64:
        raise ValueError(f"J and K must be float64, got {J.dtype} and {K.dtype}")
    entry = "qs_coulomb_exchange_batch"
    owner, ws, nbytes = _entry_workspace(entry, u.device, n, min(k, COULOMB_EXCHANGE_MAX_BATCH), p0, p1, _code(u),
                                         _code(rho))
    for d0 in range(0, k, COULOMB_EXCHANGE_MAX_BATCH):
        d1 = min(k, d0 + COULOMB_EXCHANGE_MAX_BATCH)
        _native.call(entry, _ptr(u), _code(u), _ptr(rho[d0:d1]), _code(rho), n, d1 - d0, _ptr(J[d0:d1]),
                     _ptr(K[d0:d1]), p0, p1, ws, nbytes, _stream())
    owner.record_stream(torch.cuda.current_stream())
    return J, K


def odqd_coulomb(C, inner_grid, alpha, a, planes=None):
    """Grid Coulomb elements ``u_abcd`` of the 1-D quantum dot (reference one_dim_qd.py:275-280).
    ``C``: (G', l) eigenvectors on the interior grid; ``inner_grid``: (G',).  ``planes=(a0, a1)`` builds only the
    leading-index planes ``u[a0:a1]`` (multi-GPU shard; no communication)."""
    C = _device_tensor(C, "C")
    inner_grid = _device_tensor(inner_grid, "inner_grid")
    if C.dtype != torch.float64 or inner_grid.dtype != torch.float64:
        raise TypeError("the ODQD grid build is real float64")
    Gp, l = C.shape
    if tuple(inner_grid.shape) != (Gp,):
        raise ValueError("inner_grid must have one entry per row of C")
    a0, a1 = (0, l) if planes is None else planes
    out = torch.empty((a1 - a0, l, l, l), dtype=torch.float64, device=C.device)
    nbytes = ctypes.c_int64(0)
    _native.call("qs_odqd_coulomb_workspace_bytes", l, Gp, ctypes.byref(nbytes))
    owner, ws = _workspace(nbytes.value, C.device)
    _native.call(
        "qs_odqd_coulomb_planes", _ptr(C), _ptr(inner_grid), float(alpha), float(a), l, Gp, _ptr(out), a0, a1, ws,
        nbytes.value, _stream(),
    )
    owner.record_stream(torch.cuda.current_stream())
    return out


def probe_dmma_tflops():
    """Measured FP64 tensor-pipe peak (register-resident DMMA.8x8x4 loop) in TFLOP/s."""
    val = ctypes.c_double(0.0)
    _native.call("qs_probe_dmma_tflops", ctypes.byref(val), _stream())
    return val.value


def probe_copy_gbs(nbytes=1 << 32):
    """Measured streaming-copy bandwidth in GB/s (read + write bytes)."""
    scratch = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    scratch.zero_()
    val = ctypes.c_double(0.0)
    _native.call("qs_probe_copy_gbs", ctypes.byref(val), _ptr(scratch), nbytes, _stream())
    return val.value


def spin_squared_two_body(sx, sy, sz, anti_symmetrize=False, planes=None):
    """``sum_i S_i[p,r] S_i[q,s]`` (minus the r<->s exchange when anti-symmetrised) from the three
    (n, n) spin matrices (reference basis_set.py:743-747, :523-526)."""
    mats = [_device_tensor(m, "spin matrix").to(torch.complex128).contiguous() for m in (sx, sy, sz)]
    n = mats[0].shape[0]
    p0, p1 = (0, n) if planes is None else planes
    out = torch.empty((p1 - p0, n, n, n), dtype=torch.complex128, device=mats[0].device)
    _native.call(
        "qs_spin_squared_two_body", _ptr(mats[0]), _ptr(mats[1]), _ptr(mats[2]), n, int(bool(anti_symmetrize)),
        _ptr(out), p0, p1, _stream(),
    )
    return out


def transform_functions(spf, coeff, bra):
    """Grid orbitals under a basis change, one quarter GEMM over the grid points.

    ket (``bra=False``): ``out[p, g] = sum_a C[a, p] spf[a, g]``        (reference basis_set.py:321-323)
    bra (``bra=True``):  ``out[p, g] = sum_a C_tilde[p, a] bra_spf[a, g]``  (reference basis_set.py:325-327)
    """
    spf = _device_tensor(spf, "spf")
    coeff = _device_tensor(coeff, "coefficients")
    n = spf.shape[0]
    grid_shape = tuple(spf.shape[1:])
    G = 1
    for extent in grid_shape:
        G *= extent
    if bra:
        m = coeff.shape[0]
        if coeff.shape[1] != n:
            raise ValueError("C_tilde must be (l_new, l_old)")
        sk, sw = 1, n
    else:
        m = coeff.shape[1]
        if coeff.shape[0] != n:
            raise ValueError("C must be (l_old, l_new)")
        sk, sw = m, 1
    out_dtype = _result_dtype(spf, coeff)
    # A[g, a] = spf[a, g]: the contracted index must be contiguous (pure data movement), pitch even for TMA
    pitch = n if spf.dtype == torch.complex128 else n + (n & 1)
    A = torch.zeros((G, pitch), dtype=spf.dtype, device=spf.device)
    A[:, :n] = spf.reshape(n, G).transpose(0, 1)
    image = coeff_image(coeff, n, m, spf.dtype, sk, sw)
    out = torch.empty((m,) + grid_shape, dtype=out_dtype, device=spf.device)
    quarter_transform(A, G, n, pitch, image, coeff.dtype, m, out, G, 1, 0, 1, 0, G)
    return out


def fock_gathered(h, direct, exchange, n_occ, scale_direct, scale_exchange, f=None):
    """Fock reduction on pre-gathered ``(n_occ, n, n)`` blocks (host-resident ``u``: only the needed
    elements are staged into HBM)."""
    h = _device_tensor(h, "h")
    direct = _device_tensor(direct, "direct")
    exchange = _device_tensor(exchange, "exchange") if exchange is not None else None
    n = h.shape[0]
    if f is None:
        f = torch.empty_like(h)
    else:
        _mark_written(f)
    _native.call(
        "qs_fock_gathered", _ptr(h), _code(h), _ptr(direct), _ptr(exchange), _code(direct), n, int(n_occ),
        float(scale_direct), float(scale_exchange), _ptr(f), _stream(),
    )
    return f


def tdho_coulomb(n, m, scale=1.0, planes=None, device=None):
    """Two-dimensional harmonic-oscillator Coulomb elements ``u[p,q,r,s] = scale * coulomb_ho(nm_p, nm_q,
    nm_r, nm_s)`` for host integer arrays of radial / angular quantum numbers (reference
    quantum_dots/two_dim/coulomb_elements.py:6-92 driven by two_dim_helper.py:250-268, :283-300).
    ``planes=(p0, p1)`` restricts the leading index (multi-GPU shard)."""
    import numpy as _numpy

    n = _numpy.ascontiguousarray(n, dtype=_numpy.int64)
    m = _numpy.ascontiguousarray(m, dtype=_numpy.int64)
    if n.ndim != 1 or n.shape != m.shape or n.size == 0:
        raise ValueError("n and m must be equally long 1-D integer arrays")
    l = int(n.size)
    p0, p1 = (0, l) if planes is None else planes
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else device
    i64p = ctypes.POINTER(ctypes.c_int64)
    n_ptr, m_ptr = n.ctypes.data_as(i64p), m.ctypes.data_as(i64p)
    nbytes = ctypes.c_int64(0)
    _native.call("qs_tdho_coulomb_workspace_bytes", n_ptr, m_ptr, l, ctypes.byref(nbytes))
    out = torch.empty((p1 - p0, l, l, l), dtype=torch.float64, device=device)
    owner, ws = _workspace(nbytes.value, device)
    _native.call(
        "qs_tdho_coulomb", n_ptr, m_ptr, l, float(scale), _ptr(out), p0, p1, ws, nbytes.value, _stream()
    )
    owner.record_stream(torch.cuda.current_stream())
    return out


def _bounds(sl, extent):
    """``slice`` / ``(start, stop)`` / ``None`` -> (start, stop) with numpy's clipping; unit step only."""
    if sl is None:
        return 0, extent
    if isinstance(sl, slice):
        start, stop, step = sl.indices(extent)
        if step != 1:
            raise ValueError("only unit-step slices are supported")
        return start, max(stop, start)
    start, stop = sl
    return int(start), int(stop)


def extract_block(u, a=None, b=None, c=None, d=None):
    """Dense copy of ``u[a, b, c, d]`` for unit-step slices -- the ``u[o, o, v, v]`` blocks solvers cut out
    with ``system.o`` / ``system.v`` (reference system.py:47-51).  ``u`` may be a leading-index shard
    ``(planes, n, n, n)``; ``a`` is then relative to the shard."""
    u = _device_tensor(u, "u")
    n = u.shape[-1]
    if u.dim() != 4 or tuple(u.shape[1:]) != (n, n, n):
        raise ValueError(f"u must be (planes,n,n,n), got {tuple(u.shape)}")
    (a0, a1), (b0, b1), (c0, c1), (d0, d1) = _bounds(a, u.shape[0]), _bounds(b, n), _bounds(c, n), _bounds(d, n)
    out = torch.empty((a1 - a0, b1 - b0, c1 - c0, d1 - d0), dtype=u.dtype, device=u.device)
    _native.call(
        "qs_extract_block", _ptr(u), _code(u), n, u.shape[0], a0, a1, b0, b1, c0, c1, d0, d1, _ptr(out), _stream()
    )
    return out


def scale_add(x, alpha, y=None, beta=0.0, out=None):
    """``alpha x + beta y`` (``y`` optional) in one pass; ``out`` may be ``x`` itself (reference
    system.py:189-215, time_evolution_operators/operator.py:182-196)."""
    x = _device_tensor(x, "x")
    alpha, beta = complex(alpha), complex(beta)
    if y is not None:
        y = _device_tensor(y, "y")
        if y.shape != x.shape:
            raise ValueError("x and y must have the same shape")
    needs_complex = alpha.imag != 0 or beta.imag != 0 or (y is not None and y.dtype != x.dtype)
    if needs_complex:
        x = x.to(torch.complex128)
        y = y.to(torch.complex128) if y is not None else None
    if out is None:
        out = torch.empty_like(x)
    elif out.dtype != x.dtype or out.shape != x.shape or not out.is_contiguous():
        raise ValueError("out must be a contiguous tensor of the result's shape and dtype")
    else:
        _mark_written(out)
    _native.call(
        "qs_scale_add", _ptr(x), _ptr(y), _code(x), x.numel(), alpha.real, alpha.imag, beta.real, beta.imag,
        _ptr(out), _stream(),
    )
    return out


def occupied_traces(h, u, n_occ, planes=None):
    """``(tr h[o,o], sum_ij u[i,j,i,j], sum_ij u[i,j,j,i])`` over the occupied corner as a complex128 device
    tensor of three entries (reference general_orbital_system.py:113-117, spatial_orbital_system.py:144-148).
    ``planes=(p0, p1)``: ``u`` is the leading-index shard holding planes ``[p0, p1)`` and only ``i`` in that
    range is summed (partial sums of one rank)."""
    h = _device_tensor(h, "h")
    u = _device_tensor(u, "u")
    n = h.shape[0]
    p0, p1 = (0, n) if planes is None else planes
    if tuple(h.shape) != (n, n) or tuple(u.shape) != (p1 - p0, n, n, n):
        raise ValueError(f"h must be (n,n) and u (planes,n,n,n), got {tuple(h.shape)} and {tuple(u.shape)}")
    out = torch.empty(3, dtype=torch.complex128, device=h.device)
    _native.call(
        "qs_occupied_traces", _ptr(h), _code(h), _ptr(u), _code(u), n, int(n_occ), p0, p1, _ptr(out), _stream()
    )
    return out


def transform_two_body_diagonal(w2d, C, C_tilde=None, anti_symmetrize=False):
    """``u'_pqrs = sum_ab C~[p,a] C[a,r] C~[q,b] C[b,s] W[a,b]`` for a two-body operator stored by its
    diagonal ``W`` (sinc-DVR ``u_repr = "2d"``), optionally minus the ``r <-> s`` exchange (reference
    sinc_dvr/one_dim/sinc_dvr.py:217-252)."""
    w2d = _device_tensor(w2d, "u (2d)")
    C, C_tilde = _coefficients(C, C_tilde)
    n, m = C.shape
    if tuple(w2d.shape) != (n, n):
        raise ValueError(f"the 2d two-body operator must be {(n, n)}, got {tuple(w2d.shape)}")
    out = torch.empty((m, m, m, m), dtype=_result_dtype(w2d, C), device=w2d.device)
    nbytes = ctypes.c_int64(0)
    _native.call(
        "qs_transform_two_body_diagonal_workspace_bytes", n, m, _code(w2d), _code(C), int(bool(anti_symmetrize)),
        ctypes.byref(nbytes),
    )
    owner, ws = _workspace(nbytes.value, w2d.device)
    _native.call(
        "qs_transform_two_body_diagonal", _ptr(w2d), _code(w2d), _ptr(C), _ptr(C_tilde), _code(C), n, m,
        int(bool(anti_symmetrize)), _ptr(out), ws, nbytes.value, _stream(),
    )
    owner.record_stream(torch.cuda.current_stream())
    return out
