"""The rotated epilogue of the quarter GEMM (the local store w sw1 + (x / x_inner) sx1 + x % x_inner of the dense
transforms, a kernel instantiation of its own) stores exactly what the generic strided epilogue stores.  The same
product is launched twice through ``qs_quarter_transform``: once as a plain rotated store (w_inner = 1, column stride
sw1), which takes the rotated epilogue, and once with the same addresses spelled as one block of W columns at stride
sw0, which takes the generic one.  The results are compared BIT FOR BIT, and against an exact reference: the inputs
are small integers, so every FP64 sum is exact."""

import ctypes

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

QS_F64, QS_C128 = 0, 1
SENTINEL = -7.25  # not an integer: no element the launch writes can equal it


def ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def ints(rng, shape, complex_):
    x = rng.integers(-3, 4, shape).astype(np.float64)
    return x + 1j * rng.integers(-3, 4, shape) if complex_ else x


def quarter(A, a_c, M, m_c, X, K, lda, W, x_inner, sx1, rotated):
    """out[w plane + (x / x_inner) sx1 + x % x_inner] = sum_k A[x, k] M[k, w] through the library."""
    from quantum_systems_b200 import _native

    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    a_dt, m_dt = (QS_C128 if a_c else QS_F64), (QS_C128 if m_c else QS_F64)
    nbytes = ctypes.c_int64(0)
    _native.call("qs_coeff_image_bytes", K, W, a_dt, m_dt, ctypes.byref(nbytes))
    image = torch.empty(nbytes.value // 8, dtype=torch.float64, device="cuda")
    _native.call("qs_build_coeff_image", ptr(M), m_dt, W, 1, 0, K, W, a_dt, ptr(image), stream)
    plane = -(-X // x_inner) * sx1
    out_dtype = torch.complex128 if (a_c or m_c) else torch.float64
    out = torch.full((W * plane,), SENTINEL, dtype=out_dtype, device="cuda")
    w_inner, sw0, sw1 = (1, 0, plane) if rotated else (W, plane, 0)
    _native.call("qs_quarter_transform", ptr(A), a_dt, X, K, lda, ptr(image), m_dt, W, ptr(out), x_inner, 1, sx1,
                 w_inner, sw0, sw1, stream)
    torch.cuda.synchronize()
    return out, plane


def reference(a, m, X, W, x_inner, sx1, plane, complex_):
    ref = np.full(W * plane, SENTINEL, dtype=np.complex128 if complex_ else np.float64)
    x = np.arange(X)
    rows = (x // x_inner) * sx1 + x % x_inner
    ref[(np.arange(W)[:, None] * plane + rows[None, :]).ravel()] = (a @ m).T.ravel()
    return ref


# (A complex, M complex, X, K, W, x_inner, sx1).  X not a multiple of 128, W not a multiple of 8 NT, every NT from
# 1 to 8 (real: ceil(W / 8); complex output: ceil(2 W / 8)), two tile groups, a block pitch sx1 above x_inner, and odd
# blocks and odd X for complex output (real row pairs need even ones: those launches keep the generic epilogue).
CASES = [(False, False, 312, 20, w, 24, 26) for w in (6, 14, 22, 30, 38, 46, 54, 62)] + [
    (False, False, 390, 29, 70, 30, 30),     # odd K (padded pitch), two tile groups (NT = 5 and 4)
    (False, False, 256, 16, 64, 128, 128),   # whole tiles, x_inner = sx1: the plain rotated store of the transforms
] + [(True, True, 299, 12, w, 13, 15) for w in (3, 7, 11, 15, 19, 23, 27, 31)] + [
    (False, True, 507, 13, 13, 13, 13),      # real A x complex M, odd n at its own pitch
    (True, True, 200, 24, 50, 20, 20),       # two tile groups of complex output (NT = 7 and 6)
]


@pytest.mark.parametrize("a_c,m_c,X,K,W,x_inner,sx1", CASES)
def test_rotated_epilogue_is_bit_identical_to_the_generic_one(a_c, m_c, X, K, W, x_inner, sx1):
    rng = np.random.default_rng(X * 131 + K * 7 + W)
    lda = K + (K & 1) if not a_c else K
    a = ints(rng, (X, K), a_c)
    m = ints(rng, (K, W), m_c)
    a_pad = np.zeros((X, lda), dtype=a.dtype)
    a_pad[:, :K] = a
    A = torch.from_numpy(a_pad).cuda()
    M = torch.from_numpy(np.ascontiguousarray(m)).cuda()
    rotated, plane = quarter(A, a_c, M, m_c, X, K, lda, W, x_inner, sx1, rotated=True)
    generic, _ = quarter(A, a_c, M, m_c, X, K, lda, W, x_inner, sx1, rotated=False)
    assert torch.equal(rotated, generic)
    ref = reference(a, m, X, W, x_inner, sx1, plane, a_c or m_c)
    np.testing.assert_array_equal(rotated.cpu().numpy(), ref)
