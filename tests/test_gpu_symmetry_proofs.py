"""The shortcuts of the symmetry-aware four-index transform, tested where they can go wrong without an error.

* Stale proofs: ``transform_two_body(symmetry=None)`` trusts the symmetry tag the library put on a tensor it made
  symmetric itself (``ops.proven_symmetry``), and the cached "no imaginary part" answer for complex coefficients.  A
  library entry point that writes into a caller-supplied tensor (``out=``) must void both, including a write through a
  view of the tagged tensor; otherwise the half-pair path runs on data that lost the symmetry.
* Exact sweep: with small integer inputs every product and partial sum is an integer below 2**53, so the FP64 oracle
  and any correct summation order agree BIT FOR BIT.  A dropped, duplicated or misplaced tile or pair cannot hide
  below a relative tolerance; shapes straddle the 64-column mask granule, odd extents above one tile, the
  ``SYMMETRY_MIN_N`` switch and the pair-free m = 1, 2 cases, each in both epilogue modes.
* Cached tables: tile lists and pair tables are cached per device for the life of the process; configurations that
  share a part of the key run back to back and must not pick up each other's tables."""

import numpy as np
import pytest

from conftest import assert_close_scaled
from oracle import qs_oracle as oracle

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

KIND_FLAGS = {"antisym": 1, "exchange": 2, "both": 3}


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def rand(rng, shape, complex_):
    x = rng.standard_normal(shape)
    return x + 1j * rng.standard_normal(shape) if complex_ else x


def integers(rng, shape, bound, complex_):
    x = rng.integers(-bound, bound + 1, size=shape).astype(np.float64)
    return x + 1j * rng.integers(-bound, bound + 1, size=shape) if complex_ else x


def symmetrise(u, kind):
    """The symmetries of ``symmetric_input`` of test_gpu_symmetry.py without its factor 0.5: integers stay integers."""
    if kind in ("exchange", "both"):
        u = u + u.transpose(1, 0, 3, 2)
    if kind in ("antisym", "both"):
        u = u - u.transpose(0, 1, 3, 2)
    return u


def integer_case(rng, n, m, u_complex, c_complex, biorth, kind):
    """u with entries from [-3, 3] made (anti-)symmetric, C and C_tilde from [-2, 2] (Gaussian integers when complex).
    Every partial sum of the transform is bounded by n^4 max|u| max|C|^4 (moduli): below 2**53 all of them are exact
    integers in FP64, whatever the order of summation."""
    u = symmetrise(integers(rng, (n,) * 4, 3, u_complex), kind)
    C = integers(rng, (n, m), 2, c_complex)
    Ct = integers(rng, (m, n), 2, c_complex) if biorth else None
    c_max = max(np.abs(C).max(), np.abs(Ct).max() if Ct is not None else 0.0)
    assert float(n) ** 4 * np.abs(u).max() * c_max**4 < 2.0**53, "inputs too large for exact FP64 arithmetic"
    return u, C, Ct


def assert_equal(got, expected, what):
    """Bit-for-bit comparison on the device (the 97^4 cases are 0.7 GB a tensor)."""
    if not torch.equal(got, expected):
        bad = got != expected
        idx = tuple(int(i) for i in bad.nonzero()[0])
        raise AssertionError(
            f"{what}: {int(bad.sum())} of {got.numel()} elements differ, max |diff| "
            f"{float((got - expected).abs().max()):.3e}; first at {idx}: {complex(got[idx])} != {complex(expected[idx])}"
        )


@pytest.fixture
def modes():
    from quantum_systems_b200 import _native

    lib = _native.load()
    previous = lib.qs_set_bulk_epilogue_mode(-1)  # out of range: query only

    def run(mode, fn):
        lib.qs_set_bulk_epilogue_mode(mode)
        try:
            return fn()
        finally:
            lib.qs_set_bulk_epilogue_mode(previous)

    yield run
    lib.qs_set_bulk_epilogue_mode(previous)


@pytest.fixture
def detections(monkeypatch):
    """Spy on the exact device-side test: every entry is the answer of one detection the transform ran."""
    from quantum_systems_b200 import ops

    calls = []
    real_test = ops.two_body_symmetry

    def spy(*args, **kwargs):
        calls.append(real_test(*args, **kwargs))
        return calls[-1]

    monkeypatch.setattr(ops, "two_body_symmetry", spy)
    return calls


def orthogonal(rng, n, complex_=False):
    return np.linalg.qr(rand(rng, (n, n), complex_))[0]


# ---------------------------------------------------------------------------------------------------------------
# (a) stale proofs
# ---------------------------------------------------------------------------------------------------------------
def tagged_antisymmetric(rng, n):
    from quantum_systems_b200 import ops

    t = ops.anti_symmetrize(dev(rng.standard_normal((n,) * 4)))
    assert ops.proven_symmetry(t) == ops.ANTISYMMETRIC_LAST_PAIR
    return t


def test_scale_add_into_a_tagged_tensor_voids_the_proof(detections):
    from quantum_systems_b200 import ops

    n = 48
    rng = np.random.default_rng(1)
    x = tagged_antisymmetric(rng, n)
    y = dev(rng.standard_normal((n,) * 4))
    C = orthogonal(rng, n)
    assert ops.scale_add(x, 1.0, y, 1.0, out=x) is x
    got = ops.transform_two_body(x, dev(C))
    assert_close_scaled(got.cpu().numpy(), oracle.transform_two_body_elements(x.cpu().numpy(), C))
    assert detections == [0]  # tested afresh, no symmetry found: the four full steps
    assert ops.proven_symmetry(x) == 0


def test_scale_add_through_a_view_of_a_tagged_tensor_voids_the_proof(detections):
    """The tag sits on the tensor object ``x``; the write goes through the contiguous view ``x[2:3]``."""
    from quantum_systems_b200 import ops

    n = 48
    rng = np.random.default_rng(2)
    x = tagged_antisymmetric(rng, n)
    view = x[2:3]
    assert view.is_contiguous()
    ops.scale_add(view, 1.0, dev(rng.standard_normal((1, n, n, n))), 1.0, out=view)
    C = orthogonal(rng, n)
    got = ops.transform_two_body(x, dev(C))
    assert_close_scaled(got.cpu().numpy(), oracle.transform_two_body_elements(x.cpu().numpy(), C))
    assert detections == [0]
    assert ops.proven_symmetry(x) == 0


def test_add_spin_two_body_into_a_tagged_tensor_voids_the_proof(detections):
    from quantum_systems_b200 import ops

    l = 24
    rng = np.random.default_rng(3)
    t = ops.add_spin_two_body(dev(rng.standard_normal((l,) * 4)), anti_symmetrize=True)
    assert ops.proven_symmetry(t) == ops.ANTISYMMETRIC_LAST_PAIR
    v = rng.standard_normal((l,) * 4)
    assert ops.add_spin_two_body(dev(v), anti_symmetrize=False, out=t) is t
    np.testing.assert_array_equal(t.cpu().numpy(), oracle.add_spin_two_body(v))
    C = orthogonal(rng, 2 * l)
    got = ops.transform_two_body(t, dev(C))
    assert_close_scaled(got.cpu().numpy(), oracle.transform_two_body_elements(oracle.add_spin_two_body(v), C))
    assert detections == [0]
    assert ops.proven_symmetry(t) == 0


def test_scale_add_into_real_valued_complex_coefficients_voids_the_cache():
    """Complex C with zero imaginary part: the first transform remembers "real" and runs the split kernel on C.real;
    once ``scale_add(..., out=C)`` has given C imaginary parts, the next transform must use them."""
    from quantum_systems_b200 import ops

    n = 24
    rng = np.random.default_rng(4)
    u = rand(rng, (n,) * 4, True)
    u_dev = dev(u)
    C = dev(orthogonal(rng, n).astype(np.complex128))
    first = ops.transform_two_body(u_dev, C)
    assert C._qs_has_imag[0] is False
    assert_close_scaled(first.cpu().numpy(), oracle.transform_two_body_elements(u, C.cpu().numpy()))
    ops.scale_add(C, 1.0, dev(1j * rng.standard_normal((n, n))), 1.0, out=C)
    again = ops.transform_two_body(u_dev, C)
    assert_close_scaled(again.cpu().numpy(), oracle.transform_two_body_elements(u, C.cpu().numpy()))


def test_fock_into_a_supplied_matrix_marks_it_written():
    from quantum_systems_b200 import ops

    n = 8
    rng = np.random.default_rng(5)
    h, u = dev(rng.standard_normal((n, n))), dev(rng.standard_normal((n,) * 4))
    for fock in (ops.fock_general, ops.fock_spatial):
        f = torch.empty_like(h)
        version = f._version
        assert fock(h, u, 3, f=f) is f
        assert f._version > version


def test_a_chain_on_library_made_tensors_runs_no_detection(detections):
    """Positive control: transforms, reads and writes into OTHER tensors keep the proof of a library-made tensor."""
    from quantum_systems_b200 import ops

    n = 48
    rng = np.random.default_rng(6)
    x = tagged_antisymmetric(rng, n)
    C = orthogonal(rng, n)
    h = dev(rng.standard_normal((n, n)))
    out = ops.transform_two_body(x, dev(C))
    ops.fock_general(h, out, 4, f=torch.empty_like(h))  # reads out, writes f
    ops.scale_add(out, 2.0)  # reads out, writes a new tensor
    ops.extract_block(out, slice(0, 4), slice(0, 4), slice(4, n), slice(4, n))
    out.cpu()
    assert ops.proven_symmetry(out) == ops.ANTISYMMETRIC_LAST_PAIR
    out2 = ops.transform_two_body(out, dev(C))
    assert detections == [] and ops.proven_symmetry(out2) == ops.ANTISYMMETRIC_LAST_PAIR
    expected = oracle.transform_two_body_elements(x.cpu().numpy(), C)
    assert_close_scaled(out.cpu().numpy(), expected)
    assert_close_scaled(out2.cpu().numpy(), oracle.transform_two_body_elements(expected, C), rel=1e-11)


def test_anti_symmetrising_spin_doubling_into_out_keeps_the_tag(detections):
    from quantum_systems_b200 import ops

    l = 24
    rng = np.random.default_rng(7)
    v = rng.standard_normal((l,) * 4)
    t = torch.empty((2 * l,) * 4, dtype=torch.float64, device="cuda")
    t.zero_()
    assert ops.add_spin_two_body(dev(v), anti_symmetrize=True, out=t) is t
    assert ops.proven_symmetry(t) == ops.ANTISYMMETRIC_LAST_PAIR
    C = orthogonal(rng, 2 * l)
    got = ops.transform_two_body(t, dev(C))
    assert detections == []
    spin = oracle.anti_symmetrize_u(oracle.add_spin_two_body(v))
    assert_close_scaled(got.cpu().numpy(), oracle.transform_two_body_elements(spin, C))


# ---------------------------------------------------------------------------------------------------------------
# (b) exact-arithmetic sweep of the symmetry-aware path
# ---------------------------------------------------------------------------------------------------------------
DTYPE_MIXES = [(False, False, False), (True, False, False), (True, True, True), (False, True, False)]
SHAPES = [(63, 63), (64, 64), (65, 65), (97, 97), (65, 63), (50, 97), (97, 50)]
COMPLEX_MAX = 65  # the complex oracle takes seconds per case up to here


def exact_cases():
    for n, m in SHAPES:
        for u_complex, c_complex, biorth in DTYPE_MIXES:
            if (u_complex or c_complex) and max(n, m) > COMPLEX_MAX:
                continue
            for kind in ("antisym", "exchange", "both"):
                yield pytest.param(n, m, u_complex, c_complex, biorth, kind,
                                   id=f"{n}x{m}-u{'c' if u_complex else 'r'}-C{'c' if c_complex else 'r'}"
                                      f"{'-biorth' if biorth else ''}-{kind}")


def check_exact(modes, u, C, Ct, kind, expect_detected=True):
    """Default path, symmetry=0 and every forced symmetry u has, in both epilogue modes: all bit-identical to the
    exact oracle; the result carries the symmetries exactly."""
    from quantum_systems_b200 import ops

    expected = oracle.transform_two_body_elements(u, C, Ct)
    assert np.array_equal(expected, np.round(expected)), "the oracle result is not integer-valued"
    expected = dev(expected)
    u_dev, C_dev, Ct_dev = dev(u), dev(C), None if Ct is None else dev(Ct)
    flags = KIND_FLAGS[kind]
    detected = ops.ANTISYMMETRIC_LAST_PAIR if flags & 1 else ops.PARTICLE_EXCHANGE
    runs = [(None, "default")] + [(0, "symmetry=0")] + [(s, f"symmetry={s}") for s in (1, 2) if flags & s]
    for mode in (0, 2):
        for symmetry, name in runs:
            out = modes(mode, lambda: ops.transform_two_body(u_dev, C_dev, Ct_dev, symmetry=symmetry))
            assert_equal(out, expected, f"{name}, epilogue mode {mode}")
            if symmetry is None:
                assert ops.proven_symmetry(out) == (detected if expect_detected else 0)
            del out
    if flags & 1:
        assert_equal(expected, -expected.transpose(2, 3), "anti-symmetry of the result")
        assert not (expected.diagonal(dim1=2, dim2=3) != 0).any(), "r == s diagonal of an anti-symmetric result"
    if flags & 2:
        assert_equal(expected, expected.permute(1, 0, 3, 2), "exchange symmetry of the result")


@pytest.mark.parametrize("n,m,u_complex,c_complex,biorth,kind", list(exact_cases()))
def test_symmetric_transform_is_exact_on_integers(modes, n, m, u_complex, c_complex, biorth, kind):
    rng = np.random.default_rng(1000 * n + m + 7 * u_complex + 3 * c_complex)
    u, C, Ct = integer_case(rng, n, m, u_complex, c_complex, biorth, kind)
    check_exact(modes, u, C, Ct, kind)


@pytest.mark.parametrize("n,m", SHAPES)
def test_symmetric_transform_on_normal_inputs(n, m):
    """Companion of the integer sweep: rounding is exercised only by non-integer inputs."""
    from quantum_systems_b200 import ops

    rng = np.random.default_rng(n * m)
    for kind in ("antisym", "exchange"):
        u = rand(rng, (n,) * 4, False)
        u = u - u.transpose(0, 1, 3, 2) if kind == "antisym" else 0.5 * (u + u.transpose(1, 0, 3, 2))
        C = rand(rng, (n, m), False)
        out = ops.transform_two_body(dev(u), dev(C))
        assert ops.proven_symmetry(out) == KIND_FLAGS[kind]
        assert_close_scaled(out.cpu().numpy(), oracle.transform_two_body_elements(u, C))


@pytest.mark.parametrize("n,m,detected", [(48, 47, False), (47, 48, False), (48, 48, True)])
@pytest.mark.parametrize("kind", ["antisym", "exchange"])
def test_symmetry_switch_at_the_minimum_extent(modes, detections, n, m, detected, kind):
    """Below ``SYMMETRY_MIN_N`` in n or m a symmetric u is not even tested; at 48 x 48 it is found and exploited."""
    from quantum_systems_b200 import ops

    assert ops.SYMMETRY_MIN_N == 48
    rng = np.random.default_rng(n + 2 * m)
    u, C, Ct = integer_case(rng, n, m, False, False, False, kind)
    check_exact(modes, u, C, Ct, kind, expect_detected=detected)
    assert detections == ([KIND_FLAGS[kind]] * 2 if detected else [])  # once per epilogue mode


@pytest.mark.parametrize("m", [1, 2, 3])
@pytest.mark.parametrize("n", [7, 64])
@pytest.mark.parametrize("complex_", [False, True])
@pytest.mark.parametrize("kind", ["antisym", "exchange"])
def test_forced_symmetry_with_tiny_results(modes, n, m, complex_, kind):
    """m = 1, anti-symmetric: no pair is wanted, the result is the mirror fill alone (all zero); m = 2, 3: one or
    three pairs, padded to aligned couples for real even m."""
    from quantum_systems_b200 import ops

    rng = np.random.default_rng(10 * n + m)
    u, C, _ = integer_case(rng, n, m, complex_, complex_, False, kind)
    expected = dev(oracle.transform_two_body_elements(u, C))
    symmetry = KIND_FLAGS[kind]
    for mode in (0, 2):
        out = modes(mode, lambda: ops.transform_two_body(dev(u), dev(C), symmetry=symmetry))
        assert_equal(out, expected, f"symmetry={symmetry}, epilogue mode {mode}")
        assert ops.proven_symmetry(out) == symmetry
    if kind == "antisym" and m == 1:
        assert not (expected != 0).any()


# ---------------------------------------------------------------------------------------------------------------
# (c) per-device table caches
# ---------------------------------------------------------------------------------------------------------------
def test_cached_tables_across_configurations_in_one_process():
    """Tile lists and pair tables are cached per device.  Real / complex and anti-symmetric (only r < s) / exchange
    (r <= s) alternate at the same M and pitch P = n (64 x 64 real and complex), with a different pitch (66 x 64) in
    between; each result is compared exactly."""
    from quantum_systems_b200 import ops

    sequence = [
        (64, 64, False, "antisym"), (64, 64, True, "antisym"), (66, 64, False, "antisym"),
        (64, 64, False, "exchange"), (64, 64, False, "antisym"), (66, 64, True, "exchange"),
        (64, 64, True, "exchange"), (66, 64, False, "exchange"), (64, 64, True, "antisym"),
        (64, 64, False, "antisym"),
    ]
    rng = np.random.default_rng(64)
    for n, m, complex_, kind in sequence:
        u, C, _ = integer_case(rng, n, m, complex_, complex_, False, kind)
        out = ops.transform_two_body(dev(u), dev(C))
        assert ops.proven_symmetry(out) == KIND_FLAGS[kind]
        assert_equal(out, dev(oracle.transform_two_body_elements(u, C)), f"{n}x{m} {'complex' if complex_ else 'real'} "
                                                                          f"{kind}")
