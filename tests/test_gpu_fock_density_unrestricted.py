"""qs_fock_density_unrestricted (ops.fock_from_density_unrestricted, ShardedBasisSet.fock_from_density_unrestricted):
both UHF Fock matrices of two spin densities against an einsum, against three single-density builds, and bit for bit
across shards and calls."""

import ctypes
import itertools

import numpy as np
import pytest

from conftest import assert_close_scaled

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

DTYPES = [torch.float64, torch.complex128]


def rand(gen, shape, dtype):
    x = torch.randn(shape, dtype=torch.float64, device="cuda", generator=gen)
    if dtype == torch.complex128:
        x = torch.complex(x, torch.randn(shape, dtype=torch.float64, device="cuda", generator=gen))
    return x


def reference(h, u, rho_a, rho_b):
    dt = torch.promote_types(torch.promote_types(h.dtype, u.dtype), rho_a.dtype)
    h, u, rho_a, rho_b = (t.to(dt) for t in (h, u, rho_a, rho_b))
    direct = torch.einsum("prqs,sr->pq", u, rho_a + rho_b)
    return (h + direct - torch.einsum("prsq,sr->pq", u, rho_a), h + direct - torch.einsum("prsq,sr->pq", u, rho_b))


def inputs(n, u_dt, rho_dt, h_dt, seed=None):
    gen = torch.Generator(device="cuda").manual_seed(n if seed is None else seed)
    return (rand(gen, (n,) * 4, u_dt), rand(gen, (n, n), rho_dt), rand(gen, (n, n), rho_dt), rand(gen, (n, n), h_dt))


@pytest.mark.parametrize("n", [1, 2, 3, 7, 64, 65, 130])
@pytest.mark.parametrize("u_dt,rho_dt,h_dt", list(itertools.product(DTYPES, repeat=3)),
                         ids=lambda d: "c" if d == torch.complex128 else "r")
def test_matches_einsum(n, u_dt, rho_dt, h_dt):
    from quantum_systems_b200 import ops

    u, rho_a, rho_b, h = inputs(n, u_dt, rho_dt, h_dt)
    refs = reference(h, u, rho_a, rho_b)
    got = ops.fock_from_density_unrestricted(h, u, rho_a, rho_b)
    for f, ref in zip(got, refs):
        assert f.dtype == ref.dtype
        assert_close_scaled(f.cpu().numpy(), ref.cpu().numpy(), 1e-13)
    k = n // 2
    for p0, p1 in ((k, k), (k, k + 1), (n - 1, n)):
        fa = torch.full((n, n), 7.0, dtype=refs[0].dtype, device="cuda")
        fb = torch.full((n, n), 7.0, dtype=refs[0].dtype, device="cuda")
        out = ops.fock_from_density_unrestricted(h, u[p0:p1], rho_a, rho_b, f_alpha=fa, f_beta=fb, planes=(p0, p1))
        assert out[0] is fa and out[1] is fb
        untouched = np.ones(n, dtype=bool)
        untouched[p0:p1] = False
        for f, ref in zip(out, refs):
            got_np = f.cpu().numpy()
            if p1 > p0:
                assert_close_scaled(got_np[p0:p1], ref.cpu().numpy()[p0:p1], 1e-13)
            assert np.all(got_np[untouched] == 7.0), f"rows outside [{p0}, {p1}) were written"


@pytest.mark.parametrize("n,u_dt,rho_dt", [(64, torch.float64, torch.float64), (65, torch.float64, torch.float64),
                                           (40, torch.complex128, torch.complex128), (33, torch.float64, torch.complex128)])
def test_agrees_with_three_single_density_builds(n, u_dt, rho_dt):
    """f_s = J[rho_a + rho_b] - K[rho_s] from qs_fock_density: one direct-only build, two exchange-only builds."""
    from quantum_systems_b200 import ops

    u, rho_a, rho_b, h = inputs(n, u_dt, rho_dt, u_dt)
    direct = ops.fock_from_density(h, u, rho_a + rho_b, 1.0, 0.0)
    zero = torch.zeros_like(h)
    fa, fb = ops.fock_from_density_unrestricted(h, u, rho_a, rho_b)
    assert_close_scaled(fa.cpu().numpy(), (direct + ops.fock_from_density(zero, u, rho_a, 0.0, -1.0)).cpu().numpy(), 1e-13)
    assert_close_scaled(fb.cpu().numpy(), (direct + ops.fock_from_density(zero, u, rho_b, 0.0, -1.0)).cpu().numpy(), 1e-13)


# 37 and 41 split unevenly over 2, 3 and 7 ranks; 40 (even rows, 16-byte loads) over 3 and 7
@pytest.mark.parametrize("n,u_dt,rho_dt", [(37, torch.float64, torch.float64), (40, torch.float64, torch.float64),
                                           (41, torch.complex128, torch.complex128), (40, torch.float64, torch.complex128)])
def test_deterministic_and_bit_identical_across_shards(n, u_dt, rho_dt):
    from quantum_systems_b200 import ops, sharded

    u, rho_a, rho_b, h = inputs(n, u_dt, rho_dt, u_dt, seed=2)
    first = ops.fock_from_density_unrestricted(h, u, rho_a, rho_b)
    again = ops.fock_from_density_unrestricted(h, u, rho_a, rho_b)
    assert all(torch.equal(a, b) for a, b in zip(first, again))
    for world in (2, 3, 7):
        basis = sharded.ShardedBasisSet.from_global(sharded.EmulatedContext(world), h, None, u)
        got = basis.fock_from_density_unrestricted(h, rho_a, rho_b)
        assert all(torch.equal(a, b) for a, b in zip(got, first)), f"world {world}: sharded rows differ"


def test_f_arguments_and_errors():
    from quantum_systems_b200 import _native, ops

    n = 6
    u, rho_a, rho_b, h = inputs(n, torch.float64, torch.float64, torch.float64, seed=3)
    fa = torch.empty((n, n), dtype=torch.float64, device="cuda")
    fb = torch.empty((n, n), dtype=torch.float64, device="cuda")
    va, vb = fa._version, fb._version
    ops.fock_from_density_unrestricted(h, u, rho_a, rho_b, f_alpha=fa, f_beta=fb)
    assert fa._version > va and fb._version > vb
    with pytest.raises(RuntimeError, match="complex u cannot be accumulated into a real Fock matrix"):
        ops.fock_from_density_unrestricted(h, u.to(torch.complex128), rho_a, rho_b, f_alpha=fa, f_beta=fb)
    with pytest.raises(RuntimeError, match="complex u cannot be accumulated into a real Fock matrix"):
        ops.fock_from_density_unrestricted(h, u, rho_a, rho_b.to(torch.complex128), f_alpha=fa, f_beta=fb)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.fock_from_density_unrestricted(h, u, rho_a.cpu(), rho_b)
    need = ctypes.c_int64(0)
    _native.call("qs_fock_density_unrestricted_workspace_bytes", n, 0, n, 0, 0, ctypes.byref(need))
    ws = torch.empty(need.value, dtype=torch.uint8, device="cuda")
    args = [ops._ptr(h), 0, ops._ptr(u), 0, ops._ptr(rho_a), ops._ptr(rho_b), 0, n, ops._ptr(fa), ops._ptr(fb), 0, 0, n,
            ops._ptr(ws)]
    with pytest.raises(RuntimeError, match="workspace too small"):
        _native.call("qs_fock_density_unrestricted", *args, need.value - 1, ops._stream())
    with pytest.raises(RuntimeError, match="bad row range"):
        _native.call("qs_fock_density_unrestricted", *args[:11], 0, n + 1, args[13], need.value, ops._stream())
    with pytest.raises(RuntimeError, match="bad dtype"):
        _native.call("qs_fock_density_unrestricted", *args[:6], 5, *args[7:], need.value, ops._stream())
    with pytest.raises(RuntimeError, match="bad arguments"):
        _native.call("qs_fock_density_unrestricted", *args[:5], ctypes.c_void_p(0), *args[6:], need.value,
                     ops._stream())
