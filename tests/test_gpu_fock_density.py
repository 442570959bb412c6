"""qs_fock_density (ops.fock_from_density, ShardedBasisSet.fock_from_density): the Fock matrix of a general
density matrix against an einsum, against the diagonal-density Fock kernels, and bit for bit across shards."""

import itertools

import numpy as np
import pytest

from conftest import assert_close_scaled

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

SCALES = [(1.0, 0.0), (1.0, -0.5), (1.0, -1.0), (0.0, 1.0)]
DTYPES = [torch.float64, torch.complex128]


def rand(gen, shape, dtype):
    x = torch.randn(shape, dtype=torch.float64, device="cuda", generator=gen)
    if dtype == torch.complex128:
        x = torch.complex(x, torch.randn(shape, dtype=torch.float64, device="cuda", generator=gen))
    return x


def reference(h, u, rho, a_d, a_x):
    dt = torch.promote_types(torch.promote_types(h.dtype, u.dtype), rho.dtype)
    h, u, rho = h.to(dt), u.to(dt), rho.to(dt)
    return h + a_d * torch.einsum("prqs,sr->pq", u, rho) + a_x * torch.einsum("prsq,sr->pq", u, rho)


def plane_ranges(n):
    k = n // 2
    return {"whole": (0, n), "empty": (k, k), "single": (k, k + 1), "last": (n - 1, n)}


@pytest.mark.parametrize("n", [1, 2, 3, 5, 31, 32, 33, 64, 127, 130])
@pytest.mark.parametrize("u_dt,rho_dt,h_dt", list(itertools.product(DTYPES, repeat=3)),
                         ids=lambda d: "c" if d == torch.complex128 else "r")
def test_matches_einsum(n, u_dt, rho_dt, h_dt):
    from quantum_systems_b200 import ops

    gen = torch.Generator(device="cuda").manual_seed(n)
    u, rho, h = rand(gen, (n,) * 4, u_dt), rand(gen, (n, n), rho_dt), rand(gen, (n, n), h_dt)
    for a_d, a_x in SCALES:
        ref = reference(h, u, rho, a_d, a_x)
        for name, (p0, p1) in plane_ranges(n).items():
            f = torch.full((n, n), 7.0, dtype=ref.dtype, device="cuda")
            out = ops.fock_from_density(h, u[p0:p1], rho, a_d, a_x, f=f, planes=(p0, p1))
            assert out is f
            got, want = f.cpu().numpy(), ref.cpu().numpy()
            if p1 > p0:
                assert_close_scaled(got[p0:p1], want[p0:p1], 1e-12)
            untouched = np.ones(n, dtype=bool)
            untouched[p0:p1] = False
            assert np.all(got[untouched] == 7.0), f"{name}: rows outside [{p0}, {p1}) were written"
        whole = ops.fock_from_density(h, u, rho, a_d, a_x)
        assert whole.dtype == ref.dtype
        assert_close_scaled(whole.cpu().numpy(), ref.cpu().numpy(), 1e-12)


@pytest.mark.parametrize("n", [129, 258])
def test_real_u_over_several_column_blocks(n):
    """A real row of more than 128 (odd n, 8-byte pieces) or 256 (even n, 16-byte pieces) columns takes several
    column blocks in a CTA; the reference splits a complex rho so that u is never widened to complex."""
    from quantum_systems_b200 import ops

    gen = torch.Generator(device="cuda").manual_seed(n)
    u, h = rand(gen, (n,) * 4, torch.float64), rand(gen, (n, n), torch.float64)
    for rho_dt in DTYPES:
        rho = rand(gen, (n, n), rho_dt)
        ref = reference(h, u, rho.real, 1.0, -0.5)
        if rho.is_complex():
            ref = ref + 1j * (reference(torch.zeros_like(h), u, rho.imag, 1.0, -0.5))
        got = ops.fock_from_density(h, u, rho, 1.0, -0.5)
        assert_close_scaled(got.cpu().numpy(), ref.cpu().numpy(), 1e-12)


@pytest.mark.parametrize("n,n_occ,u_dt", [(24, 5, torch.float64), (33, 7, torch.complex128), (64, 10, torch.float64)])
def test_diagonal_occupied_density_reproduces_the_occupied_fock_kernels(n, n_occ, u_dt):
    from quantum_systems_b200 import ops

    gen = torch.Generator(device="cuda").manual_seed(1)
    u, h = rand(gen, (n,) * 4, u_dt), rand(gen, (n, n), u_dt)
    occ = torch.zeros(n, dtype=torch.float64, device="cuda")
    occ[:n_occ] = 1.0
    general = ops.fock_from_density(h, u, torch.diag(occ), 1.0, 0.0)
    assert_close_scaled(general.cpu().numpy(), ops.fock_general(h, u, n_occ).cpu().numpy(), 1e-12)
    spatial = ops.fock_from_density(h, u, 2 * torch.diag(occ), 1.0, -0.5)
    assert_close_scaled(spatial.cpu().numpy(), ops.fock_spatial(h, u, n_occ).cpu().numpy(), 1e-12)


# 37 and 41 split unevenly over 2, 3 and 7 ranks; 40 (even rows, 16-byte loads) over 3 and 7
@pytest.mark.parametrize("n,u_dt", [(37, torch.float64), (40, torch.float64), (41, torch.complex128)])
def test_deterministic_and_bit_identical_across_shards(n, u_dt):
    from quantum_systems_b200 import ops, sharded

    gen = torch.Generator(device="cuda").manual_seed(2)
    u, rho, h = rand(gen, (n,) * 4, u_dt), rand(gen, (n, n), u_dt), rand(gen, (n, n), u_dt)
    first = ops.fock_from_density(h, u, rho, 1.0, -0.5)
    assert torch.equal(first, ops.fock_from_density(h, u, rho, 1.0, -0.5))
    for world in (2, 3, 7):
        ctx = sharded.EmulatedContext(world)
        basis = sharded.ShardedBasisSet.from_global(ctx, h, None, u)
        got = basis.fock_from_density(h, rho, 1.0, -0.5)
        assert torch.equal(got, first), f"world {world}: sharded rows differ from the single-tensor rows"


def test_f_argument_and_errors():
    from quantum_systems_b200 import ops

    n = 6
    gen = torch.Generator(device="cuda").manual_seed(3)
    u, rho, h = rand(gen, (n,) * 4, torch.float64), rand(gen, (n, n), torch.float64), rand(gen, (n, n), torch.float64)
    f = torch.empty((n, n), dtype=torch.float64, device="cuda")
    v0 = f._version
    ops.fock_from_density(h, u, rho, 1.0, 0.0, f=f)
    assert f._version > v0
    with pytest.raises(RuntimeError, match="complex u cannot be accumulated into a real Fock matrix"):
        ops.fock_from_density(h, u.to(torch.complex128), rho, 1.0, 0.0, f=f)
    with pytest.raises(RuntimeError, match="complex u cannot be accumulated into a real Fock matrix"):
        ops.fock_from_density(h, u, rho.to(torch.complex128), 1.0, 0.0, f=f)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.fock_from_density(h.cpu(), u, rho, 1.0, 0.0)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.fock_from_density(h, u.cpu(), rho, 1.0, 0.0)
