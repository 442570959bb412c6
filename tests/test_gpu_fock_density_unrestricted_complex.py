"""The one-read unrestricted Fock pass for complex densities on a real u (qs_fock_density_unrestricted, DESIGN
§4.11 / §4.13): both spin Fock matrices against the extended-precision reference under the rounding-error bound,
against single-density builds, bit for bit across uneven shards, and on one u past 2^31 elements."""

import numpy as np
import pytest

import large_offsets as LO
import precise as P

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def host(t):
    return t.cpu().numpy()


def complex_density(rng, n, hermitian, scale=1.0):
    g = P.graded(n)
    x = rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n))
    if hermitian:
        x = x + x.conj().T
    return scale * x * np.outer(g, g)


def summed_fock(h, u, rho_a, rho_b, dt, absolute=False):
    """``h + J[rho_a + rho_b] - K[rho_s]`` with the direct term of the summed density, as the pass forms it."""
    j = np.einsum("prqs,sr->pq", u, rho_a + rho_b)
    return np.stack([P._sub(h + j, np.einsum("prsq,sr->pq", u, r), absolute) for r in (rho_a, rho_b)])


def k_one_read(n):
    """``3 n^2 + 1`` products and sums of a real-u, complex-rho element, and the rounding of rho_a + rho_b."""
    return 3 * n * n + 2


# even n: 16-byte pieces of u; odd n: 8-byte pieces; past 128 columns a row takes two column blocks
@pytest.mark.parametrize("n,hermitian", [(64, True), (65, False), (129, True), (130, False)])
def test_within_the_rounding_bound(n, hermitian):
    from quantum_systems_b200 import ops

    rng = np.random.default_rng(n + 100 * hermitian)
    u = P.graded_two_body(rng, n)
    h = 1e-6 * (rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n)))
    ra, rb = complex_density(rng, n, hermitian), complex_density(rng, n, hermitian, scale=0.5)
    ref, absval, fp64 = P.companions(summed_fock, h, u, ra, rb)
    got = np.stack([host(f) for f in ops.fock_from_density_unrestricted(dev(h), dev(u), dev(ra), dev(rb))])
    P.assert_rounding_bound(got, ref, absval, k_one_read(n), fp64, f"n={n}")


@pytest.mark.parametrize("n", [8, 33, 64])
def test_matches_single_density_builds(n):
    """f_s = J[rho_a + rho_b] - K[rho_s] from qs_fock_density: one direct-only build, two exchange-only builds."""
    from quantum_systems_b200 import ops

    gen = torch.Generator(device="cuda").manual_seed(n)
    u = torch.randn((n,) * 4, dtype=torch.float64, device="cuda", generator=gen)
    ra, rb = (torch.randn((n, n), dtype=torch.complex128, device="cuda", generator=gen) for _ in range(2))
    h = torch.randn((n, n), dtype=torch.float64, device="cuda", generator=gen)
    direct = ops.fock_from_density(h, u, ra + rb, 1.0, 0.0)
    zero = torch.zeros_like(h)
    fa, fb = ops.fock_from_density_unrestricted(h, u, ra, rb)
    for f, rho in ((fa, ra), (fb, rb)):
        want = direct + ops.fock_from_density(zero, u, rho, 0.0, -1.0)
        assert float((f - want).abs().max() / want.abs().max()) <= 1e-13


@pytest.mark.parametrize("n", [37, 40])
def test_bit_identical_across_uneven_shards(n):
    from quantum_systems_b200 import ops, sharded

    gen = torch.Generator(device="cuda").manual_seed(n + 1)
    u = torch.randn((n,) * 4, dtype=torch.float64, device="cuda", generator=gen)
    ra, rb = (torch.randn((n, n), dtype=torch.complex128, device="cuda", generator=gen) for _ in range(2))
    h = torch.randn((n, n), dtype=torch.complex128, device="cuda", generator=gen)
    whole = ops.fock_from_density_unrestricted(h, u, ra, rb)
    assert all(torch.equal(a, b) for a, b in zip(whole, ops.fock_from_density_unrestricted(h, u, ra, rb)))
    for world in (2, 3, 7):
        basis = sharded.ShardedBasisSet.from_global(sharded.EmulatedContext(world), h, None, u)
        got = basis.fock_from_density_unrestricted(h, ra, rb)
        assert all(torch.equal(a, b) for a, b in zip(got, whole)), f"world {world}: sharded rows differ"


def test_u_past_2_31_elements():
    """n = 216 real: u[p,r,q,s] = A[p,q] B[r,s] with 216^4 > 2^31 elements, the reference in the Kronecker form."""
    from quantum_systems_b200 import ops

    n = 216
    assert n**4 > LO.S31
    need = n**4 * 8 + LO._bytes("qs_fock_density_unrestricted_workspace_bytes", n, 0, n, 0, 1) + LO.SCRATCH
    free, _ = torch.cuda.mem_get_info()
    if need > min(free, LO.BUDGET):
        pytest.skip(f"needs {need / 1e9:.1f} GB, {free / 1e9:.1f} GB free")
    rng = np.random.default_rng(216)
    g = P.pow2_graded(n)
    A, B = (P.dyadic(rng, (n, n)) * np.outer(g, g) for _ in range(2))
    Ad, Bd = dev(A), dev(B)
    u = (Ad[:, None, :, None] * Bd[None, :, None, :]).contiguous()
    del Ad, Bd
    h = 1e-6 * (rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n)))
    ra, rb = complex_density(rng, n, True), complex_density(rng, n, False, scale=1e-3)
    got = np.stack([host(f) for f in ops.fock_from_density_unrestricted(dev(h), u, dev(ra), dev(rb))])
    del u
    ref, absval, fp64 = P.companions(P.kron_fock_unrestricted, h, A, B, ra, rb)
    P.assert_rounding_bound(got, ref, absval, k_one_read(n), fp64, "n=216")
