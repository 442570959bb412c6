"""Host side of tests/test_gpu_large_offsets.py: every case's shape crosses the offset it is listed under, one step
smaller does not, its planned peak fits the per-case budget, and the two checkers (the exact comparison of hash-coded
data movement, tests/large_offsets.py, and the sweep of tests/sharded_bounds.py) fail each defect a wrapped 32-bit
offset would cause.  The defects are built by torch indexing on small CPU tensors with the boundary at 2**8."""

import numpy as np
import pytest

import large_offsets as LO
import precise as P

torch = pytest.importorskip("torch")
import sharded_bounds as SB  # noqa: E402  (needs torch)

B8 = 2**8
# more than one case may hold on one B200: the square S32 transform (u, the result and a workspace of 3 n^4 doubles)
# and the configs[5]-like shard above 2**31 with both ranks' slabs, spares, recv and scratch on one device
OVER_BUDGET = {"transform-257-real", "sharded-257-two-ranks"}


@pytest.mark.parametrize("name", sorted(LO.CASES))
def test_case_crosses_its_boundary_and_fits_the_plan(name):
    case = LO.CASES[name]
    assert case.offset(case.extent) >= case.boundary, f"{name}: largest offset {case.offset(case.extent)}"
    if case.minimal:
        assert case.offset(case.extent - 1) < case.boundary, f"{name}: extent {case.extent - 1} crosses too"
    planned = LO.planned_bytes(name)
    if name in OVER_BUDGET:
        assert planned > LO.BUDGET, f"{name}: {planned / 1e9:.1f} GB now fits; run it"
    else:
        assert planned <= LO.BUDGET, f"{name}: {planned / 1e9:.1f} GB > budget {LO.BUDGET / 1e9:.0f} GB"


def test_hash_code_is_exact_and_spread():
    lin = torch.arange(0, 2**20, dtype=torch.int64) * 4099 + (2**32 - 2**19)
    for salt in range(8):
        h = LO.hash_code(lin, salt)
        assert int(h.min()) >= 0 and int(h.max()) <= LO.MASK
        assert torch.equal(h.to(torch.float64).to(torch.int64), h)  # below 2**53: exact in FP64
        assert h.unique().numel() >= lin.numel() - 8  # 2**20 draws from 2**40 codes: a collision or two
    assert not torch.equal(LO.hash_code(lin, 0), LO.hash_code(lin, 1))
    # a difference of the hash-coded tensor depends on where it is taken, not only on the index distance
    d = LO.hash_code(lin + 5) - LO.hash_code(lin)
    assert d.unique().numel() > lin.numel() // 2


# --------------------------------------------------------------------- anti-symmetrise: the exact comparison
# u is (8, 4, 4, 4): 512 elements, planes 4..7 past the boundary 2**8 (one plane is 64 elements).


def simulated_antisymmetrize(u, wrap_direct=False, wrap_partner=False, partner_plane=None):
    """``u - u.transpose(0, 1, 3, 2)`` formed by torch indexing on the flat tensor, the direct and / or partner
    element read from ``offset mod 2**8`` past the boundary, or the partner of plane ``partner_plane[0]`` taken from
    plane ``partner_plane[1]``."""
    n = u.shape[-1]
    p, q, r, s = LO.axes(0, u.shape[0], n, "cpu")
    direct, partner = LO.lin4(p, q, r, s, n), LO.lin4(p, q, s, r, n)
    if wrap_direct:
        direct = direct % B8
    if wrap_partner:
        partner = partner % B8
    if partner_plane is not None:
        bad, src = partner_plane
        partner = torch.where(p == bad, partner - (bad - src) * n**3, partner)
    flat = u.reshape(-1)
    return flat[direct] - flat[partner]


def coded_tensor(code, shape, dtype):
    return code(torch.arange(int(np.prod(shape)), dtype=torch.int64).view(shape), dtype)


@pytest.mark.parametrize("dtype", [torch.float64, torch.complex128])
def test_exact_check_rejects_wrapped_offsets(dtype):
    shape, n = (8, 4, 4, 4), 4
    u = coded_tensor(LO.coded, shape, dtype)
    want = LO.antisymmetrized(n, dtype)
    LO.assert_exact(simulated_antisymmetrize(u), want, "correct", B8)
    for defect in ({"wrap_direct": True, "wrap_partner": True}, {"wrap_partner": True}, {"partner_plane": (6, 2)}):
        with pytest.raises(AssertionError, match="x 256"):
            LO.assert_exact(simulated_antisymmetrize(u, **defect), want, str(defect), B8)
    unwritten = simulated_antisymmetrize(u)
    unwritten[5] = float("nan")
    with pytest.raises(AssertionError, match=r"element \(5, 0, 0, 0\) at offset 320"):
        LO.assert_exact(unwritten, want, "plane 5 never written", B8)
    with pytest.raises(AssertionError, match="do not reach"):
        LO.assert_exact(simulated_antisymmetrize(u)[:4], want, "too small", B8)


def test_lin_code_hides_a_wrapped_plane_that_the_hash_exposes():
    """With ``u = lin`` every plane of the anti-symmetrised tensor is ``(r - s)(n - 1)``: reading planes past the
    boundary from ``offset mod 2**8`` still passes.  The hash-coded input fails the same defect."""
    shape, n = (8, 4, 4, 4), 4
    u = coded_tensor(LO.lin_coded, shape, torch.float64)
    wrapped = simulated_antisymmetrize(u, wrap_direct=True, wrap_partner=True)
    LO.assert_exact(wrapped, LO.antisymmetrized(n, torch.float64, code=LO.lin_coded), "lin-coded, wrapped", B8)
    u = coded_tensor(LO.coded, shape, torch.float64)
    with pytest.raises(AssertionError):
        LO.assert_exact(simulated_antisymmetrize(u, wrap_direct=True, wrap_partner=True),
                        LO.antisymmetrized(n, torch.float64), "hash-coded, wrapped", B8)


# ------------------------------------------------------------------------- the sweep of a single-GPU result
# A ⊗ B at n = 5: 625 elements, planes 2..4 past 2**8 (one plane is 125 elements).


def wrap_planes(t):
    """Every element at offset >= 2**8 read from ``offset mod 2**8``."""
    flat = t.reshape(-1).clone()
    lin = torch.arange(flat.numel())
    return flat[torch.where(lin >= B8, lin % B8, lin)].view(t.shape)


@pytest.mark.parametrize("anti", [False, True])
def test_sweep_rejects_wrapped_offsets(anti):
    n = 5
    rng = np.random.default_rng(5 + anti)
    A, B = P.dyadic(rng, (n, n)), P.dyadic(rng, (n, n))
    C = rng.standard_normal((n, n))
    arrays, k = (A, B, C, C.T), P.k_transform([n] * 4, [False] * 4)
    planes = list(range(n))
    ref = P.kron_transform_planes(*(P.cast(x, P.LD) for x in arrays), planes=planes, dt=P.LD, anti=anti)
    good = torch.from_numpy(ref.astype(P.F64))

    def sweep(t):
        return SB.sweep_slabs([("whole tensor", 0, t)], P.kron_factors, arrays, k, anti, "A ⊗ B", chunk=2,
                              boundary=B8)

    assert sweep(good) <= 1.0
    with pytest.raises(AssertionError, match="x 256"):
        sweep(wrap_planes(good))
    nan_plane = good.clone()
    nan_plane[3] = float("nan")
    with pytest.raises(AssertionError, match=r"fails at element \(3, 0, 0, 0\)"):
        sweep(nan_plane)
    if anti:
        # the exchange term of the planes past the boundary taken from the wrapped plane
        direct = torch.from_numpy(P.kron_transform_planes(*arrays, planes=planes).astype(P.F64))
        exchange = direct - good
        with pytest.raises(AssertionError, match="x 256"):
            sweep(direct - wrap_planes(exchange))
    with pytest.raises(AssertionError, match="no slab reaches"):
        SB.sweep_slabs([("", 0, good[:2])], P.kron_factors, arrays, k, anti, "small", boundary=B8)
