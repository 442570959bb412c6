"""The sharded spin-orbital system in the UHF basis: the column-table scattering store
(qs_quarter_transform_scatter_columns) against a numpy product, the sharded mixed transform under the rounding
bound of tests/precise.py, and hartree_fock.general_orbital_system_sharded on emulated ranks against the
extended-precision reference, the single-GPU hartree_fock.general_orbital_system and the spin-doubling route."""

import os
import subprocess
import sys

import numpy as np
import pytest

import precise as P

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORLDS = [1, 2, 3, 5, 8]


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def host(a):
    return a.cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)


def rand(rng, shape, complex_=False):
    return rng.standard_normal(shape) + (1j * rng.standard_normal(shape) if complex_ else 0)


class NaNEngine:
    """A CudaEngine whose scratch starts as NaN: an element nobody wrote, or one read before it was written, fails."""

    def __new__(cls):
        from quantum_systems_b200 import sharded

        class Poisoned(sharded.CudaEngine):
            def empty(self, numel, dtype):
                buf = super().empty(numel, dtype)
                buf.tensor.fill_(float("nan"))
                return buf

        return Poisoned()


# -------------------------------------------------------------------------------------- column-table store
# (label, a complex, m complex, destinations, dealt, row split)
COLUMNS = [
    ("real", False, False, 3, False, False),
    ("real dealt 16 destinations", False, False, 16, True, False),
    ("complex", True, True, 5, False, True),
    ("complex dealt", True, True, 8, True, False),
    ("split 2M", True, False, 7, False, False),
    ("split 2M dealt 16 destinations", True, False, 16, True, True),
    ("real A complex M", False, True, 2, True, True),
]


@pytest.mark.parametrize("case", COLUMNS, ids=[c[0] for c in COLUMNS])
def test_column_table_store_against_numpy(case):
    from quantum_systems_b200 import ops, sharded

    label, a_c, m_c, n_dest, dealt, split_rows = case
    rng = np.random.default_rng(len(label) + n_dest)
    X, K, W = 300, 37, 53
    A = rand(rng, (X, K), a_c)
    M = rand(rng, (K, W), m_c)
    out_c = a_c or m_c
    dtype = torch.complex128 if out_c else torch.float64
    deal = ops.scatter_deal(W) if dealt else 1
    assert (deal > 1) == dealt
    a_dtype = torch.complex128 if a_c else torch.float64
    lda = K + (K & 1) if not a_c else K
    A_pad = np.zeros((X, lda), dtype=A.dtype)
    A_pad[:, :K] = A
    A_flat = dev(A_pad).reshape(-1)
    A_buf = sharded.DeviceBuffer(A_flat.data_ptr(), X * lda, a_dtype, tensor=A_flat)
    image = ops.coeff_image(dev(M), K, W, a_dtype, W, 1, deal=deal)
    # rows: three-level split or plain
    if split_rows:
        x_inner, x_mid, sx0, sx1, sx2 = 10, 3, 1, 40, 200
    else:
        x_inner, x_mid, sx0, sx1, sx2 = X, 1, 1, 0, 0
    x = np.arange(X)
    xq = x // x_inner
    ax = (xq // x_mid) * sx2 + (xq % x_mid) * sx1 + (x % x_inner) * sx0
    span = int(ax.max()) + 4
    span += span & 1  # even: the offsets keep the promise of the last argument below
    # uneven destinations, some empty: column w goes to a random destination, in a random slot there
    weights = rng.random(n_dest) * (rng.random(n_dest) > 0.25)
    weights[0] = max(weights[0], 0.1)
    col_dest = rng.choice(n_dest, size=W, p=weights / weights.sum()).astype(np.int32)
    col_off = np.zeros(W, dtype=np.int64)
    slots = [0] * n_dest
    for w in rng.permutation(W):
        col_off[w] = slots[col_dest[w]] * span + 2 * int(rng.integers(0, 2))
        slots[col_dest[w]] += 1
    eng = sharded.CudaEngine()
    bufs = []
    for d in range(n_dest):
        b = eng.empty(max(slots[d], 1) * span, dtype)
        b.tensor.fill_(float("nan"))
        bufs.append(b)
    eng.quarter_scatter_columns(A_buf, X, K, lda, image, torch.complex128 if m_c else torch.float64, W,
                                [(b, 0) for b in bufs], dev(col_dest), dev(col_off), True, x_inner, x_mid, sx0, sx1,
                                sx2, deal=deal)
    torch.cuda.synchronize()
    product = A @ M
    for d, b in enumerate(bufs):
        got = host(b.tensor)
        written = np.zeros(got.shape, dtype=bool)
        for w in np.flatnonzero(col_dest == d):
            idx = col_off[w] + ax
            written[idx] = True
            scale = np.abs(product[:, w]).max()
            assert np.abs(got[idx] - product[:, w]).max() <= 1e-12 * scale * K, f"{label}: column {w}"
        assert np.all(np.isnan(got[~written])), f"{label}: destination {d} has stores outside its columns"


# -------------------------------------------------------------------------------------- sharded mixed transform
MIXED = [
    ("real", 13, False, False, False),
    ("complex explicit bras", 12, True, True, True),
    ("real u complex C", 17, False, True, False),
    ("complex u real C (split)", 16, True, False, True),
]


@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("case", MIXED, ids=[c[0] for c in MIXED])
def test_sharded_mixed_transform_rounding_bound(case, world):
    from quantum_systems_b200 import sharded

    label, n, u_c, c_c, explicit = case
    rng = np.random.default_rng(n * 7 + world)
    u = rand(rng, (n,) * 4, u_c)
    C_r, C_s = rand(rng, (n, n), c_c), rand(rng, (n, n), c_c)
    Ct_p = rand(rng, (n, n), c_c) if explicit else C_r.conj().T
    Ct_q = rand(rng, (n, n), c_c) if explicit else C_s.conj().T
    ref, absval, fp64 = P.companions(P.mixed_steps, u, C_r, C_s, Ct_p, Ct_q)
    ctx = sharded.EmulatedContext(world, engine=NaNEngine())
    basis = sharded.ShardedBasisSet.from_global(ctx, np.eye(n), np.eye(n), u)
    bras = (dev(Ct_p), dev(Ct_q)) if explicit else ()
    first = sharded.transform_two_body_sharded_mixed(basis.u, dev(C_r), dev(C_s), *bras)
    second = sharded.transform_two_body_sharded_mixed(basis.u, dev(C_r), dev(C_s), *bras)
    k = P.k_transform([n] * 4, [u_c or c_c] * 4)
    for out in (first, second):  # the second call neither recycles the first result nor touches u
        P.assert_rounding_bound(host(out.gather()), ref, absval, k, fp64, f"{label} W={world}")
    assert torch.equal(second.gather(), first.gather())
    assert np.array_equal(host(basis.u.gather()), u.astype(host(basis.u.gather()).dtype))
    # the input's spare set is still free for the next plain transform, which chains as before
    basis.change_basis(dev(C_r))


# -------------------------------------------------------------------------------------- the spin-orbital system
def odqd_sharded(ctx, l, potential="ho", real_one_body=False):
    """An ODQD basis sharded from its spatial arrays; ``real_one_body`` takes the real parts of the (real-valued,
    complex-typed) h and s, as a caller asking for a float64 spin-orbital system does."""
    from quantum_systems_b200 import ODQD, sharded

    pot = ODQD.HOPotential(0.25) if potential == "ho" else ODQD.DWPotential(1.0, 5)
    points = 201 if l <= 12 else 801
    od = ODQD(l, 8.0 if potential == "ho" else 10.0, points, potential=pot)
    h, s = (od.h.real, od.s.real) if real_one_body else (od.h, od.s)
    return od, sharded.ShardedBasisSet.from_global(ctx, h, s, od.u)


def random_sharded(ctx, l, complex_):
    from quantum_systems_b200 import sharded

    rng = np.random.default_rng(l)
    u = rand(rng, (l,) * 4, complex_)
    u = 0.05 * (u + u.transpose(1, 0, 3, 2)) / 2  # particle-exchange symmetric, otherwise arbitrary
    u = 0.5 * (u + u.transpose(2, 3, 0, 1).conj())
    h = np.diag(np.arange(l, dtype=np.float64)) + 0.01 * rand(rng, (l, l))
    h = 0.5 * (h + h.T)
    return u, sharded.ShardedBasisSet.from_global(ctx, h, np.eye(l), u)


def uhf_state(basis, n_alpha, n_beta):
    from quantum_systems_b200 import hartree_fock

    state = hartree_fock.ground_state_unrestricted_sharded(basis, n_alpha, n_beta)
    assert state.converged
    return state


def assemble(blocks, orbital, spin, combine):
    """``combine(B[oI,oJ,oK,oL], B[oI,oJ,oL,oK])`` where the spins allow each term (zero otherwise)."""
    n = len(orbital)
    dtype = np.result_type(*blocks.values())
    U = np.zeros((n,) * 4, dtype=dtype)
    o, s = orbital, spin
    for I in range(n):
        for J in range(n):
            A = blocks[(int(s[I]), int(s[J]))][o[I], o[J]]
            direct = np.where((s[:, None] == s[I]) & (s[None, :] == s[J]), A[o[:, None], o[None, :]], 0)
            exchange = np.where((s[None, :] == s[I]) & (s[:, None] == s[J]), A[o[None, :], o[:, None]], 0)
            U[I, J] = combine(direct, exchange)
    return U


def check_system(new, state, n_alpha, n_beta):
    """Exact anti-symmetry (rank by rank), reference energy and Fock matrix of the sharded spin-orbital basis."""
    from quantum_systems_b200 import hartree_fock

    for r in new.ctx.local_ranks:
        slab = new.u.local(r)
        assert torch.equal(slab, -slab.transpose(2, 3))
    n = n_alpha + n_beta
    assert abs(new.compute_reference_energy(n) - state.energy) <= 1e-10 * abs(state.energy)
    _, eps = hartree_fock.spin_orbital_coefficients(state)
    f = host(new.construct_fock_matrix(new.h, new.u, n))
    assert np.abs(f - np.diag(host(eps))).max() <= 1e-7


# (label, basis kind, l, n_alpha, n_beta, out dtype)
SMALL = [
    ("odqd closed shell", "odqd", 8, 2, 2, torch.complex128),
    ("odqd open shell odd l", "odqd", 9, 3, 2, torch.float64),
    ("odqd no beta electrons", "odqd", 7, 2, 0, torch.complex128),
    ("random real", "random_real", 6, 2, 1, torch.float64),
    ("random complex", "random_complex", 5, 2, 1, torch.complex128),
]


@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("case", SMALL, ids=[c[0] for c in SMALL])
def test_small_systems_against_the_extended_precision_reference(case, world):
    from quantum_systems_b200 import hartree_fock, sharded

    label, kind, l, n_alpha, n_beta, out_dtype = case
    ctx = sharded.EmulatedContext(world, engine=NaNEngine())
    if kind == "odqd":
        od, basis = odqd_sharded(ctx, l, real_one_body=out_dtype == torch.float64)
        u = host(od.u)
    else:
        u, basis = random_sharded(ctx, l, kind == "random_complex")
    state = uhf_state(basis, n_alpha, n_beta)
    u_before = basis.u.gather().clone()
    new = hartree_fock.general_orbital_system_sharded(state, basis, out_dtype=out_dtype)
    assert new.includes_spin and new.anti_symmetrized_u and new.u.proven_antisymmetric and new.l == 2 * l
    assert new.u.dtype == out_dtype and (ctx.exchange != "peer" or new.u.spare is not None)
    assert torch.equal(basis.u.gather(), u_before) and not basis.includes_spin
    check_system(new, state, n_alpha, n_beta)
    got = host(new.u.gather())

    Cs = (host(state.C_alpha), host(state.C_beta))
    refs, abss, fp64s = {}, {}, {}
    for s in (0, 1):
        for t in (0, 1):
            refs[(s, t)], abss[(s, t)], fp64s[(s, t)] = P.companions(P.mixed_steps, u, Cs[s], Cs[t],
                                                                     Cs[s].conj().T, Cs[t].conj().T)
    orbital, spin = hartree_fock.spin_orbital_order(n_alpha, n_beta, l)
    ref = assemble(refs, orbital, spin, lambda d, x: d - x)
    absval = assemble(abss, orbital, spin, lambda d, x: d + x)
    fp64 = assemble(fp64s, orbital, spin, lambda d, x: d - x)
    complex_ = np.iscomplexobj(u) or np.iscomplexobj(Cs[0])
    k = P.k_transform([l] * 4, [complex_] * 4) + 1  # + the anti-symmetrising subtraction
    P.assert_rounding_bound(got, ref, absval, k, fp64, f"{label} W={world}")


def test_one_body_side_is_bit_identical_to_the_spin_doubling_route():
    from quantum_systems_b200 import hartree_fock, sharded

    ctx = sharded.EmulatedContext(3)
    od, basis = odqd_sharded(ctx, 10)
    state = uhf_state(basis, 3, 2)
    new = hartree_fock.general_orbital_system_sharded(state, basis)
    route = sharded.ShardedBasisSet.from_spatial(ctx, od.h, od.s, od.u, anti_symmetrize=True)
    route.change_basis(hartree_fock.spin_orbital_coefficients(state)[0])
    assert torch.equal(new.h, route.h) and torch.equal(new.s, route.s)
    assert new.u.dtype == route.u.dtype
    ref = route.u.gather()
    got = new.u.gather()
    assert (got - ref).abs().max() <= 1e-13 * ref.abs().max()
    # into=: the next system is written into the buffers of this one, bit for bit the same
    again = hartree_fock.general_orbital_system_sharded(state, basis, into=new.u)
    assert again.u is new.u and again.u.proven_antisymmetric and torch.equal(again.u.gather(), got)


@pytest.mark.parametrize("world,l,potential,n_alpha,n_beta,complex_u", [
    (8, 64, "ho", 5, 3, False),
    (3, 64, "dw", 2, 2, True),
    (5, 100, "ho", 7, 6, False),
])
def test_against_the_single_gpu_system(world, l, potential, n_alpha, n_beta, complex_u, monkeypatch):
    from quantum_systems_b200 import hartree_fock, sharded

    ctx = sharded.EmulatedContext(world)
    od, basis = odqd_sharded(ctx, l, potential)
    if complex_u:  # complex u of real value: the blocks take the split (2M) quarter GEMMs
        basis = sharded.ShardedBasisSet.from_global(ctx, od.h, od.s, od.u.to(torch.complex128))
    state = uhf_state(basis, n_alpha, n_beta)
    new = hartree_fock.general_orbital_system_sharded(state, basis)
    U = hartree_fock.general_orbital_system(state, od).u
    scale = U.abs().max()
    for r in ctx.local_ranks:  # plane by plane: the whole tensor is 16 l^4 elements
        p0, p1 = new.u.planes(r)
        assert (new.u.local(r) - U[p0:p1]).abs().max() <= 1e-13 * scale, f"rank {r}"
    del U
    check_system(new, state, n_alpha, n_beta)
    # a following change_basis takes the symmetric path on the library's proof, without a device test
    monkeypatch.setattr(ctx.engine, "is_antisymmetric", lambda *a: pytest.fail("the proof was not used"))
    calls = []
    plain = sharded._RankTransform.step4_scatter_pairs
    monkeypatch.setattr(sharded._RankTransform, "step4_scatter_pairs", lambda *a: calls.append(1) or plain(*a))
    rotation = torch.linalg.qr(torch.randn((2 * l, 2 * l), dtype=torch.float64, device="cuda"))[0]
    new.change_basis(rotation)
    assert calls


def test_refusals():
    from quantum_systems_b200 import hartree_fock, sharded

    ctx = sharded.EmulatedContext(2)
    od, basis = odqd_sharded(ctx, 4)
    state = uhf_state(basis, 1, 1)
    doubled = sharded.ShardedBasisSet.from_spatial(ctx, od.h, od.s, od.u, anti_symmetrize=True)
    with pytest.raises(ValueError, match="spin-doubled"):
        hartree_fock.general_orbital_system_sharded(state, doubled)
    anti = sharded.ShardedBasisSet(ctx, 4, basis.h, basis.s, basis.u, anti_symmetrized_u=True)
    with pytest.raises(ValueError, match="anti-symmetrised"):
        hartree_fock.general_orbital_system_sharded(state, anti)
    _, other = odqd_sharded(ctx, 6)
    with pytest.raises(ValueError, match="l = 6"):
        hartree_fock.general_orbital_system_sharded(state, other)
    _, complex_basis = random_sharded(ctx, 4, True)
    with pytest.raises(TypeError):
        hartree_fock.general_orbital_system_sharded(uhf_state(complex_basis, 1, 1), complex_basis,
                                                    out_dtype=torch.float64)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_sharded_processes_agree():
    world = min(torch.cuda.device_count(), 8)
    cmd = [
        sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
        "--master-addr", "127.0.0.1", "--master-port", "29541",
        os.path.join(ROOT, "tests", "_multi_gpu_uhf_gos_worker.py"),
    ]
    proc = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert proc.returncode == 0, proc.stdout[-3000:] + proc.stderr[-3000:]
    assert "MULTI_GPU_UHF_GOS_OK" in proc.stdout
