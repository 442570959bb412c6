"""The spin-orbital system in the UHF basis from spin blocks of the spatial tensor: the four-coefficient transform
(ops.transform_two_body_mixed) under its rounding-error bound, the assembly kernel (ops.spin_orbital_two_body)
exactly against a numpy restatement of its formula, and hartree_fock.general_orbital_system against the
spin-doubling route GeneralOrbitalSystem(n, basis).change_basis(spin_orbital_coefficients(state)[0])."""

import numpy as np
import pytest

import precise as P
import uhf_oracle

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def host(a):
    return a.cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)


def rand(rng, shape, complex_=False):
    return rng.standard_normal(shape) + (1j * rng.standard_normal(shape) if complex_ else 0)


# ------------------------------------------------------------------------------------ four-coefficient transform


# (label, n, m, u complex, C complex, explicit bras)
MIXED = [
    ("real odd pitch", 13, 13, False, False, False),
    ("real explicit bras", 20, 20, False, False, True),
    ("complex", 12, 12, True, True, False),
    ("complex explicit bras", 10, 10, True, True, True),
    ("real u complex C", 15, 15, False, True, False),
    ("complex u real C (split)", 16, 16, True, False, True),
    ("rectangular m < n", 14, 9, False, False, False),
    ("complex rectangular m < n", 11, 7, True, True, True),
]


@pytest.mark.parametrize("case", MIXED, ids=[c[0] for c in MIXED])
def test_mixed_transform_rounding_bound(case):
    from quantum_systems_b200 import ops

    label, n, m, u_c, c_c, explicit = case
    rng = np.random.default_rng(n * 31 + m)
    u = rand(rng, (n,) * 4, u_c)
    C_r, C_s = rand(rng, (n, m), c_c), rand(rng, (n, m), c_c)
    Ct_p = rand(rng, (m, n), c_c) if explicit else C_r.conj().T
    Ct_q = rand(rng, (m, n), c_c) if explicit else C_s.conj().T
    ref, absval, fp64 = P.companions(P.mixed_steps, u, C_r, C_s, Ct_p, Ct_q)
    got = ops.transform_two_body_mixed(dev(u), dev(C_r), dev(C_s), *((dev(Ct_p), dev(Ct_q)) if explicit else ()))
    assert got.dtype == (torch.complex128 if (u_c or c_c) else torch.float64)
    P.assert_rounding_bound(host(got), ref, absval, P.k_transform([n] * 4, [u_c or c_c] * 4), fp64, label)


@pytest.mark.parametrize("n", [20, 33])
@pytest.mark.parametrize("u_c, c_c", [(False, False), (True, True), (True, False), (False, True)])
def test_mixed_transform_with_equal_matrices_is_the_plain_transform(n, u_c, c_c):
    from quantum_systems_b200 import ops

    rng = np.random.default_rng(n)
    u, C = dev(rand(rng, (n,) * 4, u_c)), dev(rand(rng, (n, n), c_c))
    Ct = C.conj().T.contiguous()
    plain = ops.transform_two_body(u, C, symmetry=0)
    assert torch.equal(ops.transform_two_body_mixed(u, C, C), plain)
    assert torch.equal(ops.transform_two_body_mixed(u, C, C.clone(), Ct, Ct.clone()), plain)
    assert torch.equal(ops.transform_two_body_mixed(u, C, C, Ct, Ct), ops.transform_two_body(u, C, Ct, symmetry=0))


def test_mixed_transform_takes_real_coefficients_when_exact():
    from quantum_systems_b200 import ops

    rng = np.random.default_rng(5)
    u = dev(rand(rng, (12,) * 4, True))
    C_r, C_s = dev(rand(rng, (12, 12))), dev(rand(rng, (12, 12)))
    typed = ops.transform_two_body_mixed(u, C_r.to(torch.complex128), C_s.to(torch.complex128))
    assert torch.equal(typed, ops.transform_two_body_mixed(u, C_r, C_s))


# --------------------------------------------------------------------------------------------- assembly kernel


def assemble_np(b_aa, b_ab, b_ba, b_bb, orbital, spin, out_dtype):
    """``U[I,J,K,L] = [sI=sK][sJ=sL] B[oI,oJ,oK,oL] - [sI=sL][sJ=sK] B[oI,oJ,oL,oK]`` with ``B = b_{sI sJ}``, one
    subtraction per element as in the kernel; ``b_ba=None`` is ``b_ab`` under particle exchange."""
    if b_ba is None:
        b_ba = b_ab.transpose(1, 0, 3, 2)
    B = {(0, 0): b_aa, (0, 1): b_ab, (1, 0): b_ba, (1, 1): b_bb}
    o, s = np.asarray(orbital), np.asarray(spin)
    n = len(o)
    U = np.empty((n,) * 4, dtype=out_dtype)
    for I in range(n):
        for J in range(n):
            A = B[(int(s[I]), int(s[J]))][o[I], o[J]].astype(out_dtype)
            direct = (s[:, None] == s[I]) & (s[None, :] == s[J])
            exchange = (s[None, :] == s[I]) & (s[:, None] == s[J])
            U[I, J] = np.where(direct, A[o[:, None], o[None, :]], 0) - np.where(exchange, A[o[None, :], o[:, None]], 0)
    return U


def tables(kind, l, rng):
    from quantum_systems_b200 import hartree_fock

    if kind == "uhf":
        return hartree_fock.spin_orbital_order(min(l, 3), min(l, 2) - 1, l)
    pairs = np.array([(j, s) for j in range(l) for s in (0, 1)])[rng.permutation(2 * l)]
    return pairs[:, 0], pairs[:, 1]


DTYPES = {"f64->f64": (False, torch.float64), "f64->c128": (False, torch.complex128),
          "c128->c128": (True, torch.complex128)}


@pytest.mark.parametrize("derived", [False, True], ids=["b_ba given", "b_ba derived"])
@pytest.mark.parametrize("kind", ["uhf", "permutation"])
@pytest.mark.parametrize("l", [1, 6, 33])
@pytest.mark.parametrize("dtypes", list(DTYPES))
def test_assembly_is_exact(dtypes, l, kind, derived):
    from quantum_systems_b200 import ops

    in_c, out_dtype = DTYPES[dtypes]
    rng = np.random.default_rng(l * 7 + derived)
    blocks = [rand(rng, (l,) * 4, in_c) for _ in range(4)]
    if derived:
        blocks[2] = None
    orbital, spin = tables(kind, l, rng)
    got = ops.spin_orbital_two_body(*(dev(b) if b is not None else None for b in blocks), orbital, spin,
                                    out_dtype=out_dtype)
    ref = assemble_np(*blocks, orbital, spin, np.complex128 if out_dtype == torch.complex128 else np.float64)
    assert got.dtype == out_dtype and tuple(got.shape) == (2 * l,) * 4
    assert torch.equal(got, dev(ref))
    assert ops.proven_symmetry(got) == ops.ANTISYMMETRIC_LAST_PAIR
    assert ops.two_body_symmetry(got) & ops.ANTISYMMETRIC_LAST_PAIR


@pytest.mark.parametrize("ways", [2, 3, 7])
def test_assembly_plane_ranges_are_slices_of_the_whole(ways):
    from quantum_systems_b200 import ops

    l = 7
    rng = np.random.default_rng(ways)
    blocks = [dev(rand(rng, (l,) * 4)) for _ in range(4)]
    orbital, spin = tables("permutation", l, rng)
    for b_ba in (blocks[2], None):
        whole = ops.spin_orbital_two_body(blocks[0], blocks[1], b_ba, blocks[3], orbital, spin,
                                          out_dtype=torch.complex128)
        cuts = [0] + sorted(rng.choice(np.arange(1, 2 * l), ways - 1, replace=False).tolist()) + [2 * l]
        for p0, p1 in zip(cuts[:-1], cuts[1:]):
            part = ops.spin_orbital_two_body(blocks[0], blocks[1], b_ba, blocks[3], orbital, spin,
                                             out_dtype=torch.complex128, planes=(p0, p1))
            assert torch.equal(part, whole[p0:p1])
            assert ops.proven_symmetry(part) == 0


def test_assembly_refuses_bad_tables_and_dtypes():
    from quantum_systems_b200 import ops

    l = 3
    b = dev(np.zeros((l,) * 4))
    good_o, good_s = np.repeat(np.arange(l), 2), np.tile([0, 1], l)
    with pytest.raises(ValueError, match="exactly once"):
        ops.spin_orbital_two_body(b, b, None, b, np.zeros(2 * l, dtype=int), good_s)
    with pytest.raises(ValueError, match="lie in"):
        ops.spin_orbital_two_body(b, b, None, b, good_o, np.tile([0, 2], l))
    with pytest.raises(ValueError, match="length"):
        ops.spin_orbital_two_body(b, b, None, b, good_o[:-1], good_s[:-1])
    with pytest.raises(ValueError, match="required"):
        ops.spin_orbital_two_body(b, None, b, b, good_o, good_s)
    bc = b.to(torch.complex128)
    with pytest.raises(RuntimeError, match="narrow"):
        ops.spin_orbital_two_body(bc, bc, None, bc, good_o, good_s, out_dtype=torch.float64)


# ----------------------------------------------------------------------------------------------- end to end


def odqd(l, potential="ho", **kw):
    from quantum_systems_b200 import ODQD

    pot = ODQD.HOPotential(0.25) if potential == "ho" else ODQD.DWPotential(1.0, 5)
    points = 201 if l <= 12 else 801
    return ODQD(l, 8.0 if potential == "ho" else 10.0, points, potential=pot, **kw)


def random_basis(l, exact_exchange):
    """Random Hermitian-pair ``u`` with exact particle-exchange symmetry (RandomBasisSet's construction), or that
    tensor with rounding-level noise that breaks the symmetry; a diagonal-dominant ``h`` so UHF converges."""
    from quantum_systems_b200 import RandomBasisSet

    np.random.seed(11)
    basis = RandomBasisSet(l, 1)
    u = host(basis.u)
    u = 0.5 * (u + u.transpose(2, 3, 0, 1).conj())  # keeps the exchange symmetry exact
    if not exact_exchange:
        u = u + 1e-14 * np.random.default_rng(3).standard_normal(u.shape)
    basis.h = np.diag(np.arange(l, dtype=np.float64)) + 0.1 * host(basis.h)
    basis.s = np.eye(l)
    basis.u = 0.1 * u
    return basis


def non_orthogonal_odqd():
    basis = odqd(10)
    X = np.eye(10) + 0.2 * np.random.default_rng(7).standard_normal((10, 10))
    basis.change_basis(dev(X))
    return basis


def host_odqd():
    return odqd(10, np=np)


def real_spin_doubling():
    basis = odqd(10)
    basis.cast_to_complex_on_spin_doubling = False
    return basis


def broken_guess(basis):
    _, V = np.linalg.eigh(host(basis.h).real)
    return uhf_oracle.homo_lumo_rotated(V, 1, np.pi / 4), V


# name -> (basis factory, n_alpha, n_beta, guess, exchange symmetry expected: True / False / None = whatever holds)
E2E = {
    "odqd_open_shell_l48": (lambda: odqd(48), 3, 2, None, None),
    "odqd_broken_symmetry_l48": (lambda: odqd(48, "dw"), 1, 1, broken_guess, None),
    "random_exact_exchange": (lambda: random_basis(12, True), 3, 1, None, True),
    "random_without_exchange": (lambda: random_basis(12, False), 3, 1, None, False),
    "non_orthogonal_s": (non_orthogonal_odqd, 2, 1, None, None),
    "host_numpy_basis": (host_odqd, 2, 1, None, None),
    "real_spin_doubling": (real_spin_doubling, 1, 3, None, None),
}

ONE_BODY = ("h", "s", "position", "momentum", "spf", "bra_spf", "spin_x", "spin_y", "spin_z", "spin_2", "spin_2_tb")


@pytest.mark.parametrize("case", list(E2E))
def test_against_the_spin_doubling_route(case, monkeypatch):
    from quantum_systems_b200 import GeneralOrbitalSystem, hartree_fock, ops

    make, n_a, n_b, guess, exchange = E2E[case]
    basis = make()
    state = hartree_fock.ground_state_unrestricted(basis, n_a, n_b, C=guess(basis) if guess else None)
    assert state.converged
    n = n_a + n_b
    u_before = host(basis.u).copy()
    mixed_calls = []
    plain_mixed = ops.transform_two_body_mixed
    monkeypatch.setattr(ops, "transform_two_body_mixed", lambda *a, **k: mixed_calls.append(1) or plain_mixed(*a, **k))
    new = hartree_fock.general_orbital_system(state, basis)
    monkeypatch.undo()
    C, eps = hartree_fock.spin_orbital_coefficients(state)
    ref = GeneralOrbitalSystem(n, basis.copy_basis())
    ref.change_basis(C)

    assert not basis.includes_spin and np.array_equal(host(basis.u), u_before) and basis.l == C.shape[0] // 2
    assert isinstance(new, GeneralOrbitalSystem) and (new.n, new.l) == (ref.n, ref.l) == (n, 2 * basis.l)
    if exchange is not None:
        assert len(mixed_calls) == (1 if exchange else 2)
    for name in ONE_BODY:
        a, b = getattr(new, name), getattr(ref, name)
        assert (a is None) == (b is None), name
        if a is not None:
            assert type(a) is type(b) and a.dtype == b.dtype, name
            assert np.array_equal(host(a), host(b)), f"{name} differs"
    assert type(new.u) is type(ref.u) and new.u.dtype == ref.u.dtype
    if case == "host_numpy_basis":
        assert isinstance(new.u, np.ndarray) and isinstance(new.h, np.ndarray)
    if case == "real_spin_doubling":
        assert new.u.dtype == torch.float64
    u_new, u_ref = host(new.u), host(ref.u)
    assert np.abs(u_new - u_ref).max() <= 1e-12 * np.abs(u_ref).max()

    u_dev = new.u if isinstance(new.u, torch.Tensor) else dev(new.u)
    assert ops.two_body_symmetry(u_dev) & ops.ANTISYMMETRIC_LAST_PAIR
    if isinstance(new.u, torch.Tensor):
        assert ops.proven_symmetry(new.u) == ops.ANTISYMMETRIC_LAST_PAIR
    assert abs(new.compute_reference_energy() - state.energy) <= 1e-10 * abs(state.energy)
    f = host(new.construct_fock_matrix(new.h, new.u))
    assert np.abs(f[:n, n:]).max() <= 1e-7
    assert np.abs(np.diag(f) - host(eps)).max() <= 1e-8


def test_against_an_independent_numpy_build():
    from quantum_systems_b200 import hartree_fock

    basis = odqd(6)
    state = hartree_fock.ground_state_unrestricted(basis, 2, 1)
    got = host(hartree_fock.general_orbital_system(state, basis).u)
    l = basis.l
    u = host(basis.u)
    d = np.eye(2)
    u_so = np.einsum("pr,qs,abcd->apbqcrds", d, d, u).reshape((2 * l,) * 4)
    u_so = u_so - u_so.transpose(0, 1, 3, 2)
    C = host(hartree_fock.spin_orbital_coefficients(state)[0])
    want = np.einsum("pi,qj,pqrs,rk,sl->ijkl", C.conj(), C.conj(), u_so, C, C, optimize=True)
    assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max()


def test_peak_memory():
    from quantum_systems_b200 import hartree_fock
    from quantum_systems_b200.basis_set import BasisSet
    from quantum_systems_b200.hartree_fock import UnrestrictedHartreeFockState

    l = 64
    gen = torch.Generator(device="cuda").manual_seed(0)
    basis = BasisSet(l, 1)
    basis.h = torch.eye(l, dtype=torch.float64, device="cuda")
    basis.s = torch.eye(l, dtype=torch.float64, device="cuda")
    basis.u = torch.randn((l,) * 4, dtype=torch.float64, device="cuda", generator=gen)  # no exchange symmetry
    Ca, Cb = (torch.linalg.qr(torch.randn((l, l), dtype=torch.float64, device="cuda", generator=gen))[0]
              for _ in range(2))
    e = torch.arange(l, dtype=torch.float64, device="cuda")
    state = UnrestrictedHartreeFockState(Ca, Cb, e, e.clone(), None, None, 0.0, 0.0, True, 0, 3, 2)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    system = hartree_fock.general_orbital_system(state, basis)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    s_out, s_u = 16, 8
    assert system.u.dtype == torch.complex128
    assert peak < (2 * l) ** 4 * s_out + 8 * l**4 * s_u + 64 * 2**20, f"{peak / 2**20:.1f} MiB"


def test_refusals():
    from quantum_systems_b200 import GeneralOrbitalSystem, ODSincDVR, hartree_fock

    state = hartree_fock.ground_state_unrestricted(odqd(4), 1, 1)
    with pytest.raises(ValueError, match="spin-doubled"):
        hartree_fock.general_orbital_system(state, GeneralOrbitalSystem(2, odqd(4))._basis_set)
    sinc = ODSincDVR(4, 5.0)
    assert sinc.u_repr == "2d"
    with pytest.raises(ValueError, match="4-d"):
        hartree_fock.general_orbital_system(state, sinc)
    with pytest.raises(ValueError, match="anti-symmetrised"):
        hartree_fock.general_orbital_system(state, odqd(4, anti_symmetrized_u=True))
    with pytest.raises(ValueError, match="l = 6"):
        hartree_fock.general_orbital_system(state, odqd(6))
