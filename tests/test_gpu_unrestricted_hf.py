"""Unrestricted Hartree-Fock (hartree_fock.ground_state_unrestricted) against the numpy oracle from the same guess,
through its closed-form limits, through the spin-orbital basis it hands to GeneralOrbitalSystem, and across storage
modes and shards.  Only gauge-invariant quantities are compared: energies, densities, residuals."""

import os
import subprocess
import sys

import numpy as np
import pytest

import uhf_oracle

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def host(a):
    return a.cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)


def rel(a, b):
    return abs(a - b) / abs(b)


def max_err(a, b):
    return float(np.abs(host(a) - host(b)).max())


def odqd(l=8, **kw):
    from quantum_systems_b200 import ODQD

    return ODQD(l, 8, 201, potential=ODQD.HOPotential(0.25), **kw)


def dw_basis():
    """The broken-symmetry double well of tests/test_uhf_oracle_cpu.py."""
    from quantum_systems_b200 import ODQD

    return ODQD(8, 10.0, 201, potential=ODQD.DWPotential(1.0, 5))


def oracle_state(basis, n_alpha, n_beta, C=None):
    s = host(basis.s) if basis.s is not None else None
    C = None if C is None else tuple(host(c) for c in C)
    return uhf_oracle.uhf_ground_state(host(basis.h), host(basis.u), n_alpha, n_beta, s=s, C=C,
                                      e_nuc=basis.nuclear_repulsion_energy)


def broken_guess(basis):
    _, V = np.linalg.eigh(host(basis.h).real)
    return uhf_oracle.homo_lumo_rotated(V, 1, np.pi / 4), V


def moved(basis, kind):
    """A complex unitary or a (real or complex) non-unitary basis change of ``basis``."""
    l = basis.l
    rng = np.random.default_rng(7)
    if kind == "unitary":
        X = np.linalg.qr(rng.standard_normal((l, l)) + 1j * rng.standard_normal((l, l)))[0]
    else:
        X = np.eye(l) + 0.2 * rng.standard_normal((l, l))
        if kind == "non_orthogonal_complex":
            X = X + 0.2j * rng.standard_normal((l, l))
    out = basis.copy_basis()
    out.change_basis(torch.from_numpy(X).cuda())
    return out


CASES = {
    "open_shell_2_1": (odqd, 2, 1, None),
    "open_shell_3_0": (odqd, 3, 0, None),
    "open_shell_1_3": (odqd, 1, 3, None),
    "broken_symmetry": (dw_basis, 1, 1, broken_guess),
}


def check_against_oracle(state, ref):
    assert state.converged and ref["converged"]
    assert rel(state.energy, ref["energy"]) <= 1e-10
    assert max_err(state.density_alpha, ref["density_alpha"]) <= 1e-8
    assert max_err(state.density_beta, ref["density_beta"]) <= 1e-8
    assert abs(state.spin_squared - ref["spin_squared"]) <= 1e-8


@pytest.mark.parametrize("case", list(CASES))
def test_against_the_oracle(case):
    from quantum_systems_b200 import hartree_fock

    make, n_a, n_b, guess = CASES[case]
    basis = make()
    C = guess(basis) if guess else None
    state = hartree_fock.ground_state_unrestricted(basis, n_a, n_b, C=C)
    check_against_oracle(state, oracle_state(basis, n_a, n_b, C))
    assert state.C_alpha.dtype == torch.float64
    if case == "broken_symmetry":
        assert state.spin_squared > 0.1


@pytest.mark.parametrize("kind", ["unitary", "non_orthogonal", "non_orthogonal_complex"])
def test_complex_and_non_orthogonal_problems_against_the_oracle(kind):
    from quantum_systems_b200 import hartree_fock

    e_plain = hartree_fock.ground_state_unrestricted(odqd(), 2, 1).energy
    basis = moved(odqd(), kind)
    if kind != "non_orthogonal":
        assert np.abs(host(basis.u).imag).max() > 1e-3
    state = hartree_fock.ground_state_unrestricted(basis, 2, 1)
    check_against_oracle(state, oracle_state(basis, 2, 1))
    assert rel(state.energy, e_plain) <= 1e-10
    assert state.C_alpha.dtype == (torch.float64 if kind == "non_orthogonal" else torch.complex128)


def test_one_electron_is_the_lowest_eigenvalue_of_h():
    import scipy.linalg

    from quantum_systems_b200 import hartree_fock

    basis = moved(odqd(), "non_orthogonal")
    state = hartree_fock.ground_state_unrestricted(basis, 1, 0)
    e0 = scipy.linalg.eigh(host(basis.h), host(basis.s), eigvals_only=True)[0]
    assert state.converged and rel(state.energy, e0) <= 1e-12
    assert abs(state.spin_squared - 0.75) <= 1e-12


def test_closed_shell_is_rhf():
    from quantum_systems_b200 import SpatialOrbitalSystem, hartree_fock

    system = SpatialOrbitalSystem(4, odqd())
    rhf = hartree_fock.ground_state(system)
    uhf = hartree_fock.ground_state_unrestricted(system)
    assert uhf.converged and (uhf.n_alpha, uhf.n_beta) == (2, 2)
    assert rel(uhf.energy, rhf.energy) <= 1e-12
    assert max_err(uhf.density_alpha, rhf.density_matrix / 2) <= 1e-10
    assert max_err(uhf.density_beta, rhf.density_matrix / 2) <= 1e-10
    assert abs(uhf.spin_squared) <= 1e-10
    C, eps = hartree_fock.spin_orbital_coefficients(uhf)
    assert torch.equal(C, torch.kron(uhf.C_alpha, torch.eye(2, dtype=torch.float64, device="cuda")))
    assert torch.equal(eps, torch.repeat_interleave(uhf.epsilon_alpha, 2))


@pytest.mark.parametrize("case", ["open_shell_2_1", "open_shell_1_3", "broken_symmetry"])
def test_spin_orbital_bridge(case):
    from quantum_systems_b200 import GeneralOrbitalSystem, hartree_fock, ops

    make, n_a, n_b, guess = CASES[case]
    basis = make()
    state = hartree_fock.ground_state_unrestricted(basis, n_a, n_b, C=guess(basis) if guess else None)
    C, eps = hartree_fock.spin_orbital_coefficients(state)
    n = n_a + n_b
    gos = GeneralOrbitalSystem(n, basis.copy_basis())
    ghf = hartree_fock.ground_state(gos, C=C)
    assert ghf.converged and ghf.iterations <= 3
    assert rel(ghf.energy, state.energy) <= 1e-10
    spin_z = host(ops.transform_one_body(gos.spin_z, C))
    gos.change_basis(C)
    assert rel(gos.compute_reference_energy(), state.energy) <= 1e-10
    f = host(gos.construct_fock_matrix(gos.h, gos.u))
    assert np.abs(f[:n, n:]).max() <= 1e-7
    assert np.abs(np.diag(f) - host(eps)).max() <= 1e-8
    column_spins = np.array([0.5 if abs(host(C)[0::2, k]).max() > 0 else -0.5 for k in range(C.shape[1])])
    assert np.sum(column_spins[:n] > 0) == n_a
    assert np.abs(spin_z - np.diag(column_spins)).max() <= 1e-10


def test_storage_modes():
    from quantum_systems_b200 import hartree_fock

    dev = hartree_fock.ground_state_unrestricted(odqd(), 2, 1)
    hst = hartree_fock.ground_state_unrestricted(odqd(np=np), 2, 1)
    assert isinstance(dev.C_alpha, torch.Tensor) and dev.C_alpha.is_cuda
    for name in ("C_alpha", "C_beta", "epsilon_alpha", "epsilon_beta", "density_alpha", "density_beta"):
        assert isinstance(getattr(hst, name), np.ndarray), name
    assert rel(hst.energy, dev.energy) <= 1e-12
    assert max_err(hst.density_alpha, dev.density_alpha) <= 1e-10
    C, _ = hartree_fock.spin_orbital_coefficients(hst)
    assert isinstance(C, np.ndarray) and C.shape == (16, 16)


def test_non_convergence_warns_and_returns():
    from quantum_systems_b200 import hartree_fock

    with pytest.warns(RuntimeWarning, match="did not converge"):
        state = hartree_fock.ground_state_unrestricted(odqd(), 2, 1, max_iterations=1)
    assert not state.converged and state.iterations == 1


def test_refusals():
    from quantum_systems_b200 import GeneralOrbitalSystem, ODSincDVR, SpatialOrbitalSystem, hartree_fock

    with pytest.raises(ValueError, match="ground_state"):
        hartree_fock.ground_state_unrestricted(GeneralOrbitalSystem(2, odqd(4)))
    with pytest.raises(ValueError, match="4-d"):
        hartree_fock.ground_state_unrestricted(SpatialOrbitalSystem(2, ODSincDVR(8, 5.0)))
    with pytest.raises(ValueError, match="anti-symmetrised"):
        hartree_fock.ground_state_unrestricted(odqd(4, anti_symmetrized_u=True), 1, 1)
    with pytest.raises(ValueError, match="required"):
        hartree_fock.ground_state_unrestricted(odqd(4))
    for n_a, n_b in ((5, 0), (1, -1)):
        with pytest.raises(ValueError, match=r"\[0, 4\]"):
            hartree_fock.ground_state_unrestricted(odqd(4), n_a, n_b)


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_equals_single(world):
    from quantum_systems_b200 import hartree_fock, sharded

    for make, n_a, n_b, guess in (CASES["open_shell_2_1"], CASES["broken_symmetry"]):
        basis = make()
        C = guess(basis) if guess else None
        single = hartree_fock.ground_state_unrestricted(basis, n_a, n_b, C=C)
        shards = sharded.ShardedBasisSet.from_global(sharded.EmulatedContext(world), basis.h, basis.s, basis.u)
        state = hartree_fock.ground_state_unrestricted_sharded(shards, n_a, n_b, C=C)
        assert state.converged and state.iterations == single.iterations
        assert rel(state.energy, single.energy) <= 1e-12
        assert max_err(state.density_alpha, single.density_alpha) <= 1e-10
        assert max_err(state.density_beta, single.density_beta) <= 1e-10
        assert abs(state.spin_squared - single.spin_squared) <= 1e-10
    spin = sharded.ShardedBasisSet.from_spatial(sharded.EmulatedContext(world), basis.h, basis.s, basis.u)
    with pytest.raises(ValueError, match="ground_state_sharded"):
        hartree_fock.ground_state_unrestricted_sharded(spin, 1, 1)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_sharded_processes_agree():
    world = min(torch.cuda.device_count(), 8)
    cmd = [
        sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
        "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.join(ROOT, "tests", "_multi_gpu_hf_worker.py"),
        "uhf",
    ]
    proc = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert proc.returncode == 0, proc.stdout[-3000:] + proc.stderr[-3000:]
    assert "MULTI_GPU_UHF_OK" in proc.stdout
