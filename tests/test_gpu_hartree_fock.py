"""Hartree-Fock ground states (quantum_systems_b200.hartree_fock) against the numpy oracle, through the Brillouin
condition in the HF basis, and across storage modes and shards."""

import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import hf_oracle

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def host(a):
    return a.cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)


def rel(a, b):
    return abs(a - b) / abs(b)


def max_err(a, b):
    return float(np.abs(host(a) - host(b)).max())


def rhf_system(**kw):
    from quantum_systems_b200 import ODQD, SpatialOrbitalSystem

    return SpatialOrbitalSystem(4, ODQD(10, 8, 201, potential=ODQD.HOPotential(0.25), **kw))


def ghf_system(anti_symmetrize=True, **kw):
    from quantum_systems_b200 import ODQD, GeneralOrbitalSystem

    return GeneralOrbitalSystem(4, ODQD(6, 8, 201, potential=ODQD.HOPotential(0.25), **kw),
                                anti_symmetrize=anti_symmetrize)


SYSTEMS = {
    "rhf": (rhf_system, True, False),
    "ghf": (ghf_system, False, True),
    "ghf_plain_u": (lambda **kw: ghf_system(anti_symmetrize=False, **kw), False, False),
}


def oracle_state(system, restricted, anti_symmetrized):
    s = host(system.s) if system.s is not None else None
    return hf_oracle.ground_state(host(system.h), host(system.u), system.n, restricted, anti_symmetrized, s=s,
                                  e_nuc=system.nuclear_repulsion_energy)


@pytest.mark.parametrize("kind", list(SYSTEMS))
def test_against_the_oracle(kind):
    from quantum_systems_b200 import hartree_fock

    make, restricted, anti = SYSTEMS[kind]
    system = make()
    state = hartree_fock.ground_state(system)
    ref = oracle_state(system, restricted, anti)
    assert state.converged and ref["converged"]
    assert rel(state.energy, ref["energy"]) <= 1e-10
    assert max_err(state.density_matrix, ref["density_matrix"]) <= 1e-8
    assert max_err(state.epsilon, ref["epsilon"]) <= 1e-8
    C, s = host(state.C), host(system.s)
    assert np.abs(C.conj().T @ s @ C - np.eye(C.shape[1])).max() <= 1e-10
    assert np.all(np.diff(host(state.epsilon)) >= 0)


@pytest.mark.parametrize("kind", ["rhf", "ghf"])
def test_brillouin_in_the_hf_basis(kind):
    from quantum_systems_b200 import hartree_fock

    system = SYSTEMS[kind][0]()
    state = hartree_fock.ground_state(system)
    system.change_basis(state.C)
    f = host(system.construct_fock_matrix(system.h, system.u))
    assert np.abs(f - np.diag(host(state.epsilon))).max() <= 1e-8
    assert rel(system.compute_reference_energy(), state.energy) <= 1e-10


def test_ghf_from_rhf_coefficients_stays_at_the_rhf_point():
    from quantum_systems_b200 import hartree_fock

    spas = rhf_system()
    gos = spas.construct_general_orbital_system()
    rhf = hartree_fock.ground_state(spas)
    ghf = hartree_fock.ground_state(gos, C=hf_oracle.spin_double_coefficients(host(rhf.C)))
    assert ghf.converged and ghf.iterations <= 3
    assert rel(ghf.energy, rhf.energy) <= 1e-12


@pytest.mark.parametrize("complex_", [False, True])
def test_invariant_under_a_non_orthogonal_basis(complex_):
    from quantum_systems_b200 import hartree_fock

    system = rhf_system()
    e0 = hartree_fock.ground_state(system).energy
    l = system.l
    rng = np.random.default_rng(7)
    X = np.eye(l) + 0.2 * rng.standard_normal((l, l)) + (0.2j * rng.standard_normal((l, l)) if complex_ else 0)
    moved = system.copy_system()
    moved.change_basis(torch.from_numpy(X).cuda())
    assert np.abs(host(moved.s) - np.eye(l)).max() > 0.1
    state = hartree_fock.ground_state(moved)
    assert state.converged and rel(state.energy, e0) <= 1e-10
    assert state.C.dtype == (torch.complex128 if complex_ else torch.float64)
    X[:, -1] = X[:, 0]
    singular = system.copy_system()
    singular.change_basis(torch.from_numpy(X).cuda())
    with pytest.raises(ValueError, match="singular"):
        hartree_fock.ground_state(singular)


def unitary(l, seed):
    rng = np.random.default_rng(seed)
    return np.linalg.qr(rng.standard_normal((l, l)) + 1j * rng.standard_normal((l, l)))[0]


@pytest.mark.parametrize("kind", list(SYSTEMS))
def test_complex_problem_against_the_oracle(kind):
    """A random complex unitary basis change gives h and u genuine imaginary parts; the HF energy of the real problem
    is kept, and the iteration runs in complex128."""
    from quantum_systems_b200 import hartree_fock

    make, restricted, anti = SYSTEMS[kind]
    e_real = hartree_fock.ground_state(make()).energy
    system = make()
    system.change_basis(torch.from_numpy(unitary(system.l, 11)).cuda())
    assert np.abs(host(system.u).imag).max() > 1e-3 and np.abs(host(system.h).imag).max() > 1e-3
    state = hartree_fock.ground_state(system)
    ref = oracle_state(system, restricted, anti)
    assert state.converged and ref["converged"]
    assert state.C.dtype == torch.complex128
    assert rel(state.energy, ref["energy"]) <= 1e-10
    assert rel(state.energy, e_real) <= 1e-10
    assert max_err(state.density_matrix, ref["density_matrix"]) <= 1e-8
    assert max_err(state.epsilon, ref["epsilon"]) <= 1e-8


def phase_rotated_real_h(make):
    """Orbital phases on a basis with a diagonal h: u gets imaginary parts, h and s stay real (stored as float64)."""
    system = make()
    phases = np.exp(1j * np.random.default_rng(5).uniform(0, 2 * np.pi, system.l))
    system.change_basis(torch.from_numpy(np.diag(phases)).cuda())
    basis = system._basis_set
    assert np.abs(host(system.h).imag).max() < 1e-15
    basis.h, basis.s = torch.as_tensor(host(system.h).real).cuda(), torch.as_tensor(host(system.s).real).cuda()
    assert system.h.dtype == torch.float64 and system.s.dtype == torch.float64
    assert np.abs(host(system.u).imag).max() > 1e-3
    return system


@pytest.mark.parametrize("kind", ["rhf", "ghf"])
def test_real_h_with_complex_u_iterates_in_complex(kind):
    from quantum_systems_b200 import hartree_fock

    make, restricted, anti = SYSTEMS[kind]
    e_real = hartree_fock.ground_state(make()).energy
    system = phase_rotated_real_h(make)
    state = hartree_fock.ground_state(system)
    assert state.converged and state.C.dtype == torch.complex128
    assert rel(state.energy, e_real) <= 1e-10
    assert rel(state.energy, oracle_state(system, restricted, anti)["energy"]) <= 1e-10


@pytest.mark.parametrize("kind", ["rhf", "ghf"])
def test_storage_modes_and_real_arithmetic(kind):
    from quantum_systems_b200 import hartree_fock

    make = SYSTEMS[kind][0]
    dev_state = hartree_fock.ground_state(make())
    host_state = hartree_fock.ground_state(make(np=np))
    assert isinstance(dev_state.C, torch.Tensor) and dev_state.C.is_cuda
    assert dev_state.C.dtype == torch.float64
    assert isinstance(host_state.C, np.ndarray) and host_state.C.dtype == np.float64
    assert isinstance(host_state.epsilon, np.ndarray) and isinstance(host_state.density_matrix, np.ndarray)
    assert rel(host_state.energy, dev_state.energy) <= 1e-12
    assert max_err(host_state.density_matrix, dev_state.density_matrix) <= 1e-10


def test_non_convergence_warns_and_returns():
    from quantum_systems_b200 import hartree_fock

    with pytest.warns(RuntimeWarning, match="did not converge"):
        state = hartree_fock.ground_state(rhf_system(), max_iterations=1)
    assert not state.converged and state.iterations == 1


def test_sinc_dvr_2d_storage_is_refused():
    from quantum_systems_b200 import ODSincDVR, SpatialOrbitalSystem, hartree_fock

    system = SpatialOrbitalSystem(2, ODSincDVR(8, 5.0))
    assert system._basis_set.u_repr == "2d"
    with pytest.raises(ValueError, match="4-d"):
        hartree_fock.ground_state(system)


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_equals_single(world):
    from quantum_systems_b200 import hartree_fock, sharded
    from quantum_systems_b200.odqd import ODQD

    od = ODQD(6, 8, 201, potential=ODQD.HOPotential(0.25), np=np)
    gos = ghf_system()
    single = hartree_fock.ground_state(gos)
    ctx = sharded.EmulatedContext(world)
    basis = sharded.ShardedBasisSet.from_spatial(ctx, od.h, od.s, od.u, anti_symmetrize=True)
    state = hartree_fock.ground_state_sharded(basis, gos.n)
    assert state.converged and state.C.dtype == torch.float64
    assert rel(state.energy, single.energy) <= 1e-12
    assert max_err(state.density_matrix, single.density_matrix) <= 1e-10
    basis.change_basis(state.C)
    f = host(basis.construct_fock_matrix(basis.h, basis.u, gos.n))
    assert np.abs(f - np.diag(np.diag(f))).max() <= 1e-8
    assert np.abs(np.diag(f) - host(state.epsilon)).max() <= 1e-8


def test_sharded_real_h_with_complex_u_iterates_in_complex():
    from quantum_systems_b200 import hartree_fock, sharded

    system = phase_rotated_real_h(rhf_system)
    single = hartree_fock.ground_state(system)
    basis = sharded.ShardedBasisSet.from_global(sharded.EmulatedContext(3), system.h, system.s, system.u)
    state = hartree_fock.ground_state_sharded(basis, system.n)
    assert state.converged and state.C.dtype == torch.complex128
    assert rel(state.energy, single.energy) <= 1e-12
    assert max_err(state.density_matrix, single.density_matrix) <= 1e-10


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_sharded_processes_agree():
    world = min(torch.cuda.device_count(), 8)
    cmd = [
        sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
        "--master-addr", "127.0.0.1", "--master-port", "29531", os.path.join(ROOT, "tests", "_multi_gpu_hf_worker.py"),
        "ghf",
    ]
    proc = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert proc.returncode == 0, proc.stdout[-3000:] + proc.stderr[-3000:]
    assert "MULTI_GPU_HF_OK" in proc.stdout
