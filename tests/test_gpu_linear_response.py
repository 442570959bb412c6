"""Linear-response TDHF (hartree_fock.excited_states) against the numpy oracle (tests/lr_oracle.py) for RHF singlets
and triplets, GHF on anti-symmetrised and plain u and open-shell UHF, each with TDA and RPA; the spin unions of a
closed shell, the small-kick limit of the GPU propagator, determinism, host storage, the refusals and an l = 100
double well."""

import numpy as np
import pytest
import scipy.linalg

import lr_oracle

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

TOL = 1e-8


def host(a):
    return a.cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)


def basis(l=12, **kw):
    """A stiff well: the RHF triplets of softer ODQD wells are unstable, and RPA needs a stable reference."""
    from quantum_systems_b200 import ODQD

    return ODQD(l, 6.0, 201, potential=ODQD.HOPotential(2.0), **kw)


def spatial(**kw):
    from quantum_systems_b200 import SpatialOrbitalSystem

    return SpatialOrbitalSystem(4, basis(**kw))


def general(anti_symmetrize=True):
    from quantum_systems_b200 import GeneralOrbitalSystem

    return GeneralOrbitalSystem(4, basis(l=6), anti_symmetrize=anti_symmetrize)


def separated(omega, gap=1e-3):
    """Roots whose relative distance to both neighbours exceeds ``gap``."""
    rel = np.abs(np.diff(omega)) / np.abs(omega[1:])
    left = np.concatenate([[np.inf], rel])
    right = np.concatenate([rel, [np.inf]])
    return (left > gap) & (right > gap)


def check(result, omega, XpY, XmY, mu, n_states, tda):
    got = host(result.energies)
    assert result.converged
    np.testing.assert_allclose(got, omega[:n_states], rtol=1e-10, atol=0)
    keep = separated(omega[:n_states + 1])[:n_states]
    X_ref = 0.5 * (XpY + XmY)[:n_states]
    Y_ref = 0.5 * (XpY - XmY)[:n_states]
    X = np.concatenate([host(x).reshape(n_states, -1) for x in result.X], axis=1)
    Y = np.concatenate([host(y).reshape(n_states, -1) for y in result.Y], axis=1)
    np.testing.assert_allclose((X ** 2).sum(1) - (Y ** 2).sum(1), 1.0, atol=1e-10)
    if tda:
        assert not Y.any()
    mu_got = host(result.transition_dipole)
    for n in np.flatnonzero(keep):
        sign = np.sign(X[n] @ X_ref[n])
        assert np.abs(X[n] - sign * X_ref[n]).max() <= 1e-6
        assert np.abs(Y[n] - sign * Y_ref[n]).max() <= 1e-6
        assert np.abs(mu_got[n] - sign * mu[n]).max() <= 1e-6
    np.testing.assert_allclose(host(result.oscillator_strength), 2 * got[:, None] * mu_got ** 2, rtol=1e-14)


@pytest.mark.parametrize("tda", [False, True])
@pytest.mark.parametrize("spin", ["singlet", "triplet"])
def test_rhf_matches_the_oracle(spin, tda):
    from quantum_systems_b200 import hartree_fock

    system = spatial()
    state = hartree_fock.ground_state(system, tol=1e-12)
    res = hartree_fock.excited_states(system, state, n_states=6, tda=tda, spin=spin, tol=TOL)
    h, u, d, C = host(system.h).real, host(system.u).real, host(system.dipole_moment).real, host(state.C)
    omega, XpY, XmY = lr_oracle.spectrum(*lr_oracle.matrices("rhf", h, u, C, 2, spin=spin), tda=tda)
    mu = lr_oracle.transition_dipoles("rhf", XpY, C, 2, d, spin)
    check(res, omega, XpY, XmY, mu, 6, tda)
    if spin == "triplet":
        assert not host(res.transition_dipole).any()


@pytest.mark.parametrize("tda", [False, True])
@pytest.mark.parametrize("anti_symmetrize", [True, False])
def test_ghf_matches_the_oracle(anti_symmetrize, tda):
    from quantum_systems_b200 import hartree_fock

    system = general(anti_symmetrize)
    state = hartree_fock.ground_state(system, tol=1e-12)
    res = hartree_fock.excited_states(system, state, n_states=5, tda=tda, tol=TOL)
    h, u, d, C = host(system.h).real, host(system.u).real, host(system.dipole_moment).real, host(state.C).real
    A, B = lr_oracle.matrices("ghf", h, u, C, 4, anti_symmetrized_u=anti_symmetrize)
    omega, XpY, XmY = lr_oracle.spectrum(A, B, tda=tda)
    check(res, omega, XpY, XmY, lr_oracle.transition_dipoles("ghf", XpY, C, 4, d), 5, tda)


@pytest.mark.parametrize("tda", [False, True])
def test_open_shell_uhf_matches_the_oracle(tda):
    from quantum_systems_b200 import hartree_fock

    system = spatial()
    state = hartree_fock.ground_state_unrestricted(system, 2, 1, tol=1e-12)
    res = hartree_fock.excited_states(system, state, n_states=6, tda=tda, tol=TOL)
    h, u, d = host(system.h).real, host(system.u).real, host(system.dipole_moment).real
    C = (host(state.C_alpha), host(state.C_beta))
    omega, XpY, XmY = lr_oracle.spectrum(*lr_oracle.matrices("uhf", h, u, C, (2, 1)), tda=tda)
    check(res, omega, XpY, XmY, lr_oracle.transition_dipoles("uhf", XpY, C, (2, 1), d), 6, tda)
    assert [tuple(x.shape) for x in res.X] == [(6, 2, 10), (6, 1, 11)]


@pytest.mark.parametrize("tda", [False, True])
def test_spin_unions_of_a_closed_shell(tda):
    from quantum_systems_b200 import hartree_fock

    system = spatial(l=6)
    rhf = hartree_fock.ground_state(system, tol=1e-12)
    full = 2 * 4
    singlets = host(hartree_fock.excited_states(system, rhf, full, tda=tda, tol=TOL).energies)
    triplets = host(hartree_fock.excited_states(system, rhf, full, tda=tda, spin="triplet", tol=TOL).energies)
    uhf = hartree_fock.ground_state_unrestricted(system, 2, 2, tol=1e-12)
    both = host(hartree_fock.excited_states(system, uhf, 2 * full, tda=tda, tol=TOL).energies)
    np.testing.assert_allclose(both, np.sort(np.concatenate([singlets, triplets])), rtol=1e-10)
    gsystem = general()
    ghf = hartree_fock.ground_state(gsystem, tol=1e-12)
    spin_orbital = host(hartree_fock.excited_states(gsystem, ghf, 4 * full, tda=tda, tol=TOL).energies)
    np.testing.assert_allclose(spin_orbital, np.sort(np.concatenate([singlets] + [triplets] * 3)), rtol=1e-10)


def test_a_weak_kick_in_the_gpu_propagator_follows_the_rpa_spectrum():
    """The derivation and the tolerance are those of tests/test_lr_oracle_cpu.py: to first order in kappa the dipole
    moves by 2 kappa sum_n |mu_n|^2 sin(omega_n t) over all RPA roots."""
    from quantum_systems_b200 import hartree_fock

    system = spatial(l=6)
    state = hartree_fock.ground_state(system, tol=1e-12)
    res = hartree_fock.excited_states(system, state, n_states=8, tol=1e-10)
    kappa, dt, n_steps = 1e-4, 0.01, 500
    d = host(system.dipole_moment)
    kicked = scipy.linalg.expm(1j * kappa * d[0]) @ host(state.C)[:, :2]
    start = hartree_fock.TimeDependentHartreeFockRun(None, None, None, 0.0, (torch.as_tensor(kicked).cuda(),),
                                                     (None,))
    run = hartree_fock.propagate(system, start, n_steps * dt, dt)
    d0 = float(torch.einsum("rs,sr->", host_t(state.density_matrix), host_t(d[0])).real)
    response = (host(run.dipole)[:, 0] - d0) / kappa
    predicted = 2 * np.sin(np.outer(host(run.times), host(res.energies))) @ (host(res.transition_dipole)[:, 0] ** 2)
    assert np.abs(predicted).max() > 0.1
    assert np.abs(response - predicted).max() <= 1e-3 * np.abs(predicted).max()
    assert response[1] > 0


def host_t(a):
    return torch.as_tensor(host(a)).to(torch.complex128)


def test_repeated_calls_are_bit_identical():
    from quantum_systems_b200 import hartree_fock

    system = spatial()
    state = hartree_fock.ground_state(system, tol=1e-12)
    a = hartree_fock.excited_states(system, state, n_states=4, tol=TOL)
    b = hartree_fock.excited_states(system, state, n_states=4, tol=TOL)
    assert torch.equal(a.energies, b.energies) and torch.equal(a.X[0], b.X[0]) and torch.equal(a.Y[0], b.Y[0])
    assert a.iterations == b.iterations and a.densities_built == b.densities_built > 0


def test_host_systems_get_ndarrays():
    from quantum_systems_b200 import hartree_fock

    system = spatial(np=np)
    state = hartree_fock.ground_state(system, tol=1e-12)
    res = hartree_fock.excited_states(system, state, n_states=3, tol=TOL)
    for value in (res.energies, res.X[0], res.Y[0], res.transition_dipole, res.oscillator_strength,
                  res.residual_norms):
        assert isinstance(value, np.ndarray)


def test_refusals():
    import dataclasses

    from quantum_systems_b200 import hartree_fock

    system = spatial(l=6)
    state = hartree_fock.ground_state(system, tol=1e-12)
    with pytest.raises(ValueError, match="spin"):
        hartree_fock.excited_states(system, state, spin="quintet")
    with pytest.raises(ValueError, match="n_states"):
        hartree_fock.excited_states(system, state, n_states=0)
    with pytest.raises(ValueError, match="n_states"):
        hartree_fock.excited_states(system, state, n_states=9)
    with pytest.raises(ValueError, match="not converged"):
        hartree_fock.excited_states(system, dataclasses.replace(state, converged=False))
    with pytest.raises(ValueError, match="coefficients"):
        hartree_fock.excited_states(system, dataclasses.replace(state, C=state.C[:5, :5]))
    with pytest.raises(TypeError):
        hartree_fock.excited_states(system, object())
    uhf = hartree_fock.ground_state_unrestricted(system, 2, 1, tol=1e-12)
    with pytest.raises(ValueError, match="triplet"):
        hartree_fock.excited_states(system, uhf, spin="triplet")
    gsystem = general()
    ghf = hartree_fock.ground_state(gsystem, tol=1e-12)
    with pytest.raises(ValueError, match="triplet"):
        hartree_fock.excited_states(gsystem, ghf, spin="triplet")
    with pytest.raises(ValueError, match="unrestricted"):
        hartree_fock.excited_states(gsystem, uhf)
    with pytest.raises(NotImplementedError, match="complex orbitals"):
        hartree_fock.excited_states(system, dataclasses.replace(state, C=state.C.to(torch.complex128) * 1j))
    full = spatial(l=2)
    with pytest.raises(ValueError, match="no virtual"):
        hartree_fock.excited_states(full, hartree_fock.ground_state(full, tol=1e-12))
    from quantum_systems_b200.sharded import ShardedBasisSet

    with pytest.raises(TypeError, match="ShardedBasisSet"):
        hartree_fock.excited_states(ShardedBasisSet.__new__(ShardedBasisSet), state)


def test_sinc_dvr_2d_storage_is_refused():
    from quantum_systems_b200 import hartree_fock

    system = spatial(l=4)
    state = hartree_fock.ground_state(system, tol=1e-12)
    system._basis_set.u_repr = "2d"
    with pytest.raises(ValueError, match="4-d"):
        hartree_fock.excited_states(system, state)


def test_unstable_double_well_reference():
    """The RHF state of the broken-symmetry double well of the UHF tests: a negative TDA triplet root, and RPA
    refuses it."""
    from quantum_systems_b200 import ODQD, SpatialOrbitalSystem, hartree_fock

    system = SpatialOrbitalSystem(2, ODQD(8, 10.0, 201, potential=ODQD.DWPotential(1.0, 5)))
    state = hartree_fock.ground_state(system, tol=1e-12)
    tda = hartree_fock.excited_states(system, state, n_states=2, tda=True, spin="triplet", tol=TOL)
    assert float(tda.energies[0]) < 0
    with pytest.raises(ValueError, match="not positive definite"):
        hartree_fock.excited_states(system, state, n_states=2, spin="triplet", tol=TOL)


def test_l100_double_well_twenty_electrons_ten_roots():
    from quantum_systems_b200 import ODQD, SpatialOrbitalSystem, hartree_fock

    system = SpatialOrbitalSystem(20, ODQD(100, 20, 2001, potential=ODQD.DWPotential(1, 5)))
    state = hartree_fock.ground_state(system, tol=1e-10)
    res = hartree_fock.excited_states(system, state, n_states=10, tda=True, tol=TOL)
    assert res.converged
    h, u, C = host(system.h).real, host(system.u).real, host(state.C)
    A, _ = lr_oracle.matrices("rhf", h, u, C, 10)
    omega = scipy.linalg.eigvalsh(0.5 * (A + A.T))
    np.testing.assert_allclose(host(res.energies), omega[:10], rtol=1e-10)
