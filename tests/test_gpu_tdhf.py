"""Time-dependent Hartree-Fock (hartree_fock.propagate) against the numpy RK4 oracle (tests/tdhf_oracle.py) for RHF,
GHF and UHF under a dipole pulse and an adiabatic switching, its continuation, storage modes and refusals."""

import numpy as np
import pytest

import tdhf_oracle
from oracle import hf_oracle

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

DT, STEPS = 0.02, 50
TOL = 1e-11


def host(a):
    return a.cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)


def rel_err(got, ref):
    got, ref = host(got), np.asarray(ref)
    return float(np.abs(got - ref).max() / max(np.abs(ref).max(), 1e-300))


def pulse(t):
    return 0.2 * np.sin(1.5 * t)


def odqd(l=8, **kw):
    from quantum_systems_b200 import ODQD

    return ODQD(l, 8, 201, potential=ODQD.HOPotential(0.25), **kw)


def spatial(**kw):
    """Four electrons: RHF with two doubly occupied orbitals."""
    from quantum_systems_b200 import SpatialOrbitalSystem

    return SpatialOrbitalSystem(4, odqd(**kw))


def general(**kw):
    from quantum_systems_b200 import GeneralOrbitalSystem

    return GeneralOrbitalSystem(2, odqd(l=5, **kw))


def with_pulse(system, *extra, **kw):
    from quantum_systems_b200.time_evolution_operators import DipoleFieldInteraction

    system.set_time_evolution_operator([DipoleFieldInteraction(pulse), *extra], **kw)
    return system


def oracle_run(system, kind, C_occ, n_steps=STEPS, u_t=None, scales=None):
    h0, u, d = host(system.h), host(system.u), host(system.dipole_moment)
    return tdhf_oracle.propagate(kind, tdhf_oracle.dipole_field(h0, d, pulse), u_t or (lambda t: u), C_occ, 0.0,
                                 n_steps, DT, dipole=d, scales=scales, e_nuc=system.nuclear_repulsion_energy)


def assert_matches(run, ref):
    for got, want in zip(run.C, ref["C"]):
        assert rel_err(got, want) <= TOL
    assert rel_err(run.energy, ref["energy"]) <= TOL
    assert rel_err(run.dipole, ref["dipole"]) <= TOL
    np.testing.assert_array_equal(host(run.times), ref["times"])
    assert run.t == ref["t"]


def test_rhf_matches_the_oracle():
    from quantum_systems_b200 import hartree_fock

    system = spatial()
    state = hartree_fock.ground_state(system)
    run = hartree_fock.propagate(with_pulse(system), state, STEPS * DT, DT)
    assert run.energy.shape == (STEPS,) and run.dipole.shape == (STEPS, 1) and len(run.C) == 1
    ref = oracle_run(system, "rhf", (host(state.C)[:, :system.n],), scales=hf_oracle.scales(True, False))
    assert_matches(run, ref)
    assert np.ptp(ref["dipole"][:, 0]) > 1e-4  # the pulse drives the dipole


def test_ghf_matches_the_oracle():
    from quantum_systems_b200 import hartree_fock

    system = general()
    state = hartree_fock.ground_state(system)
    run = hartree_fock.propagate(with_pulse(system), state, STEPS * DT, DT)
    ref = oracle_run(system, "ghf", (host(state.C)[:, :system.n],), scales=hf_oracle.scales(False, True))
    assert_matches(run, ref)


def test_uhf_matches_the_oracle():
    from quantum_systems_b200 import hartree_fock

    system = spatial()
    state = hartree_fock.ground_state_unrestricted(system, 2, 1)
    run = hartree_fock.propagate(with_pulse(system), state, STEPS * DT, DT)
    assert len(run.C) == 2 and tuple(run.C[1].shape) == (8, 1)
    assert system.n == 2
    ref = oracle_run(system, "uhf", (host(state.C_alpha)[:, :2], host(state.C_beta)[:, :1]))
    assert_matches(run, ref)


@pytest.mark.parametrize("kind", ["rhf", "uhf"])
def test_adiabatic_switching_matches_the_oracle_on_a_scaled_u(kind):
    from quantum_systems_b200 import hartree_fock
    from quantum_systems_b200.time_evolution_operators import AdiabaticSwitching

    def switch(t):
        return 0.5 * np.cos(t)

    system = spatial()
    if kind == "rhf":
        state = hartree_fock.ground_state(system)
        C_occ, scales = (host(state.C)[:, :system.n],), hf_oracle.scales(True, False)
    else:
        state = hartree_fock.ground_state_unrestricted(system, 2, 1)
        C_occ, scales = (host(state.C_alpha)[:, :2], host(state.C_beta)[:, :1]), None
    u = host(system.u)
    run = hartree_fock.propagate(with_pulse(system, AdiabaticSwitching(switch)), state, STEPS * DT, DT)
    ref = oracle_run(system, kind, C_occ, u_t=lambda t: (1.0 + switch(t)) * u, scales=scales)
    assert_matches(run, ref)


def test_closed_shell_uhf_matches_rhf():
    from quantum_systems_b200 import hartree_fock

    system = with_pulse(spatial())
    rhf = hartree_fock.ground_state(system)
    uhf = hartree_fock.UnrestrictedHartreeFockState(
        C_alpha=rhf.C, C_beta=rhf.C, epsilon_alpha=rhf.epsilon, epsilon_beta=rhf.epsilon,
        density_alpha=rhf.density_matrix / 2, density_beta=rhf.density_matrix / 2, energy=rhf.energy,
        spin_squared=0.0, converged=True, iterations=0, n_alpha=system.n, n_beta=system.n)
    a = hartree_fock.propagate(system, rhf, STEPS * DT, DT)
    b = hartree_fock.propagate(system, uhf, STEPS * DT, DT)
    assert rel_err(b.energy, host(a.energy)) <= TOL
    assert rel_err(b.dipole, host(a.dipole)) <= TOL
    assert rel_err(b.density_matrix[0] + b.density_matrix[1], host(a.density_matrix[0])) <= TOL


def test_chained_calls_are_bit_identical_to_one_call():
    from quantum_systems_b200 import hartree_fock

    system = with_pulse(spatial())
    state = hartree_fock.ground_state_unrestricted(system, 2, 1)
    whole = hartree_fock.propagate(system, state, 2 * STEPS * DT, DT)
    first = hartree_fock.propagate(system, state, STEPS * DT, DT)
    second = hartree_fock.propagate(system, first, 2 * STEPS * DT, DT)
    assert second.t == whole.t
    for name in ("times", "energy", "dipole"):
        assert torch.equal(torch.cat([getattr(first, name), getattr(second, name)]), getattr(whole, name)), name
    assert all(torch.equal(a, b) for a, b in zip(second.C, whole.C))
    assert all(torch.equal(a, b) for a, b in zip(second.density_matrix, whole.density_matrix))


def test_observe_every_keeps_every_kth_observation():
    from quantum_systems_b200 import hartree_fock

    system = with_pulse(spatial())
    state = hartree_fock.ground_state(system)
    every = hartree_fock.propagate(system, state, STEPS * DT, DT)
    fifth = hartree_fock.propagate(system, state, STEPS * DT, DT, observe_every=5)
    assert torch.equal(fifth.energy, every.energy[::5]) and torch.equal(fifth.times, every.times[::5])
    assert torch.equal(fifth.C[0], every.C[0])


def test_host_system_gets_ndarrays():
    from quantum_systems_b200 import hartree_fock

    dev = with_pulse(spatial())
    hst = with_pulse(spatial(np=np))
    state = hartree_fock.ground_state(hst)
    run = hartree_fock.propagate(hst, state, 10 * DT, DT)
    for value in (run.times, run.energy, run.dipole, *run.C, *run.density_matrix):
        assert isinstance(value, np.ndarray)
    ref = hartree_fock.propagate(dev, hartree_fock.ground_state(dev), 10 * DT, DT)
    assert rel_err(run.energy, host(ref.energy)) <= TOL
    assert rel_err(run.C[0], host(ref.C[0])) <= TOL


def test_device_resident_call_does_not_synchronise():
    """A device system with a real u and no overlap matrix: the whole call, set-up included, runs without a host
    synchronisation; the first read is the caller's."""
    from quantum_systems_b200 import hartree_fock

    system = with_pulse(spatial())
    system._basis_set.s = None
    state = hartree_fock.ground_state_unrestricted(system, 2, 1)
    hartree_fock.propagate(system, state, 2 * DT, DT)  # warm-up: the library is loaded, the allocator primed
    torch.cuda.set_sync_debug_mode("error")
    try:
        run = hartree_fock.propagate(system, state, 10 * DT, DT)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert np.all(np.isfinite(host(run.energy)))


def test_refusals():
    from quantum_systems_b200 import ODSincDVR, SpatialOrbitalSystem, hartree_fock, sharded
    from quantum_systems_b200.time_evolution_operators import AdiabaticSwitching, TimeEvolutionOperator

    system = spatial()
    state = hartree_fock.ground_state(system)
    with pytest.raises(ValueError, match="dt must be positive"):
        hartree_fock.propagate(system, state, 1.0, 0.0)
    with pytest.raises(ValueError, match="dt must be positive"):
        hartree_fock.propagate(system, state, 1.0, -0.1)
    with pytest.raises(ValueError, match="lies before the start time"):
        hartree_fock.propagate(system, state, -0.1, DT)
    run = hartree_fock.propagate(system, state, 2 * DT, DT)
    with pytest.raises(ValueError, match="lies before the start time"):
        hartree_fock.propagate(system, run, DT, DT)

    # states that do not fit the system
    with pytest.raises(ValueError, match="shape"):
        hartree_fock.propagate(SpatialOrbitalSystem(2, odqd(l=6)), state, 1.0, DT)
    with pytest.raises(ValueError, match="shape"):
        hartree_fock.propagate(SpatialOrbitalSystem(6, odqd()), run, 1.0, DT)
    with pytest.raises(ValueError, match="unrestricted"):
        hartree_fock.propagate(general(), hartree_fock.ground_state_unrestricted(system, 2, 1), 1.0, DT)
    with pytest.raises(TypeError, match="state must be"):
        hartree_fock.propagate(system, state.C, 1.0, DT)

    # two-body operators on anything but system.u
    class OtherTensor(TimeEvolutionOperator):
        is_two_body_operator = True

        def u_t_scaled(self, t):
            return 1.0, self._system.u.clone()

    class ReferenceOnly(TimeEvolutionOperator):
        is_two_body_operator = True

        def u_t(self, t):
            return self._system.u

    for op in (OtherTensor(), ReferenceOnly()):
        system.set_time_evolution_operator(op)
        with pytest.raises(ValueError, match="does not scale system.u"):
            hartree_fock.propagate(system, state, 1.0, DT)
    system.set_time_evolution_operator(AdiabaticSwitching(1.0))
    hartree_fock.propagate(system, state, DT, DT)

    # 2-d sinc-DVR storage and sharded bases
    dvr = SpatialOrbitalSystem(2, ODSincDVR(8, 5.0))
    with pytest.raises(ValueError, match="4-d two-body tensor"):
        hartree_fock.propagate(dvr, state, 1.0, DT)
    h = torch.as_tensor(host(system.h)).cuda()
    basis = sharded.ShardedBasisSet.from_global(sharded.EmulatedContext(2), h, None, system.u)
    with pytest.raises(TypeError, match="ShardedBasisSet"):
        hartree_fock.propagate(basis, state, 1.0, DT)
