"""The numpy TDHF oracle (tests/tdhf_oracle.py) against the invariants of a Hartree-Fock propagation (no GPU)."""

import numpy as np
import pytest
import scipy.linalg

import tdhf_oracle
import uhf_oracle
from oracle import hf_oracle
from oracle import qs_oracle as oracle
from quantum_systems_b200.potentials import HOPotential


@pytest.fixture(scope="module")
def odqd():
    return oracle.odqd_setup_basis(6, 10.0, 201, HOPotential(0.25))


def rk4_density_bound(eps, dt, n_steps, weight):
    """Drift of a stationary density under RK4: each occupied orbital keeps its direction and loses norm,
    |R(-i eps dt)|^2 = 1 - (eps dt)^6 / 72 + O((eps dt)^8) per step; summed over the orbitals, times the channel
    weight and a slack of 1.5."""
    return 1.5 * weight * n_steps * np.sum((np.abs(eps) * dt) ** 6) / 72


def test_converged_state_without_field_keeps_its_density(odqd):
    h, u = odqd["h"].real, odqd["u"].real
    state = hf_oracle.ground_state(h, u, 2, restricted=True, tol=1e-12)
    dt, n_steps = 0.05, 200
    run = tdhf_oracle.propagate("rhf", lambda t: h, lambda t: u, (state["C"][:, :2],), 0.0, n_steps, dt,
                                scales=hf_oracle.scales(True, False))
    drift = np.abs(run["density_matrix"][0] - state["density_matrix"]).max()
    # the SCF residual (tol) also moves the density, at most by its size per unit time
    assert drift <= rk4_density_bound(state["epsilon"][:2], dt, n_steps, 2) + 1e-12 * n_steps * dt * 10


def test_energy_is_conserved_after_a_dipole_kick(odqd):
    h, u, d = odqd["h"].real, odqd["u"].real, odqd["position"]
    state = hf_oracle.ground_state(h, u, 2, restricted=True)
    kick = scipy.linalg.expm(-0.1j * d[0])
    C = kick @ state["C"][:, :2]
    run = tdhf_oracle.propagate("rhf", lambda t: h, lambda t: u, (C,), 0.0, 200, 0.01, dipole=d,
                                scales=hf_oracle.scales(True, False))
    assert abs(run["energy"][0] - state["energy"]) > 1e-4  # the kick put energy in
    assert np.ptp(run["energy"]) <= 1e-9 * abs(run["energy"][0])
    assert np.ptp(run["dipole"][:, 0]) > 1e-3  # and the dipole oscillates


def test_closed_shell_uhf_reproduces_rhf(odqd):
    h, u, d = odqd["h"].real, odqd["u"].real, odqd["position"]
    state = hf_oracle.ground_state(h, u, 2, restricted=True)
    h_t = tdhf_oracle.dipole_field(h, d, lambda t: 0.3 * np.sin(2.0 * t))
    C = state["C"][:, :2]
    rhf = tdhf_oracle.propagate("rhf", h_t, lambda t: u, (C,), 0.0, 100, 0.02, dipole=d,
                                scales=hf_oracle.scales(True, False))
    uhf = tdhf_oracle.propagate("uhf", h_t, lambda t: u, (C, C), 0.0, 100, 0.02, dipole=d)
    np.testing.assert_allclose(uhf["energy"], rhf["energy"], rtol=1e-12)
    np.testing.assert_allclose(uhf["dipole"], rhf["dipole"], rtol=1e-11, atol=1e-12)
    total = uhf["density_matrix"][0] + uhf["density_matrix"][1]
    assert np.abs(total - rhf["density_matrix"][0]).max() <= 1e-12
    assert np.ptp(rhf["dipole"][:, 0]) > 1e-3  # the field drives the system
    # the UHF Fock matrices are the RHF one for equal spin densities
    Fa, Fb = uhf_oracle.uhf_fock(h, u, *uhf["density_matrix"])
    F = hf_oracle.fock_from_density(h, u, total, 1.0, -0.5)
    assert np.abs(Fa - F).max() <= 1e-12 and np.abs(Fb - F).max() <= 1e-12
