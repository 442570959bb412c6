"""The numpy linear-response oracle (tests/lr_oracle.py) against the relations its spectra must satisfy (no GPU):
spin unions of closed shells, the small-kick limit of real-time TDHF and the instability of a stretched RHF."""

import numpy as np
import pytest
import scipy.linalg

import lr_oracle
import tdhf_oracle
from oracle import hf_oracle
from oracle import qs_oracle as oracle
from quantum_systems_b200.potentials import DWPotential, HOPotential

N_OCC = 2  # doubly occupied orbitals of the closed shell


@pytest.fixture(scope="module")
def closed_shell():
    # a stiff well (omega = 2): the RHF triplets of softer ODQD wells are unstable, and RPA needs a stable reference
    basis = oracle.odqd_setup_basis(6, 6.0, 201, HOPotential(2.0))
    h, u, d = basis["h"].real, basis["u"].real, basis["position"].real
    state = hf_oracle.ground_state(h, u, N_OCC, restricted=True, tol=1e-12)
    assert state["converged"]
    return h, u, d, state["C"]


def rhf(closed_shell, spin, tda):
    h, u, _, C = closed_shell
    return lr_oracle.spectrum(*lr_oracle.matrices("rhf", h, u, C, N_OCC, spin=spin), tda=tda)[0]


def spin_doubled(u):
    """The spin-orbital ``u`` of a spatial one, spin index fastest (the order of add_spin)."""
    l = u.shape[0]
    eye = np.eye(2)
    return np.einsum("PQRS,ac,bd->PaQbRcSd", u, eye, eye).reshape((2 * l,) * 4)


@pytest.mark.parametrize("tda", [False, True])
def test_closed_shell_uhf_is_the_union_of_rhf_singlets_and_triplets(closed_shell, tda):
    h, u, _, C = closed_shell
    omega = lr_oracle.spectrum(*lr_oracle.matrices("uhf", h, u, (C, C), (N_OCC, N_OCC)), tda=tda)[0]
    union = np.sort(np.concatenate([rhf(closed_shell, "singlet", tda), rhf(closed_shell, "triplet", tda)]))
    np.testing.assert_allclose(omega, union, rtol=1e-10, atol=1e-12)


@pytest.mark.parametrize("anti_symmetrized", [False, True])
@pytest.mark.parametrize("tda", [False, True])
def test_closed_shell_ghf_is_singlets_plus_three_of_each_triplet(closed_shell, tda, anti_symmetrized):
    h, u, _, C = closed_shell
    u_so = spin_doubled(u)
    if anti_symmetrized:
        u_so = u_so - u_so.transpose(0, 1, 3, 2)
    h_so = np.kron(h, np.eye(2))
    C_so = hf_oracle.spin_double_coefficients(C)
    A, B = lr_oracle.matrices("ghf", h_so, u_so, C_so, 2 * N_OCC, anti_symmetrized_u=anti_symmetrized)
    omega = lr_oracle.spectrum(A, B, tda=tda)[0]
    triplets = rhf(closed_shell, "triplet", tda)
    # the GHF space also holds the spin-flip excitations: two more copies of each triplet (M_s = +-1)
    expected = np.sort(np.concatenate([rhf(closed_shell, "singlet", tda), triplets, triplets, triplets]))
    np.testing.assert_allclose(omega, expected, rtol=1e-10, atol=1e-12)


def test_a_weak_kick_follows_the_rpa_spectrum(closed_shell):
    """``C_o -> expm(i kappa d) C_o`` multiplies the determinant by ``exp(i kappa D)``, D the summed dipole.  To first
    order the state is ``|0> + i kappa sum_n <n|D|0> |n>``, whose dipole moves by
    ``sum_n 2 Re(i kappa |mu_n|^2 exp(-i omega_n t)) = 2 kappa sum_n |mu_n|^2 sin(omega_n t)``: positive slope at
    t = 0 for kappa > 0.  TDHF linearised about a stable reference is RPA, so the same holds with the RPA roots and
    ``mu_n``.  The rest is O(kappa^2) (relative O(kappa) after dividing by kappa; the quadratic response of a
    symmetric well is small as well) and the RK4 error, O((omega dt)^4) per unit time, below 1e-8 here."""
    h, u, d, C = closed_shell
    kappa, dt, n_steps = 1e-4, 0.01, 500
    A, B = lr_oracle.matrices("rhf", h, u, C, N_OCC)
    omega, XpY, _ = lr_oracle.spectrum(A, B)
    mu = lr_oracle.transition_dipoles("rhf", XpY, C, N_OCC, d)
    kicked = scipy.linalg.expm(1j * kappa * d[0]) @ C[:, :N_OCC]
    run = tdhf_oracle.propagate("rhf", lambda t: h, lambda t: u, (kicked,), 0.0, n_steps, dt, dipole=d,
                                scales=hf_oracle.scales(True, False))
    d0 = np.einsum("rs,sr->", hf_oracle.density(C, N_OCC, True), d[0]).real
    response = (run["dipole"][:, 0] - d0) / kappa
    predicted = 2 * np.sin(np.outer(run["times"], omega)) @ (mu[:, 0] ** 2)
    assert np.abs(predicted).max() > 0.1  # the kick excites the system
    assert np.abs(response - predicted).max() <= 1e-3 * np.abs(predicted).max()
    assert response[1] > 0  # the sign: the dipole first moves up


def test_stretched_double_well_rhf_is_triplet_unstable():
    """The broken-symmetry double well of tests/test_uhf_oracle_cpu.py: its RHF singlet lies above a UHF state, so
    the triplet instability shows as a negative TDA root, and RPA has no real spectrum."""
    basis = oracle.odqd_setup_basis(8, 10.0, 201, DWPotential(1.0, 5))
    h, u = basis["h"].real, basis["u"].real
    state = hf_oracle.ground_state(h, u, 1, restricted=True, tol=1e-12)
    assert state["converged"]
    A, B = lr_oracle.matrices("rhf", h, u, state["C"], 1, spin="triplet")
    assert lr_oracle.spectrum(A, B, tda=True)[0][0] < 0
    with pytest.raises(ValueError, match="not positive definite"):
        lr_oracle.spectrum(A, B)
