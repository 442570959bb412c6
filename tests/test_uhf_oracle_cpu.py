"""The numpy UHF oracle (tests/uhf_oracle.py) against closed forms, the RHF oracle and the stationarity
conditions of an unrestricted determinant (no GPU)."""

import numpy as np
import pytest
import scipy.linalg

import uhf_oracle
from oracle import hf_oracle
from oracle import qs_oracle as oracle
from quantum_systems_b200.potentials import DWPotential, HOPotential


@pytest.fixture(scope="module")
def odqd():
    return oracle.odqd_setup_basis(6, 10.0, 201, HOPotential(0.25))


def non_orthogonal(basis, seed=5):
    h, u = basis["h"].real, basis["u"]
    X = np.eye(h.shape[0]) + 0.2 * np.random.default_rng(seed).standard_normal(h.shape)
    return oracle.transform_one_body_elements(h, X), oracle.transform_two_body_elements(u, X), X.T @ X


def brillouin_residual(h, u, s, state):
    w, V = np.linalg.eigh(s)
    X = (V * w ** -0.5) @ V.conj().T
    Fa, Fb = uhf_oracle.uhf_fock(h, u, state["density_alpha"], state["density_beta"])
    return max(np.abs(X.conj().T @ (F @ r @ s - s @ r @ F) @ X).max()
               for F, r in ((Fa, state["density_alpha"]), (Fb, state["density_beta"])))


def test_one_electron_is_the_lowest_eigenvalue_of_h(odqd):
    """One electron sees no interaction (its direct and exchange terms cancel), in any metric."""
    h, u, s = non_orthogonal(odqd)
    state = uhf_oracle.uhf_ground_state(h, u, 1, 0, s=s)
    assert state["converged"]
    e0 = scipy.linalg.eigh(h, s, eigvals_only=True)[0]
    assert abs(state["energy"] - e0) <= 1e-12 * abs(e0)
    assert abs(state["spin_squared"] - 0.75) <= 1e-12


def test_closed_shell_from_the_core_guess_is_rhf(odqd):
    h, u = odqd["h"], odqd["u"]
    rhf = hf_oracle.ground_state(h, u, 2, restricted=True)
    uhf = uhf_oracle.uhf_ground_state(h, u, 2, 2)
    assert rhf["converged"] and uhf["converged"]
    assert abs(uhf["energy"] - rhf["energy"]) <= 1e-12 * abs(rhf["energy"])
    for rho in (uhf["density_alpha"], uhf["density_beta"]):
        assert np.abs(rho - rhf["density_matrix"] / 2).max() <= 1e-10
    assert abs(uhf["spin_squared"]) <= 1e-10


@pytest.mark.parametrize("metric", ["orthonormal", "non_orthogonal"])
def test_open_shell_is_stationary_and_idempotent(odqd, metric):
    if metric == "orthonormal":
        h, u, s = odqd["h"].real, odqd["u"], np.eye(6)
    else:
        h, u, s = non_orthogonal(odqd)
    state = uhf_oracle.uhf_ground_state(h, u, 2, 1, s=s)
    assert state["converged"]
    assert brillouin_residual(h, u, s, state) <= 1e-8
    for rho, n_occ in ((state["density_alpha"], 2), (state["density_beta"], 1)):
        assert np.abs(rho @ s @ rho - rho).max() <= 1e-10
        assert abs(np.trace(rho @ s) - n_occ) <= 1e-10
    assert state["spin_squared"] >= 0.75  # <S^2> of a doublet determinant is at least s(s+1)


# Two electrons (n_alpha = n_beta = 1) in the cusped double well ODQD(8, 10.0, 201, DWPotential(omega=1, l=5)):
# the wells are far enough apart that the singlet breaks spin symmetry (one electron per well).  Found with this
# oracle: E_RHF = 1.92905, E_UHF = 1.20582 with <S^2> = 0.99997 from a HOMO/LUMO rotation by pi/4 of the alpha guess.
BROKEN_SYMMETRY = dict(l=8, grid_length=10.0, num_grid_points=201, omega=1.0, separation=5, angle=np.pi / 4)


def test_broken_symmetry_in_a_stretched_double_well():
    p = BROKEN_SYMMETRY
    basis = oracle.odqd_setup_basis(p["l"], p["grid_length"], p["num_grid_points"], DWPotential(p["omega"], p["separation"]))
    h, u = basis["h"], basis["u"]
    rhf = hf_oracle.ground_state(h, u, 1, restricted=True)
    _, C_core = np.linalg.eigh(h.real)
    uhf = uhf_oracle.uhf_ground_state(h, u, 1, 1, C=(uhf_oracle.homo_lumo_rotated(C_core, 1, p["angle"]), C_core))
    assert rhf["converged"] and uhf["converged"]
    assert uhf["energy"] < rhf["energy"] - 1e-3
    assert uhf["spin_squared"] > 0.1
    assert brillouin_residual(h.real, u, np.eye(p["l"]), uhf) <= 1e-8
