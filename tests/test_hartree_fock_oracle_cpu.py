"""The numpy Hartree-Fock oracle against closed forms and its own invariances (no GPU)."""

import numpy as np
import pytest

from oracle import hf_oracle
from oracle import qs_oracle as oracle


@pytest.fixture(scope="module")
def odqd():
    return oracle.odqd_setup_basis(6, 10.0, 201, _HO(0.25))


class _HO:
    def __init__(self, omega):
        self.omega = omega

    def __call__(self, x):
        return 0.5 * self.omega**2 * x**2


def test_no_interaction_gives_the_aufbau_sum_of_h():
    rng = np.random.default_rng(3)
    A = rng.standard_normal((7, 7))
    h = A + A.T
    u = np.zeros((7,) * 4)
    eig = np.linalg.eigvalsh(h)
    rhf = hf_oracle.ground_state(h, u, 3, restricted=True)
    ghf = hf_oracle.ground_state(h, u, 3, restricted=False, anti_symmetrized_u=True)
    assert rhf["converged"] and ghf["converged"]
    assert abs(rhf["energy"] - 2 * eig[:3].sum()) <= 1e-12 * abs(eig).max()
    assert abs(ghf["energy"] - eig[:3].sum()) <= 1e-12 * abs(eig).max()


def test_one_spatial_orbital():
    h = np.array([[-0.7]])
    u = np.full((1, 1, 1, 1), 0.3)
    state = hf_oracle.ground_state(h, u, 1, restricted=True)
    assert abs(state["energy"] - (2 * -0.7 + 0.3)) <= 1e-15


def test_rhf_equals_ghf_on_the_spin_doubled_basis(odqd):
    h, u = odqd["h"], odqd["u"]
    rhf = hf_oracle.ground_state(h, u, 2, restricted=True)
    assert rhf["converged"]
    h2 = oracle.add_spin_one_body(h)
    u2 = oracle.anti_symmetrize_u(oracle.add_spin_two_body(u))
    ghf = hf_oracle.ground_state(h2, u2, 4, restricted=False, anti_symmetrized_u=True,
                                 C=hf_oracle.spin_double_coefficients(rhf["C"]))
    assert ghf["converged"] and ghf["iterations"] <= 3
    assert abs(ghf["energy"] - rhf["energy"]) <= 1e-12 * abs(rhf["energy"])


def test_energy_is_invariant_under_a_non_orthogonal_basis_change(odqd):
    h, u = odqd["h"], odqd["u"]
    l = h.shape[0]
    X = np.eye(l) + 0.2 * np.random.default_rng(5).standard_normal((l, l))
    ref = hf_oracle.ground_state(h, u, 2, restricted=True)
    h_x = oracle.transform_one_body_elements(h, X)
    u_x = oracle.transform_two_body_elements(u, X)
    state = hf_oracle.ground_state(h_x, u_x, 2, restricted=True, s=X.T @ X)
    assert state["converged"]
    assert abs(state["energy"] - ref["energy"]) <= 1e-10 * abs(ref["energy"])
    with pytest.raises(ValueError):
        X_sing = X.copy()
        X_sing[:, -1] = X_sing[:, 0]
        hf_oracle.ground_state(h, u, 2, restricted=True, s=X_sing.T @ X_sing)
