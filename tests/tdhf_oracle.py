"""Plain numpy time-dependent Hartree-Fock: the propagation of quantum_systems_b200.hartree_fock.propagate, written
for reading, not for speed.  The occupied columns of each spin channel move under i dC'/dt = X^H F(t) X C' in the
Loewdin basis X = S^(-1/2), C = X C', with classical RK4 and fixed dt; the Fock matrices are einsums over the whole
u(t).  Test infrastructure only.
"""

import numpy as np

import uhf_oracle
from oracle import hf_oracle


def fock(kind, h, u, rho, scales=None):
    """The channel Fock matrices: one channel with ``scales`` (RHF, GHF) or the two UHF channels (``kind == "uhf"``)."""
    if kind == "uhf":
        return uhf_oracle.uhf_fock(h, u, *rho)
    return (hf_oracle.fock_from_density(h, u, rho[0], *scales),)


def propagate(kind, h_t, u_t, C_occ, t0, n_steps, dt, s=None, dipole=None, scales=None, e_nuc=0.0, observe_every=1):
    """RK4 from the occupied columns ``C_occ`` (one per channel) at ``t0``.  ``h_t(t)`` and ``u_t(t)`` give the
    one- and two-body elements at time t; ``kind`` is "rhf" (weight 2), "ghf" or "uhf" (weight 1).  The observables
    are taken at the start of every ``observe_every``-th step: ``E = 1/2 sum_s tr rho_s (h + F_s) + e_nuc`` and
    ``sum_s tr rho_s d_i``.  Time advances by repeated addition of dt.  Returns a dict with times, energy, dipole,
    t, C and density_matrix (tuples per channel)."""
    weight = 2.0 if kind == "rhf" else 1.0
    l = C_occ[0].shape[0]
    S = np.eye(l) if s is None else np.asarray(s)
    w, V = np.linalg.eigh(S)
    X = (V * w ** -0.5) @ V.conj().T
    X_inv = X @ S

    def densities(Cp):
        return tuple(weight * (X @ c) @ (X @ c).conj().T for c in Cp)

    def derivative(t, h, Cp):
        rho = densities(Cp)
        F = fock(kind, h, u_t(t), rho, scales)
        return [-1j * (X.conj().T @ f @ X @ c) for f, c in zip(F, Cp)], rho, F

    Cp = [X_inv @ np.asarray(c, dtype=np.complex128) for c in C_occ]
    times, energy, dip = [], [], []
    t = t0
    for step in range(n_steps):
        h = h_t(t)
        k1, rho, F = derivative(t, h, Cp)
        if step % observe_every == 0:
            times.append(t)
            energy.append(0.5 * sum(np.sum(r.T * (h + f)) for r, f in zip(rho, F)).real + e_nuc)
            if dipole is not None:
                total = sum(rho)
                dip.append(np.einsum("rs,isr->i", total, dipole).real)
        t_mid, t_end = t + 0.5 * dt, t + dt
        k2 = derivative(t_mid, h_t(t_mid), [c + 0.5 * dt * k for c, k in zip(Cp, k1)])[0]
        k3 = derivative(t_mid, h_t(t_mid), [c + 0.5 * dt * k for c, k in zip(Cp, k2)])[0]
        k4 = derivative(t_end, h_t(t_end), [c + dt * k for c, k in zip(Cp, k3)])[0]
        Cp = [c + dt / 6.0 * (a + 2 * b + 2 * e + g) for c, a, b, e, g in zip(Cp, k1, k2, k3, k4)]
        t = t_end
    dim = 0 if dipole is None else dipole.shape[0]
    return {"times": np.array(times), "energy": np.array(energy), "dipole": np.array(dip).reshape(len(times), dim),
            "t": t, "C": tuple(X @ c for c in Cp), "density_matrix": densities(Cp)}


def dipole_field(h0, dipole, strength, axis=0):
    """``h(t) = h0 - E(t) d_axis``: the length-gauge DipoleFieldInteraction."""
    return lambda t: h0 - strength(t) * dipole[axis]
