"""Plain numpy Hartree-Fock: the same SCF as quantum_systems_b200.hartree_fock, written for reading, not for speed.

Fock matrix from a density (einsum over the whole u), symmetric Loewdin orthogonalisation, Pulay DIIS with 8
vectors on the error X^H (F rho S - S rho F) X, Aufbau in eigh order.  Test infrastructure only.
"""

import numpy as np

DIIS_VECTORS = 8


def fock_from_density(h, u, rho, scale_direct, scale_exchange):
    """f[p,q] = h[p,q] + a_d sum_rs u[p,r,q,s] rho[s,r] + a_x sum_rs u[p,r,s,q] rho[s,r]."""
    return (
        h
        + scale_direct * np.einsum("prqs,sr->pq", u, rho, optimize=True)
        + scale_exchange * np.einsum("prsq,sr->pq", u, rho, optimize=True)
    )


def scales(restricted, anti_symmetrized_u):
    if restricted:
        return 1.0, -0.5
    return (1.0, 0.0) if anti_symmetrized_u else (1.0, -1.0)


def density(C, n_occ, restricted):
    C_o = C[:, :n_occ]
    rho = C_o @ C_o.conj().T
    return 2 * rho if restricted else rho


def energy(h, f, rho, e_nuc=0.0):
    return 0.5 * np.sum(rho.T * (h + f)).real + e_nuc


def ground_state(h, u, n_occ, restricted, anti_symmetrized_u=False, s=None, tol=1e-9, max_iterations=100, C=None,
                 e_nuc=0.0):
    """Returns a dict with C, epsilon, energy, density_matrix, converged, iterations."""
    h = np.asarray(h)
    u = np.asarray(u)
    if not (np.iscomplexobj(h) and np.any(h.imag)) and not (s is not None and np.iscomplexobj(s) and np.any(s.imag)) \
            and not (np.iscomplexobj(u) and np.any(u.imag)):
        h, u = h.real, u.real
        s = None if s is None else np.asarray(s).real
    n = h.shape[0]
    S = np.eye(n) if s is None else np.asarray(s)
    w, V = np.linalg.eigh(S)
    if not (w.max() > 0 and w.min() > 1e-12 * w.max()):
        raise ValueError("the overlap matrix is numerically singular or not positive definite")
    X = (V * w ** -0.5) @ V.conj().T
    a_d, a_x = scales(restricted, anti_symmetrized_u)

    def diagonalise(F):
        eps, Cp = np.linalg.eigh(X.conj().T @ F @ X)
        return X @ Cp, eps

    if C is None:
        C, eps = diagonalise(h)
    else:
        C, eps = np.asarray(C), None
    rho = density(C, n_occ, restricted)
    fs, errs = [], []
    converged, it, E = False, 0, 0.0
    for it in range(1, max_iterations + 1):
        F = fock_from_density(h, u, rho, a_d, a_x)
        E = energy(h, F, rho, e_nuc)
        err = X.conj().T @ (F @ rho @ S - S @ rho @ F) @ X
        converged = np.abs(err).max() <= tol
        if not converged:
            fs.append(F)
            errs.append(err)
            fs, errs = fs[-DIIS_VECTORS:], errs[-DIIS_VECTORS:]
            if len(fs) > 1:
                k = len(fs)
                gram = np.array([[np.vdot(a, b).real for b in errs] for a in errs])
                B = -np.ones((k + 1, k + 1))
                B[:k, :k] = gram / gram.diagonal().max()
                B[k, k] = 0.0
                rhs = np.zeros(k + 1)
                rhs[k] = -1.0
                c = np.linalg.solve(B, rhs)[:k]
                F = sum(ci * Fi for ci, Fi in zip(c, fs))
        C, eps = diagonalise(F)
        rho = density(C, n_occ, restricted)
        if converged:
            break
    return {"C": C, "epsilon": eps, "energy": E, "density_matrix": rho, "converged": converged, "iterations": it}


def spin_double_coefficients(C):
    """Spatial orbitals C (l, l) -> spin-orbitals (2l, 2l) in the order of add_spin (spin index fastest): orbital j
    with spin sigma is column 2 j + sigma, so the Aufbau order of a closed shell is kept."""
    return np.kron(C, np.eye(2))
