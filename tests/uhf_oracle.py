"""Plain numpy unrestricted Hartree-Fock: the same SCF as quantum_systems_b200.hartree_fock.ground_state_unrestricted,
written for reading, not for speed.  It follows oracle/hf_oracle.py (Loewdin orthogonalisation, Pulay DIIS with 8
vectors, Aufbau in eigh order) with one Fock matrix per spin.  Test infrastructure only.
"""

import numpy as np

from oracle.hf_oracle import DIIS_VECTORS, density


def uhf_fock(h, u, rho_alpha, rho_beta):
    """f_s[p,q] = h[p,q] + sum_rs u[p,r,q,s] (rho_a + rho_b)[s,r] - sum_rs u[p,r,s,q] rho_s[s,r] on a spatial u."""
    direct = np.einsum("prqs,sr->pq", u, rho_alpha + rho_beta, optimize=True)
    return (h + direct - np.einsum("prsq,sr->pq", u, rho_alpha, optimize=True),
            h + direct - np.einsum("prsq,sr->pq", u, rho_beta, optimize=True))


def uhf_ground_state(h, u, n_alpha, n_beta, s=None, tol=1e-9, max_iterations=100, C=None, e_nuc=0.0):
    """Unrestricted HF on a spatial u: the SCF of ground_state with one Fock matrix per spin, one DIIS over the
    stacked errors of both spins, converged when the larger of the two errors is at most tol.  C = (C_alpha, C_beta)
    or None (core Hamiltonian for both).  Returns a dict with the fields of UnrestrictedHartreeFockState."""
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

    def diagonalise(F):
        eps, Cp = np.linalg.eigh(X.conj().T @ F @ X)
        return X @ Cp, eps

    if C is None:
        Ca, ea = diagonalise(h)
        Cb, eb = Ca.copy(), ea.copy()
    else:
        (Ca, Cb), ea, eb = (np.asarray(c) for c in C), None, None
    ra, rb = density(Ca, n_alpha, False), density(Cb, n_beta, False)
    fs, errs = [], []
    converged, it, E = False, 0, 0.0
    for it in range(1, max_iterations + 1):
        Fa, Fb = uhf_fock(h, u, ra, rb)
        E = 0.5 * (np.sum(ra.T * (h + Fa)) + np.sum(rb.T * (h + Fb))).real + e_nuc
        err = np.stack([X.conj().T @ (F @ r @ S - S @ r @ F) @ X for F, r in ((Fa, ra), (Fb, rb))])
        converged = np.abs(err).max() <= tol
        if not converged:
            fs.append(np.stack([Fa, Fb]))
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
                Fa, Fb = sum(ci * Fi for ci, Fi in zip(c, fs))
        Ca, ea = diagonalise(Fa)
        Cb, eb = diagonalise(Fb)
        ra, rb = density(Ca, n_alpha, False), density(Cb, n_beta, False)
        if converged:
            break
    ov = Ca[:, :n_alpha].conj().T @ S @ Cb[:, :n_beta]
    s_z = 0.5 * (n_alpha - n_beta)
    return {"C_alpha": Ca, "C_beta": Cb, "epsilon_alpha": ea, "epsilon_beta": eb, "density_alpha": ra,
            "density_beta": rb, "energy": E, "spin_squared": s_z * (s_z + 1) + n_beta - np.sum(np.abs(ov) ** 2),
            "converged": converged, "iterations": it}


def homo_lumo_rotated(C, n_occ, angle):
    """C with its HOMO (column n_occ - 1) and LUMO (column n_occ) rotated by angle: a guess that breaks the spin
    symmetry of a core guess when given to one spin only."""
    C = np.array(C, copy=True)
    homo, lumo = C[:, n_occ - 1].copy(), C[:, n_occ].copy()
    C[:, n_occ - 1] = np.cos(angle) * homo + np.sin(angle) * lumo
    C[:, n_occ] = -np.sin(angle) * homo + np.cos(angle) * lumo
    return C
