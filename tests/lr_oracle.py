"""Plain numpy linear-response TDHF: the A and B matrices of RHF (singlet and triplet), GHF and UHF built element by
element from the MO two-body tensor, and their spectra from scipy's dense eigensolver.  Written for reading, not for
speed; test infrastructure only.

Conventions of quantum_systems_b200.hartree_fock.excited_states: ``u`` is physicists' ``<pq|rs> = u[p,q,r,s]``, so
chemists' ``(pq|rs) = u[p,r,q,s]``; ``F`` is the Fock matrix of the reference density and ``dF`` the orbital term
``delta_ij F_ab - delta_ab F_ij`` in the MO basis.  Vectors are indexed (i, a) with i occupied and a virtual, i
slowest; UHF stacks the alpha block before the beta block.
"""

import numpy as np
import scipy.linalg

import uhf_oracle
from oracle import hf_oracle


def mo_tensor(u, C_p, C_q, C_r, C_s):
    """``sum_{PQRS} C_p[P,p] C_q[Q,q] C_r[R,r] C_s[S,s] u[P,Q,R,S]`` (real coefficients)."""
    return np.einsum("PQRS,Pp,Qq,Rr,Ss->pqrs", u, C_p, C_q, C_r, C_s, optimize=True)


def orbital_term(F_mo, n_occ):
    """``delta_ij F_ab - delta_ab F_ij`` as a matrix over (i, a) pairs."""
    F_oo, F_vv = F_mo[:n_occ, :n_occ], F_mo[n_occ:, n_occ:]
    n_virt = F_vv.shape[0]
    return np.kron(np.eye(n_occ), F_vv) - np.kron(F_oo, np.eye(n_virt))


def pairs(T4):
    """A (o, v, o', v') array as the (o v, o' v') matrix of (i a, j b)."""
    o, v, o2, v2 = T4.shape
    return T4.reshape(o * v, o2 * v2)


def matrices(kind, h, u, C, n_occ, spin="singlet", anti_symmetrized_u=False):
    """``(A, B)`` of a reference.  ``kind``: "rhf" (``C`` (l, l), ``n_occ`` doubly occupied, ``spin`` singlet or
    triplet), "ghf" (``C`` and ``n_occ`` of the spin-orbitals; ``u`` anti-symmetrised or not) or "uhf" (``C`` and
    ``n_occ`` are (alpha, beta) pairs on the spatial ``u``)."""
    if kind == "uhf":
        Cs, occ = C, n_occ
        rhos = [hf_oracle.density(c, n, False) for c, n in zip(Cs, occ)]
        Fs = uhf_oracle.uhf_fock(h, u, *rhos)
    else:
        Cs, occ = (C,), (n_occ,)
        restricted = kind == "rhf"
        rho = hf_oracle.density(C, n_occ, restricted)
        Fs = (hf_oracle.fock_from_density(h, u, rho, *hf_oracle.scales(restricted, anti_symmetrized_u)),)
    o = [c[:, :n] for c, n in zip(Cs, occ)]
    v = [c[:, n:] for c, n in zip(Cs, occ)]
    dF = [orbital_term(c.T @ f @ c, n) for c, f, n in zip(Cs, Fs, occ)]

    if kind == "ghf":
        def antisym(p, q, r, s):  # <pq||rs> over the four blocks
            t = mo_tensor(u, p, q, r, s)
            return t if anti_symmetrized_u else t - mo_tensor(u, p, q, s, r).transpose(0, 1, 3, 2)

        # A_ia,jb = <aj||ib>, B_ia,jb = <ab||ij>: (a, j, i, b) and (a, b, i, j) reordered to (i, a, j, b)
        A2 = antisym(v[0], o[0], o[0], v[0]).transpose(2, 0, 1, 3)
        B2 = antisym(v[0], v[0], o[0], o[0]).transpose(2, 0, 3, 1)
        return dF[0] + pairs(A2), pairs(B2)

    def chem(p, q, r, s):  # (pq|rs) = <pr|qs>
        return mo_tensor(u, p, r, q, s).transpose(0, 2, 1, 3)

    if kind == "rhf":
        ovov = chem(o[0], v[0], o[0], v[0])                          # (ia|jb)
        oovv = chem(o[0], o[0], v[0], v[0]).transpose(0, 2, 1, 3)    # (ij|ab) at (i, a, j, b)
        ib_ja = chem(o[0], v[0], o[0], v[0]).transpose(0, 3, 2, 1)   # (ib|ja) at (i, a, j, b)
        if spin == "singlet":
            return dF[0] + pairs(2 * ovov - oovv), pairs(2 * ovov - ib_ja)
        if spin == "triplet":
            return dF[0] - pairs(oovv), -pairs(ib_ja)
        raise ValueError(spin)

    # UHF: blocks (sigma, tau) of A = delta dF + (ia|jb) - delta (ij|ab), B = (ia|jb) - delta (ib|ja)
    A_blocks, B_blocks = [[None, None], [None, None]], [[None, None], [None, None]]
    for s in range(2):
        for t in range(2):
            coulomb = pairs(chem(o[s], v[s], o[t], v[t]))
            A_st, B_st = coulomb.copy(), coulomb.copy()
            if s == t:
                A_st += dF[s] - pairs(chem(o[s], o[s], v[s], v[s]).transpose(0, 2, 1, 3))
                B_st -= pairs(chem(o[s], v[s], o[s], v[s]).transpose(0, 3, 2, 1))
            A_blocks[s][t], B_blocks[s][t] = A_st, B_st
    return np.block(A_blocks), np.block(B_blocks)


def spectrum(A, B, tda=False):
    """All roots ascending: ``(omega, X + Y, X - Y)`` with the vectors as rows and ``(X + Y) . (X - Y) = 1``.
    TDA: ``eigh(A)``, ``Y = 0``.  RPA: ``eigh`` of ``(A - B)^(1/2) (A + B) (A - B)^(1/2)``, whose eigenvalues are
    ``omega^2``; raises ``ValueError`` when ``A - B`` or ``A + B`` is not positive definite."""
    A, B = 0.5 * (A + A.T), 0.5 * (B + B.T)
    if tda:
        w, z = scipy.linalg.eigh(A)
        return w, z.T, z.T
    em, Vm = scipy.linalg.eigh(A - B)
    ep = scipy.linalg.eigvalsh(A + B)
    if em.min() <= 0 or ep.min() <= 0:
        raise ValueError("A - B or A + B is not positive definite: unstable reference")
    root = (Vm * np.sqrt(em)) @ Vm.T
    root_inv = (Vm / np.sqrt(em)) @ Vm.T
    w2, z = scipy.linalg.eigh(root @ (A + B) @ root)
    omega = np.sqrt(w2)
    return omega, ((root @ z) / np.sqrt(omega)).T, ((root_inv @ z) * np.sqrt(omega)).T


def transition_dipoles(kind, XpY, C, n_occ, dipole, spin="singlet"):
    """``<0|d|n>`` (roots, axes): ``sum_ia d_ia (X + Y)_ia`` over the channels, times sqrt 2 for RHF singlets and
    zero for RHF triplets."""
    Cs, occ = (C, n_occ) if kind == "uhf" else ((C,), (n_occ,))
    blocks = [(c[:, :n].T @ dipole @ c[:, n:]).reshape(dipole.shape[0], -1) for c, n in zip(Cs, occ)]
    d_ov = np.concatenate(blocks, axis=1)
    mu = XpY @ d_ov.T
    if kind == "rhf":
        mu = mu * (np.sqrt(2.0) if spin == "singlet" else 0.0)
    return mu
