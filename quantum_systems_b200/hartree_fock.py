"""Hartree-Fock ground states: the coefficients ``C`` a user passes to ``change_basis`` before CC or CI.

``ground_state(system)`` solves restricted HF (RHF) for a ``SpatialOrbitalSystem`` and general HF (GHF) for a
``GeneralOrbitalSystem``; ``ground_state_sharded(basis, n_occ)`` does the same for a ``ShardedBasisSet`` whose
``u`` is spread over several GPUs.  ``QuantumSystem.change_to_hf_basis`` keeps raising ``NotImplementedError``, as
in the reference; this module is the separate entry point::

    state = hartree_fock.ground_state(system)
    system.change_basis(state.C)     # the system is now in the HF basis

The only O(n^4) step of an iteration, the Fock build from the density matrix, is the CUDA kernel behind
``ops.fock_from_density``.  Everything else is O(n^3) plumbing in torch on the device: Loewdin orthogonalisation
``X = S^(-1/2)``, Pulay DIIS on the error ``X^dagger (F rho S - S rho F) X`` with 8 vectors, ``torch.linalg.eigh`` and
Aufbau filling of the lowest orbitals (in ``eigh`` order).  When ``h``, ``s``, ``u`` and a given initial ``C`` have no
imaginary part the iteration runs in float64 and ``C`` is real, so that ``change_basis(state.C)`` takes the real
quarter GEMM; otherwise it runs in complex128.  One SCF loop serves every solver of this module: it iterates over
spin channels, one for RHF and GHF, two for UHF.

``ground_state_unrestricted(system, n_alpha, n_beta)`` solves unrestricted HF (UHF) on the spatial ``u``: one
coefficient matrix per spin, for open shells and spin-polarised or broken-symmetry states.  Its Fock build,
``ops.fock_from_density_unrestricted``, reads a real ``u`` once for both spins.  ``general_orbital_system`` moves
the spin-orbital system into the UHF basis, ready for CC or CI::

    state = hartree_fock.ground_state_unrestricted(basis, n_alpha=2, n_beta=1)
    system = hartree_fock.general_orbital_system(state, basis)    # GeneralOrbitalSystem(3, ...) in the UHF basis

It transforms the spin blocks of the spatial ``u`` and assembles the anti-symmetrised ``(2l)^4`` tensor from them
in one pass.  ``spin_orbital_coefficients`` gives the ``(2l, 2l)`` coefficients and orbital energies of the same
basis; ``GeneralOrbitalSystem(3, basis).change_basis(C)`` with them computes the same system through the
spin-doubled ``u``: eight to ten times the tensor-core flops (twice that on a complex128 ``u``) and four
``(2l)^4`` buffers.

``propagate(system, state, t_final, dt)`` is time-dependent Hartree-Fock: it moves the occupied orbitals of an RHF,
GHF or UHF state under ``system.h_t(t)`` and the two-body weight of the system's time-evolution operators with
classical RK4, one Fock build of the same kernels per stage, and records the energy and the dipole moment::

    system.set_time_evolution_operator(DipoleFieldInteraction(pulse))
    run = hartree_fock.propagate(system, state, t_final=5.0, dt=1e-2)
    run.times, run.energy, run.dipole                     # (k,), (k,), (k, dim)
    run = hartree_fock.propagate(system, run, t_final=10.0, dt=1e-2)    # continues from run.t
"""

import dataclasses
import warnings

import numpy as np
import torch

from . import _arrays, ops

DIIS_VECTORS = 8
# S is refused when its smallest eigenvalue is below this fraction of its largest: S^(-1/2) would amplify rounding
# errors past the accuracy the iteration is asked for
SINGULAR_OVERLAP = 1e-12


@dataclasses.dataclass
class HartreeFockState:
    """``C`` (l, l): orbitals as columns in ascending orbital energy ``epsilon``, ``C^dagger S C = I``.
    ``density_matrix`` is ``C_o C_o^dagger`` (GHF) or ``2 C_o C_o^dagger`` (RHF) of the occupied columns ``C_o``;
    ``energy`` includes the nuclear repulsion.  ``converged`` is False when ``max_iterations`` ran out."""

    C: object
    epsilon: object
    energy: float
    density_matrix: object
    converged: bool
    iterations: int


@dataclasses.dataclass
class TimeDependentHartreeFockRun:
    """One ``propagate`` call.  ``times`` (k,), ``energy`` (k,) and ``dipole`` (k, dim) are the observables at the
    start of every ``observe_every``-th step: ``energy`` is ``1/2 sum_s tr rho_s (h(t) + F_s(t))`` plus the nuclear
    repulsion, ``dipole`` is ``sum_s tr rho_s d`` for each axis of ``system.dipole_moment``.  ``t`` is the time the
    run ended at and ``C`` / ``density_matrix`` the state there, one entry per spin channel (one for RHF and GHF,
    alpha and beta for UHF): the occupied columns ``C_o`` (l, n_occ) in complex128 and ``C_o C_o^dagger`` (times 2 for
    RHF).  Passing the run back to ``propagate`` continues from ``t``; the observables of ``t`` itself are the first
    ones of that next call."""

    times: object
    energy: object
    dipole: object
    t: float
    C: tuple
    density_matrix: tuple


@dataclasses.dataclass
class UnrestrictedHartreeFockState:
    """``C_alpha``, ``C_beta`` (l, l): orbitals of each spin as columns in ascending orbital energy
    ``epsilon_alpha``, ``epsilon_beta``, ``C^dagger S C = I``; the first ``n_alpha`` (``n_beta``) are occupied.
    ``density_alpha`` / ``density_beta`` are ``C_o C_o^dagger``; ``energy`` includes the nuclear repulsion;
    ``spin_squared`` is ``<S^2>`` of the UHF determinant.  ``converged`` is False when ``max_iterations`` ran out."""

    C_alpha: object
    C_beta: object
    epsilon_alpha: object
    epsilon_beta: object
    density_alpha: object
    density_beta: object
    energy: float
    spin_squared: float
    converged: bool
    iterations: int
    n_alpha: int
    n_beta: int


def ground_state(system, tol=1e-9, max_iterations=100, C=None):
    """RHF (``SpatialOrbitalSystem``: ``system.n`` doubly occupied orbitals, scales ``(1, -1/2)``) or GHF
    (``GeneralOrbitalSystem``: scales ``(1, 0)`` on an anti-symmetrised ``u``, else ``(1, -1)``) ground state.
    ``C`` is the initial guess (default: the core Hamiltonian).  Host (numpy) systems upload ``u`` once and get
    ndarrays back; device systems get tensors.

    The iteration runs in complex128 as soon as one of ``h``, ``s``, ``u`` or ``C`` has a non-zero imaginary part,
    else in float64.  A complex128 ``u`` without imaginary part (every ``GeneralOrbitalSystem`` built from a real
    basis) is then copied to a float64 tensor for the duration of the call: ``n^4 * 8`` more bytes of HBM (2.1 GB at
    n = 128), in exchange for half the bytes read by every Fock build.  ``ground_state_sharded`` does not make that
    copy, see there."""
    from .spatial_orbital_system import SpatialOrbitalSystem

    basis = system._basis_set
    _require_4d(basis)
    restricted = isinstance(system, SpatialOrbitalSystem)
    h, s, u, C = _device_inputs(system, (C,))
    fock = _density_fock(u, _scales(restricted, basis.anti_symmetrized_u))
    occupations = ((system.n, 2 if restricted else 1),)
    result = _scf(h, s, lambda rho: fock(h, rho), occupations, tol, max_iterations, C, system.nuclear_repulsion_energy,
                  None)
    return _host_results(system, _hf_state(result))


def ground_state_sharded(basis, n_occ, tol=1e-9, max_iterations=100, C=None, nuclear_repulsion_energy=0.0):
    """The same SCF on a ``ShardedBasisSet``: ``basis.includes_spin`` selects GHF (else RHF with ``n_occ`` doubly
    occupied orbitals) and ``basis.anti_symmetrized_u`` the exchange scale.  ``h`` and ``s`` are replicated; only the
    Fock build is distributed (``ShardedBasisSet.fock_from_density``).  Rank 0's coefficients, orbital energies,
    energy and convergence decision are broadcast every iteration, so every rank holds bit-identical ``C`` and takes
    the same number of iterations.  A given initial ``C`` must have the same shape and dtype on every rank; rank 0's
    values are used everywhere.

    The working dtype follows the same rule as ``ground_state``, with the imaginary-part test of ``u`` combined over
    all ranks.  A real-valued complex128 ``u`` is NOT copied to float64 here: the slabs of a tensor that needs several
    GPUs are sized to fill them, so the Fock build reads the complex slabs and keeps the real part of ``f`` (its
    imaginary part is exactly zero for a real density)."""
    restricted = not basis.includes_spin
    h, s, C, agree = _sharded_inputs(basis, (C,))
    scales = _scales(restricted, basis.anti_symmetrized_u)
    fock = _sharded_fock(lambda rho: (basis.fock_from_density(h, rho[0], *scales),), h.dtype)
    occupations = ((n_occ, 2 if restricted else 1),)
    return _hf_state(_scf(h, s, fock, occupations, tol, max_iterations, C, nuclear_repulsion_energy, agree))


def ground_state_unrestricted(system, n_alpha=None, n_beta=None, tol=1e-9, max_iterations=100, C=None):
    """UHF ground state with ``n_alpha`` spin-up and ``n_beta`` spin-down electrons on the spatial ``u`` of
    ``system``: a ``SpatialOrbitalSystem`` (both default to ``system.n``, its number of doubly occupied orbitals)
    or a spatial ``BasisSet`` (both required).  ``C = (C_alpha, C_beta)`` is the initial guess (default: the core
    Hamiltonian for both spins; a spin-symmetric guess stays spin-symmetric, so a broken-symmetry solution needs a
    guess that breaks it).  Fock matrices ``f_s = h + J[rho_a + rho_b] - K[rho_s]`` from
    ``ops.fock_from_density_unrestricted``, one Pulay DIIS over the errors of both spins with one coefficient set,
    converged when the larger error of the two is at most ``tol``.  Working dtype and the float64 copy of a
    real-valued complex ``u`` as in ``ground_state``.  Host (numpy) systems get ndarrays back."""
    basis = getattr(system, "_basis_set", system)
    _require_plain_spatial_u(basis, "ground_state")
    if system is not basis:
        n_alpha = system.n if n_alpha is None else n_alpha
        n_beta = system.n if n_beta is None else n_beta
    n_alpha, n_beta = _occupations(n_alpha, n_beta, basis.l)
    h, s, u, C = _device_inputs(basis, (None, None) if C is None else C)
    fock = _density_fock(u, None)
    occupations = ((n_alpha, 1), (n_beta, 1))
    result = _scf(h, s, lambda rho: fock(h, rho), occupations, tol, max_iterations, C, basis.nuclear_repulsion_energy,
                  None)
    return _host_results(basis, _uhf_state(result, h, s, n_alpha, n_beta))


def ground_state_unrestricted_sharded(basis, n_alpha, n_beta, tol=1e-9, max_iterations=100, C=None,
                                      nuclear_repulsion_energy=0.0):
    """The UHF iteration of ``ground_state_unrestricted`` on a ``ShardedBasisSet`` with ``includes_spin=False``:
    only the Fock build is distributed (``ShardedBasisSet.fock_from_density_unrestricted``); rank 0's coefficients,
    orbital energies, energy and convergence decision are broadcast, the working dtype and the given guesses are
    handled as in ``ground_state_sharded`` (a real-valued complex ``u`` is not copied to float64)."""
    _require_plain_spatial_u(basis, "ground_state_sharded")
    n_alpha, n_beta = _occupations(n_alpha, n_beta, basis.u.n)
    h, s, C, agree = _sharded_inputs(basis, (None, None) if C is None else C)
    fock = _sharded_fock(lambda rho: basis.fock_from_density_unrestricted(h, *rho), h.dtype)
    occupations = ((n_alpha, 1), (n_beta, 1))
    result = _scf(h, s, fock, occupations, tol, max_iterations, C, nuclear_repulsion_energy, agree)
    return _uhf_state(result, h, s, n_alpha, n_beta)


def propagate(system, state, t_final, dt, observe_every=1):
    """Time-dependent Hartree-Fock from ``state`` to ``t_final`` in fixed steps ``dt``: a ``HartreeFockState`` of
    ``ground_state(system)`` (RHF on a ``SpatialOrbitalSystem``, GHF on a ``GeneralOrbitalSystem``), an
    ``UnrestrictedHartreeFockState`` of ``ground_state_unrestricted(system, ...)`` on a ``SpatialOrbitalSystem``, or
    a ``TimeDependentHartreeFockRun`` of an earlier call, which continues from its ``t`` (a state starts at t = 0).
    Returns a ``TimeDependentHartreeFockRun``; a chain of calls computes bit for bit what one call over the whole
    interval computes.

    The occupied columns ``C_o`` of each spin channel are propagated in complex128 in the Loewdin basis
    ``X = S^(-1/2)``: ``i dC'/dt = X^dagger F(t) X C'`` with ``C = X C'``, classical RK4, one Fock build per stage.
    ``F(t) = h(t) + w(t) G[rho]``: ``h(t)`` is ``system.h_t(t)``; the two-body operators enter as the weight
    ``w(t) = [add_u_0] + sum_k w_k(t)`` of their ``u_t_scaled`` pairs, whose operand must be the system's own ``u``,
    so the n^4 tensor is never scaled or copied.  The Fock builds and channels are those of the ground-state solvers
    (``ops.fock_from_density`` with the RHF or GHF scales, ``ops.fock_from_density_unrestricted`` for UHF).  The
    first stage of a step gives the observables at its start without another build.  ``round((t_final - t) / dt)``
    steps are taken; time advances by repeated addition of ``dt``.

    On a device-resident system no step synchronises with the host and the observables stay in device buffers; only
    the set-up reads the host (the overlap check of ``S``, the imaginary-part test of a complex ``u``).  Host
    (numpy) systems upload ``u`` once and get ndarrays, read once at the end.  A complex128 ``u`` without imaginary
    part is copied to float64 for the call, as in ``ground_state``.  2-D sinc-DVR storage, a ``ShardedBasisSet`` and
    two-body operators on any other tensor than ``system.u`` are refused."""
    from .sharded import ShardedBasisSet
    from .spatial_orbital_system import SpatialOrbitalSystem

    if isinstance(system, ShardedBasisSet) or isinstance(getattr(system, "_basis_set", None), ShardedBasisSet):
        raise TypeError("propagate runs on one GPU: a ShardedBasisSet has no dipole matrices or time-evolution "
                        "operators")
    basis = system._basis_set
    _require_4d(basis)
    restricted = isinstance(system, SpatialOrbitalSystem)
    dt, t_final, observe_every = float(dt), float(t_final), int(observe_every)
    if not dt > 0:
        raise ValueError(f"dt must be positive, got {dt}")
    if observe_every < 1:
        raise ValueError(f"observe_every must be at least 1, got {observe_every}")
    C_occ, t, unrestricted = _propagation_start(system, basis, state, restricted)
    if not t_final >= t:
        raise ValueError(f"t_final = {t_final} lies before the start time {t}")
    n_steps = int(round((t_final - t) / dt))

    s = _arrays.to_device(basis.s) if basis.s is not None else None
    u = _arrays.to_device(basis.u)
    if _has_imag(s):
        s = s.to(torch.complex128)
    elif s is not None:
        s = _as_dtype(s, torch.float64)
    if u.is_complex() and not _has_imag(u):
        u = _as_dtype(u, torch.float64)
    device, cdt = u.device, torch.complex128
    l = basis.l
    X = _orthogonaliser(s, l, s.dtype if s is not None else torch.float64, device).to(cdt)
    X_inv = X @ (s.to(cdt) if s is not None else torch.eye(l, dtype=cdt, device=device))  # S^(1/2)
    Xh = X.mH.contiguous()
    weight = 2 if restricted and not unrestricted else 1
    fock = _density_fock(u, None if unrestricted else _scales(restricted, basis.anti_symmetrized_u))
    d = system.dipole_moment
    d = _arrays.to_device(d).to(cdt) if d is not None else None
    dim = 0 if d is None else d.shape[0]
    e_nuc = float(system.nuclear_repulsion_energy)

    # the two-body weight and its checks, before any step
    _two_body_weight(system, t)

    def h_at(time):
        return _arrays.to_device(system.h_t(time))

    def derivative(time, h, Cp):
        """``-i X^dagger F X C'`` of every channel, the densities and the Fock matrices."""
        Cs = [X @ c for c in Cp]
        rho = tuple(_density(c, c.shape[1], weight) for c in Cs)
        F = fock(h, rho, _two_body_weight(system, time))
        return [-1j * (Xh @ (f @ c)) for f, c in zip(F, Cs)], rho, F

    n_obs = (n_steps + observe_every - 1) // observe_every
    energy = torch.empty(n_obs, dtype=torch.float64, device=device)
    dipole = torch.empty((n_obs, dim), dtype=torch.float64, device=device)
    times = []
    Cp = [X_inv @ _arrays.to_device(c).to(cdt) for c in C_occ]
    h = h_at(t)
    for step in range(n_steps):
        k1, rho, F = derivative(t, h, Cp)
        if step % observe_every == 0:
            j = len(times)
            times.append(t)
            energy[j] = 0.5 * sum(torch.sum(r.transpose(0, 1) * (h + f)) for r, f in zip(rho, F)).real + e_nuc
            if d is not None:
                rho_total = sum(rho[1:], rho[0])
                dipole[j] = torch.einsum("rs,isr->i", rho_total, d).real
        t_mid, t_end = t + 0.5 * dt, t + dt
        h_mid = h_at(t_mid)
        k2 = derivative(t_mid, h_mid, [c + (0.5 * dt) * k for c, k in zip(Cp, k1)])[0]
        k3 = derivative(t_mid, h_mid, [c + (0.5 * dt) * k for c, k in zip(Cp, k2)])[0]
        h = h_at(t_end)
        k4 = derivative(t_end, h, [c + dt * k for c, k in zip(Cp, k3)])[0]
        Cp = [c + (dt / 6.0) * (a + 2.0 * b + 2.0 * e + g) for c, a, b, e, g in zip(Cp, k1, k2, k3, k4)]
        t = t_end
    C = tuple(X @ c for c in Cp)
    rho = tuple(_density(c, c.shape[1], weight) for c in C)
    times = torch.tensor(times, dtype=torch.float64).to(device, non_blocking=True)
    return _read_run(system, TimeDependentHartreeFockRun(times, energy, dipole, t, C, rho))


@dataclasses.dataclass
class ExcitedStates:
    """Linear-response excited states of one ``excited_states`` call, roots in ascending ``energies`` (n_states,).
    ``X`` and ``Y`` hold one ``(n_states, n_occ, n_virt)`` array per spin channel (one for RHF and GHF, alpha and
    beta for UHF), normalised to ``sum X^2 - sum Y^2 = 1`` over all channels; ``Y`` is zero for TDA.
    ``transition_dipole`` (n_states, dim) is ``<0|d|n>`` for each axis of ``system.dipole_moment`` (sqrt 2 times the
    spatial sum for RHF singlets, zero for RHF triplets) and ``oscillator_strength`` is ``2 omega |mu_a|^2`` per
    axis.  ``residual_norms`` are the final residuals of the roots, ``converged`` says whether all are at most
    ``tol``, ``iterations`` counts subspace iterations and ``densities_built`` the AO densities contracted with u."""

    energies: object
    X: tuple
    Y: tuple
    transition_dipole: object
    oscillator_strength: object
    residual_norms: object
    converged: bool
    iterations: int
    densities_built: int


def excited_states(system, state, n_states=5, tda=False, spin="singlet", tol=1e-6, max_iterations=100):
    """Linear-response TDHF (RPA, or the Tamm-Dancoff approximation with ``tda=True``) excitation energies of a
    converged reference: a ``HartreeFockState`` on a ``SpatialOrbitalSystem`` (RHF, ``spin="singlet"`` or
    ``"triplet"``) or a ``GeneralOrbitalSystem`` (GHF), or an ``UnrestrictedHartreeFockState`` on a
    ``SpatialOrbitalSystem`` (UHF, spin-conserving).  Returns ``ExcitedStates``; host (numpy) systems get ndarrays.

    With ``F`` the Fock matrix of the state's density and ``(pq|rs) = u[p,r,q,s]``, ``A = dF + <aj||ib>`` and
    ``B = <ab||ij>`` (GHF; RHF and UHF in their spin-adapted forms), ``dF = delta_ij F_ab - delta_ab F_ij``.  ``A +- B``
    act on a trial vector ``Z`` of each channel through the AO density ``T = C_o Z C_v^T``: the two-electron part of
    ``(A +- B) Z`` is ``C_v^T G[T^T +- T] C_o`` and that of ``A Z`` is ``C_v^T G[T^T] C_o``, with ``G`` the Coulomb and
    exchange combination of the channel (RHF singlet ``2J - K``, triplet ``-K``, GHF the ground-state scales, UHF
    ``J[D_alpha] + J[D_beta] - K[D_sigma]``).  All densities of an iteration go through one
    ``ops.coulomb_exchange`` call, the only O(n^4) step; the rest is torch on the device.  TDA is a Davidson
    iteration on ``A``; RPA the real symmetric subspace method of Stratmann, Scuseria and Frisch (J. Chem. Phys. 109,
    8218 (1998)): ``A + B`` and ``A - B`` projected onto one expansion space, ``(A-B)^(1/2) (A+B) (A-B)^(1/2) z =
    omega^2 z``, residuals preconditioned with ``(dF_diag - omega)^-1``.  The space starts from the unit vectors of
    the lowest ``dF`` diagonal and is capped at the dimension ``n_occ n_virt``, where Rayleigh-Ritz is exact.  A
    projected ``A - B`` or ``A + B`` that is not positive definite means an unstable reference: RPA raises
    ``ValueError``; TDA returns the negative root.

    Refused: a ``ShardedBasisSet`` and 2-D sinc-DVR storage, a complex working dtype (complex orbitals), an
    unconverged state or one that does not fit ``system``, ``spin`` other than singlet or triplet or a triplet of
    GHF or UHF, ``n_states`` outside ``[1, n_occ n_virt]`` and a reference without virtual orbitals.  A complex128
    ``u`` without imaginary part is copied to float64 for the call, as in ``ground_state``."""
    from .sharded import ShardedBasisSet
    from .spatial_orbital_system import SpatialOrbitalSystem

    if isinstance(system, ShardedBasisSet) or isinstance(getattr(system, "_basis_set", None), ShardedBasisSet):
        raise TypeError("excited_states runs on one GPU: a ShardedBasisSet is not supported")
    basis = system._basis_set
    _require_4d(basis)
    restricted = isinstance(system, SpatialOrbitalSystem)
    if spin not in ("singlet", "triplet"):
        raise ValueError(f"spin must be 'singlet' or 'triplet', got {spin!r}")
    l = basis.l
    if isinstance(state, UnrestrictedHartreeFockState):
        if not restricted:
            raise ValueError("an unrestricted state is solved on the SpatialOrbitalSystem it came from")
        _require_plain_spatial_u(basis, "excited_states")
        kind = "uhf"
        coefficients = (state.C_alpha, state.C_beta)
        occupied = (state.n_alpha, state.n_beta)
    elif isinstance(state, HartreeFockState):
        kind = "rhf" if restricted else "ghf"
        coefficients, occupied = (state.C,), (system.n,)
    else:
        raise TypeError("state must be a HartreeFockState or an UnrestrictedHartreeFockState, "
                        f"got {type(state).__name__}")
    if spin == "triplet" and kind != "rhf":
        raise ValueError(f"spin='triplet' is an RHF option; a {kind.upper()} reference has no spin adaptation")
    if not state.converged:
        raise ValueError("the reference state is not converged")
    for C in coefficients:
        if tuple(C.shape) != (l, l):
            raise ValueError(f"the state has {tuple(C.shape)} coefficients, the system needs {(l, l)}")
    if not all(0 <= n_occ <= l for n_occ in occupied):
        raise ValueError(f"occupations {occupied} do not fit l = {l}")
    sizes = [n_occ * (l - n_occ) for n_occ in occupied]
    dim = sum(sizes)
    if dim == 0:
        raise ValueError("the reference has no virtual orbitals (or no occupied ones): nothing to excite")
    n_states = int(n_states)
    if not 1 <= n_states <= dim:
        raise ValueError(f"n_states = {n_states} must lie in [1, {dim}] (n_occ * n_virt)")

    h = _arrays.to_device(basis.h)
    u = _arrays.to_device(basis.u)
    Cs = [_arrays.to_device(C) for C in coefficients]
    if any(_has_imag(t) for t in (h, u, *Cs)):
        raise NotImplementedError("excited_states needs real orbitals and a real u: complex orbitals are not "
                                  "supported")
    h, u = _as_dtype(h, torch.float64), _as_dtype(u, torch.float64)
    Cs = [_as_dtype(C, torch.float64) for C in Cs]

    # the Fock matrices of the reference from one existing build, and the response scales (J, K) of each channel
    if kind == "uhf":
        F = _density_fock(u, None)(h, tuple(_density(C, n_occ, 1) for C, n_occ in zip(Cs, occupied)))
        scales = (1.0, -1.0)
    else:
        F = _density_fock(u, _scales(restricted, basis.anti_symmetrized_u))(
            h, (_density(Cs[0], occupied[0], 2 if restricted else 1),))
        if kind == "rhf":
            scales = (2.0, -1.0) if spin == "singlet" else (0.0, -1.0)
        else:
            scales = _scales(False, basis.anti_symmetrized_u)
    channels = []
    for C, f, n_occ in zip(Cs, F, occupied):
        C_o, C_v = C[:, :n_occ].contiguous(), C[:, n_occ:].contiguous()
        channels.append((C_o, C_v, C_o.T @ f @ C_o, C_v.T @ f @ C_v))
    diagonal = torch.cat([(torch.diagonal(F_vv)[None, :] - torch.diagonal(F_oo)[:, None]).reshape(-1)
                          for _, _, F_oo, F_vv in channels])
    counter = [0]

    def products(V, signs):
        """``(A + s B) V`` for each ``s`` in ``signs`` (None: ``A`` alone) on the rows of ``V`` (m, dim)."""
        m = V.shape[0]
        Zs, Ts, offset = [], [], 0
        for (C_o, C_v, _, _), size in zip(channels, sizes):
            Z = V[:, offset:offset + size].reshape(m, C_o.shape[1], C_v.shape[1])
            offset += size
            Zs.append(Z)
            Ts.append(C_o @ Z @ C_v.T)
        densities = [T.transpose(1, 2) + (0.0 if s is None else s) * T for s in signs for T in Ts]
        J, K = ops.coulomb_exchange(u, torch.cat(densities).contiguous())
        counter[0] += J.shape[0]
        J = J.reshape(len(signs), len(Ts), m, l, l)
        K = K.reshape(len(signs), len(Ts), m, l, l)
        out = []
        for a in range(len(signs)):
            J_total = J[a].sum(dim=0) if kind == "uhf" else J[a, 0]
            parts = []
            for c, ((C_o, C_v, F_oo, F_vv), Z) in enumerate(zip(channels, Zs)):
                G = scales[0] * J_total + scales[1] * K[a, c]
                parts.append((Z @ F_vv - F_oo @ Z + C_o.T @ G.transpose(1, 2) @ C_v).reshape(m, -1))
            out.append(torch.cat(parts, dim=1))
        return out

    solve = _davidson_tda if tda else _davidson_rpa
    omega, XpY, XmY, residuals, converged, iterations = solve(products, diagonal, n_states, tol, max_iterations)
    X, Y = 0.5 * (XpY + XmY), 0.5 * (XpY - XmY)
    # one sign per root: the largest component of X positive
    pick = torch.argmax(X.abs(), dim=1)
    sign = torch.sign(X.gather(1, pick[:, None]))
    sign[sign == 0] = 1.0
    X, Y, XpY = X * sign, Y * sign, XpY * sign

    d = system.dipole_moment
    n_axes = 0 if d is None else d.shape[0]
    mu = torch.zeros((n_states, n_axes), dtype=torch.float64, device=u.device)
    if d is not None and not (kind == "rhf" and spin == "triplet"):
        d = _arrays.to_device(d)
        if _has_imag(d):
            raise NotImplementedError("excited_states needs a real dipole moment")
        d = _as_dtype(d, torch.float64)
        offset = 0
        for (C_o, C_v, _, _), size in zip(channels, sizes):
            d_ov = (C_o.T @ d @ C_v).reshape(n_axes, -1)
            mu += XpY[:, offset:offset + size] @ d_ov.T
            offset += size
        if kind == "rhf":
            mu *= 2.0 ** 0.5
    strength = 2.0 * omega[:, None] * mu ** 2

    def split(M):
        out, offset = [], 0
        for (C_o, C_v, _, _), size in zip(channels, sizes):
            out.append(M[:, offset:offset + size].reshape(n_states, C_o.shape[1], C_v.shape[1]).contiguous())
            offset += size
        return tuple(out)

    result = ExcitedStates(energies=omega, X=split(X), Y=split(Y), transition_dipole=mu, oscillator_strength=strength,
                           residual_norms=residuals, converged=converged, iterations=iterations,
                           densities_built=counter[0])
    if _arrays.is_host_module(system.np):
        host = _arrays.to_host
        result = dataclasses.replace(result, energies=host(result.energies), X=tuple(host(x) for x in result.X),
                                     Y=tuple(host(y) for y in result.Y),
                                     transition_dipole=host(result.transition_dipole),
                                     oscillator_strength=host(result.oscillator_strength),
                                     residual_norms=host(result.residual_norms))
    return result


# a correction whose norm falls below this fraction of its length before projection adds nothing new to the space
_DEPENDENT = 1e-8


def _expand(basis, vectors, dim):
    """``basis`` (m, dim), orthonormal rows, extended by the parts of ``vectors`` orthogonal to it and to each other
    (two Gram-Schmidt passes), at most to ``dim`` rows.  Returns ``(basis, new rows)``."""
    new = []
    for v in vectors:
        if basis.shape[0] + len(new) >= dim:
            break
        length = torch.linalg.vector_norm(v)
        if not length > 0:
            continue
        v = v / length
        Q = torch.cat([basis, *[w[None] for w in new]]) if new else basis
        for _ in range(2):
            v = v - (Q @ v) @ Q
        norm = float(torch.linalg.vector_norm(v))
        if norm > _DEPENDENT:
            new.append(v / norm)
    if not new:
        return basis, basis[:0]
    added = torch.stack(new)
    return torch.cat([basis, added]), added


def _start(diagonal, n_states):
    """Unit vectors at the lowest entries of the orbital-energy diagonal: ``2 n_states`` of them, at most all."""
    dim = diagonal.shape[0]
    count = min(dim, 2 * n_states)
    order = torch.argsort(diagonal, stable=True)[:count]
    return torch.eye(dim, dtype=torch.float64, device=diagonal.device)[order]


def _precondition(R, diagonal, omega):
    den = diagonal[None, :] - omega[:, None]
    den = torch.where(den.abs() < 1e-8, torch.copysign(torch.full_like(den, 1e-8), den), den)
    return R / den


def _davidson_tda(products, diagonal, n_states, tol, max_iterations):
    """Davidson on ``A``; returns ``(omega, X, X, residual norms, converged, iterations)``."""
    dim = diagonal.shape[0]
    basis = diagonal.new_zeros((0, dim))
    AV = diagonal.new_zeros((0, dim))
    basis, new = _expand(basis, _start(diagonal, n_states), dim)
    it = 0
    for it in range(1, max_iterations + 1):
        AV = torch.cat([AV, products(new, (None,))[0]])
        a = basis @ AV.T
        w, z = torch.linalg.eigh(0.5 * (a + a.T))
        omega, z = w[:n_states], z[:, :n_states]
        x = z.T @ basis
        R = z.T @ AV - omega[:, None] * x
        norms = torch.linalg.vector_norm(R, dim=1)
        done = norms <= tol
        if bool(done.all()) or it == max_iterations:
            break
        basis, new = _expand(basis, _precondition(R[~done], diagonal, omega[~done]), dim)
        if new.shape[0] == 0:
            break
    return omega, x, x, norms, bool(done.all()), it


def _davidson_rpa(products, diagonal, n_states, tol, max_iterations):
    """Stratmann-Scuseria-Frisch on ``A + B`` and ``A - B``; returns ``(omega, X + Y, X - Y, residual norms,
    converged, iterations)`` with ``(X + Y) . (X - Y) = 1``."""
    dim = diagonal.shape[0]
    basis = diagonal.new_zeros((0, dim))
    PV = diagonal.new_zeros((0, dim))
    MV = diagonal.new_zeros((0, dim))
    basis, new = _expand(basis, _start(diagonal, n_states), dim)
    it = 0
    for it in range(1, max_iterations + 1):
        plus, minus = products(new, (1.0, -1.0))
        PV, MV = torch.cat([PV, plus]), torch.cat([MV, minus])
        mp, mm = basis @ PV.T, basis @ MV.T
        mp, mm = 0.5 * (mp + mp.T), 0.5 * (mm + mm.T)
        em, Vm = torch.linalg.eigh(mm)
        ep = torch.linalg.eigvalsh(mp)
        if not float(em.min()) > 0:
            raise ValueError(f"A - B is not positive definite in the subspace (eigenvalue {float(em.min()):.3e}): "
                             "the reference is unstable, RPA has no real excitation energies")
        if not float(ep.min()) > 0:
            raise ValueError(f"A + B is not positive definite in the subspace (eigenvalue {float(ep.min()):.3e}): "
                             "the reference is unstable, RPA has no real excitation energies")
        root = (Vm * em.sqrt()) @ Vm.T
        root_inv = (Vm * em.rsqrt()) @ Vm.T
        H = root @ mp @ root
        w2, z = torch.linalg.eigh(0.5 * (H + H.T))
        omega = w2[:n_states].sqrt()
        z = z[:, :n_states]
        xp = (root @ z) / omega.sqrt()
        xm = (root_inv @ z) * omega.sqrt()
        XpY, XmY = xp.T @ basis, xm.T @ basis
        R_plus = xp.T @ PV - omega[:, None] * XmY
        R_minus = xm.T @ MV - omega[:, None] * XpY
        norms = torch.sqrt(torch.linalg.vector_norm(R_plus, dim=1) ** 2
                           + torch.linalg.vector_norm(R_minus, dim=1) ** 2)
        done = norms <= tol
        if bool(done.all()) or it == max_iterations:
            break
        open_ = ~done
        corrections = torch.cat([_precondition(R_plus[open_], diagonal, omega[open_]),
                                 _precondition(R_minus[open_], diagonal, omega[open_])])
        basis, new = _expand(basis, corrections, dim)
        if new.shape[0] == 0:
            break
    return omega, XpY, XmY, norms, bool(done.all()), it


def _propagation_start(system, basis, state, restricted):
    """The occupied columns of each channel, the start time and whether the state is unrestricted, after checking
    that ``state`` fits ``system``."""
    l = basis.l

    def shaped(C, n_occ, what):
        if tuple(C.shape) != (l, n_occ):
            raise ValueError(f"{what} has shape {tuple(C.shape)}, the system needs {(l, n_occ)}")
        return C

    if isinstance(state, UnrestrictedHartreeFockState):
        if not restricted:
            raise ValueError("an unrestricted state propagates on the SpatialOrbitalSystem it was solved on")
        _require_plain_spatial_u(basis, "propagate")
        shaped(state.C_alpha, l, "C_alpha")
        shaped(state.C_beta, l, "C_beta")
        return (state.C_alpha[:, :state.n_alpha], state.C_beta[:, :state.n_beta]), 0.0, True
    if isinstance(state, HartreeFockState):
        return (shaped(state.C, l, "C")[:, :system.n],), 0.0, False
    if isinstance(state, TimeDependentHartreeFockRun):
        if len(state.C) == 2:
            if not restricted:
                raise ValueError("an unrestricted run propagates on a SpatialOrbitalSystem")
            _require_plain_spatial_u(basis, "propagate")
            return tuple(shaped(c, c.shape[1], f"C[{k}]") for k, c in enumerate(state.C)), float(state.t), True
        if len(state.C) != 1:
            raise ValueError(f"a run has one or two spin channels, got {len(state.C)}")
        return (shaped(state.C[0], system.n, "C[0]"),), float(state.t), False
    raise TypeError("state must be a HartreeFockState, an UnrestrictedHartreeFockState or a "
                    f"TimeDependentHartreeFockRun, got {type(state).__name__}")


def _two_body_weight(system, t):
    """``w(t) = [add_u_0] + sum_k w_k(t)`` over the two-body operators of ``system``, from their ``u_t_scaled`` pairs;
    an operator without one, or whose operand is not ``system.u``, is refused."""
    w = 1.0 if system._add_u_0 else 0.0
    for op in system._time_evolution_operator:
        if not op.is_two_body_operator:
            continue
        scaled = getattr(op, "u_t_scaled", None)
        weight, operand = scaled(t) if scaled is not None else (None, None)
        if operand is not system.u:
            raise ValueError(f"propagate folds two-body operators into the Fock build as a weight on system.u; "
                             f"{type(op).__name__} does not scale system.u")
        w = w + weight
    return w


def _read_run(system, run):
    """``run`` with its tensors as ndarrays when ``system`` keeps its arrays on the host: the one read of the call."""
    if not _arrays.is_host_module(system.np):
        return run
    host = _arrays.to_host
    return dataclasses.replace(run, times=host(run.times), energy=host(run.energy), dipole=host(run.dipole),
                               C=tuple(host(c) for c in run.C),
                               density_matrix=tuple(host(r) for r in run.density_matrix))


def _density_fock(u, scales):
    """The Fock build of the single-GPU solvers and the propagator: ``fock(h, rho, w=1)`` maps the tuple of channel
    densities to the tuple of Fock matrices ``h + w G[rho]``.  ``scales`` (direct, exchange) give one channel through
    ``ops.fock_from_density`` (``w`` multiplies the scales); None gives the two UHF channels through
    ``ops.fock_from_density_unrestricted``, which takes no scales, so ``w != 1`` builds ``G`` on a zero ``h`` and adds
    ``h + w G`` on the n^2 side."""
    if scales is not None:
        a_d, a_x = scales

        def fock(h, rho, w=1.0):
            return (ops.fock_from_density(h, u, rho[0], w * a_d, w * a_x),)

        return fock

    def fock(h, rho, w=1.0):
        if w == 1.0:
            return ops.fock_from_density_unrestricted(h, u, *rho)
        return tuple(h + w * g for g in ops.fock_from_density_unrestricted(torch.zeros_like(h), u, *rho))

    return fock


def _device_inputs(source, guesses):
    """``h``, ``s``, ``u`` and the initial guesses of a system or basis on the device in the working dtype, with a
    complex ``u`` without imaginary part copied to float64 (see ``ground_state``)."""
    h = _arrays.to_device(source.h)
    s = _arrays.to_device(source.s) if source.s is not None else None
    u = _arrays.to_device(source.u)  # uploaded once for a host system, resident for the iterations
    guesses = [_arrays.to_device(C) if C is not None else None for C in guesses]
    dtype = _working_dtype(_has_imag(h), _has_imag(s), _has_imag(u), *(_has_imag(C) for C in guesses))
    h, s = _as_dtype(h, dtype), _as_dtype(s, dtype)
    guesses = tuple(_as_dtype(C, dtype) for C in guesses)
    if dtype == torch.float64:
        u = _as_dtype(u, dtype)
    return h, s, u, guesses


def _host_results(source, state):
    """``state`` with its tensors as ndarrays when ``source`` keeps its arrays on the host."""
    if _arrays.is_host_module(source.np):
        for field in dataclasses.fields(state):
            value = getattr(state, field.name)
            if isinstance(value, torch.Tensor):
                setattr(state, field.name, _arrays.to_host(value))
    return state


def _sharded_inputs(basis, guesses):
    """``h``, ``s`` and the initial guesses (rank 0's everywhere) of a ``ShardedBasisSet`` on the device in the working
    dtype, and the callback that broadcasts rank 0's tensors (None on one process)."""
    from .sharded import ProcessContext

    ctx = basis.ctx
    h = _arrays.to_device(basis.h)
    s = _arrays.to_device(basis.s) if basis.s is not None else None
    collective = isinstance(ctx, ProcessContext) and ctx.world > 1

    def agree(*tensors):
        for t in tensors:
            ctx.dist.broadcast(torch.view_as_real(t) if t.is_complex() else t, src=0, group=ctx.group)

    guesses = [_arrays.to_device(C).contiguous() if C is not None else None for C in guesses]
    if collective:
        agree(*(C for C in guesses if C is not None))
    u_imag = any(_has_imag(basis.u.local(r)) for r in ctx.local_ranks)
    if collective:
        flag = torch.tensor([float(u_imag)], dtype=torch.float64, device=h.device)
        ctx.dist.all_reduce(flag, op=ctx.dist.ReduceOp.MAX, group=ctx.group)
        u_imag = bool(flag.item())
    dtype = _working_dtype(_has_imag(h), _has_imag(s), u_imag, *(_has_imag(C) for C in guesses))
    h, s = _as_dtype(h, dtype), _as_dtype(s, dtype)
    guesses = tuple(_as_dtype(C, dtype) for C in guesses)
    return h, s, guesses, agree if collective else None


def _sharded_fock(build, dtype):
    """The ``fock`` of the sharded solvers from ``build``, which maps the densities to the distributed Fock builds."""

    def fock(rho):
        # real working dtype: u has no imaginary part, so with real densities the imaginary parts are exactly zero
        return tuple(f.real.contiguous() if dtype == torch.float64 and f.is_complex() else f for f in build(rho))

    return fock


def _require_4d(basis):
    if getattr(basis, "u_repr", "4d") == "2d":
        raise ValueError("Hartree-Fock needs the 4-d two-body tensor; call set_u_repr('4d') on a sinc-DVR basis first")


def _require_plain_spatial_u(basis, ghf_entry):
    """Refuses a basis whose ``u`` is not the plain spatial 4-d tensor of UHF; a spin-doubled one is pointed to the
    GHF solver ``ghf_entry``."""
    if basis.includes_spin:
        raise ValueError("UHF needs the spatial two-body tensor; a spin-doubled basis is solved by "
                         f"hartree_fock.{ghf_entry} (GHF)")
    _require_4d(basis)
    if basis.anti_symmetrized_u:
        raise ValueError("UHF needs the plain spatial u, not an anti-symmetrised one")


def spin_orbital_order(n_alpha, n_beta, l):
    """The spin-orbital order of an unrestricted state: ``(orbital, spin)``, integer ndarrays of length ``2l`` with
    spin-orbital ``I`` the spatial orbital ``orbital[I]`` of spin ``spin[I]`` (0 = alpha).  The occupied spin-orbitals
    come first, then the virtual ones, each block ordered by (orbital index, spin) with alpha before beta.  The one
    order of ``spin_orbital_coefficients`` and ``general_orbital_system``."""
    occ = (n_alpha, n_beta)
    pairs = ([(j, s) for j in range(l) for s in (0, 1) if j < occ[s]]
             + [(j, s) for j in range(l) for s in (0, 1) if j >= occ[s]])
    table = np.array(pairs, dtype=np.int64).reshape(2 * l, 2)
    return table[:, 0].copy(), table[:, 1].copy()


def spin_orbital_coefficients(state):
    """The UHF state as ``(C, epsilon)`` of the spin-doubled basis: ``C`` is ``(2l, 2l)`` for
    ``GeneralOrbitalSystem(n_alpha + n_beta, basis).change_basis(C)``.  Rows follow ``add_spin`` (row ``2a + s``,
    ``s = 0`` the spin-up component); the columns follow ``spin_orbital_order``: the occupied spin-orbitals, then the
    virtual ones, each block ordered by (orbital index, spin) with alpha before beta.  A closed shell with
    ``C_alpha = C_beta`` gives ``kron(C, I_2)``.  Returns tensors or ndarrays, as the state holds."""
    Ca, Cb = state.C_alpha, state.C_beta
    xp = torch if isinstance(Ca, torch.Tensor) else np
    l = Ca.shape[0]
    orbital, spin_of = spin_orbital_order(state.n_alpha, state.n_beta, l)
    dtype = Ca.dtype if Ca.dtype == Cb.dtype else (torch.complex128 if xp is torch else np.complex128)
    kw = {"device": Ca.device} if xp is torch else {}
    C = xp.zeros((2 * l, 2 * l), dtype=dtype, **kw)
    eps = xp.zeros(2 * l, dtype=state.epsilon_alpha.dtype, **kw)
    for spin, (Cs, es) in enumerate(((Ca, state.epsilon_alpha), (Cb, state.epsilon_beta))):
        cols = [int(k) for k in np.flatnonzero(spin_of == spin)]
        orbs = [int(j) for j in orbital[cols]]
        C[spin::2, cols] = Cs[:, orbs].to(dtype) if xp is torch else Cs[:, orbs]
        eps[cols] = es[orbs]
    return C, eps


def general_orbital_system(state, basis):
    """``GeneralOrbitalSystem(state.n_alpha + state.n_beta, ...)`` in the spin-orbital basis of the UHF ``state`` of
    the spatial ``basis``, which is left unmodified: what ``GeneralOrbitalSystem(n, basis.copy_basis())
    .change_basis(spin_orbital_coefficients(state)[0])`` computes, without the spin-doubled ``(2l)^4`` input and its
    ``(2l)^4`` four-index transform.

    ``u`` is built from the spin blocks ``B_st = C_s^dagger C_t^dagger u C_s C_t`` of the spatial tensor
    (``ops.transform_two_body`` for the same-spin blocks, with the symmetry found by one exact test of ``u``, and
    ``ops.transform_two_body_mixed`` for alpha-beta, and for beta-alpha only when ``u`` lacks particle-exchange
    symmetry) and one assembly pass into the anti-symmetrised result (``ops.spin_orbital_two_body``), whose dtype
    follows ``cast_to_complex_on_spin_doubling`` as on the spin-doubling route.  The one-body elements, the grid
    orbitals and the spin operators take the code of ``change_to_general_orbital_basis`` and ``change_basis`` and are
    bit-identical to that route.  A host (numpy) basis gets ndarrays."""
    from .general_orbital_system import GeneralOrbitalSystem

    _require_plain_spatial_u(basis, "ground_state")
    l = basis.l
    if tuple(state.C_alpha.shape) != (l, l) or tuple(state.C_beta.shape) != (l, l):
        raise ValueError(f"the state has {tuple(state.C_alpha.shape)} coefficients, the basis l = {l}")
    C, _ = spin_orbital_coefficients(state)
    U = _spin_orbital_u(_arrays.to_device(basis.u), _arrays.to_device(state.C_alpha),
                        _arrays.to_device(state.C_beta), state.n_alpha, state.n_beta,
                        basis.cast_to_complex_on_spin_doubling)
    # the one-body side of GeneralOrbitalSystem(n, basis.copy_basis()).change_basis(C): the same calls without u
    gos_basis = basis._copy_basis(with_u=False)
    gos_basis._spin_double(a=[1, 0], b=[0, 1], anti_symmetrize=True, two_body=False)
    system = GeneralOrbitalSystem(state.n_alpha + state.n_beta, gos_basis)
    gos_basis._change_basis(C, None, two_body=False)
    gos_basis.u = _arrays.to_module(U, basis.np)
    system.set_system_size(system.n, gos_basis.l)
    return system


def general_orbital_system_sharded(state, basis, out_dtype=torch.complex128, into=None):
    """The spin-orbital system in the basis of the UHF ``state`` of the spatial ``ShardedBasisSet`` ``basis``, as a
    ``ShardedBasisSet`` of extent 2l (``includes_spin=True``, ``anti_symmetrized_u=True``): what
    ``ShardedBasisSet.from_spatial_planes(...)`` followed by ``change_basis(spin_orbital_coefficients(state)[0])``
    computes, without the spin-doubled input and its ``(2l)^4`` transform.

    ``u`` comes from the four spin blocks of the spatial tensor (``sharded.spin_orbital_two_body_sharded``): each rank
    receives only the spatial planes its own spin-orbital planes are assembled from.  The result carries the proof of
    its exact anti-symmetry and a spare buffer set (peer schedule), so a following ``change_basis`` takes the
    symmetry-aware path without testing.  ``h`` and ``s`` are ``transform_one_body(add_spin_one_body(., out_dtype), C)``
    with the ``C`` of ``spin_orbital_coefficients``, the calls of the spin-doubling route.  ``state`` may come from
    ``ground_state_unrestricted_sharded`` or from the single-GPU solver; rank 0's coefficients are used on every rank.
    ``out_dtype=torch.float64`` needs real spin blocks.  ``basis`` and its ``u`` are left untouched.

    Each call allocates the result and its spare set as new peer-visible buffers, which live until ``ctx.close()``;
    ``into`` (a ``ShardedTwoBody`` of extent 2l and dtype ``out_dtype``, e.g. the ``u`` of an earlier result that is
    no longer needed) receives ``u`` instead, see ``sharded.spin_orbital_two_body_sharded``."""
    from .sharded import ProcessContext, ShardedBasisSet, spin_orbital_two_body_sharded

    _require_plain_spatial_u(basis, "ground_state_sharded")
    ctx, l = basis.ctx, basis.u.n
    if tuple(state.C_alpha.shape) != (l, l) or tuple(state.C_beta.shape) != (l, l):
        raise ValueError(f"the state has {tuple(state.C_alpha.shape)} coefficients, the basis l = {l}")
    if out_dtype not in (torch.float64, torch.complex128):
        raise TypeError(f"out_dtype must be float64 or complex128, got {out_dtype}")
    fields = {name: _arrays.to_device(getattr(state, name)).contiguous()
              for name in ("C_alpha", "C_beta", "epsilon_alpha", "epsilon_beta")}
    if isinstance(ctx, ProcessContext) and ctx.world > 1:
        fields = {name: t.clone() for name, t in fields.items()}  # the caller's state keeps its own tensors
        for t in fields.values():
            ctx.dist.broadcast(torch.view_as_real(t) if t.is_complex() else t, src=0, group=ctx.group)
    state = dataclasses.replace(state, **fields)
    n_alpha, n_beta = _occupations(state.n_alpha, state.n_beta, l)
    u = spin_orbital_two_body_sharded(basis.u, state.C_alpha, state.C_beta, n_alpha, n_beta, out_dtype=out_dtype,
                                      into=into)
    # the one-body side of from_spatial_planes + change_basis, call for call
    C, _ = spin_orbital_coefficients(state)
    C, _ = ops.real_coefficients_if_exact(out_dtype == torch.complex128, C, None)
    h = ops.transform_one_body(ops.add_spin_one_body(_arrays.to_device(basis.h), out_dtype=out_dtype), C)
    s = None
    if basis.s is not None:
        s = ops.transform_one_body(ops.add_spin_one_body(_arrays.to_device(basis.s), out_dtype=out_dtype), C)
    return ShardedBasisSet(ctx, 2 * l, h, s, u, includes_spin=True, anti_symmetrized_u=True)


def _spin_orbital_u(u, Ca, Cb, n_alpha, n_beta, widen):
    """The anti-symmetrised ``(2l)^4`` tensor of ``general_orbital_system`` from the spin blocks of ``u``."""
    l = u.shape[0]
    flags = ops.proven_symmetry(u)
    if flags != ops.PARTICLE_EXCHANGE:
        flags = ops.two_body_symmetry(u)
    exchange = bool(flags & ops.PARTICLE_EXCHANGE)
    # the same-spin blocks keep both symmetries of u (one matrix for both kets and both bras); below
    # ops.SYMMETRY_MIN_N the plain steps are cheaper, as in transform_two_body
    same_spin = 0
    if ops.EXPLOIT_SYMMETRY and l >= ops.SYMMETRY_MIN_N:
        same_spin = (ops.ANTISYMMETRIC_LAST_PAIR if flags & ops.ANTISYMMETRIC_LAST_PAIR
                     else ops.PARTICLE_EXCHANGE if exchange else 0)
    b_aa = ops.transform_two_body(u, Ca, symmetry=same_spin)
    b_bb = ops.transform_two_body(u, Cb, symmetry=same_spin)
    b_ab = ops.transform_two_body_mixed(u, Ca, Cb)
    b_ba = None if exchange else ops.transform_two_body_mixed(u, Cb, Ca)
    out_dtype = torch.complex128 if (widen or b_aa.is_complex()) else torch.float64
    orbital, spin = spin_orbital_order(n_alpha, n_beta, l)
    U = ops.spin_orbital_two_body(b_aa, b_ab, b_ba, b_bb, orbital, spin, out_dtype=out_dtype)
    del b_aa, b_ab, b_ba, b_bb  # consumed: back to the allocator before the caller goes on
    return U


def _occupations(n_alpha, n_beta, l):
    if n_alpha is None or n_beta is None:
        raise ValueError("n_alpha and n_beta are required for a basis set")
    n_alpha, n_beta = int(n_alpha), int(n_beta)
    if not (0 <= n_alpha <= l and 0 <= n_beta <= l):
        raise ValueError(f"n_alpha = {n_alpha} and n_beta = {n_beta} must lie in [0, {l}]")
    return n_alpha, n_beta

def _working_dtype(*has_imag):
    return torch.complex128 if any(has_imag) else torch.float64


def _as_dtype(t, dtype):
    """``t`` in the working dtype.  float64 is chosen only when no operand has an imaginary part, so taking the real
    part of a complex operand then drops exact zeros only."""
    if t is None or t.dtype == dtype:
        return t
    return t.real.contiguous() if dtype == torch.float64 else t.to(dtype).contiguous()


def _has_imag(t):
    return t is not None and t.is_complex() and ops._has_imaginary_part(t)


def _scales(restricted, anti_symmetrized_u):
    if restricted:
        return 1.0, -0.5
    return (1.0, 0.0) if anti_symmetrized_u else (1.0, -1.0)


def _orthogonaliser(s, n, dtype, device):
    """Symmetric Loewdin ``X = S^(-1/2)`` (identity when ``s is None``)."""
    if s is None:
        return torch.eye(n, dtype=dtype, device=device)
    w, V = torch.linalg.eigh(s)
    w_min, w_max = float(w.min()), float(w.max())
    if not (w_max > 0 and w_min > SINGULAR_OVERLAP * w_max):
        raise ValueError(
            f"the overlap matrix is numerically singular or not positive definite "
            f"(eigenvalues in [{w_min:.3e}, {w_max:.3e}])"
        )
    return (V * w.rsqrt().to(dtype)) @ V.mH


def _density(C, n_occ, weight):
    C_o = C[:, :n_occ]
    rho = C_o @ C_o.mH
    return rho if weight == 1 else weight * rho


def _stacked(ts):
    """The matrices of all channels as one tensor for DIIS: one channel's matrix itself, without a copy, else the
    (channels, n, n) stack."""
    return ts[0] if len(ts) == 1 else torch.stack(ts)


def _diis(fs, errs):
    """Pulay extrapolation ``sum_i c_i F_i`` with ``sum_i c_i = 1`` minimising ``|sum_i c_i e_i|``."""
    k = len(fs)
    E = torch.stack([e.reshape(-1) for e in errs])
    B = torch.zeros((k + 1, k + 1), dtype=torch.float64, device=E.device)
    gram = (E.conj() @ E.T).real
    B[:k, :k] = gram / gram.diagonal().max()  # scaled to O(1): only the ratios matter, and they stay resolvable
    B[:k, k] = B[k, :k] = -1.0
    rhs = torch.zeros(k + 1, dtype=torch.float64, device=E.device)
    rhs[k] = -1.0
    c = torch.linalg.solve(B, rhs)[:k]
    return sum(ci.to(fs[0].dtype) * Fi for ci, Fi in zip(c, fs))


def _scf(h, s, fock, occupations, tol, max_iterations, C, e_nuc, agree):
    """The SCF iteration over spin channels, ``(n_occ, weight)`` each in ``occupations``: RHF is one channel of weight
    2, GHF one of weight 1, UHF two of weight 1.  ``fock`` maps the tuple of channel densities to the tuple of Fock
    matrices; ``C`` holds one initial guess per channel, or None for the core Hamiltonian (one ``eigh`` of ``h``,
    copied to every channel).  The energy is ``1/2 sum_s tr rho_s (h + F_s) + e_nuc``; DIIS extrapolates the
    stacked Fock matrices of all channels with one coefficient set from their stacked errors, and the largest error
    decides convergence.  ``h``, ``s``, ``C`` and what ``fock`` returns are all in the working dtype, the dtype of
    ``h``.  Returns ``(C, epsilon, rho, energy, converged, iterations)``, the first three a tuple per channel."""
    n = h.shape[0]
    dtype, device = h.dtype, h.device
    X = _orthogonaliser(s, n, dtype, device)
    S = _metric(s, h)

    def diagonalise(F):
        eps, Cp = torch.linalg.eigh(X.mH @ F @ X)
        C_new = X @ Cp
        if agree is not None:
            agree(C_new, eps)
        return C_new, eps

    if C[0] is None:
        C0, eps0 = diagonalise(h)
        C = (C0,) + tuple(C0.clone() for _ in occupations[1:])
        eps = (eps0,) + tuple(eps0.clone() for _ in occupations[1:])
    else:
        eps = (None,) * len(occupations)
    rho = tuple(_density(Cs, n_occ, weight) for Cs, (n_occ, weight) in zip(C, occupations))
    fs, errs = [], []
    converged, it, energy = False, 0, 0.0
    for it in range(1, max_iterations + 1):
        F = fock(rho)
        traces = [torch.sum(r.transpose(0, 1) * (h + f)) for r, f in zip(rho, F)]
        energy_t = 0.5 * sum(traces[1:], traces[0]).real + e_nuc
        err = _stacked([X.mH @ (f @ r @ S - S @ r @ f) @ X for f, r in zip(F, rho)])
        decision = torch.stack([energy_t.to(torch.float64), err.abs().max().to(torch.float64)])
        if agree is not None:
            agree(decision)
        energy, err_max = (float(x) for x in decision.tolist())
        converged = err_max <= tol
        if not converged:
            fs.append(_stacked(F))
            errs.append(err)
            if len(fs) > DIIS_VECTORS:
                fs.pop(0)
                errs.pop(0)
            if len(fs) > 1:
                F = _diis(fs, errs)
                F = (F,) if len(occupations) == 1 else tuple(F)
        C, eps = zip(*(diagonalise(f) for f in F))
        rho = tuple(_density(Cs, n_occ, weight) for Cs, (n_occ, weight) in zip(C, occupations))
        if converged:
            break
    if not converged:
        warnings.warn(f"Hartree-Fock did not converge in {max_iterations} iterations", RuntimeWarning, stacklevel=3)
    return C, eps, rho, energy, converged, it


def _metric(s, h):
    """The overlap matrix, the identity when ``s is None``, in the dtype of ``h``."""
    return s if s is not None else torch.eye(h.shape[0], dtype=h.dtype, device=h.device)


def _hf_state(result):
    """The ``HartreeFockState`` of a one-channel ``_scf`` result."""
    (C,), (eps,), (rho,), energy, converged, it = result
    return HartreeFockState(C=C, epsilon=eps, energy=energy, density_matrix=rho, converged=converged, iterations=it)


def _uhf_state(result, h, s, n_alpha, n_beta):
    """The ``UnrestrictedHartreeFockState`` of a two-channel ``_scf`` result, with ``<S^2>``."""
    (Ca, Cb), (ea, eb), (rho_a, rho_b), energy, converged, it = result
    overlap = Ca[:, :n_alpha].mH @ _metric(s, h) @ Cb[:, :n_beta]
    s_z = 0.5 * (n_alpha - n_beta)
    spin_squared = s_z * (s_z + 1) + n_beta - float((overlap.abs() ** 2).sum())
    return UnrestrictedHartreeFockState(
        C_alpha=Ca, C_beta=Cb, epsilon_alpha=ea, epsilon_beta=eb, density_alpha=rho_a, density_beta=rho_b,
        energy=energy, spin_squared=spin_squared, converged=converged, iterations=it, n_alpha=n_alpha, n_beta=n_beta,
    )
