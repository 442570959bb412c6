"""``BasisSet`` -- container of second-quantised matrix elements, B200 edition.

Mirror of the reference's ``quantum_systems/basis_set.py`` (class at :7, public surface listed in
SURVEY.md section 8b): same constructor, attributes, method names, argument meaning, assertion and
warning behaviour.  What differs is where the work happens:

* storage follows the injected array module ``np`` (``_arrays``): HBM-resident torch tensors for the
  default ``quantum_systems_b200.xp``, host ndarrays for ``numpy``;
* every O(n^4)/O(n^5) operation -- four-index transform, spin doubling, anti-symmetrisation -- is
  dispatched to hand-written sm_100a kernels through the C ABI (``ops``), never to numpy/torch math;
* spin doubling + anti-symmetrisation + complex cast are ONE fused pass instead of four;
* ``spin_2_tb`` is built lazily from three (n, n) factors, and a basis change transforms the factors
  (O(n^3)) instead of running a second O(n^5) transform on an n^4 tensor (exact; SURVEY.md section 8f).
"""

import copy
import types
import warnings

import torch

from . import _arrays, ops, streamed


def _is_complex(a):
    return a.is_complex() if isinstance(a, torch.Tensor) else a.dtype.kind == "c"


class BasisSet:
    """Container for ``h``, ``u``, ``s``, position/momentum, spin operators and grid orbitals.

    Parameters (reference basis_set.py:14-38)
    ----------
    l : int
        Number of basis functions.
    dim : int
        Dimensionality of the system.
    np : module
        Array module deciding where arrays are stored: ``quantum_systems_b200.xp`` (default, HBM)
        or ``numpy`` (host, staged through the GPU per call).
    includes_spin : bool
        The basis functions are spin-orbitals already.
    anti_symmetrized_u : bool
        ``u`` is anti-symmetrised already.
    """

    # names visited by change_module / cast_to_complex (reference basis_set.py:281-294, :304-317)
    _ARRAY_SLOTS = (
        "_h", "_s", "_u", "_spf", "_bra_spf", "_position", "_momentum",
        "_spin_x", "_spin_y", "_spin_z", "_spin_2", "_spin_2_tb",
    )

    def __init__(self, l, dim, np=None, includes_spin=False, anti_symmetrized_u=False):
        self.np = _arrays.default_module() if np is None else np
        self.l = l
        self.dim = dim
        self._grid = None
        for slot in self._ARRAY_SLOTS:
            setattr(self, slot, None)
        self._sigma_x = self._sigma_y = self._sigma_z = None
        # (S_x, S_y, S_z) in the CURRENT basis, from which spin_2_tb is materialised on demand
        self._spin_tb_factors = None
        self._spin_tb_anti_symmetrized = False
        self._nuclear_repulsion_energy = 0
        self.particle_charge = -1  # electrons, reference basis_set.py:65-66
        self._includes_spin = includes_spin
        self._anti_symmetrized_u = anti_symmetrized_u
        # Reference behaviour: spin doubling casts everything to complex128 (basis_set.py:632-634).
        # Set False to keep real matrix elements real (needed for the 205 GB FP64 tensor of config 5).
        self.cast_to_complex_on_spin_doubling = True

    # ------------------------------------------------------------------ storage helpers
    def _store(self, arr):
        return _arrays.store(arr, self.np)

    @staticmethod
    def check_axis_lengths(arr, length):
        return [length == axis for axis in arr.shape]

    def _checked(self, arr, needs_spin=False):
        if needs_spin:
            assert self.includes_spin
        if arr is None:
            return None
        arr = self._store(arr)
        assert all(self.check_axis_lengths(arr, self.l))
        return arr

    # ------------------------------------------------------------------ plain properties
    @property
    def includes_spin(self):
        return self._includes_spin

    @property
    def anti_symmetrized_u(self):
        return self._anti_symmetrized_u

    @property
    def grid(self):
        return self._grid

    @grid.setter
    def grid(self, grid):
        self._grid = grid

    @property
    def h(self):
        return self._h

    @h.setter
    def h(self, h):
        self._h = self._checked(h)

    @property
    def u(self):
        return self._u

    @u.setter
    def u(self, u):
        self._u = self._checked(u)

    @property
    def s(self):
        return self._s

    @s.setter
    def s(self, s):
        self._s = self._checked(s)

    def _checked_vector_operator(self, value):
        assert len(value) == self.dim
        value = self._store(value)
        for i in range(self.dim):
            assert all(self.check_axis_lengths(value[i], self.l))
        return value

    @property
    def position(self):
        return self._position

    @position.setter
    def position(self, position):
        self._position = self._checked_vector_operator(position)

    @property
    def dipole_moment(self):
        return self.particle_charge * self.position

    @property
    def momentum(self):
        return self._momentum

    @momentum.setter
    def momentum(self, momentum):
        self._momentum = self._checked_vector_operator(momentum)

    @property
    def spin_x(self):
        return self._spin_x

    @spin_x.setter
    def spin_x(self, spin_x):
        self._spin_x = self._checked(spin_x, needs_spin=True)

    @property
    def spin_y(self):
        return self._spin_y

    @spin_y.setter
    def spin_y(self, spin_y):
        self._spin_y = self._checked(spin_y, needs_spin=True)

    @property
    def spin_z(self):
        return self._spin_z

    @spin_z.setter
    def spin_z(self, spin_z):
        self._spin_z = self._checked(spin_z, needs_spin=True)

    @property
    def spin_2(self):
        return self._spin_2

    @spin_2.setter
    def spin_2(self, spin_2):
        self._spin_2 = self._checked(spin_2, needs_spin=True)

    @property
    def spin_2_tb(self):
        """Two-body part of S^2.  Materialised on first access from the (n, n) spin factors."""
        if self._spin_2_tb is None and self._spin_tb_factors is not None:
            sx, sy, sz = self._spin_tb_factors
            dense = ops.spin_squared_two_body(sx, sy, sz, anti_symmetrize=self._spin_tb_anti_symmetrized)
            self._spin_2_tb = _arrays.to_module(dense, self.np)
        return self._spin_2_tb

    @spin_2_tb.setter
    def spin_2_tb(self, spin_2_tb):
        self._spin_2_tb = self._checked(spin_2_tb, needs_spin=True)
        self._spin_tb_factors = None  # an explicit tensor overrides the factorised form

    @property
    def sigma_x(self):
        return self._sigma_x

    @sigma_x.setter
    def sigma_x(self, sigma_x):
        assert self.includes_spin
        self._sigma_x = sigma_x

    @property
    def sigma_y(self):
        return self._sigma_y

    @sigma_y.setter
    def sigma_y(self, sigma_y):
        assert self.includes_spin
        self._sigma_y = sigma_y

    @property
    def sigma_z(self):
        return self._sigma_z

    @sigma_z.setter
    def sigma_z(self, sigma_z):
        assert self.includes_spin
        self._sigma_z = sigma_z

    def _checked_spf(self, spf):
        if spf is None:
            return None
        spf = self._store(spf)
        assert spf.shape[0] == self.l
        assert len(tuple(spf.shape[1:])) == self.dim
        return spf

    @property
    def spf(self):
        return self._spf

    @spf.setter
    def spf(self, spf):
        self._spf = self._checked_spf(spf)

    @property
    def bra_spf(self):
        if self._bra_spf is None and self._spf is not None:
            # Hermitian basis: the dual functions are the complex conjugates (basis_set.py:246-251)
            self._bra_spf = self._store(_conj(self._spf))
        return self._bra_spf

    @bra_spf.setter
    def bra_spf(self, bra_spf):
        self._bra_spf = self._checked_spf(bra_spf)

    @property
    def nuclear_repulsion_energy(self):
        return self._nuclear_repulsion_energy

    @nuclear_repulsion_energy.setter
    def nuclear_repulsion_energy(self, nuclear_repulsion_energy):
        self._nuclear_repulsion_energy = nuclear_repulsion_energy

    # ------------------------------------------------------------------ the `np` hook
    @staticmethod
    def change_arr_module(arr, np):
        return _arrays.store(arr, np) if arr is not None else None

    def change_module(self, np):
        """Move every stored array to the storage of the new module (basis_set.py:272-296)."""
        self.bra_spf  # noqa: B018 - materialise the default dual functions first, as the reference does
        self.np = np
        for slot in self._ARRAY_SLOTS:
            setattr(self, slot, self.change_arr_module(getattr(self, slot), self.np))

    def cast_to_complex(self):
        """Cast every stored array to complex128 (basis_set.py:298-319)."""
        self.bra_spf  # noqa: B018
        for slot in self._ARRAY_SLOTS:
            arr = getattr(self, slot)
            if arr is not None and not _is_complex(arr):
                setattr(self, slot, _astype_complex(arr))

    # ------------------------------------------------------------------ basis changes
    @staticmethod
    def transform_spf(spf, C, np):
        """``tensordot(C, spf, axes=(0, 0))`` (basis_set.py:321-323) as one quarter GEMM."""
        return _arrays.to_module(ops.transform_functions(_arrays.to_device(spf), _arrays.to_device(C), False), np)

    @staticmethod
    def transform_bra_spf(bra_spf, C_tilde, np):
        """``tensordot(C_tilde, bra_spf, axes=(1, 0))`` (basis_set.py:325-327)."""
        return _arrays.to_module(
            ops.transform_functions(_arrays.to_device(bra_spf), _arrays.to_device(C_tilde), True), np
        )

    @staticmethod
    def transform_one_body_elements(h, C, np, C_tilde=None):
        """``C_tilde (h C)`` with ``C_tilde = C^dagger`` by default (basis_set.py:329-334)."""
        out = ops.transform_one_body(_arrays.to_device(h), _arrays.to_device(C), _arrays.to_device(C_tilde))
        return _arrays.to_module(out, np)

    @staticmethod
    def transform_two_body_elements(u, C, np, C_tilde=None):
        """Four-index transform (basis_set.py:336-350) on the FP64 tensor cores.  A large host-resident ``u``
        (``np = numpy``) takes the streamed schedule that hides the PCIe copies behind the kernels."""
        C_dev, C_tilde_dev = _arrays.to_device(C), _arrays.to_device(C_tilde)
        if _arrays.is_host_module(np) and streamed.applicable(u, C_dev):
            return streamed.transform_two_body(u, C_dev, C_tilde_dev)
        out = ops.transform_two_body(_arrays.to_device(u), C_dev, C_tilde_dev)
        return _arrays.to_module(out, np)

    def get_transformed_h(self, C):
        return self.transform_one_body_elements(self.h, C, np=self.np)

    def get_transformed_u(self, C):
        return self.transform_two_body_elements(self.u, C, np=self.np)

    def _change_basis_one_body_elements(self, C, C_tilde):
        self.h = self.transform_one_body_elements(self.h, C, np=self.np, C_tilde=C_tilde)
        if self.s is not None:
            self.s = self.transform_one_body_elements(self.s, C, np=self.np, C_tilde=C_tilde)
        # spin_x/y/z/spin_2 are deliberately NOT updated: the reference computes the transformed
        # matrices into a loop-local and drops them (basis_set.py:368-372); a drop-in keeps that.

    def _change_basis_two_body_elements(self, C, C_tilde):
        self.u = self.transform_two_body_elements(self.u, C, np=self.np, C_tilde=C_tilde)
        self._change_basis_spin_2_tb(C, C_tilde)

    def _change_basis_spin_2_tb(self, C, C_tilde):
        if self._spin_tb_factors is not None:
            # transform of sum_i S_i (x) S_i == sum_i (C~ S_i C) (x) (C~ S_i C): O(n^3), exact
            self._spin_tb_factors = tuple(
                ops.transform_one_body(f, _arrays.to_device(C), _arrays.to_device(C_tilde))
                for f in self._spin_tb_factors
            )
            self._spin_2_tb = None
        elif self._spin_2_tb is not None:
            self.spin_2_tb = self.transform_two_body_elements(self._spin_2_tb, C, np=self.np, C_tilde=C_tilde)

    def _change_basis_vector_operator(self, value, C, C_tilde):
        parts = [
            _arrays.to_device(self.transform_one_body_elements(value[i], C, np=self.np, C_tilde=C_tilde))
            for i in range(value.shape[0])
        ]
        return torch.stack(parts)

    def _change_basis_position_elements(self, C, C_tilde):
        self.position = self._change_basis_vector_operator(self.position, C, C_tilde)

    def _change_basis_momentum_elements(self, C, C_tilde):
        self.momentum = self._change_basis_vector_operator(self.momentum, C, C_tilde)

    def _change_basis_spf(self, C, C_tilde):
        self.bra_spf = self.transform_bra_spf(self.bra_spf, C_tilde, self.np)
        self.spf = self.transform_spf(self.spf, C, self.np)

    def change_basis(self, C, C_tilde=None):
        r"""Change basis with ket coefficients ``C`` (shape ``(l_old, l_new)``) and bra coefficients
        ``C_tilde`` (shape ``(l_new, l_old)``, default ``C^dagger``); rectangular matrices change the
        number of basis functions.  Same contract as the reference's ``BasisSet.change_basis``
        (basis_set.py:413-464): h, s, u, spin_2_tb, position, momentum, spf and bra_spf are replaced
        by new arrays; inputs are never modified in place.
        """
        self._change_basis(C, C_tilde, two_body=True)

    def _change_basis(self, C, C_tilde, two_body):
        """``change_basis``; ``two_body=False`` leaves ``u`` alone (the caller stores the transformed one)."""
        C_dev = _arrays.to_device(C)
        self.l = C_dev.shape[1]
        if C_tilde is None:
            C_tilde = torch.conj(C_dev).transpose(0, 1).resolve_conj().contiguous()
        C_tilde_dev = _arrays.to_device(C_tilde)

        self._change_basis_one_body_elements(C_dev, C_tilde_dev)
        if two_body:
            self._change_basis_two_body_elements(C_dev, C_tilde_dev)
        else:
            self._change_basis_spin_2_tb(C_dev, C_tilde_dev)
        if self.position is not None:
            self._change_basis_position_elements(C_dev, C_tilde_dev)
        if self.momentum is not None:
            self._change_basis_momentum_elements(C_dev, C_tilde_dev)
        if self.spf is not None:
            self._change_basis_spf(C_dev, C_tilde_dev)

    def compute_particle_density(self, rho_qp, C=None, C_tilde=None):
        r"""``rho(r) = sum_pq bra_p(r) rho_qp[q, p] ket_q(r)`` (basis_set.py:466-509,
        system_helper.py:14-27); optionally in a basis changed by ``C`` / ``C_tilde``."""
        assert self._spf is not None, "Set up single-particle functions prior to calling this function"
        ket, bra = self.spf, self.bra_spf
        if C is not None:
            ket = self.transform_spf(ket, C, self.np)
            C_tilde = C_tilde if C_tilde is not None else _conj(_arrays.to_device(C)).transpose(0, 1).contiguous()
            bra = self.transform_bra_spf(bra, C_tilde, self.np)
        ket_d, bra_d, rho_d = _arrays.to_device(ket), _arrays.to_device(bra), _arrays.to_device(rho_qp)
        assert bra_d.shape == ket_d.shape
        dt = torch.promote_types(torch.promote_types(ket_d.dtype, bra_d.dtype), rho_d.dtype)
        rho = torch.einsum("p...,qp,q...->...", bra_d.to(dt), rho_d.to(dt), ket_d.to(dt))
        return _arrays.to_module(rho, self.np)

    # ------------------------------------------------------------------ spin doubling / anti-symmetry
    def anti_symmetrize_two_body_elements(self):
        r"""``u_pqrs <- u_pqrs - u_pqsr`` once (idempotent through the flag), also for ``spin_2_tb``
        (basis_set.py:511-528)."""
        if not self._anti_symmetrized_u:
            self.u = self.anti_symmetrize_u(self.u)
            if self._spin_tb_factors is not None:
                self._spin_tb_anti_symmetrized = True
                self._spin_2_tb = None
            elif self._spin_2_tb is not None:
                self.spin_2_tb = self.anti_symmetrize_u(self._spin_2_tb)
            self._anti_symmetrized_u = True

    def change_to_general_orbital_basis(self, a=[1, 0], b=[0, 1], anti_symmetrize=True):
        r"""Spin-double the basis in place: every spatial orbital becomes two spin-orbitals
        (spin index fastest).  Same contract as basis_set.py:530-636: returns ``self``; on a basis that
        is spin-doubled already it warns and returns ``None``.

        ``u`` goes through ONE fused kernel (kron with the spin deltas + anti-symmetrisation + cast to
        complex128) instead of the reference's kron / subtract-transpose / astype passes.
        """
        if self._includes_spin:
            warnings.warn("The basis has already been spin-doubled. Avoiding a second doubling.")
            return
        return self._spin_double(a, b, anti_symmetrize, two_body=True)

    def _spin_double(self, a, b, anti_symmetrize, two_body):
        """``change_to_general_orbital_basis``; ``two_body=False`` leaves ``u`` alone and records it as
        anti-symmetrised when ``anti_symmetrize`` is set (the caller stores that tensor)."""
        self._includes_spin = True
        self.l = 2 * self.l
        widen = self.cast_to_complex_on_spin_doubling

        overlap = _arrays.to_device(self.s)
        self.h = self.add_spin_one_body(self.h, np=self.np)
        self.s = self.add_spin_one_body(self.s, np=self.np)

        # A subclass that overrides the static hooks (reference dispatch through `self`, basis_set.py:523, :576;
        # e.g. the 2-D sinc-DVR storage) gets its own add_spin_two_body / anti_symmetrize_u, un-fused.  Without the
        # u step the hooks do not run and the anti-symmetrisation is recorded as fused.
        hooks_overridden = two_body and (
            type(self).add_spin_two_body is not BasisSet.add_spin_two_body
            or type(self).anti_symmetrize_u is not BasisSet.anti_symmetrize_u
        )
        fuse_as = bool(anti_symmetrize) and not self._anti_symmetrized_u and not hooks_overridden
        if hooks_overridden:
            self.u = self.add_spin_two_body(self._u, np=self.np)
        elif two_body:
            u_dev = _arrays.to_device(self._u)
            out_dtype = torch.complex128 if (widen or u_dev.is_complex()) else torch.float64
            self.u = _arrays.to_module(
                ops.add_spin_two_body(u_dev, anti_symmetrize=fuse_as, out_dtype=out_dtype), self.np
            )

        if getattr(self, "u_repr", "4d") != "2d":
            np_host = _host_numpy()
            self.a = np_host.array(a).astype(np_host.complex128).reshape(-1, 1)
            self.b = np_host.array(b).astype(np_host.complex128).reshape(-1, 1)
            # spin basis must be orthonormal (basis_set.py:586-589)
            assert abs(np_host.dot(self.a.conj().T, self.a) - 1) < 1e-12
            assert abs(np_host.dot(self.b.conj().T, self.b) - 1) < 1e-12
            assert abs(np_host.dot(self.a.conj().T, self.b)) < 1e-12

            self.sigma_x, self.sigma_y, self.sigma_z = self.setup_pauli_matrices(self.a, self.b, np_host)
            half_overlap = 0.5 * overlap.to(torch.complex128)
            spins = [
                torch.kron(half_overlap, _arrays.to_device(sigma).contiguous())
                for sigma in (self.sigma_x, self.sigma_y, self.sigma_z)
            ]
            self.spin_x, self.spin_y, self.spin_z = spins
            s_dev = _arrays.to_device(self.s)
            spin_2 = torch.zeros_like(spins[0])
            for s_i in spins:
                spin_2 += ops.transform_one_body(s_dev, s_i, s_i)  # S_i s S_i, basis_set.py:746
            self.spin_2 = spin_2
            self._spin_tb_factors = tuple(spins)
            self._spin_tb_anti_symmetrized = False
            self._spin_2_tb = None

        if anti_symmetrize:
            if fuse_as:
                # u was anti-symmetrised by the fused kernel above; spin_2_tb follows lazily
                if self._spin_tb_factors is not None:
                    self._spin_tb_anti_symmetrized = True
                elif self._spin_2_tb is not None:
                    self.spin_2_tb = self.anti_symmetrize_u(self._spin_2_tb)
                self._anti_symmetrized_u = True
            else:
                self.anti_symmetrize_two_body_elements()

        if self.position is not None:
            self.position = torch.stack(
                [_arrays.to_device(self.add_spin_one_body(self.position[i], np=self.np)) for i in range(len(self.position))]
            )
        if self.momentum is not None:
            self.momentum = torch.stack(
                [_arrays.to_device(self.add_spin_one_body(self.momentum[i], np=self.np)) for i in range(len(self.momentum))]
            )
        if self.spf is not None:
            had_bra = self._bra_spf is not None
            bra = self._bra_spf
            self._bra_spf = None
            self.spf = self.add_spin_spf(self.spf, self.np)
            if had_bra:
                self.bra_spf = self.add_spin_bra_spf(bra, self.np)

        if widen:
            self.cast_to_complex()
        return self

    @staticmethod
    def setup_pauli_matrices(a, b, np):
        r"""Pauli matrices ``(sigma_i)_{rho gamma} = <rho| sigma_i |gamma>`` in the spin basis
        ``{a, b}`` (column vectors), in the order x, y, z (basis_set.py:638-697).  2x2 host work."""
        np_host = _host_numpy()
        a = np_host.asarray(_arrays.to_host(a) if isinstance(a, torch.Tensor) else a).reshape(-1, 1)
        b = np_host.asarray(_arrays.to_host(b) if isinstance(b, torch.Tensor) else b).reshape(-1, 1)
        cartesian = (
            np_host.array([[0, 1], [1, 0]], dtype=np_host.complex128),
            np_host.array([[0, -1j], [1j, 0]], dtype=np_host.complex128),
            np_host.array([[1, 0], [0, -1]], dtype=np_host.complex128),
        )
        kets = (a, b)
        result = []
        for pauli in cartesian:
            m = np_host.zeros((2, 2), dtype=np_host.complex128)
            for i, bra in enumerate(kets):
                for j, ket in enumerate(kets):
                    m[i, j] = (bra.conj().T @ pauli @ ket)[0, 0]
            result.append(m)
        return tuple(result)

    @staticmethod
    def setup_spin_squared_operator(spin_x, spin_y, spin_z, overlap, np):
        r"""One-body ``sum_i S_i s S_i`` and two-body ``sum_i S_i (x) S_i`` parts of ``S^2``
        (basis_set.py:699-749).  Returns dense ``(l, l)`` and ``(l, l, l, l)`` arrays."""
        sx, sy, sz = (_arrays.to_device(m, torch.complex128) for m in (spin_x, spin_y, spin_z))
        s_dev = _arrays.to_device(overlap)
        spin_2 = torch.zeros_like(sx)
        for s_i in (sx, sy, sz):
            spin_2 += ops.transform_one_body(s_dev, s_i, s_i)
        spin_2_tb = ops.spin_squared_two_body(sx, sy, sz, anti_symmetrize=False)
        return _arrays.to_module(spin_2, np), _arrays.to_module(spin_2_tb, np)

    @staticmethod
    def add_spin_spf(spf, np):
        """Row interleave ``new[2p] = new[2p+1] = spf[p]`` (basis_set.py:751-759); data movement only."""
        dev = _arrays.to_device(spf)
        return _arrays.to_module(torch.repeat_interleave(dev, 2, dim=0), np)

    @staticmethod
    def add_spin_bra_spf(bra_spf, np):
        if bra_spf is None:
            return None
        return BasisSet.add_spin_spf(bra_spf, np)

    @staticmethod
    def add_spin_one_body(h, np):
        """``kron(h, I_2)`` (basis_set.py:768-770)."""
        return _arrays.to_module(ops.add_spin_one_body(_arrays.to_device(h)), np)

    @staticmethod
    def add_spin_two_body(_u, np):
        """``kron(u, delta_pr delta_qs)`` (basis_set.py:772-774)."""
        return _arrays.to_module(ops.add_spin_two_body(_arrays.to_device(_u)), np)

    @staticmethod
    def anti_symmetrize_u(_u):
        """``u - u.transpose(0, 1, 3, 2)`` as a new array of the input's kind (basis_set.py:776-778)."""
        out = ops.anti_symmetrize(_arrays.to_device(_u))
        return out if isinstance(_u, torch.Tensor) else _arrays.to_host(out)

    # ------------------------------------------------------------------ copies
    def copy_basis(self):
        """Deep copy (basis_set.py:784-805).  Array modules are shared, never copied."""
        return self._copy_basis(with_u=True)

    def _copy_basis(self, with_u):
        """``copy_basis``; ``with_u=False`` gives a copy whose ``u`` is None instead of a copy of ``u``."""
        memo = {}
        if not with_u and self._u is not None:
            memo[id(self._u)] = None  # deepcopy takes a memo entry as the copy of that object
        for value in vars(self).values():
            if isinstance(value, types.ModuleType):
                memo[id(value)] = value
        memo[id(self.np)] = self.np
        potential = getattr(self, "potential", None)
        if potential is not None:
            for value in vars(potential).values():
                if isinstance(value, types.ModuleType):
                    memo[id(value)] = value
        new_basis = copy.deepcopy(self, memo)
        assert new_basis.np is self.np
        return new_basis


def _host_numpy():
    import numpy

    return numpy


def _conj(a):
    if isinstance(a, torch.Tensor):
        return torch.conj(a).resolve_conj()
    return a.conj()


def _astype_complex(a):
    if isinstance(a, torch.Tensor):
        return a.to(torch.complex128)
    return a.astype("complex128")
