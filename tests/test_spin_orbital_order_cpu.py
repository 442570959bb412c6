"""The spin-orbital order of an unrestricted state, on the host: ``hartree_fock.spin_orbital_order`` is the column
order of ``spin_orbital_coefficients``.  And the spin-orbital assembly kernel compiles for sm_100a without spills."""

import os
import re
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def numpy_state(n_alpha, n_beta, l, seed=0):
    from quantum_systems_b200.hartree_fock import UnrestrictedHartreeFockState

    rng = np.random.default_rng(seed)
    Ca, Cb = rng.uniform(1.0, 2.0, (l, l)), rng.uniform(-2.0, -1.0, (l, l))  # no zero element, signs tell spins
    ea, eb = np.sort(rng.standard_normal(l)), np.sort(rng.standard_normal(l))
    return UnrestrictedHartreeFockState(
        C_alpha=Ca, C_beta=Cb, epsilon_alpha=ea, epsilon_beta=eb, density_alpha=None, density_beta=None,
        energy=0.0, spin_squared=0.0, converged=True, iterations=0, n_alpha=n_alpha, n_beta=n_beta,
    )


@pytest.mark.parametrize("n_alpha, n_beta, l", [
    (1, 1, 1), (1, 0, 1), (0, 0, 3), (2, 1, 5), (3, 0, 4), (4, 4, 4), (1, 3, 6), (0, 2, 3), (11, 10, 23), (5, 5, 9),
])
def test_order_is_the_column_order_of_the_coefficients(n_alpha, n_beta, l):
    from quantum_systems_b200 import hartree_fock

    state = numpy_state(n_alpha, n_beta, l)
    orbital, spin = hartree_fock.spin_orbital_order(n_alpha, n_beta, l)
    assert orbital.shape == spin.shape == (2 * l,)
    assert sorted(zip(orbital.tolist(), spin.tolist())) == [(j, s) for j in range(l) for s in (0, 1)]
    C, eps = hartree_fock.spin_orbital_coefficients(state)
    assert isinstance(C, np.ndarray) and C.shape == (2 * l, 2 * l)
    for I in range(2 * l):
        o, s = int(orbital[I]), int(spin[I])
        col = C[:, I]
        # the column lives on the rows of its spin only and is that spin's coefficient column o
        assert not col[1 - s::2].any()
        assert np.array_equal(col[s::2], (state.C_alpha, state.C_beta)[s][:, o])
        assert eps[I] == (state.epsilon_alpha, state.epsilon_beta)[s][o]
    # the occupied spin-orbitals come first
    occupied = [int(orbital[I]) < (n_alpha, n_beta)[int(spin[I])] for I in range(2 * l)]
    assert occupied == [True] * (n_alpha + n_beta) + [False] * (2 * l - n_alpha - n_beta)


def test_closed_shell_order_is_spin_fastest():
    from quantum_systems_b200 import hartree_fock

    orbital, spin = hartree_fock.spin_orbital_order(3, 3, 7)
    assert orbital.tolist() == np.repeat(np.arange(7), 2).tolist()
    assert spin.tolist() == [0, 1] * 7


def test_assembly_kernel_has_no_spills(tmp_path):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc is not installed")
    from quantum_systems_b200.build import NVCC_FLAGS

    src = os.path.join(ROOT, "quantum_systems_b200", "csrc", "spin_antisym.cu")
    proc = subprocess.run([nvcc, *NVCC_FLAGS, "-Xptxas", "-v", "-c", "-o", str(tmp_path / "spin.o"), src],
                          capture_output=True, text=True)
    assert proc.returncode == 0, proc.stderr[-3000:]
    assert "arch=compute_100a,code=sm_100a" in NVCC_FLAGS
    # ptxas reports each entry, then its properties: pair every spin_orbital_kernel entry with its spill line
    reports = re.findall(r"Compiling entry function '(\w+)' for 'sm_100a'.*?Function properties for \1\n\s*(.*?)\n",
                         proc.stderr, flags=re.S)
    spills = {name: line for name, line in reports if "spin_orbital_kernel" in name}
    assert len(spills) == 3, proc.stderr[-3000:]  # F64 -> F64, F64 -> C128, C128 -> C128
    for name, line in spills.items():
        assert "0 bytes spill stores, 0 bytes spill loads" in line, f"{name}: {line}"
