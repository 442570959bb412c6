"""quantum_systems_b200 -- B200-native two-body integral pipeline behind the HyQD/quantum-systems API.

Drop-in for the hot path of ``quantum_systems`` (reference ``quantum_systems/__init__.py:1-21``):
``BasisSet``, ``QuantumSystem``, ``GeneralOrbitalSystem``, ``SpatialOrbitalSystem``, ``ODQD`` and
``RandomBasisSet`` keep the reference's names, signatures and error behaviour; the O(n^4)/O(n^5) work
(``change_basis``, ``add_spin`` + ``anti_symmetrize_u``, ``construct_fock_matrix``, the ODQD grid
Coulomb build) runs in hand-written sm_100a CUDA kernels behind a C ABI (``include/qsb200.h``).
"""

__version__ = "0.1.0"

from . import xp  # noqa: F401  (the device array module for the `np=` hook)
from .basis_set import BasisSet
from .system import QuantumSystem
from .general_orbital_system import GeneralOrbitalSystem
from .spatial_orbital_system import SpatialOrbitalSystem
from .random_basis import RandomBasisSet
from .odqd import ODHO, ODQD
from .sinc_dvr import ODSincDVR
from . import time_evolution_operators  # noqa: F401
from . import hartree_fock  # noqa: F401
from . import two_dim_ho  # noqa: F401
from .two_dim_ho import (
    get_coulomb_elements,
    TwoDimensionalHarmonicOscillator,
    TwoDimensionalDoubleWell,
    TwoDimSmoothDoubleWell,
    TwoDimHarmonicOscB,
)

__all__ = [
    "BasisSet",
    "QuantumSystem",
    "GeneralOrbitalSystem",
    "SpatialOrbitalSystem",
    "RandomBasisSet",
    "ODQD",
    "ODHO",
    "ODSincDVR",
    "TwoDimensionalHarmonicOscillator",
    "TwoDimensionalDoubleWell",
    "TwoDimSmoothDoubleWell",
    "TwoDimHarmonicOscB",
    "get_coulomb_elements",
    "hartree_fock",
    "xp",
]
