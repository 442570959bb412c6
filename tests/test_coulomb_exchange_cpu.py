"""The large-offset case of tests/test_gpu_coulomb_exchange.py checked without a GPU, as tests/test_large_offsets_cpu.py
checks the cases of tests/large_offsets.py: n = 216 is the smallest extent whose u passes 2^31 elements, and the
memory plan covers u, the workspace the library asks for and the checks' scratch, within the per-case budget."""

import pytest

pytest.importorskip("torch")

import large_offsets as LO  # noqa: E402
from test_gpu_coulomb_exchange import LARGE, LARGE_K  # noqa: E402


@pytest.fixture(scope="module")
def library():
    from quantum_systems_b200 import _native
    from quantum_systems_b200.build import build

    build()
    return _native.load()


def test_the_extent_is_the_smallest_that_crosses_the_boundary():
    n = LARGE.extent
    assert LARGE.offset(n) >= LARGE.boundary > LARGE.offset(n - 1)


def test_the_plan_covers_u_and_the_workspace(library):
    n = LARGE.extent
    ws = LO._bytes("qs_coulomb_exchange_batch_workspace_bytes", n, LARGE_K, 0, n, 0, 0)
    assert ws > 0
    assert LARGE.nbytes(n) >= 8 * n**4 + ws + LO.SCRATCH
    assert LARGE.nbytes(n) <= LO.BUDGET
