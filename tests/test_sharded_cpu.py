"""Host-side logic of the sharded schedule on a CPU-only box: block partition, stride plans and both
exchange layouts, checked against the numpy oracle.  The arithmetic of the quarter steps is supplied
by tests/_numpy_engine.py (test infrastructure); the schedule under test is the product's
``quantum_systems_b200.sharded``.  The multi-process test runs world_size 2 under gloo."""

import os
import socket
import sys

import numpy as np
import pytest
import torch

from oracle import qs_oracle as oracle

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from _numpy_engine import NumpyEngine  # noqa: E402


def rand(rng, shape, complex_):
    x = rng.standard_normal(shape)
    return x + 1j * rng.standard_normal(shape) if complex_ else x


def test_scatter_deal_rule_is_a_permutation():
    """The numpy stand-in and the library agree on the dealing multiplier, and it permutes the columns."""
    import ctypes
    from math import gcd

    from quantum_systems_b200 import _native
    from quantum_systems_b200.build import build

    build()
    lib = _native.load()
    for W in list(range(1, 70)) + [128, 148, 192, 256, 400, 401]:
        deal = ctypes.c_int64(0)
        assert lib.qs_scatter_deal(W, ctypes.byref(deal)) == 0
        assert deal.value == NumpyEngine().scatter_deal(W)
        assert 1 <= deal.value < max(W, 2) and gcd(deal.value, W) == 1
        assert sorted((j * deal.value) % W for j in range(W)) == list(range(W))
        if W >= 64:  # any 32 consecutive logical columns touch every eighth of the range
            for start in (0, W // 3):
                hit = {((j * deal.value) % W) * 8 // W for j in range(start, start + 32)}
                assert hit == set(range(8))


def test_block_partition():
    from quantum_systems_b200.sharded import block_partition

    assert block_partition(400, 8) == (50, [0, 50, 100, 150, 200, 250, 300, 350, 400])
    assert block_partition(10, 4) == (3, [0, 3, 6, 9, 10])
    assert block_partition(3, 4) == (1, [0, 1, 2, 3, 3])  # trailing rank empty
    for n in range(1, 40):
        for w in range(1, 9):
            block, off = block_partition(n, w)
            assert off[0] == 0 and off[-1] == n and all(0 <= b - a <= block for a, b in zip(off, off[1:]))


@pytest.mark.parametrize("world", [1, 2, 3, 4])
@pytest.mark.parametrize("n,m,u_complex,c_complex,biorth", [
    (8, 8, False, False, False),
    (9, 9, False, False, False),   # odd real extent: padded pitch
    (7, 10, False, False, False),  # rectangular, grows
    (10, 6, True, True, True),     # rectangular, shrinks, bi-orthogonal complex
    (6, 6, False, True, False),    # real u, complex C
    (8, 8, True, False, False),    # complex u, real C
    (12, 17, False, False, False),  # >= 16 new columns: the scattering steps deal their columns (qs_scatter_deal)
    (16, 16, True, True, True),
])
def test_emulated_peer_schedule_matches_oracle(world, n, m, u_complex, c_complex, biorth):
    from quantum_systems_b200 import sharded

    rng = np.random.default_rng(100 * n + m + world)
    u = rand(rng, (n,) * 4, u_complex)
    C = rand(rng, (n, m), c_complex)
    Ct = rand(rng, (m, n), c_complex) if biorth else None
    ctx = sharded.EmulatedContext(world, engine=NumpyEngine())
    basis = sharded.ShardedBasisSet.from_global(ctx, np.eye(n), np.eye(n), u)
    out = sharded.transform_two_body_sharded(basis.u, torch.from_numpy(C), None if Ct is None else torch.from_numpy(Ct))
    expected = oracle.transform_two_body_elements(u, C, Ct)
    got = out.gather().numpy()
    assert got.shape == expected.shape and got.dtype == expected.dtype
    np.testing.assert_allclose(got, expected, rtol=1e-12, atol=1e-12 * np.abs(expected).max())
    # result is sharded on the leading index again, with the same block rule
    assert [out.planes(r) for r in range(world)] == list(zip(out.offsets[:-1], out.offsets[1:]))
    if m == n and not (u_complex != (c_complex or u_complex)):
        # second transform recycles the first tensor's buffers (ping-pong) and must still be right
        out2 = sharded.transform_two_body_sharded(out, torch.from_numpy(C), None if Ct is None else torch.from_numpy(Ct))
        expected2 = oracle.transform_two_body_elements(expected, C, Ct)
        np.testing.assert_allclose(out2.gather().numpy(), expected2, rtol=1e-11, atol=1e-11 * np.abs(expected2).max())


@pytest.mark.parametrize("world", [1, 2, 3, 4])
@pytest.mark.parametrize("n,m,complex_", [(8, 8, False), (9, 9, False), (10, 7, True), (6, 11, False), (12, 12, True)])
def test_emulated_symmetry_aware_schedule_matches_oracle(world, n, m, complex_):
    """Anti-symmetric u through the pair schedule (forced: the automatic switch needs n >= 48): cyclic r, source-major
    T2 read through block tables -- one launch when every source holds equally many planes, one per source
    otherwise -- packed pairs, scattering store through the pair table, mirror fill."""
    from quantum_systems_b200 import sharded

    rng = np.random.default_rng(10 * n + m + world)
    u = rand(rng, (n,) * 4, complex_)
    u = u - u.transpose(0, 1, 3, 2)
    C = rand(rng, (n, m), complex_)
    ctx = sharded.EmulatedContext(world, engine=NumpyEngine())
    basis = sharded.ShardedBasisSet.from_global(ctx, np.eye(n), np.eye(n), u)
    out = sharded.transform_two_body_sharded(basis.u, torch.from_numpy(C), symmetry=1)
    expected = oracle.transform_two_body_elements(u, C)
    got = out.gather().numpy()
    np.testing.assert_allclose(got, expected, rtol=1e-12, atol=1e-12 * np.abs(expected).max())
    np.testing.assert_array_equal(got, -got.transpose(0, 1, 3, 2))
    assert out.proven_antisymmetric
    if m == n:  # the chain goes on without a new test of the symmetry
        out2 = sharded.transform_two_body_sharded(out, torch.from_numpy(C), symmetry=1)
        expected2 = oracle.transform_two_body_elements(expected, C)
        np.testing.assert_allclose(out2.gather().numpy(), expected2, rtol=1e-11, atol=1e-11 * np.abs(expected2).max())


@pytest.mark.parametrize("world,n", [(3, 72), (2, 70)])
def test_symmetry_aware_schedule_with_many_tiles(world, n):
    """Large enough for several row AND column tiles per launch: the first exchange sends only the tiles that hold a
    wanted pair (the stand-in writes exactly the tiles the library's planner lists; everything else stays NaN), and
    steps 3 and 4 must never touch what was not sent."""
    from quantum_systems_b200 import sharded

    rng = np.random.default_rng(n)
    u = rng.standard_normal((n,) * 4)
    u = u - u.transpose(0, 1, 3, 2)
    C = np.linalg.qr(rng.standard_normal((n, n)))[0]
    ctx = sharded.EmulatedContext(world, engine=NumpyEngine())
    basis = sharded.ShardedBasisSet.from_global(ctx, np.eye(n), np.eye(n), u)
    out = sharded.transform_two_body_sharded(basis.u, torch.from_numpy(C))  # n >= 48: found anti-symmetric, exploited
    assert out.proven_antisymmetric
    got = out.gather().numpy()
    assert not np.isnan(got).any()
    expected = oracle.transform_two_body_elements(u, C)
    np.testing.assert_allclose(got, expected, rtol=1e-12, atol=1e-12 * np.abs(expected).max())
    np.testing.assert_array_equal(got, -got.transpose(0, 1, 3, 2))


def test_recycled_handle_raises_instead_of_showing_new_data():
    """A transform writes into the buffers of the tensor replaced one call earlier (ping-pong).  A caller that
    still holds that older handle must get an error, not silently the newer tensor; copy() keeps data alive."""
    from quantum_systems_b200 import sharded

    n = 6
    rng = np.random.default_rng(3)
    u = rng.standard_normal((n,) * 4)
    C = torch.from_numpy(np.linalg.qr(rng.standard_normal((n, n)))[0])
    ctx = sharded.EmulatedContext(2, engine=NumpyEngine())
    u0 = sharded.ShardedBasisSet.from_global(ctx, np.eye(n), np.eye(n), u).u
    kept = u0.copy()
    u1 = sharded.transform_two_body_sharded(u0, C)
    np.testing.assert_array_equal(u0.gather().numpy(), u)  # one call later the input is still intact
    u2 = sharded.transform_two_body_sharded(u1, C)  # writes into u0's buffers
    with pytest.raises(RuntimeError, match="recycled"):
        u0.gather()
    with pytest.raises(RuntimeError, match="recycled"):
        u0.local(0)
    np.testing.assert_array_equal(kept.gather().numpy(), u)
    expected = oracle.transform_two_body_elements(oracle.transform_two_body_elements(u, C.numpy()), C.numpy())
    np.testing.assert_allclose(u2.gather().numpy(), expected, rtol=1e-11, atol=1e-11)
    assert u1.gather().shape == (n,) * 4  # the tensor replaced ONE call earlier is still valid


@pytest.mark.parametrize("world", [1, 2, 3, 5])
@pytest.mark.parametrize("complex_", [False, True])
def test_emulated_consumers_of_a_sharded_tensor(world, complex_):
    """u[o,o,v,v]-style blocks, scaled copies and the reference energy on a sharded tensor
    (SURVEY.md section 8f-3) against plain numpy slicing and the oracle."""
    from quantum_systems_b200 import sharded

    n, n_occ = 7, 3
    rng = np.random.default_rng(17 + world)
    u = rand(rng, (n,) * 4, complex_)
    h = rand(rng, (n, n), complex_)
    ctx = sharded.EmulatedContext(world, engine=NumpyEngine())
    basis = sharded.ShardedBasisSet.from_global(ctx, h, np.eye(n), u, includes_spin=True)
    o, v = slice(0, n_occ), slice(n_occ, n)
    for sl in [(o, o, v, v), (v, o, v, o), (o, o, o, o), (v, v, v, v), (slice(2, 6), None, slice(0, 1), v),
               (slice(5, 5), o, o, o)]:
        np.testing.assert_array_equal(basis.u.extract(*sl).numpy(), u[tuple(slice(None) if s is None else s for s in sl)])
    np.testing.assert_allclose(
        basis.compute_reference_energy(n_occ, nuclear_repulsion_energy=0.25),
        oracle.reference_energy_general(h, u, n_occ, 0.25), rtol=1e-13,
    )
    spatial = sharded.ShardedBasisSet.from_global(ctx, h, np.eye(n), u)
    np.testing.assert_allclose(
        spatial.compute_reference_energy(n_occ), oracle.reference_energy_spatial(h, u, n_occ), rtol=1e-13
    )
    scaled = basis.u.copy().axpby_(0.5)
    np.testing.assert_array_equal(scaled.gather().numpy(), 0.5 * u)
    # u_t = u_0 + f(t) u on a sharded tensor (reference system.py:203-215): one new handle, shard-local passes
    from quantum_systems_b200.system import scaled_sum

    np.testing.assert_array_equal(basis.u.scaled(2.0, scaled, -1.0).gather().numpy(), 2.0 * u - 0.5 * u)
    total = scaled_sum(None, [(1.0, basis.u), (0.25, basis.u), (-3.0, scaled)])
    np.testing.assert_allclose(total.gather().numpy(), (1.25 - 1.5) * u, rtol=1e-15)
    np.testing.assert_array_equal(basis.u.gather().numpy(), u)  # the copy left the original alone
    combo = basis.u.copy().axpby_(2.0, scaled, -3.0)
    np.testing.assert_allclose(combo.gather().numpy(), 2.0 * u - 1.5 * u, rtol=1e-15)
    if not complex_:
        with pytest.raises(TypeError):
            basis.u.axpby_(1j)


@pytest.mark.parametrize("world", [1, 2, 3, 4])
@pytest.mark.parametrize("n,m,complex_", [(8, 8, False), (9, 9, False), (7, 10, True), (10, 6, True), (16, 16, False)])
def test_emulated_symmetry_aware_schedule(world, n, m, complex_, monkeypatch):
    """Anti-symmetric u: steps 3-4 on the pairs the cyclic rule selects (balanced over the r-partition), packed by
    pair, local mirror fill -- against the oracle's four full steps; the result is exactly anti-symmetric."""
    from quantum_systems_b200 import sharded

    monkeypatch.setattr(sharded, "SYMMETRY_MIN_N", 4)
    rng = np.random.default_rng(10 * n + m + world)
    u = rand(rng, (n,) * 4, complex_)
    u = u - u.transpose(0, 1, 3, 2)
    C = rand(rng, (n, m), complex_)
    ctx = sharded.EmulatedContext(world, engine=NumpyEngine())
    basis = sharded.ShardedBasisSet.from_global(ctx, np.eye(n), np.eye(n), u)
    assert sharded.is_antisymmetric_last_pair(basis.u)
    out = sharded.transform_two_body_sharded(basis.u, torch.from_numpy(C))
    expected = oracle.transform_two_body_elements(u, C)
    got = out.gather().numpy()
    np.testing.assert_allclose(got, expected, rtol=1e-12, atol=1e-12 * np.abs(expected).max())
    np.testing.assert_array_equal(got, -got.transpose(0, 1, 3, 2))
    # a tensor without the symmetry takes the four full steps
    basis2 = sharded.ShardedBasisSet.from_global(ctx, np.eye(n), np.eye(n), u + 1.0)
    assert not sharded.is_antisymmetric_last_pair(basis2.u)


def test_cyclic_rule_picks_each_pair_once_and_balances_r():
    from quantum_systems_b200.sharded import cyclic_wanted

    for m in (1, 2, 3, 8, 9, 50, 400):
        r, s = np.arange(m)[:, None], np.arange(m)[None, :]
        w = cyclic_wanted(r, s, m)
        assert not w.diagonal().any()
        assert np.array_equal(w ^ w.T, ~np.eye(m, dtype=bool))  # exactly one of (r, s), (s, r)
        per_r = w.sum(axis=1)
        assert per_r.max() - per_r.min() <= 1  # every r has the same number of partners (+-1 for even m)


def _free_port():
    with socket.socket() as sock:
        sock.bind(("127.0.0.1", 0))
        return sock.getsockname()[1]


def _gloo_worker(rank, world, port, n, m, complex_, results):
    import torch.distributed as dist

    from quantum_systems_b200 import sharded

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        rng = np.random.default_rng(7)
        u = rand(rng, (n,) * 4, complex_)
        C = rand(rng, (n, m), complex_)
        ctx = sharded.ProcessContext(engine=NumpyEngine())
        assert ctx.exchange == "collective"
        basis = sharded.ShardedBasisSet.from_global(ctx, np.eye(n), np.eye(n), u)
        p0, p1 = basis.u.planes(rank)
        np.testing.assert_array_equal(basis.u.local().numpy(), u[p0:p1])
        out = sharded.transform_two_body_sharded(basis.u, torch.from_numpy(C))
        expected = oracle.transform_two_body_elements(u, C)
        q0, q1 = out.planes(rank)
        np.testing.assert_allclose(out.local().numpy(), expected[q0:q1], rtol=1e-12, atol=1e-12 * np.abs(expected).max())
        full = out.gather().numpy()
        np.testing.assert_allclose(full, expected, rtol=1e-12, atol=1e-12 * np.abs(expected).max())
        # consumers: replicated blocks (all-gather) and the reference energy (6-double all-reduce)
        if m >= 4:
            o, v = slice(0, 3), slice(3, m)
            np.testing.assert_allclose(out.extract(o, o, v, v).numpy(), expected[o, o, v, v], rtol=1e-12,
                                       atol=1e-12 * np.abs(expected).max())
            np.testing.assert_allclose(out.extract(v, o, None, o).numpy(), expected[v, o, :, o], rtol=1e-12,
                                       atol=1e-12 * np.abs(expected).max())
            h = rand(np.random.default_rng(3), (m, m), complex_)
            holder = sharded.ShardedBasisSet(ctx, m, torch.from_numpy(h), None, out, includes_spin=True)
            np.testing.assert_allclose(holder.compute_reference_energy(3), oracle.reference_energy_general(h, expected, 3),
                                       rtol=1e-11)
            doubled = out.copy().axpby_(2.0)
            np.testing.assert_allclose(doubled.local().numpy(), 2.0 * expected[q0:q1], rtol=1e-12,
                                       atol=1e-12 * np.abs(expected).max())
        results[rank] = "ok"
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("n,m,complex_", [(8, 8, False), (7, 9, True)])
def test_collective_schedule_world2_gloo(n, m, complex_):
    import torch.multiprocessing as mp

    world = 2
    port = _free_port()
    manager = mp.get_context("spawn").Manager()
    results = manager.dict()
    mp.spawn(_gloo_worker, args=(world, port, n, m, complex_, results), nprocs=world, join=True)
    assert dict(results) == {0: "ok", 1: "ok"}


# ------------------------------------------------------- the rounding-bound check of the sharded schedule, on the host
# tests/sharded_bounds.py holds the sharded transform of an exact A ⊗ B tensor to the rounding-error bound on whole
# planes and on every element (tests/test_gpu_rounding_bounds.py runs it on the device).  Here it runs unchanged on
# the numpy engine, whose buffers start as NaN: a correct schedule passes, and three broken engines fail it.


class DroppedPairTile(NumpyEngine):
    """Step 2 of the anti-symmetric pair schedule leaves out one of the tiles its planner keeps."""

    @staticmethod
    def _pair_tiles(*args):
        tiles = NumpyEngine._pair_tiles(*args)
        return np.delete(tiles, len(tiles) // 2, axis=0)


class SwappedDealtColumns(NumpyEngine):
    """The dealt store of step 4 (deal > 1) exchanges two output columns."""

    def quarter_scatter(self, A, X, K, lda, image, m_dtype, W, dests, *args, deal=1, cyclic=False):
        if deal > 1:
            image = image.copy()
            image[:, [0, 1]] = image[:, [1, 0]]
        super().quarter_scatter(A, X, K, lda, image, m_dtype, W, dests, *args, deal=deal, cyclic=cyclic)


class Step1In46Bits(NumpyEngine):
    """Step 1 rounds its operands to 46-bit mantissas (with every source holding equally many planes, step 1 is the
    only plain ``quarter`` launch of the peer schedule)."""

    def quarter(self, A, X, K, lda, image, *args):
        import precise as P
        from _numpy_engine import HostBuffer

        chopped = HostBuffer(torch.from_numpy(P.chop(A.flat()[: X * lda], 46)))
        super().quarter(chopped, X, K, lda, P.chop(image, 46), *args)


def graded_kron_case(n, seed):
    """Graded family on an exact tensor: dyadic ``A``, ``B`` scaled by power-of-two ``g_a g_c`` and a near-identity
    ``C``, so that the result spans 16 decades and small elements carry the rounding of every step."""
    import precise as P

    rng = np.random.default_rng(seed)
    g = P.pow2_graded(n)
    A, B = (P.dyadic(rng, (n, n)) * np.outer(g, g) for _ in range(2))
    C = P.near_identity(rng, n)
    return rng, A, B, C


def run_sharded_bound(engine, n, anti, world=3):
    """The sharded transform of the graded exact tensor through ``engine``, checked by tests/sharded_bounds.py.
    Returns the result and its reference arrays."""
    import precise as P
    import sharded_bounds as SB
    from quantum_systems_b200 import sharded

    rng, A, B, C = graded_kron_case(n, seed=n + anti)
    ctx = sharded.EmulatedContext(world, engine=engine)
    u = SB.exact_sharded(ctx, A, B, anti, torch.float64, "cpu")
    out = sharded.transform_two_body_sharded(u, torch.from_numpy(C))
    assert out.proven_antisymmetric == anti, "the case did not take the schedule it is there for"
    SB.check_sharded(P.assert_rounding_bound, out, P.kron_factors, (A, B, C, C.T), P.k_transform([n] * 4, [False] * 4),
                     anti, rng, f"n={n} W={world} anti={anti}")
    return out, (A, B, C, C.T)


@pytest.fixture
def pair_schedule_below_48(monkeypatch):
    from quantum_systems_b200 import sharded
    from quantum_systems_b200.build import build

    build()  # the numpy pair step asks the library's planner for its tiles
    monkeypatch.setattr(sharded, "SYMMETRY_MIN_N", 4)


# n = 21 over 3 ranks: equal sources (7 planes each), an odd real pitch and 21 >= 16 dealt columns in step 4.
# n = 20 anti-symmetric: uneven sources (7, 7, 6, per-source pair tables) and pair lists padded to couples.
@pytest.mark.parametrize("n,anti", [(21, False), (20, True)], ids=["full steps", "pair schedule"])
def test_sharded_bound_harness_passes_the_numpy_schedule(n, anti, pair_schedule_below_48):
    from quantum_systems_b200 import sharded

    assert np.isnan(NumpyEngine().empty(4, torch.float64).flat()).all(), "the stand-in's buffers must start as NaN"
    _, off = sharded.block_partition(n, 3)
    assert len({b - a for a, b in zip(off, off[1:])}) == (2 if anti else 1)
    assert NumpyEngine().scatter_deal(n) > 1
    run_sharded_bound(NumpyEngine(), n, anti)


def test_sharded_bound_harness_rejects_a_dropped_pair_tile(pair_schedule_below_48):
    with pytest.raises(AssertionError, match="non-finite|sweep"):
        run_sharded_bound(DroppedPairTile(), 20, True)


def test_sharded_bound_harness_rejects_swapped_dealt_columns(pair_schedule_below_48):
    with pytest.raises(AssertionError, match="criterion"):
        run_sharded_bound(SwappedDealtColumns(), 21, False)


def test_sharded_bound_harness_rejects_a_46_bit_step_the_scaled_check_accepts(pair_schedule_below_48):
    import precise as P
    from conftest import assert_close_scaled

    with pytest.raises(AssertionError, match="criterion B"):
        run_sharded_bound(Step1In46Bits(), 21, False)
    # the same mutant, end to end, is well inside the 1e-12 max-scaled tolerance
    from quantum_systems_b200 import sharded
    import sharded_bounds as SB

    _, A, B, C = graded_kron_case(21, seed=21)
    ctx = sharded.EmulatedContext(3, engine=Step1In46Bits())
    out = sharded.transform_two_body_sharded(SB.exact_sharded(ctx, A, B, False, torch.float64, "cpu"),
                                             torch.from_numpy(C))
    assert_close_scaled(out.gather().numpy(), P.kron_transform_planes(A, B, C, C.T, planes=range(21), dt=np.float64))
