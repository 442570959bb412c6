"""The sharded spin-orbital system of an unrestricted basis on a CPU-only box: the plane routing of
``sharded.spin_plane_routing`` by brute force, and the whole schedule of ``sharded.spin_orbital_two_body_sharded``
(emulated ranks and two gloo processes) against an independent einsum build.  The column-table store and the
assembly kernel are stood in for by the numpy engine below, which implements their documented semantics
(include/qsb200.h: qs_quarter_transform_scatter_columns, qs_spin_orbital_two_body) on NaN-initialised buffers, so
a plane that is read before anyone wrote it shows up."""

import os
import socket
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from _numpy_engine import NumpyEngine  # noqa: E402


class SpinBlockEngine(NumpyEngine):
    """The numpy engine plus the column-table store and the spin-orbital assembly."""

    def quarter_scatter_columns(self, A, X, K, lda, image, m_dtype, W, dests, col_dest, col_off, offsets_even,
                                x_inner, x_mid, sx0, sx1, sx2, deal=1):
        if X <= 0:
            return
        res = self._product(A, X, K, lda, image)
        if deal > 1:  # column j of the product is physical column (j * deal) % W
            physical = np.empty_like(res)
            physical[:, (np.arange(W) * deal) % W] = res
            res = physical
        dest, off = col_dest.numpy(), col_off.numpy()
        assert dest.dtype == np.int32 and off.dtype == np.int64 and len(dest) == len(off) == W
        assert np.all((0 <= dest) & (dest < len(dests)))
        if offsets_even:
            assert np.all(off % 2 == 0)
        x = np.arange(X)
        xq = x // x_inner
        ax = (xq // max(x_mid, 1)) * sx2 + (xq % max(x_mid, 1)) * sx1 + (x % x_inner) * sx0
        for w in range(W):
            buf, base = dests[dest[w]]
            idx = base + off[w] + ax
            assert idx.min() >= 0 and idx.max() < buf.numel
            buf.flat()[idx] = res[:, w]

    def spin_orbital_planes(self, blocks, l, orbital, spin, out, p0, p1):
        orbital, spin = orbital.numpy(), spin.numpy()
        n = 2 * l

        def plane(b, o):  # spatial plane o of block b; must lie inside the staged planes
            buf, off = blocks[b]
            start = off + int(o) * l**3
            assert 0 <= start and start + l**3 <= buf.numel, "assembly reads outside the staged planes"
            return buf.flat()[start : start + l**3].reshape(l, l, l)

        sK, sL = spin[:, None], spin[None, :]
        oK, oL = orbital[:, None], orbital[None, :]
        res = np.zeros((p1 - p0, n, n, n), dtype=out.flat().dtype)
        for I in range(p0, p1):
            for J in range(n):
                B = plane(2 * spin[I] + spin[J], orbital[I])[orbital[J]]  # b[oI, oJ, :, :]
                res[I - p0, J] = (np.where((sK == spin[I]) & (sL == spin[J]), B[oK, oL], 0)
                                  - np.where((sL == spin[I]) & (sK == spin[J]), B[oL, oK], 0))
        out.flat()[: res.size] = res.reshape(-1)


def rand(rng, shape, complex_):
    x = rng.standard_normal(shape)
    return x + 1j * rng.standard_normal(shape) if complex_ else x


def reference_spin_orbital_u(u, Ca, Cb, n_alpha, n_beta):
    """Spin-double and anti-symmetrise u, then one einsum transform with the (2l, 2l) spin-orbital coefficients."""
    from quantum_systems_b200.hartree_fock import spin_orbital_order

    l = u.shape[0]
    u2 = np.zeros((2 * l,) * 4, dtype=u.dtype)
    for s in (0, 1):
        for t in (0, 1):
            u2[s::2, t::2, s::2, t::2] = u
    anti = u2 - u2.transpose(0, 1, 3, 2)
    orbital, spin = spin_orbital_order(n_alpha, n_beta, l)
    C = np.zeros((2 * l, 2 * l), dtype=np.result_type(Ca, Cb))
    for I in range(2 * l):
        C[spin[I] :: 2, I] = (Ca, Cb)[spin[I]][:, orbital[I]]
    return np.einsum("ap,bq,abcd,cr,ds->pqrs", C.conj(), C.conj(), anti, C, C, optimize=True)


# ------------------------------------------------------------------------------------------------ routing
def brute_force_owner(n_alpha, n_beta, l, world):
    from quantum_systems_b200.hartree_fock import spin_orbital_order
    from quantum_systems_b200.sharded import block_partition

    orbital, spin = spin_orbital_order(n_alpha, n_beta, l)
    _, offsets = block_partition(2 * l, world)
    owner = np.full((2, l), -1)
    for P in range(2 * l):
        owner[spin[P], orbital[P]] = [j for j in range(world) if offsets[j] <= P < offsets[j + 1]][0]
    return owner, offsets, orbital, spin


def routing_cases():
    rng = np.random.default_rng(2026)
    cases = {(1, 0, 0, 1), (1, 1, 0, 2), (1, 1, 1, 3), (5, 0, 0, 2), (5, 5, 5, 4), (6, 3, 0, 4), (6, 6, 0, 5),
             (7, 7, 2, 16), (3, 2, 1, 9), (10, 4, 4, 8), (200, 13, 0, 8), (200, 200, 0, 8), (100, 21, 20, 8)}
    while len(cases) < 400:
        l = int(rng.integers(1, 40))
        cases.add((l, int(rng.integers(0, l + 1)), int(rng.integers(0, l + 1)), int(rng.integers(1, 17))))
    return sorted(cases)


def test_plane_routing_by_brute_force():
    from quantum_systems_b200.sharded import spin_plane_routing

    for l, n_alpha, n_beta, world in routing_cases():
        expected_owner, offsets, orbital, spin = brute_force_owner(n_alpha, n_beta, l, world)
        owner, ranges = spin_plane_routing(n_alpha, n_beta, l, world)
        assert ranges.shape == (world, 2, 2)
        np.testing.assert_array_equal(owner, expected_owner)
        for s in (0, 1):
            # the ranges tile [0, l) in rank order
            assert ranges[0, s, 0] == 0 and ranges[-1, s, 1] == l
            assert np.all(ranges[1:, s, 0] == ranges[:-1, s, 1]) and np.all(ranges[:, s, 1] >= ranges[:, s, 0])
        for j in range(world):
            # rank j's planes map to one contiguous orbital range per spin, the one the routing names
            planes = range(offsets[j], offsets[j + 1])
            for s in (0, 1):
                orbs = sorted(int(orbital[P]) for P in planes if spin[P] == s)
                assert orbs == list(range(ranges[j, s, 0], ranges[j, s, 1])), (l, n_alpha, n_beta, world, j, s)
        # every (block, p) lands exactly once, on the rank that owns plane P(p, sigma)
        for sigma in (0, 1):
            for _tau in (0, 1):
                for p in range(l):
                    hits = [j for j in range(world) if ranges[j, sigma, 0] <= p < ranges[j, sigma, 1]]
                    assert hits == [expected_owner[sigma, p]]


def test_routing_with_no_beta_electrons_leaves_ranks_without_alpha_planes():
    from quantum_systems_b200.sharded import spin_plane_routing

    _, ranges = spin_plane_routing(8, 0, 8, 8)
    alpha = ranges[:, 0, 1] - ranges[:, 0, 0]
    assert sorted(alpha.tolist()) == [0, 0, 0, 0, 2, 2, 2, 2]  # the uneven split a block partition cannot express


def test_column_table_store_refusals():
    """qs_quarter_transform_scatter_columns refuses, before touching a device, a missing column table, more than 16
    destinations and a dealing multiplier that is not coprime to W."""
    import ctypes

    from quantum_systems_b200 import _native
    from quantum_systems_b200.build import build

    build()
    lib = _native.load()
    fake = ctypes.c_void_p(1 << 20)  # never dereferenced: every call below is refused by its argument checks

    def call(n_dest, col_dest, col_off, W=32, deal=1):
        table = (ctypes.c_void_p * max(n_dest, 1))(*([fake] * max(n_dest, 1)))
        return lib.qs_quarter_transform_scatter_columns(fake, 0, 128, 16, 16, fake, 0, W, table, n_dest, col_dest,
                                                        col_off, 0, 128, 1, 1, 0, 0, deal, ctypes.c_void_p(0))

    assert call(2, ctypes.c_void_p(0), fake) != 0 and b"null pointer" in lib.qs_last_error()
    assert call(2, fake, ctypes.c_void_p(0)) != 0 and b"null pointer" in lib.qs_last_error()
    assert call(0, fake, fake) != 0 and b"empty destination table" in lib.qs_last_error()
    assert call(17, fake, fake) != 0 and b"at most 16 destinations" in lib.qs_last_error()
    assert call(2, fake, fake, W=32, deal=2) != 0 and b"not coprime" in lib.qs_last_error()


# ------------------------------------------------------------------------------------------------ end to end
CASES = [
    # l, n_alpha, n_beta, u complex, C complex
    (4, 2, 2, False, False),
    (5, 3, 1, False, False),
    (5, 2, 0, True, False),
    (6, 6, 1, False, True),
    (3, 1, 1, True, True),
    (1, 1, 0, False, False),
    (17, 5, 3, False, False),  # 17 >= 16 new columns: step 4 deals its columns
]


@pytest.mark.parametrize("world", [1, 2, 3, 4])
@pytest.mark.parametrize("l,n_alpha,n_beta,u_complex,c_complex", CASES)
def test_emulated_spin_orbital_two_body_sharded(world, l, n_alpha, n_beta, u_complex, c_complex):
    from quantum_systems_b200 import sharded

    if l >= 16 and world not in (1, 3):
        pytest.skip("the dealt case runs at two rank counts")
    rng = np.random.default_rng(17 * l + world)
    u = rand(rng, (l,) * 4, u_complex)
    Ca, Cb = rand(rng, (l, l), c_complex), rand(rng, (l, l), c_complex)
    ctx = sharded.EmulatedContext(world, engine=SpinBlockEngine())
    basis = sharded.ShardedBasisSet.from_global(ctx, np.eye(l), np.eye(l), u)
    before = basis.u.gather().numpy().copy()
    out = sharded.spin_orbital_two_body_sharded(basis.u, torch.from_numpy(Ca), torch.from_numpy(Cb), n_alpha, n_beta)
    expected = reference_spin_orbital_u(u, Ca, Cb, n_alpha, n_beta)
    got = out.gather().numpy()
    assert out.n == 2 * l and out.dtype == torch.complex128 and out.proven_antisymmetric
    np.testing.assert_allclose(got, expected, rtol=0, atol=1e-12 * np.abs(expected).max())
    np.testing.assert_array_equal(got, -got.transpose(0, 1, 3, 2))
    np.testing.assert_array_equal(basis.u.gather().numpy(), before)  # the input stays as it was
    # a second call reuses the cached staging buffers and gives the same planes; with into= it writes into the
    # buffers of the first result and allocates no new ones
    again = sharded.spin_orbital_two_body_sharded(basis.u, torch.from_numpy(Ca), torch.from_numpy(Cb), n_alpha,
                                                  n_beta)
    np.testing.assert_array_equal(again.gather().numpy(), got)
    for r in ctx.local_ranks:
        again.local(r).fill_(float("nan"))
    reused = sharded.spin_orbital_two_body_sharded(basis.u, torch.from_numpy(Ca), torch.from_numpy(Cb), n_alpha,
                                                   n_beta, into=again)
    assert reused is again and reused.proven_antisymmetric
    np.testing.assert_array_equal(reused.gather().numpy(), got)
    with pytest.raises(ValueError, match="into"):
        sharded.spin_orbital_two_body_sharded(basis.u, torch.from_numpy(Ca), torch.from_numpy(Cb), n_alpha, n_beta,
                                              into=basis.u)


def test_real_blocks_give_a_real_result_and_complex_blocks_refuse_one():
    from quantum_systems_b200 import sharded

    rng = np.random.default_rng(5)
    l = 4
    u = rand(rng, (l,) * 4, False)
    Ca, Cb = rand(rng, (l, l), False), rand(rng, (l, l), False)
    ctx = sharded.EmulatedContext(2, engine=SpinBlockEngine())
    basis = sharded.ShardedBasisSet.from_global(ctx, np.eye(l), np.eye(l), u)
    out = sharded.spin_orbital_two_body_sharded(basis.u, torch.from_numpy(Ca), torch.from_numpy(Cb), 2, 1,
                                                out_dtype=torch.float64)
    assert out.dtype == torch.float64
    expected = reference_spin_orbital_u(u, Ca, Cb, 2, 1)
    np.testing.assert_allclose(out.gather().numpy(), expected, rtol=0, atol=1e-12 * np.abs(expected).max())
    with pytest.raises(TypeError):
        sharded.spin_orbital_two_body_sharded(basis.u, torch.from_numpy(Ca + 1j), torch.from_numpy(Cb), 2, 1,
                                              out_dtype=torch.float64)


@pytest.mark.parametrize("world", [1, 2, 3])
@pytest.mark.parametrize("n,u_complex,c_complex,bras", [(6, False, False, False), (7, True, True, True),
                                                        (17, False, True, False)])
def test_emulated_mixed_transform_leaves_its_input_valid(world, n, u_complex, c_complex, bras):
    from quantum_systems_b200 import sharded

    rng = np.random.default_rng(n + world)
    u = rand(rng, (n,) * 4, u_complex)
    C_r, C_s = rand(rng, (n, n), c_complex), rand(rng, (n, n), c_complex)
    Ct_p = rand(rng, (n, n), c_complex) if bras else None
    Ct_q = rand(rng, (n, n), c_complex) if bras else None
    ctx = sharded.EmulatedContext(world, engine=SpinBlockEngine())
    basis = sharded.ShardedBasisSet.from_global(ctx, np.eye(n), np.eye(n), u)
    t = lambda M: None if M is None else torch.from_numpy(M)  # noqa: E731
    first = sharded.transform_two_body_sharded_mixed(basis.u, t(C_r), t(C_s), t(Ct_p), t(Ct_q))
    second = sharded.transform_two_body_sharded_mixed(basis.u, t(C_r), t(C_s), t(Ct_p), t(Ct_q))
    Ct_p = C_r.conj().T if Ct_p is None else Ct_p
    Ct_q = C_s.conj().T if Ct_q is None else Ct_q
    expected = np.einsum("pa,qb,abcd,cr,ds->pqrs", Ct_p, Ct_q, u, C_r, C_s, optimize=True)
    for out in (first, second):  # the first handle is not recycled by the second call
        np.testing.assert_allclose(out.gather().numpy(), expected, rtol=0, atol=1e-12 * np.abs(expected).max())
    np.testing.assert_array_equal(basis.u.gather().numpy(), u)


def _free_port():
    with socket.socket() as sock:
        sock.bind(("127.0.0.1", 0))
        return sock.getsockname()[1]


def _gloo_worker(rank, world, port, results):
    import torch.distributed as dist

    from quantum_systems_b200 import sharded

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        for l, n_alpha, n_beta, u_complex, c_complex in [(5, 3, 1, False, False), (4, 4, 0, True, True),
                                                          (6, 2, 2, False, True)]:
            rng = np.random.default_rng(l)
            u = rand(rng, (l,) * 4, u_complex)
            Ca, Cb = rand(rng, (l, l), c_complex), rand(rng, (l, l), c_complex)
            ctx = sharded.ProcessContext(engine=SpinBlockEngine())
            assert ctx.exchange == "collective"
            basis = sharded.ShardedBasisSet.from_global(ctx, np.eye(l), np.eye(l), u)
            out = sharded.spin_orbital_two_body_sharded(basis.u, torch.from_numpy(Ca), torch.from_numpy(Cb),
                                                        n_alpha, n_beta)
            expected = reference_spin_orbital_u(u, Ca, Cb, n_alpha, n_beta)
            p0, p1 = out.planes(rank)
            np.testing.assert_allclose(out.local().numpy(), expected[p0:p1], rtol=0,
                                       atol=1e-12 * np.abs(expected).max())
            np.testing.assert_allclose(out.gather().numpy(), expected, rtol=0, atol=1e-12 * np.abs(expected).max())
            mixed = sharded.transform_two_body_sharded_mixed(basis.u, torch.from_numpy(Ca), torch.from_numpy(Cb))
            ref = np.einsum("ap,bq,abcd,cr,ds->pqrs", Ca.conj(), Cb.conj(), u, Ca, Cb, optimize=True)
            np.testing.assert_allclose(mixed.gather().numpy(), ref, rtol=0, atol=1e-12 * np.abs(ref).max())
        results[rank] = "ok"
    finally:
        dist.destroy_process_group()


def test_collective_schedule_world2_gloo():
    import torch.multiprocessing as mp

    world = 2
    port = _free_port()
    manager = mp.get_context("spawn").Manager()
    results = manager.dict()
    mp.spawn(_gloo_worker, args=(world, port, results), nprocs=world, join=True)
    assert dict(results) == {0: "ok", 1: "ok"}
