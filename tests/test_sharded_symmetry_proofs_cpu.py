"""The anti-symmetry proof of a ``ShardedTwoBody`` (``proven_antisymmetric``) on a CPU-only box: it lets the sharded
transform skip the exact device-side test and run steps 3 and 4 on half of the (r, s) pairs, so a proof that outlives
the data it was made for gives a wrong result without any error.  Writes into ``local()`` must void it, every library
operation must leave it exactly as true as the data, and reads must keep it (a chain of basis changes that inspects
its tensors would otherwise pay one detection per step).  Also: the pair tables cached per context must not be shared
between real and complex transforms of the same shape.  The arithmetic runs in tests/_numpy_engine.py."""

import os
import socket
import sys

import numpy as np
import pytest
import torch

from oracle import qs_oracle as oracle

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from _numpy_engine import NumpyEngine  # noqa: E402

WORLDS = [1, 2, 3, 5]  # world 5 at n = 12: the last rank holds no plane


def rand(rng, shape, complex_):
    x = rng.standard_normal(shape)
    return x + 1j * rng.standard_normal(shape) if complex_ else x


def antisymmetric(rng, n, complex_=False):
    u = rand(rng, (n,) * 4, complex_)
    return u - u.transpose(0, 1, 3, 2)


def truly_antisymmetric(t):
    got = t.gather().numpy()
    return bool(np.array_equal(got, -got.transpose(0, 1, 3, 2)))


def assert_matches_oracle(got, u, C):
    expected = oracle.transform_two_body_elements(u, C)
    np.testing.assert_allclose(got, expected, rtol=0, atol=1e-12 * np.abs(expected).max())


@pytest.fixture
def detections(monkeypatch):
    """Automatic detection at the small extents of these tests; records the answer of every test of u that read the
    data (a process whose slabs carry the proof skips the read)."""
    from quantum_systems_b200 import sharded

    monkeypatch.setattr(sharded, "SYMMETRY_MIN_N", 4)
    calls, reads = [], []
    real_read = NumpyEngine.is_antisymmetric

    def read(self, buf, n, planes):
        reads.append(real_read(self, buf, n, planes))
        return reads[-1]

    real_test = sharded.is_antisymmetric_last_pair

    def spy(u, trust_proof=False):
        del reads[:]
        answer = real_test(u, trust_proof)
        if reads:
            calls.append(answer)
        return answer

    monkeypatch.setattr(NumpyEngine, "is_antisymmetric", read)
    monkeypatch.setattr(sharded, "is_antisymmetric_last_pair", spy)
    return calls


def proven_result(world, n, complex_=False, seed=0):
    """A transform result the library has proven anti-symmetric, the context, the coefficients and the input."""
    from quantum_systems_b200 import sharded

    rng = np.random.default_rng(seed + world)
    u = antisymmetric(rng, n, complex_)
    C = np.linalg.qr(rand(rng, (n, n), complex_))[0]
    ctx = sharded.EmulatedContext(world, engine=NumpyEngine())
    basis = sharded.ShardedBasisSet.from_global(ctx, np.eye(n), np.eye(n), u)
    out = sharded.transform_two_body_sharded(basis.u, torch.from_numpy(C))
    assert out.proven_antisymmetric
    return out, ctx, C, u


@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("complex_", [False, True])
def test_write_through_local_voids_the_proof(world, complex_, detections):
    from quantum_systems_b200 import sharded

    out, _, C, _ = proven_result(world, 12, complex_)
    assert detections == [True]
    rank = world - 1 if out.planes(world - 1)[1] > out.planes(world - 1)[0] else 0
    out.local(rank)[0, 1, 2, 3] += 1.0  # breaks u[p,q,r,s] = -u[p,q,s,r] for one (r, s) pair
    assert not out.proven_antisymmetric
    mutated = out.gather().numpy().copy()
    again = sharded.transform_two_body_sharded(out, torch.from_numpy(C))
    assert detections == [True, False]  # the exact test ran and said no: four full steps
    assert not again.proven_antisymmetric
    assert_matches_oracle(again.gather().numpy(), mutated, C)


@pytest.mark.parametrize("world", WORLDS)
def test_a_write_through_a_view_of_a_plane_voids_the_proof(world, detections):
    """A whole plane overwritten through a view of ``local()`` (``copy_``), i.e. not through the handle."""
    from quantum_systems_b200 import sharded

    out, _, C, _ = proven_result(world, 12, seed=10)
    plane = out.local(0)[1]
    plane.copy_(torch.from_numpy(np.random.default_rng(1).standard_normal(plane.shape)))
    assert not out.proven_antisymmetric
    mutated = out.gather().numpy().copy()
    assert_matches_oracle(sharded.transform_two_body_sharded(out, torch.from_numpy(C)).gather().numpy(), mutated, C)
    assert detections == [True, False]


@pytest.mark.parametrize("world", WORLDS)
def test_reads_keep_the_proof(world, detections, monkeypatch):
    """gather(), extract(), occupied_traces() and local() used read-only do not void the proof: the next transform
    of the chain runs no detection (bench.py reads ``tensor.local()`` between timed transforms)."""
    from quantum_systems_b200 import sharded

    n, n_occ = 12, 4
    out, _, C, _ = proven_result(world, n, seed=20)
    before = out.gather().numpy().copy()
    o, v = slice(0, n_occ), slice(n_occ, n)
    np.testing.assert_array_equal(out.extract(o, o, v, v).numpy(), before[o, o, v, v])
    traces = out.occupied_traces(torch.eye(n, dtype=torch.float64), n_occ)
    direct = np.einsum("ijij->", before[o, o, o, o])
    assert abs(traces[1] - direct) <= 1e-12 * np.abs(before).sum()
    for r in range(world):
        local = out.local(r)
        local.abs().sum()
        local.clone()
        local.numpy().sum()
    assert out.proven_antisymmetric
    assert detections == [True]
    decided, inner = [], sharded.is_antisymmetric_last_pair
    monkeypatch.setattr(sharded, "is_antisymmetric_last_pair",
                        lambda u, trust_proof=False: decided.append(trust_proof) or inner(u, trust_proof))
    again = sharded.transform_two_body_sharded(out, torch.from_numpy(C))
    assert detections == [True]  # no second read of u ...
    assert decided == [True]  # ... but the (collective) decision still ran, trusting the proof
    assert again.proven_antisymmetric
    assert_matches_oracle(again.gather().numpy(), before, C)
    np.testing.assert_array_equal(again.gather().numpy(), -again.gather().numpy().transpose(0, 1, 3, 2))


@pytest.mark.parametrize("world", WORLDS)
def test_library_writers_leave_the_flag_as_true_as_the_data(world, detections):
    """axpby_, scaled and copy: the result is proven exactly when every operand was, and then really is
    anti-symmetric; a write into a copy leaves the original's proof alone (separate buffers)."""
    from quantum_systems_b200 import sharded

    n = 12
    proven, ctx, C, _ = proven_result(world, n, seed=30)
    rng = np.random.default_rng(31)
    plain = sharded.ShardedBasisSet.from_global(ctx, np.eye(n), np.eye(n), rng.standard_normal((n,) * 4)).u
    assert not plain.proven_antisymmetric
    del detections[:]

    def check(t, proven_expected):
        assert t.proven_antisymmetric == proven_expected
        assert truly_antisymmetric(t) == proven_expected  # the flag tells the truth, all of it
        data = t.gather().numpy().copy()
        result = sharded.transform_two_body_sharded(t, torch.from_numpy(C))
        assert_matches_oracle(result.gather().numpy(), data, C)
        assert detections[-1:] == ([] if proven_expected else [False])
        del detections[:]

    check(proven.scaled(0.5), True)
    check(proven.scaled(0.5, proven, -2.0), True)
    check(proven.scaled(1.0, plain, 1.0), False)
    check(plain.scaled(1.0, proven, 1.0), False)
    check(proven.copy(), True)
    check(proven.copy().axpby_(-0.25), True)
    check(proven.copy().axpby_(1.0, proven, 3.0), True)
    check(proven.copy().axpby_(1.0, plain, 1e-3), False)

    dirty = proven.copy()
    dirty.local(0)[0, 0, 0, 1] -= 1.0
    assert not dirty.proven_antisymmetric and proven.proven_antisymmetric
    check(dirty, False)
    check(proven, True)


def _add_spin_two_body_stand_in(u, anti_symmetrize=False, out_dtype=None, planes=None, out=None,
                                first_spatial_plane=0):
    """Documented semantics of ``ops.add_spin_two_body`` on host tensors, writing through torch as the library's
    entry point does through the C ABI (both bump the version counter of ``out``)."""
    slab = u.numpy()
    l = slab.shape[-1]
    p0, p1 = (0, 2 * l) if planes is None else planes
    P = np.arange(p0, p1)[:, None, None, None]
    Q, R, S = (np.arange(2 * l).reshape(shape) for shape in ((1, -1, 1, 1), (1, 1, -1, 1), (1, 1, 1, -1)))
    spin = slab[P // 2 - first_spatial_plane, Q // 2, R // 2, S // 2] * ((P % 2 == R % 2) & (Q % 2 == S % 2))
    if anti_symmetrize:
        spin = spin - spin.transpose(0, 1, 3, 2)
    out.copy_(torch.from_numpy(np.ascontiguousarray(spin)))
    return out


@pytest.fixture
def host_spin_doubling(monkeypatch):
    from quantum_systems_b200 import _arrays, ops

    monkeypatch.setattr(ops, "add_spin_two_body", _add_spin_two_body_stand_in)
    monkeypatch.setattr(ops, "add_spin_one_body", lambda h, out_dtype=None: torch.kron(h, torch.eye(2, dtype=h.dtype))
                        .to(out_dtype or h.dtype))
    monkeypatch.setattr(_arrays, "to_device", lambda a, dtype=None: NumpyEngine().asarray(a, dtype))


@pytest.mark.parametrize("world", WORLDS)
def test_spin_doubling_into_a_successor(world, detections, host_spin_doubling):
    """successor() hands out the spare buffers unproven; from_spatial_planes(into=...) proves them exactly when it
    anti-symmetrises, and a rebuild without anti-symmetrisation into a proven tensor takes the proof away."""
    from quantum_systems_b200 import sharded

    l = 6
    rng = np.random.default_rng(40 + world)
    u_spatial = rng.standard_normal((l,) * 4)
    u_spatial = 0.5 * (u_spatial + u_spatial.transpose(1, 0, 3, 2))
    spin = oracle.add_spin_two_body(u_spatial)
    C = np.linalg.qr(rng.standard_normal((2 * l, 2 * l)))[0]
    ctx = sharded.EmulatedContext(world, engine=NumpyEngine())

    def build(anti, into):
        return sharded.ShardedBasisSet.from_spatial_planes(ctx, np.eye(l), np.eye(l), l, lambda a0, a1: u_spatial[a0:a1],
                                                           anti_symmetrize=anti, out_dtype=torch.float64, into=into).u

    u = build(True, None)
    assert u.proven_antisymmetric
    np.testing.assert_array_equal(u.gather().numpy(), oracle.anti_symmetrize_u(spin))
    result = sharded.transform_two_body_sharded(u, torch.from_numpy(C))
    assert detections == [] and result.proven_antisymmetric
    assert_matches_oracle(result.gather().numpy(), oracle.anti_symmetrize_u(spin), C)

    nxt = result.successor()
    assert not nxt.proven_antisymmetric
    nxt = build(True, nxt)
    assert nxt.proven_antisymmetric and truly_antisymmetric(nxt)
    plain = build(False, nxt)  # same buffers, rebuilt without the anti-symmetrisation
    assert plain is nxt and not plain.proven_antisymmetric
    assert not truly_antisymmetric(plain)
    np.testing.assert_array_equal(plain.gather().numpy(), spin)
    assert_matches_oracle(sharded.transform_two_body_sharded(plain, torch.from_numpy(C)).gather().numpy(), spin, C)
    assert detections == [False]


@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("n", [8, 12])
def test_pair_tables_across_dtypes_in_one_context(world, n):
    """Real, then complex, then real again: same (n, m, world, pitch) in one context, so the pair tables cached per
    context must be keyed on the dtype -- real even extents pad the pair lists to aligned couples, complex ones do
    not.  Tiles the first exchange does not send stay NaN in the stand-in, so a table that reads one shows up."""
    from quantum_systems_b200 import sharded

    ctx = sharded.EmulatedContext(world, engine=NumpyEngine())
    rng = np.random.default_rng(n + world)
    for complex_ in (False, True, False):
        u = antisymmetric(rng, n, complex_)
        C = rand(rng, (n, n), complex_)
        basis = sharded.ShardedBasisSet.from_global(ctx, np.eye(n), np.eye(n), u)
        got = sharded.transform_two_body_sharded(basis.u, torch.from_numpy(C), symmetry=1).gather().numpy()
        assert not np.isnan(got).any()
        assert_matches_oracle(got, u, C)
        np.testing.assert_array_equal(got, -got.transpose(0, 1, 3, 2))


def _free_port():
    with socket.socket() as sock:
        sock.bind(("127.0.0.1", 0))
        return sock.getsockname()[1]


def _gloo_proof_worker(rank, world, port, results):
    import datetime

    import torch.distributed as dist

    from quantum_systems_b200 import sharded

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    # a rank that issued one collective more than the others fails here instead of hanging
    dist.init_process_group("gloo", rank=rank, world_size=world, timeout=datetime.timedelta(seconds=60))
    try:
        n = 6
        u = antisymmetric(np.random.default_rng(5), n)
        ctx = sharded.ProcessContext(engine=NumpyEngine())
        handle = sharded.ShardedBasisSet.from_global(ctx, np.eye(n), np.eye(n), u).u
        handle.proven_antisymmetric = True  # as the fused spin doubling leaves it on every rank
        answers = [sharded.is_antisymmetric_last_pair(handle, trust_proof=True)]
        if rank == 0:
            handle.local()[0, 1, 2, 3] += 1.0  # only the owner of plane 0 writes
        answers.append(handle.proven_antisymmetric)  # local: void on rank 0 only
        answers.append(sharded.is_antisymmetric_last_pair(handle, trust_proof=True))
        answers.append(sharded.is_antisymmetric_last_pair(handle))
        ctx.barrier()
        results[rank] = answers
    finally:
        dist.destroy_process_group()


def test_one_rank_writing_through_local_changes_the_answer_of_every_rank():
    """One process per rank: the proof is rank-local, so a write through ``local()`` on rank 0 voids it there only.
    The decision of the transform must still be the same on every rank (it selects the schedule and the collectives
    that follow), so the proven ranks take part in the all-reduce of the exact test without reading their planes."""
    import torch.multiprocessing as mp

    world = 3
    manager = mp.get_context("spawn").Manager()
    results = manager.dict()
    mp.spawn(_gloo_proof_worker, args=(world, _free_port(), results), nprocs=world, join=True)
    assert results[0] == [True, False, False, False]
    for rank in range(1, world):
        assert results[rank] == [True, True, False, False]
