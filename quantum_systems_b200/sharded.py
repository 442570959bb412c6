"""Sharded two-body pipeline: one tensor ``u`` spread over the GPUs of an NVSwitch domain.

Once ``u`` no longer fits one GPU (n >~ 300 spin-orbitals) it is block-partitioned on its LEADING
index, ``ceil(n / W)`` planes per rank (SURVEY.md section 8e).  The four-index transform of
``BasisSet.transform_two_body_elements`` (reference basis_set.py:336-350) then runs as

    u[a_loc,b,c,d] --C--> T1[s,a_loc,b,c] --C--> T2[r,s,a_loc,b]           steps 1-2: local contractions
                                   \\=> T2[src][r_loc][s][a_loc][b]         re-partition a -> r (exchange; r dealt
                                                                           cyclically, tiles kept source-major)
    T2[src][r_loc][s][a_loc][b] --C~--> T3[q,r_loc,s,a] --C~--> u'[p,q,r,s]  steps 3-4: local contractions
                                   \\=> u'[p_loc,q,r,s]                     re-partition r -> p (exchange)

like the transpose steps of a distributed FFT.  Both exchanges are FUSED into the producing GEMM: the
epilogue of steps 2 and 4 stores every tile straight into the buffer of the rank that owns it, through
peer pointers mapped with CUDA IPC over NVLink (``qs_quarter_transform_scatter``), so no tile is
written locally, re-read and sent.  ``torch.distributed`` is used for the rendezvous (exchange of IPC
handles), for stream-ordered barriers and for the tiny all-gather of the Fock matrix; it never
carries tensor data on this path.  ``exchange="collective"`` selects the plain
``all_to_all_single`` schedule instead (validation, and CPU/gloo tests of the partition logic).

An exactly anti-symmetric ``u`` (every spin-doubled, anti-symmetrised tensor) is known from its producer or detected
on the device and transformed with steps 3-4 on half of the (r, s) pairs (``cyclic_wanted`` keeps the ranks
balanced) and with a first exchange that sends only the tiles holding such a pair; see
``transform_two_body_sharded`` and DESIGN.md sections 4.9 and 5.

One process per GPU drives one rank (``ProcessContext``).  ``EmulatedContext`` drives all W ranks
from one process on one device; it exists to test the schedule and the scattering kernel on a
single GPU.

The arithmetic runs in the ``engine``: ``CudaEngine`` (the kernels of ``libqsb200.so``) is the only
engine this package provides -- there is no CPU fallback.  Tests inject their own numpy engine to
check the schedule under gloo without a GPU.
"""

import ctypes
import os
import weakref

import torch

from . import _native
from ._native import QS_C128, QS_F64

_CODES = {torch.float64: QS_F64, torch.complex128: QS_C128}
_ITEMSIZE = {torch.float64: 8, torch.complex128: 16}


def block_partition(n, world):
    """Contiguous blocks of ``ceil(n / world)`` indices; trailing ranks may be short or empty.
    Returns ``(block, offsets)`` with rank r owning ``[offsets[r], offsets[r + 1])``."""
    block = -(-n // world)
    return block, [min(r * block, n) for r in range(world + 1)]


# below this extent the symmetry test costs more than the tiles it saves
SYMMETRY_MIN_N = 48
# False: `transform_two_body_sharded(symmetry=None)` never tests for anti-symmetry and runs the four full quarter steps
EXPLOIT_SYMMETRY = True
# Where the scattered tiles land in the peer schedule (see _RankTransform): "source_major" = cyclic intermediate index
# and source-major T2; "interleaved" = block partition of r and T2[r_loc][s][a][b] (the round-1 layout).
# ROTATE_TILES: every rank starts its walk over the tiles of a scattering launch at a different place (rank / world
# of the way through), so that the ranks are never in the same block of a destination at the same time.
SCATTER_LAYOUT = os.environ.get("QS_SHARD_LAYOUT", "source_major")
ROTATE_TILES = os.environ.get("QS_SHARD_ROTATE", "0") == "1"
# False (QS_SHARD_MASK=0): the first exchange of the anti-symmetric schedule sends every tile, as in round 1.
MASK_FIRST_EXCHANGE = os.environ.get("QS_SHARD_MASK", "1") != "0"


def cyclic_wanted(r, s, m):
    """Which of the ordered pairs (r, s), (s, r) the sharded symmetry-aware transform computes: the one whose
    cyclic distance ``(s - r) mod m`` is the shorter; ties (``2 d = m``) go to ``r < s``.  Same rule as
    ``qs_cyclic_pair_wanted`` (csrc/symmetry.cu); works on numpy index arrays."""
    d = (s - r) % m
    return (d > 0) & ((2 * d < m) | ((2 * d == m) & (r < s)))


def padded_pitch(n, dtype):
    """Row pitch (elements) of a contracted axis of extent n: real rows must be a multiple of 16 bytes
    to be described to TMA (csrc/transform.cu)."""
    return n if dtype == torch.complex128 else n + (n & 1)


# ------------------------------------------------------------------------------------------------
# engine: where the arithmetic runs
# ------------------------------------------------------------------------------------------------
class DeviceBuffer:
    """A flat device allocation of ``numel`` elements of ``dtype``: either a torch tensor (scratch from
    the caching allocator) or a raw pointer (an IPC-exported cudaMalloc block or a peer's mapping)."""

    def __init__(self, ptr, numel, dtype, tensor=None):
        self.ptr = int(ptr)
        self.numel = int(numel)
        self.dtype = dtype
        self.tensor = tensor

    def at(self, offset):
        return self.ptr + int(offset) * _ITEMSIZE[self.dtype]

    def as_tensor(self):
        """torch view of the buffer (local memory only)."""
        if self.tensor is None:
            self.tensor = torch.as_tensor(_CudaArray(self.ptr, self.numel, self.dtype), device="cuda")
        return self.tensor


class _CudaArray:
    def __init__(self, ptr, numel, dtype):
        self.__cuda_array_interface__ = {
            "shape": (numel,),
            "typestr": "<c16" if dtype == torch.complex128 else "<f8",
            "data": (ptr, False),
            "version": 3,
            "strides": None,
        }


class CudaEngine:
    """Quarter GEMMs of libqsb200.so on the current CUDA stream."""

    def empty(self, numel, dtype):
        t = torch.empty(max(int(numel), 1), dtype=dtype, device="cuda")
        return DeviceBuffer(t.data_ptr(), numel, dtype, tensor=t)

    @staticmethod
    def _stream():
        return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def asarray(self, a, dtype=None):
        from . import _arrays

        return _arrays.to_device(a, dtype)

    def scatter_deal(self, W):
        from . import ops

        return ops.scatter_deal(W)

    def image(self, M, K, W, a_dtype, stride_k, stride_w, conj=False, deal=1):
        from . import ops

        return ops.coeff_image(M, K, W, a_dtype, stride_k, stride_w, conj=conj, deal=deal)

    def pad_rows(self, src, rows, n, pitch, dst):
        _native.call(
            "qs_pad_rows", ctypes.c_void_p(src.at(0)), ctypes.c_void_p(dst.at(0)), rows, n, pitch, _CODES[src.dtype],
            self._stream(),
        )

    def quarter(self, A, X, K, lda, image, m_dtype, W, out, out_offset, x_inner, sx0, sx1, w_inner, sw0, sw1):
        if X <= 0:
            return
        _native.call(
            "qs_quarter_transform", ctypes.c_void_p(A.at(0)), _CODES[A.dtype], X, K, lda,
            ctypes.c_void_p(image.data_ptr()), _CODES[m_dtype], W, ctypes.c_void_p(out.at(out_offset)), x_inner, sx0,
            sx1, w_inner, sw0, sw1, self._stream(),
        )

    # symmetry-aware steps (csrc/symmetry.cu, tabulated row placement of csrc/quarter_gemm.cu)
    def index_table(self, host_int64):
        return torch.from_numpy(host_int64).cuda()

    def is_antisymmetric(self, buf, n, planes):
        flag = ctypes.c_int(1)
        scratch = torch.empty(2, dtype=torch.int32, device="cuda")
        _native.call(
            "qs_is_antisymmetric_last_pair", ctypes.c_void_p(buf.at(0)), _CODES[buf.dtype], n, planes,
            ctypes.byref(flag), ctypes.c_void_p(scratch.data_ptr()), self._stream(),
        )
        return bool(flag.value)

    def cyclic_fill(self, buf, m, planes):
        _native.call("qs_cyclic_antisymmetric_fill", ctypes.c_void_p(buf.at(0)), _CODES[buf.dtype], m, planes,
                     self._stream())

    def quarter_rows(self, A, X, K, lda, image, m_dtype, W, out, x_inner, sx0, host_table, dev_table, w_inner, sw0,
                     sw1):
        if X <= 0:
            return
        nbytes = ctypes.c_int64(0)
        _native.call("qs_quarter_tile_list_bytes", X, K, W, _CODES[A.dtype], _CODES[m_dtype], ctypes.byref(nbytes))
        lists = torch.empty(nbytes.value, dtype=torch.uint8, device="cuda")
        _native.call(
            "qs_quarter_transform_rows", ctypes.c_void_p(A.at(0)), _CODES[A.dtype], X, K, lda,
            ctypes.c_void_p(image.data_ptr()), _CODES[m_dtype], W, ctypes.c_void_p(out.at(0)), x_inner, sx0,
            ctypes.c_void_p(host_table.ctypes.data), ctypes.c_void_p(dev_table.data_ptr()), w_inner, sw0, sw1,
            ctypes.c_void_p(lists.data_ptr()), nbytes.value, self._stream(),
        )
        lists.record_stream(torch.cuda.current_stream())

    def quarter_scatter_rows(self, A, X, K, lda, image, m_dtype, W, dests, x_inner, sx1, xr_table, w_inner, sw0,
                             deal=1, tile_start=0, rows_paired=False):
        if X <= 0:
            return
        table = (ctypes.c_void_p * len(dests))(*[buf.at(off) for buf, off in dests])
        _native.call(
            "qs_quarter_transform_scatter_rows", ctypes.c_void_p(A.at(0)), _CODES[A.dtype], X, K, lda,
            ctypes.c_void_p(image.data_ptr()), _CODES[m_dtype], W, table, len(dests), x_inner, sx1,
            ctypes.c_void_p(xr_table.data_ptr()), w_inner, sw0, int(deal), int(tile_start), int(bool(rows_paired)),
            self._stream(),
        )

    def quarter_scatter_pairs(self, A, X, K, lda, image, m_dtype, W, dests, x_inner, x_mid, sx0, sx1, sx2, sw0,
                              rows_per_s, padded):
        """The first exchange of the anti-symmetric schedule: cyclic destinations, only the tiles that hold a pair
        (r, s) the cyclic pair rule wants (qs_quarter_transform_scatter_pairs)."""
        if X <= 0:
            return
        nbytes = ctypes.c_int64(0)
        _native.call("qs_quarter_tile_list_bytes", X, K, W, _CODES[A.dtype], _CODES[m_dtype], ctypes.byref(nbytes))
        lists = torch.empty(nbytes.value, dtype=torch.uint8, device="cuda")
        table = (ctypes.c_void_p * len(dests))(*[buf.at(off) for buf, off in dests])
        _native.call(
            "qs_quarter_transform_scatter_pairs", ctypes.c_void_p(A.at(0)), _CODES[A.dtype], X, K, lda,
            ctypes.c_void_p(image.data_ptr()), _CODES[m_dtype], W, table, len(dests), x_inner, max(x_mid, 1), sx0, sx1,
            sx2, sw0, rows_per_s, int(bool(padded)), ctypes.c_void_p(lists.data_ptr()), nbytes.value, self._stream(),
        )
        lists.record_stream(torch.cuda.current_stream())

    # consumers of a shard (csrc/consumers.cu)
    def extract_block(self, buf, planes, n, bounds):
        (a0, a1), (b0, b1), (c0, c1), (d0, d1) = bounds
        out = torch.empty((a1 - a0, b1 - b0, c1 - c0, d1 - d0), dtype=buf.dtype, device="cuda")
        _native.call(
            "qs_extract_block", ctypes.c_void_p(buf.at(0)), _CODES[buf.dtype], n, planes, a0, a1, b0, b1, c0, c1, d0,
            d1, ctypes.c_void_p(out.data_ptr()), self._stream(),
        )
        return out

    def scale_add(self, x, y, count, alpha, beta, out):
        alpha, beta = complex(alpha), complex(beta)
        _native.call(
            "qs_scale_add", ctypes.c_void_p(x.at(0)), ctypes.c_void_p(y.at(0) if y is not None else 0),
            _CODES[x.dtype], count, alpha.real, alpha.imag, beta.real, beta.imag, ctypes.c_void_p(out.at(0)),
            self._stream(),
        )

    def occupied_traces(self, h, buf, n, n_occ, p0, p1):
        from . import ops

        out = torch.empty(3, dtype=torch.complex128, device="cuda")
        _native.call(
            "qs_occupied_traces", ops._ptr(h), ops._code(h), ctypes.c_void_p(buf.at(0)), _CODES[buf.dtype], n,
            int(n_occ), p0, p1, ctypes.c_void_p(out.data_ptr()), self._stream(),
        )
        return out

    def quarter_scatter(self, A, X, K, lda, image, m_dtype, W, dests, x_inner, x_mid, sx0, sx1, sx2, w_inner, sw0,
                        deal=1, cyclic=False, tile_start=0):
        if X <= 0:
            return
        table = (ctypes.c_void_p * len(dests))(*[buf.at(off) for buf, off in dests])
        _native.call(
            "qs_quarter_transform_scatter", ctypes.c_void_p(A.at(0)), _CODES[A.dtype], X, K, lda,
            ctypes.c_void_p(image.data_ptr()), _CODES[m_dtype], W, table, len(dests), x_inner, max(x_mid, 1), sx0, sx1,
            sx2, max(w_inner, 1), sw0, int(deal), int(bool(cyclic)), int(tile_start), self._stream(),
        )


# ------------------------------------------------------------------------------------------------
# contexts: who drives which rank, and how ranks reach each other's memory
# ------------------------------------------------------------------------------------------------
class EmulatedContext:
    """All ``world`` ranks driven by this process on the current device (single-GPU tests)."""

    def __init__(self, world, engine=None):
        self.world = world
        self.local_ranks = list(range(world))
        self.engine = engine if engine is not None else CudaEngine()
        self.exchange = "peer"

    def shared_empty(self, numels, dtype):
        """One buffer per rank, visible to every rank.  Returns ``{rank: [buffer of rank 0, ...]}``."""
        buffers = [self.engine.empty(numels[r], dtype) for r in range(self.world)]
        return {r: buffers for r in self.local_ranks}

    def shared_cached(self, tag, numels, dtype):
        return _cached(self, tag, numels, dtype)

    def barrier(self):
        pass  # one stream, program order


class ProcessContext:
    """This process drives one rank of an initialised ``torch.distributed`` group (one process per GPU).

    ``exchange="peer"`` (default on CUDA): destination buffers are cudaMalloc blocks exported with CUDA
    IPC and opened by every peer; the GEMM epilogues store into them over NVLink.
    ``exchange="collective"``: ``all_to_all_single`` of a locally written send buffer.
    """

    def __init__(self, group=None, engine=None, exchange=None):
        import torch.distributed as dist

        if not dist.is_initialized():
            raise RuntimeError("ProcessContext needs an initialised torch.distributed process group")
        self.dist = dist
        self.group = group
        self.rank = dist.get_rank(group)
        self.world = dist.get_world_size(group)
        self.local_ranks = [self.rank]
        self.engine = engine if engine is not None else CudaEngine()
        self.on_cuda = isinstance(self.engine, CudaEngine)
        self.exchange = exchange or ("peer" if self.on_cuda else "collective")
        self._flag = None
        self._allocations = []  # (local pointer, [opened peer pointers]) for close()

    def barrier(self):
        """Stream-ordered barrier: a one-element all-reduce on the current stream (no host block)."""
        if self._flag is None:
            self._flag = torch.zeros(1, dtype=torch.float32, device="cuda" if self.on_cuda else "cpu")
        self.dist.all_reduce(self._flag, op=self.dist.ReduceOp.MAX, group=self.group)

    def shared_empty(self, numels, dtype):
        if self.exchange != "peer":
            raise RuntimeError("shared buffers exist only for exchange='peer'")
        hb = _native.load().qs_ipc_handle_bytes()
        handle = ctypes.create_string_buffer(hb)
        local = ctypes.c_void_p()
        nbytes = max(int(numels[self.rank]), 1) * _ITEMSIZE[dtype]
        _native.call("qs_ipc_alloc", nbytes, ctypes.byref(local), handle)
        handles = [None] * self.world
        self.dist.all_gather_object(handles, handle.raw, group=self.group)
        buffers, opened = [], []
        for r in range(self.world):
            if r == self.rank:
                buffers.append(DeviceBuffer(local.value, numels[r], dtype))
            else:
                peer = ctypes.c_void_p()
                _native.call("qs_ipc_open", ctypes.c_char_p(handles[r]), ctypes.byref(peer))
                opened.append(peer.value)
                buffers.append(DeviceBuffer(peer.value, numels[r], dtype))
        self._allocations.append((local.value, opened))
        return {self.rank: buffers}

    def shared_cached(self, tag, numels, dtype):
        """Peer-visible scratch that persists across calls (the IPC rendezvous is paid once)."""
        return _cached(self, tag, numels, dtype)

    def close(self):
        """Unmap the peers' buffers and free the local ones (collective: every rank must call it)."""
        if self.on_cuda:
            torch.cuda.synchronize()
        self.barrier()
        for local, opened in self._allocations:
            for ptr in opened:
                _native.call("qs_ipc_close", ctypes.c_void_p(ptr))
        if self.on_cuda:
            torch.cuda.synchronize()
        self.barrier()
        if self.on_cuda:
            torch.cuda.synchronize()
        for local, _ in self._allocations:
            _native.call("qs_ipc_free", ctypes.c_void_p(local))
        self._allocations = []

    # collective exchange (validation path)
    def all_to_all(self, send, send_splits, recv, recv_splits):
        """``all_to_all_single`` on flat float64 views (complex buffers are pairs of doubles)."""
        s, r = send.as_tensor(), recv.as_tensor()
        scale = 1
        if s.is_complex():
            s, r = torch.view_as_real(s).reshape(-1), torch.view_as_real(r).reshape(-1)
            scale = 2
        self.dist.all_to_all_single(
            r[: scale * sum(recv_splits)], s[: scale * sum(send_splits)], [scale * x for x in recv_splits],
            [scale * x for x in send_splits], group=self.group,
        )


def _owners(ctx):
    return ctx.__dict__.setdefault("_buffer_owners", {})


def _recycle(ctx, buffers, keep=None):
    """``buffers`` are about to be overwritten: the handle that still points at them (if any, and unless it is
    ``keep``) becomes invalid instead of silently showing the new contents."""
    ref = _owners(ctx).pop(id(buffers), None)
    old = ref() if ref is not None else None
    if old is not None and old is not keep:
        old._buffers = None


def _cached(ctx, tag, numels, dtype):
    cache = ctx.__dict__.setdefault("_shared_cache", {})
    key = (tag, tuple(int(x) for x in numels), dtype)
    if key not in cache:
        cache[key] = ctx.shared_empty(numels, dtype)
    return cache[key]


# ------------------------------------------------------------------------------------------------
# the sharded tensor handle
# ------------------------------------------------------------------------------------------------
class ShardedTwoBody:
    """``u`` of shape ``(n, n, n, n)`` block-partitioned on its leading index.

    ``local[r]`` is rank r's ``(planes_r, n, n, n)`` slab (only the ranks this process drives).  The
    slabs live in peer-visible buffers; ``spare`` is the second set the next transform writes into
    (ping-pong: a transform recycles the buffers of the tensor it replaced one call earlier).
    """

    def __init__(self, ctx, n, dtype, buffers, spare=None):
        self.ctx = ctx
        self.n = n
        self.dtype = dtype
        self._buffers = buffers  # {rank: [buffer of every rank]}
        self.spare = spare
        self.block, self.offsets = block_partition(n, ctx.world)
        self.proven_antisymmetric = False
        # who currently owns a buffer set: a transform that recycles the set invalidates that handle
        _owners(ctx)[id(buffers)] = weakref.ref(self)

    def _slab_versions(self):
        # as_tensor() is cached per buffer, so every local() view shares its tensor's version counter
        return tuple(self._buffers[r][r].as_tensor()._version for r in self.ctx.local_ranks)

    @property
    def proven_antisymmetric(self):
        """True once the library itself has made the slabs of THIS process EXACTLY anti-symmetric in their last pair
        (fused spin doubling, cyclic mirror fill): the transform then skips the device-side read of them.  Setting it
        stamps the version counters of the local slabs; any write through torch into ``local()`` (or through an
        ``ops`` entry point with ``out=local()``) bumps a counter and voids the proof, reads keep it.  Writes that
        bypass torch (raw pointers) are not seen.  The proof is local: with one process per rank, a write on some ranks
        voids it on those ranks only, so the transform combines the ranks' answers in one all-reduce
        (``is_antisymmetric_last_pair(trust_proof=True)``) and every rank takes the same schedule."""
        return self._proof is not None and self._buffers is not None and self._proof == self._slab_versions()

    @proven_antisymmetric.setter
    def proven_antisymmetric(self, value):
        self._proof = self._slab_versions() if value else None

    @property
    def buffers(self):
        """The peer-visible slabs.  Raises once a later transform has recycled them (the reference's
        ``change_basis`` returns fresh arrays; here a tensor replaced TWO calls earlier donates its memory --
        ``copy()`` keeps an old tensor alive)."""
        if self._buffers is None:
            raise RuntimeError(
                "this ShardedTwoBody was recycled: a later change_basis wrote its result into these buffers "
                "(ping-pong); take .copy() before the second transform to keep an old tensor"
            )
        return self._buffers

    @property
    def shape(self):
        return (self.n,) * 4

    def planes(self, rank):
        return self.offsets[rank], self.offsets[rank + 1]

    def local(self, rank=None):
        rank = self.ctx.local_ranks[0] if rank is None else rank
        p0, p1 = self.planes(rank)
        n = self.n
        flat = self.buffers[rank][rank].as_tensor()
        return flat[: (p1 - p0) * n**3].view(p1 - p0, n, n, n)

    @classmethod
    def empty(cls, ctx, n, dtype, with_spare=True):
        _, offsets = block_partition(n, ctx.world)
        numels = [(offsets[r + 1] - offsets[r]) * n**3 for r in range(ctx.world)]
        if ctx.exchange == "peer":
            buffers = ctx.shared_empty(numels, dtype)
            spare = ctx.shared_empty(numels, dtype) if with_spare else None
        else:
            buffers = {r: {r: ctx.engine.empty(numels[r], dtype)} for r in ctx.local_ranks}
            spare = None
        return cls(ctx, n, dtype, buffers, spare)

    def gather(self):
        """The full tensor on every rank (small n only: tests, inspection)."""
        ctx = self.ctx
        if isinstance(ctx, EmulatedContext):
            return torch.cat([self.local(r) for r in range(ctx.world)], dim=0)
        local = self.local()
        n = self.n
        padded = torch.zeros((self.block, n, n, n), dtype=local.dtype, device=local.device)
        padded[: local.shape[0]] = local
        parts = [torch.empty_like(padded) for _ in range(ctx.world)]  # equal sizes: short trailing blocks are padded
        if padded.is_complex():
            ctx.dist.all_gather([torch.view_as_real(p) for p in parts], torch.view_as_real(padded), group=ctx.group)
        else:
            ctx.dist.all_gather(parts, padded, group=ctx.group)
        parts = [parts[r][: self.offsets[r + 1] - self.offsets[r]] for r in range(ctx.world)]
        return torch.cat(parts, dim=0)


    # -------------------------------------------------------------- consumers (SURVEY.md section 8f-3)
    def _bounds(self, a, b, c, d):
        from .ops import _bounds

        n = self.n
        return _bounds(a, n), _bounds(b, n), _bounds(c, n), _bounds(d, n)

    def extract(self, a=None, b=None, c=None, d=None):
        """Dense ``u[a, b, c, d]`` (unit-step slices), replicated on every rank -- the ``u[o, o, v, v]``
        blocks of the solvers.  Each rank cuts its own planes out of its shard (``qs_extract_block``);
        the pieces are all-gathered (the only communication: the block itself)."""
        ctx = self.ctx
        (a0, a1), *rest = self._bounds(a, b, c, d)
        rest = tuple(rest)
        pieces = {}
        for r in ctx.local_ranks:
            p0, p1 = self.planes(r)
            lo, hi = min(max(a0, p0), p1), max(min(a1, p1), p0)
            hi = max(hi, lo)
            pieces[r] = ctx.engine.extract_block(self.buffers[r][r], p1 - p0, self.n, ((lo - p0, hi - p0),) + rest)
        if isinstance(ctx, EmulatedContext):
            return torch.cat([pieces[r] for r in range(ctx.world)], dim=0)
        piece = pieces[ctx.rank]
        padded = torch.zeros((self.block,) + tuple(piece.shape[1:]), dtype=piece.dtype, device=piece.device)
        padded[: piece.shape[0]] = piece
        parts = [torch.empty_like(padded) for _ in range(ctx.world)]
        if padded.is_complex():
            ctx.dist.all_gather([torch.view_as_real(p) for p in parts], torch.view_as_real(padded), group=ctx.group)
        else:
            ctx.dist.all_gather(parts, padded, group=ctx.group)
        rows = []
        for r in range(ctx.world):
            p0, p1 = self.planes(r)
            rows.append(parts[r][: max(min(a1, p1) - max(a0, p0), 0)])
        return torch.cat(rows, dim=0)

    def axpby_(self, alpha, other=None, beta=0.0):
        """In place ``u <- alpha u + beta other`` on every shard (``other`` sharded alike); no communication.
        ``u_t = f(t) u`` of an adiabatic switching is ``axpby_(f(t))`` on a copy."""
        if other is not None and (other.n != self.n or other.dtype != self.dtype):
            raise ValueError("operands must share extent and dtype")
        alpha, beta = complex(alpha), complex(beta)
        if self.dtype != torch.complex128 and (alpha.imag != 0 or beta.imag != 0):
            raise TypeError("complex factor on a real sharded tensor")
        for r in self.ctx.local_ranks:
            p0, p1 = self.planes(r)
            count = (p1 - p0) * self.n**3
            if count:
                mine = self.buffers[r][r]
                self.ctx.engine.scale_add(mine, other.buffers[r][r] if other is not None else None, count, alpha, beta,
                                          mine)
        self.proven_antisymmetric = self.proven_antisymmetric and (other is None or other.proven_antisymmetric)
        return self

    def successor(self):
        """A handle over this tensor's SPARE buffers whose own spare is this tensor's memory, for a caller that is
        done with this tensor and wants to build the next one in place (``from_spatial_planes(..., into=...)`` of
        the next spatial tensor) without new peer allocations.  This handle stays valid until a transform of the
        successor recycles its buffers."""
        if self.spare is None:
            raise RuntimeError("this ShardedTwoBody has no spare buffer set")
        _recycle(self.ctx, self.spare, keep=self)
        return ShardedTwoBody(self.ctx, self.n, self.dtype, self.spare, self.buffers)

    def scaled(self, alpha, other=None, beta=0.0):
        """A NEW sharded tensor ``alpha u + beta other`` in one pass per shard (``qs_scale_add``), no
        communication: ``u_t = u_0 + f(t) u`` of reference system.py:203-215 / operator.py:182-196."""
        if other is not None and (other.n != self.n or other.dtype != self.dtype):
            raise ValueError("operands must share extent and dtype")
        alpha, beta = complex(alpha), complex(beta)
        if self.dtype != torch.complex128 and (alpha.imag != 0 or beta.imag != 0):
            raise TypeError("complex factor on a real sharded tensor")
        new = ShardedTwoBody.empty(self.ctx, self.n, self.dtype, with_spare=False)
        for r in self.ctx.local_ranks:
            p0, p1 = self.planes(r)
            count = (p1 - p0) * self.n**3
            if count:
                self.ctx.engine.scale_add(self.buffers[r][r], other.buffers[r][r] if other is not None else None,
                                          count, alpha, beta, new.buffers[r][r])
        self.ctx.barrier()
        new.proven_antisymmetric = self.proven_antisymmetric and (other is None or other.proven_antisymmetric)
        return new

    def copy(self):
        """A new sharded tensor (own buffers, no spare) with the same contents."""
        new = ShardedTwoBody.empty(self.ctx, self.n, self.dtype, with_spare=False)
        for r in self.ctx.local_ranks:
            p0, p1 = self.planes(r)
            count = (p1 - p0) * self.n**3
            if count:
                self.ctx.engine.scale_add(self.buffers[r][r], None, count, 1.0, 0.0, new.buffers[r][r])
        self.ctx.barrier()
        new.proven_antisymmetric = self.proven_antisymmetric
        return new

    def occupied_traces(self, h, n_occ):
        """``(tr h[o,o], sum_ij u[i,j,i,j], sum_ij u[i,j,j,i])`` as Python complex numbers: every rank reduces
        the occupied rows it owns, then a 6-double all-reduce."""
        ctx = self.ctx
        total = None
        for r in ctx.local_ranks:
            p0, p1 = self.planes(r)
            part = ctx.engine.occupied_traces(h, self.buffers[r][r], self.n, n_occ, p0, p1)  # rows [p0, p1) only
            total = part if total is None else total + part
        if isinstance(ctx, ProcessContext) and ctx.world > 1:
            ctx.dist.all_reduce(torch.view_as_real(total), group=ctx.group)
        return tuple(complex(x) for x in total.cpu().tolist())


# ------------------------------------------------------------------------------------------------
# one rank's share of a sharded four-index transform
# ------------------------------------------------------------------------------------------------
class _RankTransform:
    """One rank's share of a sharded four-index transform.

    Where the tiles land (peer schedule).  Eight ranks that each fill ONE OF EIGHT ADJACENT CHUNKS of a block in a
    destination's memory at the same time get position-dependent NVLink throughput: at n = 192 on 8 B200s the ranks
    writing the outermost chunks needed 2.9 ms for a scattering step, the middle ones 2.2 ms, and the slow ranks
    followed the chunk position when it was rotated, not the physical GPU (profiles/r02g_*, r02h_*).  With streams
    that are far apart or interleaved row by row every rank needs 2.04 ms (profiles/r02i_*).  Hence

    * the intermediate index r is dealt to the ranks CYCLICALLY (rank j owns r = j, j + W, ...): in the final
      store u'[p_loc, q, r, s] a rank's rows interleave with the other ranks' rows inside every (r, s) block, and
      in the first exchange consecutive columns go to different destinations by themselves;
    * the received half-transformed tensor is kept SOURCE-MAJOR, ``T2[src][r_loc][s][a_loc][b]``: each source
      writes one contiguous region of the destination instead of a chunk of every (a, b) block.

    Both are internal: the input stays block-partitioned on its leading index a, the result on p.  The collective
    schedule (validation path) keeps the block partition of r.
    """

    def __init__(self, ctx, rank, n, m, u_dtype, c_dtype):
        self.ctx, self.rank, self.n, self.m = ctx, rank, n, m
        self.engine = ctx.engine
        self.u_dtype, self.c_dtype = u_dtype, c_dtype
        self.t_dtype = torch.complex128 if torch.complex128 in (u_dtype, c_dtype) else torch.float64
        self.a_block, self.a_off = block_partition(n, ctx.world)  # partition of the old leading index
        self.r_block, self.r_off = block_partition(m, ctx.world)  # partition of the new leading index p (and of r
        #                                                           in the collective schedule)
        self.cyclic = ctx.exchange == "peer" and SCATTER_LAYOUT == "source_major"  # r dealt cyclically
        self.tile_start = (rank * 65536) // ctx.world if (ROTATE_TILES and ctx.exchange == "peer") else 0
        self.Pu = padded_pitch(n, u_dtype)
        self.P = padded_pitch(n, self.t_dtype)
        self.A = self.a_off[rank + 1] - self.a_off[rank]
        self.R = self.r_count(rank)
        # every source holds the same number of planes: step 3 reads the source-major T2 in one launch
        self.even_sources = all(self.a_off[j + 1] - self.a_off[j] == self.A for j in range(ctx.world))

    def r_count(self, rank):
        """Number of intermediate indices r that `rank` owns."""
        if self.cyclic:
            return len(range(rank, self.m, self.ctx.world))
        return self.r_off[rank + 1] - self.r_off[rank]

    def r_values(self):
        """The intermediate indices r of this rank, in the order of its local index r_loc."""
        import numpy

        if self.cyclic:
            return numpy.arange(self.rank, self.m, self.ctx.world, dtype=numpy.int64)
        return self.r_off[self.rank] + numpy.arange(self.R, dtype=numpy.int64)

    # sizes (elements of t_dtype unless noted)
    def recv_numel(self, rank):
        return self.r_count(rank) * self.m * self.n * self.P

    def out_numel(self, rank):
        return (self.r_off[rank + 1] - self.r_off[rank]) * self.m**3

    def scratch_numel(self):
        return max(self.m * self.A * self.n * self.P, self.m * self.R * self.m * self.P, 1)

    def prepare(self, C, C_tilde):
        eng, n, m = self.engine, self.n, self.m
        self.img1 = eng.image(C, n, m, self.u_dtype, m, 1)
        self.img2 = eng.image(C, n, m, self.t_dtype, m, 1)
        if C_tilde is not None:
            self.img3 = eng.image(C_tilde, n, m, self.t_dtype, 1, n)
        else:
            self.img3 = eng.image(C, n, m, self.t_dtype, m, 1, conj=True)  # C~ = C^dagger, basis_set.py:338-339
        # The last step scatters BLOCKS of the new leading index p (the result is block-partitioned), so it deals
        # its output columns over all destinations (uniform NVLink traffic): its image holds the columns of C~ in
        # dealt order.  The first exchange sends cyclic columns and needs no dealing.
        self.deal = eng.scatter_deal(m) if self.ctx.exchange == "peer" and self.ctx.world > 1 else 1
        self.img2_scatter = self.img2
        if self.deal > 1 and not self.cyclic:  # block partition of r: the first exchange deals its columns too
            self.img2_scatter = eng.image(C, n, m, self.t_dtype, m, 1, deal=self.deal)
        if self.deal > 1:
            if C_tilde is not None:
                self.img4_scatter = eng.image(C_tilde, n, m, self.t_dtype, 1, n, deal=self.deal)
            else:
                self.img4_scatter = eng.image(C, n, m, self.t_dtype, m, 1, conj=True, deal=self.deal)
        else:
            self.img4_scatter = self.img3
        self.scratch = eng.empty(self.scratch_numel(), self.t_dtype)

    def step1(self, u_in):
        """T1[s, a_loc, b, c] = sum_d u[a_loc, b, c, d] C[d, s]  (new index slowest, c at pitch P)."""
        eng, n, m, A, P = self.engine, self.n, self.m, self.A, self.P
        if A == 0:
            return
        src = u_in
        if self.Pu != n:
            padded = eng.empty(A * n * n * self.Pu, self.u_dtype)
            eng.pad_rows(u_in, A * n * n, n, self.Pu, padded)
            src = padded
        eng.quarter(src, A * n * n, n, self.Pu, self.img1, self.c_dtype, m, self.scratch, 0, n, 1, P, 1, 0, A * n * P)

    def step2_scatter(self, recv, pairs_only=False):
        """T2[r, s, a, b] = sum_c T1[s, a_loc, b, c] C[c, r], stored into the rank that owns r (cyclic: r % W) at
        [src = this rank][r_loc = r // W][s][a_loc][b] (b at pitch P): the a -> r re-partition rides on the epilogue,
        and this rank's tiles fill ONE contiguous region of every destination.  ``pairs_only`` (anti-symmetric u):
        only the tiles that hold a pair (r, s) which steps 3 and 4 will use are computed and sent."""
        eng, n, m, A, P = self.engine, self.n, self.m, self.A, self.P
        a0 = self.a_off[self.rank]
        if not self.cyclic:  # interleaved layout: [r_loc][s][a][b], this rank's planes between the others'
            dests = [(recv[j], a0 * P) for j in range(self.ctx.world)]
            eng.quarter_scatter(self.scratch, m * A * n, n, P, self.img2_scatter, self.c_dtype, m, dests, n, A, 1, P,
                                n * P, self.r_block, m * n * P, deal=self.deal, tile_start=self.tile_start)
            return
        # region of this source in destination j: behind the regions of the sources before it
        dests = [(recv[j], a0 * self.r_count(j) * m * P) for j in range(self.ctx.world)]
        if pairs_only and MASK_FIRST_EXCHANGE and not self.tile_start:
            # the tiles sent here must cover the pairs of the (cached) tables steps 3 and 4 read
            self.prepare_pairs()
            assert self.rows_paired == self.pairs_padded(), "cached pair tables of another T2 dtype"
            eng.quarter_scatter_pairs(self.scratch, m * A * n, n, P, self.img2, self.c_dtype, m, dests, n, A, 1, P,
                                      A * P, m * A * P, A * n, self.rows_paired)
            return
        eng.quarter_scatter(self.scratch, m * A * n, n, P, self.img2, self.c_dtype, m, dests, n, A, 1, P, A * P,
                            0, m * A * P, deal=1, cyclic=True, tile_start=self.tile_start)

    def step2_local(self, send):
        """Collective schedule: T2[r, s, a_loc, b] written locally, blocks of r contiguous per destination."""
        eng, n, m, A, P = self.engine, self.n, self.m, self.A, self.P
        eng.quarter(self.scratch, m * A * n, n, P, self.img2, self.c_dtype, m, send, 0, n, 1, P, 1, 0, m * A * P)

    def step3(self, recv_local):
        """T3[q, r_loc, s, a] = sum_b T2[src][r_loc][s][a_loc][b] C~[q, b]: the rows arrive source-major and are
        stored with a = a_off[src] + a_loc.  One launch when every source holds the same number of planes (three-level
        row split through the single-destination form of the scattering store), else one launch per source."""
        eng, n, m, R, P = self.engine, self.n, self.m, self.R, self.P
        if R == 0:
            return
        if not self.cyclic:  # interleaved layout: rows (r_loc, s, a) in place
            eng.quarter(recv_local, R * m * n, n, P, self.img3, self.c_dtype, m, self.scratch, 0, n, 1, P, 1, 0, R * m * P)
        elif self.even_sources:
            eng.quarter_scatter(recv_local, R * m * n, n, P, self.img3, self.c_dtype, m, [(self.scratch, 0)], self.A,
                                R * m, 1, P, self.A, m, R * m * P, deal=1)
        else:
            self.step3_blocked(recv_local)

    def step3_blocked(self, recv_blocks):
        """The received buffer is [src][r_loc][s][a_loc(src)][b]; one launch per source drops its planes between the
        others' (a at pitch P in T3).  Also the collective schedule's step 3."""
        eng, n, m, R, P = self.engine, self.n, self.m, self.R, self.P
        offset = 0
        for src in range(self.ctx.world):
            A_src = self.a_off[src + 1] - self.a_off[src]
            if A_src == 0 or R == 0:
                continue
            block = _slice(recv_blocks, offset, R * m * A_src * P)
            eng.quarter(block, R * m * A_src, n, P, self.img3, self.c_dtype, m, self.scratch, self.a_off[src], A_src,
                        1, P, 1, 0, R * m * P)
            offset += R * m * A_src * P

    def step4_scatter(self, out):
        """u'[p, q, r, s] = sum_a T3[q, r_loc, s, a] C~[p, a], stored into the rank that owns p at
        [p_loc][q][r][s]: the result is sharded on its leading index again.  r = rank + W r_loc: this rank's rows
        of every (r, s) block interleave with the other ranks' rows."""
        eng, n, m, R, P, W = self.engine, self.n, self.m, self.R, self.P, self.ctx.world
        if not self.cyclic:  # block partition of r: this rank's rows are one chunk of every (r, s) block
            dests = [(out[j], self.r_off[self.rank] * m) for j in range(W)]
            eng.quarter_scatter(self.scratch, m * R * m, n, P, self.img4_scatter, self.c_dtype, m, dests, m, R, 1, m,
                                m * m, self.r_block, m**3, deal=self.deal, tile_start=self.tile_start)
            return
        dests = [(out[j], self.rank * m) for j in range(W)]
        eng.quarter_scatter(self.scratch, m * R * m, n, P, self.img4_scatter, self.c_dtype, m, dests, m, R, 1, W * m,
                            m * m, self.r_block, m**3, deal=self.deal, tile_start=self.tile_start)

    # ---- anti-symmetric u: steps 3 and 4 on half of the (r, s) pairs (cyclic rule), packed by pair -------------
    def pairs_padded(self):
        """Real tensors with an even extent pad the pair lists to aligned couples (s even, s + 1), see prepare_pairs."""
        return self.t_dtype == torch.float64 and self.m % 2 == 0

    def prepare_pairs(self):
        """Pair tables of this rank: for every owned r the partners s the cyclic-distance rule assigns to (r, s)."""
        import numpy

        m, R, P, W = self.m, self.R, self.P, self.ctx.world
        # built and uploaded once per (rank, n, m, world, P, dtype of T2), then reused by every transform; the dtype
        # decides whether the lists are padded to aligned couples (pairs_padded)
        cache = self.ctx.__dict__.setdefault("_pair_tables", {})
        key = (self.rank, self.n, m, W, P, self.cyclic, self.t_dtype)
        if key in cache:
            (self.npairs, self.step3_tables, self.rs_of_pair, self.rs_of_pair_dev, self.rows_paired) = cache[key]
            return
        r = self.r_values()[:, None]
        sI = numpy.arange(m, dtype=numpy.int64)[None, :]
        wanted = cyclic_wanted(r, sI, m)
        # Real tensors with an even extent: complete every aligned couple (s even, s + 1) that holds a wanted partner.
        # The extra element of a couple -- (r, r), or a pair whose mirror image the owner of s computes anyway -- is
        # overwritten by the cyclic fill afterwards; rows 2k and 2k + 1 of step 4 are then neighbours in the result
        # and cross NVLink as 16-byte stores forming whole lines instead of scattered 8-byte ones.
        self.rows_paired = self.pairs_padded()
        if self.rows_paired:
            wanted = wanted | wanted[:, sI[0] ^ 1]
        self.npairs = int(wanted.sum())
        slot = numpy.full((R, m), -1, dtype=numpy.int64)
        slot[wanted] = numpy.arange(self.npairs, dtype=numpy.int64) * P  # row-major (r_loc, s) order
        self.rs_of_pair = numpy.ascontiguousarray((r * m + sI)[wanted])
        self.rs_of_pair_dev = self.engine.index_table(self.rs_of_pair) if self.npairs else None
        # step 3 reads the source-major T2: rows (src, r_loc, s, a_loc) -> T3p[q, pair(r_loc, s), a_off[src] + a_loc]
        self.step3_tables = []
        if self.npairs:
            if not self.cyclic:  # interleaved layout: rows (r_loc, s, a), blocks of n rows
                table = numpy.ascontiguousarray(slot.reshape(-1))
                self.step3_tables = [("interleaved", table, self.engine.index_table(table))]
            elif self.even_sources:
                per_source = [slot.reshape(-1) + numpy.where(slot.reshape(-1) >= 0, self.a_off[src], 0)
                              for src in range(W)]
                table = numpy.ascontiguousarray(numpy.concatenate(per_source))
                self.step3_tables = [(None, table, self.engine.index_table(table))]
            else:
                for src in range(W):
                    if self.a_off[src + 1] > self.a_off[src]:
                        table = numpy.ascontiguousarray(slot.reshape(-1) + numpy.where(slot.reshape(-1) >= 0, self.a_off[src], 0))
                        self.step3_tables.append((src, table, self.engine.index_table(table)))
        cache[key] = (self.npairs, self.step3_tables, self.rs_of_pair, self.rs_of_pair_dev, self.rows_paired)

    def step3_pairs(self, recv_local):
        """T3p[q, pair(r_loc, s), a] = sum_b T2[src][r_loc][s][a_loc][b] C~[q, b] for the wanted pairs only."""
        eng, n, m, R, P = self.engine, self.n, self.m, self.R, self.P
        if self.npairs == 0:
            return
        for src, host_table, dev_table in self.step3_tables:
            if src == "interleaved":
                eng.quarter_rows(recv_local, R * m * n, n, P, self.img3, self.c_dtype, m, self.scratch, n, 1,
                                 host_table, dev_table, 1, 0, self.npairs * P)
            elif src is None:  # all sources in one launch: blocks of A rows, table over (src, r_loc, s)
                eng.quarter_rows(recv_local, R * m * n, n, P, self.img3, self.c_dtype, m, self.scratch, self.A, 1,
                                 host_table, dev_table, 1, 0, self.npairs * P)
            else:
                A_src = self.a_off[src + 1] - self.a_off[src]
                block = _slice(recv_local, self.a_off[src] * R * m * P, R * m * A_src * P)
                eng.quarter_rows(block, R * m * A_src, n, P, self.img3, self.c_dtype, m, self.scratch, A_src, 1,
                                 host_table, dev_table, 1, 0, self.npairs * P)

    def step4_scatter_pairs(self, out):
        """u'[p, q, r, s] = sum_a T3p[q, pair, a] C~[p, a] for the wanted pairs, stored into the rank that owns p."""
        eng, n, m, P = self.engine, self.n, self.m, self.P
        if self.npairs == 0:
            return
        dests = [(out[j], 0) for j in range(self.ctx.world)]
        eng.quarter_scatter_rows(self.scratch, m * self.npairs, n, P, self.img4_scatter, self.c_dtype, m, dests,
                                 self.npairs, m * m, self.rs_of_pair_dev, self.r_block, m**3, deal=self.deal,
                                 tile_start=self.tile_start, rows_paired=self.rows_paired)

    def step4_local(self, out_local):
        """Collective schedule: u'[p, q, r_loc, s] dense on this rank (sharded on the third index)."""
        eng, n, m, R, P = self.engine, self.n, self.m, self.R, self.P
        eng.quarter(self.scratch, m * R * m, n, P, self.img3, self.c_dtype, m, out_local, 0, m * R * m, 1, 0, 1, 0,
                    m * R * m)


def _slice(buf, offset, numel):
    if isinstance(buf, DeviceBuffer):
        return DeviceBuffer(buf.at(offset), numel, buf.dtype)
    return buf.slice(offset, numel)


def is_antisymmetric_last_pair(u, trust_proof=False):
    """Exact, collective test of ``u[p,q,r,s] == -u[p,q,s,r]`` on a ``ShardedTwoBody``: every rank tests its own
    planes on the device (``qs_is_antisymmetric_last_pair``), the flags are combined with a one-element all-reduce.
    ``trust_proof``: a process whose slabs carry the library's proof (``proven_antisymmetric``) skips the read of its
    planes but still takes part in the all-reduce, so every rank returns the same answer after the same collectives."""
    ctx = u.ctx
    ok = trust_proof and u.proven_antisymmetric
    if not ok:
        ok = True
        for r in ctx.local_ranks:
            p0, p1 = u.planes(r)
            ok = ok and ctx.engine.is_antisymmetric(u.buffers[r][r], u.n, p1 - p0)
    if isinstance(ctx, ProcessContext) and ctx.world > 1:
        flag = torch.tensor([1.0 if ok else 0.0], dtype=torch.float32, device="cuda" if ctx.on_cuda else "cpu")
        ctx.dist.all_reduce(flag, op=ctx.dist.ReduceOp.MIN, group=ctx.group)
        ok = bool(flag.item() > 0.5)
    return ok


def transform_two_body_sharded(u, C, C_tilde=None, symmetry=None):
    """Four-index transform of a ``ShardedTwoBody``; returns a new handle sharded on the leading index.

    Same contraction order (s, r, q, p) and operands as the single-GPU ``ops.transform_two_body``
    (reference basis_set.py:336-350).  Rectangular ``C`` (n, m) changes the extent; ``C_tilde`` (m, n)
    defaults to ``C^dagger``.

    ``symmetry=None``: in the peer schedule an exactly anti-symmetric ``u`` (``u_pqrs = -u_pqsr``, tested on the
    device) runs steps 3 and 4 on half of the (r, s) pairs -- of (r, s) and (s, r) the rank owning r computes the
    one at the shorter cyclic distance, so the ranks stay balanced -- and every rank completes its own planes with
    the mirror image (no extra communication).  ``symmetry=0`` forces the four full steps.
    """
    ctx = u.ctx
    n, m = C.shape
    if n != u.n:
        raise ValueError(f"C has {n} rows but u has {u.n} orbitals")
    if symmetry is None:
        symmetry = 1 if (EXPLOIT_SYMMETRY and ctx.exchange == "peer" and min(n, m) >= SYMMETRY_MIN_N
                         and is_antisymmetric_last_pair(u, trust_proof=True)) else 0
    if symmetry and ctx.exchange != "peer":
        raise ValueError("the symmetry-aware sharded transform needs the peer exchange")
    work = {r: _RankTransform(ctx, r, n, m, u.dtype, C.dtype) for r in ctx.local_ranks}
    t_dtype = next(iter(work.values())).t_dtype
    for w in work.values():
        w.prepare(C, C_tilde)
    any_w = next(iter(work.values()))

    if ctx.exchange == "peer":
        recv = ctx.shared_cached("recv", [any_w.recv_numel(r) for r in range(ctx.world)], t_dtype)
        out_numels = [any_w.out_numel(r) for r in range(ctx.world)]
        if u.spare is not None and u.dtype == t_dtype and m == n:
            out = u.spare  # ping-pong: reuse the buffers of the tensor replaced one call earlier
            _recycle(ctx, out, keep=u)  # a caller still holding that older tensor gets an error, not new data
        else:
            out = ctx.shared_empty(out_numels, t_dtype)
        ctx.barrier()  # every rank is done with whatever it last read from these buffers
        for r, w in work.items():
            w.step1(u.buffers[r][r])
            w.step2_scatter(recv[r], pairs_only=bool(symmetry))
        ctx.barrier()  # all tiles of T2 have landed
        for r, w in work.items():
            if symmetry:
                w.prepare_pairs()
                w.step3_pairs(recv[r][r])
                w.step4_scatter_pairs(out[r])
            else:
                w.step3(recv[r][r])
                w.step4_scatter(out[r])
        ctx.barrier()  # all tiles of u' have landed
        if symmetry:
            for r, w in work.items():
                # the other half of every local plane p: -u'[p,q,s,r]
                ctx.engine.cyclic_fill(out[r][r], m, w.r_off[r + 1] - w.r_off[r])
        spare = u.buffers if (u.dtype == t_dtype and m == n) else None
        result = ShardedTwoBody(ctx, m, t_dtype, out, spare)
        result.proven_antisymmetric = bool(symmetry)  # the cyclic fill wrote exact negatives and a zero diagonal
        return result

    # collective schedule (one rank per process)
    (r, w), = work.items()
    eng, P = ctx.engine, w.P
    send = eng.empty(m * m * w.A * P, t_dtype)
    recv = eng.empty(w.R * m * n * P, t_dtype)
    w.step1(u.buffers[r][r])
    w.step2_local(send)
    send_splits = [(w.r_off[j + 1] - w.r_off[j]) * m * w.A * P for j in range(ctx.world)]
    recv_splits = [w.R * m * (w.a_off[k + 1] - w.a_off[k]) * P for k in range(ctx.world)]
    ctx.all_to_all(send, send_splits, recv, recv_splits)
    w.step3_blocked(recv)
    out_local = eng.empty(m * w.R * m * m, t_dtype)  # u'[p, q, r_loc, s]
    w.step4_local(out_local)
    # r -> p re-partition: send [p in P_j][q][r_loc][s], receive [p_loc][q][r_loc(k)][s] from every k
    send_splits = [(w.r_off[j + 1] - w.r_off[j]) * m * w.R * m for j in range(ctx.world)]
    recv_splits = [w.R * m * (w.r_off[k + 1] - w.r_off[k]) * m for k in range(ctx.world)]
    staged = eng.empty(sum(recv_splits), t_dtype)
    ctx.all_to_all(out_local, send_splits, staged, recv_splits)
    result = ShardedTwoBody(ctx, m, t_dtype, {r: {r: eng.empty(w.R * m**3, t_dtype)}})
    dense = result.local(r)
    offset = 0
    for k in range(ctx.world):
        Rk = w.r_off[k + 1] - w.r_off[k]
        block = staged.as_tensor()[offset : offset + recv_splits[k]].view(w.R, m, Rk, m)
        dense[:, :, w.r_off[k] : w.r_off[k + 1], :] = block  # data movement only
        offset += recv_splits[k]
    return result


def odqd_spatial_planes(C, inner_grid, alpha=1.0, a=0.25):
    """Plane builder for :meth:`ShardedBasisSet.from_spatial_planes`: the shielded-Coulomb elements of a 1-D
    quantum dot (reference one_dim_qd.py:275-280) for leading-index planes ``[p0, p1)`` only -- ``C`` (G', l) and
    the interior grid are replicated, each rank runs the two DMMA GEMMs for its own rows of ``T = D W``."""
    from . import _arrays, ops

    C_dev, grid_dev = _arrays.to_device(C), _arrays.to_device(inner_grid)
    return lambda p0, p1: ops.odqd_coulomb(C_dev, grid_dev, alpha, a, planes=(p0, p1))


# ------------------------------------------------------------------------------------------------
# the reference-facing container, sharded
# ------------------------------------------------------------------------------------------------
class ShardedBasisSet:
    """``h``, ``s`` replicated on every rank, ``u`` a ``ShardedTwoBody``.

    Mirrors the part of ``BasisSet`` that the hot path needs at multi-GPU scale: ``change_basis``
    (reference basis_set.py:413-464), spin doubling fused with anti-symmetrisation
    (:530-636, :772-778) and the general Fock matrix (general_orbital_system.py:119-159).
    """

    def __init__(self, ctx, l, h, s, u, includes_spin=False, anti_symmetrized_u=False):
        self.ctx = ctx
        self.l = l
        self.h = h
        self.s = s
        self.u = u
        self.includes_spin = includes_spin
        self.anti_symmetrized_u = anti_symmetrized_u

    @classmethod
    def from_slabs(cls, ctx, n, h, s, slab_fn, dtype=torch.float64, **flags):
        """``slab_fn(p0, p1)`` returns this rank's ``(p1 - p0, n, n, n)`` planes (host or device array)."""
        eng = ctx.engine
        u = ShardedTwoBody.empty(ctx, n, dtype)
        for r in ctx.local_ranks:
            p0, p1 = u.planes(r)
            if p1 > p0:
                u.local(r).copy_(eng.asarray(slab_fn(p0, p1), dtype), non_blocking=True)
        ctx.barrier()
        return cls(ctx, n, eng.asarray(h), eng.asarray(s) if s is not None else None, u, **flags)

    @classmethod
    def from_global(cls, ctx, h, s, u, **flags):
        """Every rank holds the same full array ``u`` (small n) and keeps its own planes."""
        n = u.shape[0]
        dtype = torch.complex128 if (u.is_complex() if isinstance(u, torch.Tensor) else u.dtype.kind == "c") else torch.float64
        return cls.from_slabs(ctx, n, h, s, lambda p0, p1: u[p0:p1], dtype=dtype, **flags)

    @classmethod
    def from_spatial(cls, ctx, h, s, u_spatial, anti_symmetrize=True, out_dtype=torch.complex128, into=None):
        """Spin-double a replicated spatial basis into a sharded spin-orbital one: every rank writes its
        own planes P = 2p + sigma of the (2l)^4 tensor with the fused add_spin + anti-symmetrise (+ cast)
        kernel -- no communication (SURVEY.md section 8e)."""
        from . import _arrays, ops

        u_dev = _arrays.to_device(u_spatial)
        l = u_dev.shape[0]
        n = 2 * l
        if u_dev.is_complex():
            out_dtype = torch.complex128
        u = into if into is not None else ShardedTwoBody.empty(ctx, n, out_dtype)
        if u.n != n or u.dtype != out_dtype:
            raise ValueError("`into` must be a ShardedTwoBody of extent 2 l and the requested dtype")
        for r in ctx.local_ranks:
            p0, p1 = u.planes(r)
            if p1 > p0:
                ops.add_spin_two_body(u_dev, anti_symmetrize=anti_symmetrize, out_dtype=out_dtype, planes=(p0, p1),
                                      out=u.local(r))
        ctx.barrier()
        u.proven_antisymmetric = bool(anti_symmetrize)  # the fused pass writes a - b and b - a: exact negatives
        h2 = ops.add_spin_one_body(_arrays.to_device(h), out_dtype=out_dtype)
        s2 = ops.add_spin_one_body(_arrays.to_device(s), out_dtype=out_dtype)
        return cls(ctx, n, h2, s2, u, includes_spin=True, anti_symmetrized_u=bool(anti_symmetrize))

    @classmethod
    def from_spatial_planes(cls, ctx, h, s, l, spatial_planes, anti_symmetrize=True, out_dtype=torch.complex128,
                            into=None):
        """Like :meth:`from_spatial`, but no rank ever holds the whole spatial tensor: ``spatial_planes(p0, p1)``
        returns (builds) the planes ``u_spatial[p0:p1]`` as a ``(p1 - p0, l, l, l)`` device tensor, and every rank
        asks only for the planes behind its own spin-orbital planes ``P = 2p + sigma``.  With
        :func:`odqd_spatial_planes` the grid Coulomb build itself is sharded (SURVEY.md section 8e): ODQD build ->
        add_spin + anti-symmetrise -> change_basis without a replicated l^4 tensor and without communication
        before the transform."""
        from . import _arrays, ops

        n = 2 * l
        u = into if into is not None else ShardedTwoBody.empty(ctx, n, out_dtype)
        if u.n != n or u.dtype != out_dtype:
            raise ValueError("`into` must be a ShardedTwoBody of extent 2 l and the requested dtype")
        for r in ctx.local_ranks:
            p0, p1 = u.planes(r)
            if p1 > p0:
                sp0, sp1 = p0 // 2, (p1 - 1) // 2 + 1
                slab = _arrays.to_device(spatial_planes(sp0, sp1))
                if slab.is_complex() and out_dtype != torch.complex128:
                    raise TypeError("complex spatial integrals need a complex128 sharded tensor")
                ops.add_spin_two_body(slab, anti_symmetrize=anti_symmetrize, out_dtype=out_dtype, planes=(p0, p1),
                                      out=u.local(r), first_spatial_plane=sp0)
        ctx.barrier()
        u.proven_antisymmetric = bool(anti_symmetrize)  # the fused pass writes a - b and b - a: exact negatives
        h2 = ops.add_spin_one_body(_arrays.to_device(h), out_dtype=out_dtype)
        s2 = ops.add_spin_one_body(_arrays.to_device(s), out_dtype=out_dtype)
        return cls(ctx, n, h2, s2, u, includes_spin=True, anti_symmetrized_u=bool(anti_symmetrize))

    @classmethod
    def from_odqd(cls, ctx, l, grid_length, num_grid_points, a=0.25, alpha=1.0, potential=None,
                  anti_symmetrize=True, out_dtype=torch.complex128, into=None):
        """The sharded counterpart of ``GeneralOrbitalSystem(n, ODQD(l, grid_length, num_grid_points, ...))``
        (reference one_dim_qd.py:258-289 -> general_orbital_system.py:39-53 -> basis_set.py:530-636): the O(G l)
        eigenproblem on the host of every rank (replicated, microseconds to seconds), then the grid Coulomb build,
        spin doubling and anti-symmetrisation of this rank's planes only.  The eigenvectors are kept as
        ``grid_coefficients`` (G', l) and the interior grid as ``inner_grid``."""
        from . import potentials
        from .odqd import grid_orbitals

        potential = potentials.HOPotential(0.25) if potential is None else potential
        grid, eps, Cg = grid_orbitals(l, grid_length, num_grid_points, potential)
        import numpy

        basis = cls.from_spatial_planes(
            ctx, numpy.diag(eps), numpy.eye(l), l, odqd_spatial_planes(Cg, grid[1:-1], alpha, a),
            anti_symmetrize=anti_symmetrize, out_dtype=out_dtype, into=into,
        )
        basis.grid_coefficients, basis.inner_grid = Cg, grid[1:-1]
        return basis

    def change_basis(self, C, C_tilde=None):
        """``h, s <- C~ X C`` on every rank (replicated, O(n^3)); ``u`` through the sharded transform."""
        from . import _arrays, ops

        C = _arrays.to_device(C)
        C_tilde = _arrays.to_device(C_tilde) if C_tilde is not None else None
        if C_tilde is not None:
            dt = torch.complex128 if torch.complex128 in (C.dtype, C_tilde.dtype) else torch.float64
            C, C_tilde = C.to(dt), C_tilde.to(dt)
        # real-valued coefficients of complex dtype select the split (2M) quarter GEMM, see ops
        C, C_tilde = ops.real_coefficients_if_exact(self.u.dtype == torch.complex128, C, C_tilde)
        self.l = C.shape[1]
        self.h = ops.transform_one_body(self.h, C, C_tilde)
        if self.s is not None:
            self.s = ops.transform_one_body(self.s, C, C_tilde)
        self.u = transform_two_body_sharded(self.u, C, C_tilde)

    def compute_reference_energy(self, n_occ, h=None, u=None, nuclear_repulsion_energy=0.0):
        """``E_0 = h_ii + 1/2 u_ijij + E_n`` over the occupied spin-orbitals (reference
        general_orbital_system.py:75-117) for a spin-orbital basis, ``2 h_ii + 2 u_ijij - u_ijji + E_n``
        (spatial_orbital_system.py:106-148) for a spatial one."""
        h = self.h if h is None else h
        u = self.u if u is None else u
        tr_h, direct, exchange = u.occupied_traces(h, n_occ)
        if self.includes_spin:
            energy = tr_h + 0.5 * direct + nuclear_repulsion_energy
        else:
            energy = 2 * tr_h + 2 * direct - exchange + nuclear_repulsion_energy
        is_complex = u.dtype == torch.complex128 or h.is_complex()
        return energy if is_complex else energy.real

    def construct_fock_matrix(self, h, u, n_occ, f=None):
        """``f = h + sum_i u[p,i,q,i]``: every rank reduces the rows p it owns, then the rows are
        all-gathered (n^2 elements)."""
        from . import ops

        ctx = self.ctx
        n = u.n
        if f is None:
            f = torch.empty_like(h)
        for r in ctx.local_ranks:
            p0, p1 = u.planes(r)
            if p1 > p0:
                _native.call(
                    "qs_fock_general", ops._ptr(h), ops._code(h), ctypes.c_void_p(u.buffers[r][r].at(0)),
                    _CODES[u.dtype], n, int(n_occ), ops._ptr(f), p0, p1, ops._stream(),
                )
        if isinstance(ctx, ProcessContext) and ctx.world > 1:
            block, offsets = u.block, u.offsets
            padded = torch.zeros((ctx.world, block, n), dtype=f.dtype, device=f.device)
            p0, p1 = u.planes(ctx.rank)
            padded[ctx.rank, : p1 - p0] = f[p0:p1]
            flat = torch.view_as_real(padded) if padded.is_complex() else padded
            ctx.dist.all_reduce(flat, group=ctx.group)  # disjoint rows: sum == gather
            for r in range(ctx.world):
                q0, q1 = offsets[r], offsets[r + 1]
                f[q0:q1] = padded[r, : q1 - q0]
        return f
