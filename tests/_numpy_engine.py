"""TEST INFRASTRUCTURE: a numpy stand-in for ``quantum_systems_b200.sharded.CudaEngine``.

It implements the documented semantics of ``qs_quarter_transform`` / ``qs_quarter_transform_scatter``
(include/qsb200.h) on host buffers so that the sharded SCHEDULE (partition, strides, exchange
layouts) can be exercised under gloo on a CPU-only box.  The product package never imports it.
"""

import numpy as np
import torch


class HostBuffer:
    def __init__(self, tensor):
        self.tensor = tensor
        self.dtype = tensor.dtype
        self.numel = tensor.numel()

    def as_tensor(self):
        return self.tensor

    def slice(self, offset, numel):
        return HostBuffer(self.tensor[offset : offset + numel])

    def flat(self):
        return self.tensor.numpy()


class NumpyEngine:
    def empty(self, numel, dtype):
        return HostBuffer(torch.full((max(int(numel), 1),), float("nan"), dtype=dtype))

    def asarray(self, a, dtype=None):
        t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))
        return t if dtype is None else t.to(dtype)

    def scatter_deal(self, W):
        """Same rule as qs_scatter_deal (include/qsb200.h): nearest integer to W / golden ratio coprime to W."""
        from math import gcd

        if W < 16:
            return 1
        s = int(W * 0.6180339887498949 + 0.5)
        while s < W and gcd(s, W) != 1:
            s += 1
        return s if 1 < s < W else 1

    def image(self, M, K, W, a_dtype, stride_k, stride_w, conj=False, deal=1):
        flat = (M.numpy() if isinstance(M, torch.Tensor) else np.asarray(M)).reshape(-1)
        k = np.arange(K)[:, None] * stride_k
        w = ((np.arange(W) * deal) % W)[None, :] * stride_w  # image column j holds M[:, (j * deal) % W]
        dense = flat[k + w]
        return dense.conj() if conj else dense

    def pad_rows(self, src, rows, n, pitch, dst):
        out = dst.flat()[: rows * pitch].reshape(rows, pitch)
        out[:, :n] = src.flat()[: rows * n].reshape(rows, n)
        out[:, n:] = 0

    @staticmethod
    def _product(A, X, K, lda, image):
        rows = A.flat()[: X * lda].reshape(X, lda)[:, :K]
        return rows @ image

    def quarter(self, A, X, K, lda, image, m_dtype, W, out, out_offset, x_inner, sx0, sx1, w_inner, sw0, sw1):
        if X <= 0:
            return
        res = self._product(A, X, K, lda, image)
        x = np.arange(X)
        w = np.arange(W)
        ax = (x // x_inner) * sx1 + (x % x_inner) * sx0
        aw = (w // w_inner) * sw1 + (w % w_inner) * sw0
        out.flat()[out_offset + ax[:, None] + aw[None, :]] = res

    def quarter_scatter(self, A, X, K, lda, image, m_dtype, W, dests, x_inner, x_mid, sx0, sx1, sx2, w_inner, sw0,
                        deal=1, cyclic=False):
        if X <= 0:
            return
        res = self._product(A, X, K, lda, image)
        if deal > 1:  # column j of the product is physical column (j * deal) % W
            physical = np.empty_like(res)
            physical[:, (np.arange(W) * deal) % W] = res
            res = physical
        x = np.arange(X)
        x_mid = max(x_mid, 1)
        xq = x // x_inner
        ax = (xq // x_mid) * sx2 + (xq % x_mid) * sx1 + (x % x_inner) * sx0
        for j, (buf, off) in enumerate(dests):
            if cyclic:  # column w goes to destination w % n_dest and is column w // n_dest there
                cols = np.arange(j, W, len(dests))
                aw = (cols // len(dests)) * sw0
            else:
                cols = np.arange(j * w_inner, min((j + 1) * w_inner, W))
                aw = (cols % max(w_inner, 1)) * sw0
            if len(cols) == 0:
                continue
            buf.flat()[off + ax[:, None] + aw[None, :]] = res[:, cols]

    def quarter_scatter_pairs(self, A, X, K, lda, image, m_dtype, W, dests, x_inner, x_mid, sx0, sx1, sx2, sw0,
                              rows_per_s, padded):
        """qs_quarter_transform_scatter_pairs: cyclic destinations, and ONLY the CTA tiles the library's own host-side
        planner (qs_quarter_plan_tiles, mask kind 3; no device involved) would launch are written -- everything else
        keeps the NaN the buffers were created with, so a later read of a tile that was never sent shows up."""
        if X <= 0:
            return
        res = self._product(A, X, K, lda, image)
        launched = np.zeros((X, W), dtype=bool)
        for x0, x1, w0, w1 in self._pair_tiles(X, K, W, A.dtype, m_dtype, x_inner, rows_per_s, padded):
            launched[x0 : x1 + 1, w0 : w1 + 1] = True
        x = np.arange(X)
        xq = x // x_inner
        ax = (xq // max(x_mid, 1)) * sx2 + (xq % max(x_mid, 1)) * sx1 + (x % x_inner) * sx0
        n_dest = len(dests)
        for j, (buf, off) in enumerate(dests):
            cols = np.arange(j, W, n_dest)
            if len(cols) == 0:
                continue
            aw = (cols // n_dest) * sw0
            flat = buf.flat()
            rows, cidx = np.nonzero(launched[:, cols])
            flat[off + ax[rows] + aw[cidx]] = res[rows, cols[cidx]]

    @staticmethod
    def _pair_tiles(X, K, W, a_dtype, m_dtype, x_inner, rows_per_s, padded):
        """The tiles ``(x0, x1, w0, w1)`` (inclusive) that qs_quarter_transform_scatter_pairs launches."""
        import ctypes

        from quantum_systems_b200 import _native

        lib = _native.load()
        code = {torch.float64: 0, torch.complex128: 1}
        args = (X, K, W, code[a_dtype], code[m_dtype], x_inner, 3, 0 if padded else 1, 1, 1, rows_per_s, W,
                ctypes.c_void_p(0))
        count = ctypes.c_int64(0)
        assert lib.qs_quarter_plan_tiles(*args, ctypes.c_void_p(0), 0, ctypes.byref(count)) == 0
        tiles = np.zeros((count.value, 4), dtype=np.int64)
        assert lib.qs_quarter_plan_tiles(*args, ctypes.c_void_p(tiles.ctypes.data), count.value, ctypes.byref(count)) == 0
        return tiles

    # consumers of a shard: documented semantics of qs_extract_block / qs_scale_add / qs_occupied_traces
    def extract_block(self, buf, planes, n, bounds):
        (a0, a1), (b0, b1), (c0, c1), (d0, d1) = bounds
        slab = buf.flat()[: planes * n**3].reshape(planes, n, n, n)
        return torch.from_numpy(np.ascontiguousarray(slab[a0:a1, b0:b1, c0:c1, d0:d1]))

    def scale_add(self, x, y, count, alpha, beta, out):
        if not x.dtype.is_complex:
            alpha, beta = complex(alpha).real, complex(beta).real
        res = alpha * x.flat()[:count]
        if y is not None:
            res = res + beta * y.flat()[:count]
        out.flat()[:count] = res

    def occupied_traces(self, h, buf, n, n_occ, p0, p1):
        h = h.numpy() if isinstance(h, torch.Tensor) else np.asarray(h)
        slab = buf.flat()[: (p1 - p0) * n**3].reshape(p1 - p0, n, n, n)
        tr_h = direct = exchange = 0.0
        for i in range(p0, min(p1, n_occ)):
            tr_h += h[i, i]
            for j in range(n_occ):
                direct += slab[i - p0, j, i, j]
                exchange += slab[i - p0, j, j, i]
        return torch.tensor([tr_h, direct, exchange], dtype=torch.complex128)

    # symmetry-aware steps: documented semantics of qs_quarter_transform_rows / _scatter_rows /
    # qs_is_antisymmetric_last_pair / qs_cyclic_antisymmetric_fill
    def index_table(self, host_int64):
        return torch.from_numpy(host_int64)

    def is_antisymmetric(self, buf, n, planes):
        slab = buf.flat()[: planes * n**3].reshape(planes, n, n, n)
        return bool(np.array_equal(slab, -slab.transpose(0, 1, 3, 2)))

    def cyclic_fill(self, buf, m, planes):
        from quantum_systems_b200.sharded import cyclic_wanted

        slab = buf.flat()[: planes * m**3].reshape(planes, m, m, m)
        r, s = np.arange(m)[:, None], np.arange(m)[None, :]
        wanted = cyclic_wanted(r, s, m)
        mirrored = -slab.transpose(0, 1, 3, 2)
        slab[...] = np.where(wanted, slab, np.where(r == s, 0, mirrored))

    def quarter_rows(self, A, X, K, lda, image, m_dtype, W, out, x_inner, sx0, host_table, dev_table, w_inner, sw0, sw1):
        if X <= 0:
            return
        res = self._product(A, X, K, lda, image)
        x = np.arange(X)
        base = host_table[x // x_inner]
        keep = base >= 0
        ax = base[keep] + (x[keep] % x_inner) * sx0
        w = np.arange(W)
        aw = (w // w_inner) * sw1 + (w % w_inner) * sw0
        out.flat()[ax[:, None] + aw[None, :]] = res[keep]

    def quarter_scatter_rows(self, A, X, K, lda, image, m_dtype, W, dests, x_inner, sx1, xr_table, w_inner, sw0, deal=1,
                             rows_paired=False):
        if X <= 0:
            return
        res = self._product(A, X, K, lda, image)
        if deal > 1:
            physical = np.empty_like(res)
            physical[:, (np.arange(W) * deal) % W] = res
            res = physical
        table = xr_table.numpy() if isinstance(xr_table, torch.Tensor) else np.asarray(xr_table)
        if rows_paired:  # the promise behind the 16-byte stores: rows 2k, 2k + 1 adjacent at an even offset
            assert x_inner % 2 == 0 and np.all(table[0::2] % 2 == 0) and np.all(table[1::2] == table[0::2] + 1)
        x = np.arange(X)
        ax = (x // x_inner) * sx1 + table[x % x_inner]
        for j, (buf, off) in enumerate(dests):
            cols = np.arange(j * w_inner, min((j + 1) * w_inner, W))
            if len(cols) == 0:
                continue
            aw = (cols % w_inner) * sw0
            buf.flat()[off + ax[:, None] + aw[None, :]] = res[:, cols]
