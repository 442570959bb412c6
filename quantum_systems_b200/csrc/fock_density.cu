// Fock matrix from a general density matrix (the O(n^4) step of a Hartree-Fock iteration):
//
//   f[p,q] = h[p,q] + a_d sum_{r,s} u[p,r,q,s] rho[s,r] + a_x sum_{r,s} u[p,r,s,q] rho[s,r],   p in [p_begin, p_end)
//
// For fixed (p, r) the block B = u[p,r,:,:] is contiguous (rows q, columns s).  The direct term of row q is the dot
// product B[q,:] . rho[:,r]; the exchange term of column q is the weighted column sum sum_s rho[s,r] B[s,q].  Both
// come from the same coalesced 16-byte loads of B, so every element of u is read from HBM once.
//
// Pass 1: one CTA per (plane p, chunk of r).  A warp owns the rows q = warp, warp + 8, ...; its lanes sweep the
// columns of a row in 16-byte pieces.  The direct partial of row q accumulates in the lane over the r of the chunk
// and is reduced with a warp butterfly once per (q, column block); the exchange partials of the lane's columns stay
// in registers over all rows and r, and the 8 warps are summed through shared memory in warp order.  The chunk's
// partial row a_d D + a_x X goes to the caller's workspace.
// Pass 2: f[p,q] = h[p,q] + sum over chunks in chunk order.
//
// Unrestricted (two spin densities, qs_fock_density_unrestricted):
//
//   f_s[p,q] = h[p,q] + sum_{r,s} u[p,r,q,s] (rho_a + rho_b)[s,r] - sum_{r,s} u[p,r,s,q] rho_s[s,r],   s in {a, b}
//
// Real u and real densities: rho_c = rho_a + i rho_b goes through the real-u x complex-rho pass once in kSplit mode,
// which writes a chunk's direct row D and exchange row X as two rows instead of a_d D + a_x X: D = J[rho_a] +
// i J[rho_b], X = K[rho_a] + i K[rho_b].  Real u and complex densities: the kUnrestricted pass stages the chunk's
// columns of rho_a + rho_b, rho_a and rho_b and writes three rows, D = J[rho_a + rho_b], X_a = K[rho_a] and
// X_b = K[rho_b].  Either way u is read once for both spins.  Complex u: the split pass runs once per density and
// u is read twice.  The unrestricted sum kernel forms both matrices from those rows in chunk order.
//
// No floating-point atomics.  The chunking depends on n only (fd_chunk), never on the plane range, so a row computed
// on a shard is bit-identical to the same row computed on the whole tensor.
#include "common.cuh"

namespace {

constexpr int kFdThreads = 256;
constexpr int kFdWarps = kFdThreads / 32;
constexpr int kFdTiles = 4;  // 16-byte column pieces a lane holds per column block

// What pass 1 writes per (plane, chunk): a_d D + a_x X (one row), D and X (two rows), or D[rho_a + rho_b],
// X[rho_a] and X[rho_b] (three rows) of the two densities rho and rho_b.
enum : int { kCombined = 0, kSplit = 1, kUnrestricted = 2 };
// densities staged in shared memory, exchange rows written
__host__ __device__ constexpr int fd_densities(int mode) { return mode == kUnrestricted ? 3 : 1; }
__host__ __device__ constexpr int fd_exchange_rows(int mode) { return mode == kUnrestricted ? 2 : 1; }
// column pieces per lane and block: kUnrestricted holds twice the exchange accumulators of a complex density, so it
// takes blocks of 128 columns for both piece widths
__host__ __device__ constexpr int fd_tiles(int mode, int v) { return mode == kUnrestricted ? kFdTiles / v : kFdTiles; }

// r per CTA: about 1024 / n rows of r, between 1 and 16 -- enough CTAs for a few planes, few partial rows.
inline int64_t fd_chunk(int64_t n) {
    int64_t c = 1024 / n;
    return c < 1 ? 1 : (c > 16 ? 16 : c);
}

struct cplx {
    double x, y;
};

template <bool C>
struct Val;
template <>
struct Val<false> {
    using T = double;
};
template <>
struct Val<true> {
    using T = cplx;
};

__device__ __forceinline__ double mul(double a, double b) { return a * b; }
__device__ __forceinline__ cplx mul(cplx a, double b) { return {a.x * b, a.y * b}; }
__device__ __forceinline__ cplx mul(double a, cplx b) { return {a * b.x, a * b.y}; }
__device__ __forceinline__ cplx mul(cplx a, cplx b) { return {a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x}; }
__device__ __forceinline__ double add(double a, double b) { return a + b; }
__device__ __forceinline__ cplx add(cplx a, cplx b) { return {a.x + b.x, a.y + b.y}; }
__device__ __forceinline__ void zero(double& a) { a = 0.0; }
__device__ __forceinline__ void zero(cplx& a) { a = {0.0, 0.0}; }

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}
__device__ __forceinline__ cplx warp_sum(cplx v) { return {warp_sum(v.x), warp_sum(v.y)}; }

// V elements of u per lane piece: 2 for real u with an even row (one 16-byte load), else 1 (8 or 16 bytes).
template <bool UC, int V>
struct Piece {
    typename Val<UC>::T e[V];
};

template <bool UC, int V>
__device__ __forceinline__ Piece<UC, V> load_piece(const double* __restrict__ p) {
    Piece<UC, V> r;
    if constexpr (UC) {
        const double2 v = __ldg(reinterpret_cast<const double2*>(p));
        r.e[0] = {v.x, v.y};
    } else if constexpr (V == 2) {
        const double2 v = __ldg(reinterpret_cast<const double2*>(p));
        r.e[0] = v.x;
        r.e[1] = v.y;
    } else {
        r.e[0] = __ldg(p);
    }
    return r;
}

// UC: u complex, RC: rho complex, V: elements per piece.  Accumulators are complex when either is.  Real u with
// complex rho and 16-byte pieces holds twice the exchange accumulators: two CTAs per SM give it the registers, and
// kUnrestricted the same with half the column pieces (fd_tiles) for its two exchange rows.
// (Unrolling the r loop of real u four times instead of two needs that register budget for every real kernel and
// was measured slower at n = 128: 0.508 against 0.412 ms on a B200.)
// MODE: kCombined writes a_d D + a_x X; kSplit writes D and X (a_d, a_x unused); kUnrestricted (real u, complex
// rho) stages rho + rho_b, rho and rho_b and writes D of the first and X of the other two.
template <bool UC, bool RC, int V, int MODE>
__global__ void __launch_bounds__(kFdThreads, (!UC && RC && (V == 2 || MODE == kUnrestricted)) ? 2 : 3)
    fock_density_kernel(const double* __restrict__ u, const double* __restrict__ rho,
                        const double* __restrict__ rho_b, int n, int chunk, int n_chunks, double a_d, double a_x,
                        double* __restrict__ ws) {
    using R = typename Val<RC>::T;
    using A = typename Val<UC || RC>::T;
    constexpr int kTiles = fd_tiles(MODE, V);
    constexpr int kBlockCols = 32 * V * kTiles;
    constexpr int kDens = fd_densities(MODE), kX = fd_exchange_rows(MODE);
    static_assert(MODE != kUnrestricted || (!UC && RC), "the one-read unrestricted pass is for real u, complex rho");

    extern __shared__ double4 fd_smem[];
    // [kDens][chunk][n]: rho_s[d][rl][s] = rho_d[s, r0 + rl]; density 0 feeds the direct row, the last kX the
    // exchange rows (the same one density unless kUnrestricted)
    R* rho_s = reinterpret_cast<R*>(fd_smem);
    const size_t staged = (size_t)chunk * n;
    A* dacc = reinterpret_cast<A*>(rho_s + kDens * staged);  // [n] direct partials (row q owned by warp q % 8)
    A* xcol = dacc + n;                                      // [kX][n] exchange partials
    A* xs = xcol + kX * n;                                   // [kFdWarps][kBlockCols]

    const int pl = blockIdx.x / n_chunks;  // plane relative to p_begin
    const int c_idx = blockIdx.x - pl * n_chunks;
    const int r0 = c_idx * chunk;
    const int rc = min(chunk, n - r0);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    for (int i = threadIdx.x; i < rc * n; i += kFdThreads) {
        const int s = i / rc, rl = i - s * rc;
        const size_t src = (size_t)s * n + r0 + rl, dst = (size_t)rl * n + s;
        const R a = reinterpret_cast<const R*>(rho)[src];
        if constexpr (MODE == kUnrestricted) {
            const R b = reinterpret_cast<const R*>(rho_b)[src];
            rho_s[dst] = add(a, b);
            rho_s[staged + dst] = a;
            rho_s[2 * staged + dst] = b;
        } else {
            rho_s[dst] = a;
        }
    }
    for (int q = threadIdx.x; q < n; q += kFdThreads) zero(dacc[q]);
    __syncthreads();

    const size_t n2 = (size_t)n * n;
    const double* plane = u + (size_t)pl * n * n2 * (UC ? 2 : 1);
    for (int cb = 0; cb < n; cb += kBlockCols) {
        A x[kX][kTiles][V];
#pragma unroll
        for (int j = 0; j < kX; ++j)
#pragma unroll
            for (int k = 0; k < kTiles; ++k)
#pragma unroll
                for (int v = 0; v < V; ++v) zero(x[j][k][v]);
        for (int q = warp; q < n; q += kFdWarps) {
            A d;
            zero(d);
#pragma unroll 2
            for (int rl = 0; rl < rc; ++rl) {
                R rq[kX];
#pragma unroll
                for (int j = 0; j < kX; ++j) rq[j] = rho_s[(kDens - kX + j) * staged + (size_t)rl * n + q];
                const double* row = plane + ((size_t)(r0 + rl) * n2 + (size_t)q * n) * (UC ? 2 : 1);
                Piece<UC, V> pc[kTiles];
#pragma unroll
                for (int k = 0; k < kTiles; ++k) {
                    const int c = cb + (k * 32 + lane) * V;
                    if (c < n) pc[k] = load_piece<UC, V>(row + (size_t)c * (UC ? 2 : 1));
                }
#pragma unroll
                for (int k = 0; k < kTiles; ++k) {
                    const int c = cb + (k * 32 + lane) * V;
                    if (c < n) {
#pragma unroll
                        for (int v = 0; v < V; ++v) {
                            d = add(d, mul(pc[k].e[v], rho_s[(size_t)rl * n + c + v]));
#pragma unroll
                            for (int j = 0; j < kX; ++j) x[j][k][v] = add(x[j][k][v], mul(rq[j], pc[k].e[v]));
                        }
                    }
                }
            }
            d = warp_sum(d);
            if (lane == 0) dacc[q] = add(dacc[q], d);
        }
#pragma unroll
        for (int j = 0; j < kX; ++j) {
#pragma unroll
            for (int k = 0; k < kTiles; ++k)
#pragma unroll
                for (int v = 0; v < V; ++v) xs[warp * kBlockCols + (k * 32 + lane) * V + v] = x[j][k][v];
            __syncthreads();
            for (int jc = threadIdx.x; jc < kBlockCols && cb + jc < n; jc += kFdThreads) {
                A t = xs[jc];
                for (int w = 1; w < kFdWarps; ++w) t = add(t, xs[w * kBlockCols + jc]);
                xcol[j * n + cb + jc] = t;
            }
            __syncthreads();
        }
    }
    if constexpr (MODE == kCombined) {
        A* out = reinterpret_cast<A*>(ws) + ((size_t)pl * n_chunks + c_idx) * n;
        for (int q = threadIdx.x; q < n; q += kFdThreads) out[q] = add(mul(dacc[q], a_d), mul(xcol[q], a_x));
    } else {
        A* out = reinterpret_cast<A*>(ws) + ((size_t)pl * n_chunks + c_idx) * (1 + kX) * n;
        for (int q = threadIdx.x; q < n; q += kFdThreads) {
            out[q] = dacc[q];
#pragma unroll
            for (int j = 0; j < kX; ++j) out[(1 + j) * n + q] = xcol[j * n + q];
        }
    }
}

// f[p,q] = h[p,q] + sum_c ws[p][c][q] in chunk order.
__global__ void fock_density_sum_kernel(const double* __restrict__ h, bool h_c, const double* __restrict__ ws,
                                        bool ws_c, double* __restrict__ f, bool f_c, int n, int n_chunks,
                                        long long p_begin, long long rows) {
    const long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (e >= rows * n) return;
    const long long pl = e / n, q = e - pl * n;
    const long long o = (p_begin + pl) * n + q;
    double re = h_c ? h[2 * o] : h[o];
    double im = h_c ? h[2 * o + 1] : 0.0;
    for (int c = 0; c < n_chunks; ++c) {
        const long long w = (pl * n_chunks + c) * n + q;
        if (ws_c) {
            re += ws[2 * w];
            im += ws[2 * w + 1];
        } else {
            re += ws[w];
        }
    }
    if (f_c) {
        f[2 * o] = re;
        f[2 * o + 1] = im;
    } else {
        f[o] = re;
    }
}

// Where the unrestricted sum kernel finds the rows of pass 1 (complex, per plane and chunk): kPackedRows, [D, X] of
// rho_a + i rho_b with D = J_a + i J_b and X = K_a + i K_b (u, rho real); kOneReadRows, [D, X_a, X_b]; kTwoReadRows,
// [D, X] of rho_a and, at element offset `second`, of rho_b, whose D rows are added.
enum : int { kPackedRows = 0, kOneReadRows = 1, kTwoReadRows = 2 };

// f_a, f_b from the rows of pass 1, summed in chunk order.
__global__ void fock_density_unrestricted_sum_kernel(const double* __restrict__ h, bool h_c,
                                                     const cplx* __restrict__ ws, int layout, long long second,
                                                     double* __restrict__ fa, double* __restrict__ fb, bool f_c,
                                                     int n, int n_chunks, long long p_begin, long long rows) {
    const long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (e >= rows * n) return;
    const long long pl = e / n, q = e - pl * n;
    const long long o = (p_begin + pl) * n + q;
    double ar = h_c ? h[2 * o] : h[o];
    double ai = h_c ? h[2 * o + 1] : 0.0;
    double br = ar, bi = ai;
    const int per_chunk = layout == kOneReadRows ? 3 : 2;
    for (int c = 0; c < n_chunks; ++c) {
        const long long w = (pl * n_chunks + c) * per_chunk * n + q;
        const cplx d = ws[w], x = ws[w + n];
        if (layout == kPackedRows) {
            const double j = d.x + d.y;
            ar += j - x.x;
            br += j - x.y;
        } else if (layout == kOneReadRows) {
            const cplx xb = ws[w + 2 * n];
            ar += d.x - x.x;
            ai += d.y - x.y;
            br += d.x - xb.x;
            bi += d.y - xb.y;
        } else {
            const cplx d2 = ws[second + w], x2 = ws[second + w + n];
            const double jr = d.x + d2.x, ji = d.y + d2.y;
            ar += jr - x.x;
            ai += ji - x.y;
            br += jr - x2.x;
            bi += ji - x2.y;
        }
    }
    if (f_c) {
        fa[2 * o] = ar;
        fa[2 * o + 1] = ai;
        fb[2 * o] = br;
        fb[2 * o + 1] = bi;
    } else {
        fa[o] = ar;
        fb[o] = br;
    }
}

// rho_c = rho_a + i rho_b for two real (n, n) densities
__global__ void pack_densities_kernel(const double* __restrict__ ra, const double* __restrict__ rb,
                                      cplx* __restrict__ rc, long long n2) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n2) rc[i] = {ra[i], rb[i]};
}

size_t fd_smem_bytes(int64_t n, int u_dtype, int rho_dtype, int mode) {
    const bool acc_c = u_dtype == QS_C128 || rho_dtype == QS_C128;
    const int v = (u_dtype == QS_F64 && n % 2 == 0) ? 2 : 1;
    const size_t a = acc_c ? 16 : 8;
    return (size_t)fd_densities(mode) * fd_chunk(n) * n * (rho_dtype == QS_C128 ? 16 : 8) +
           (size_t)(1 + fd_exchange_rows(mode)) * n * a + (size_t)kFdWarps * 32 * v * fd_tiles(mode, v) * a;
}

// Launch geometry of both entries, from fd_geometry.
struct FdGeometry {
    int n, chunk, n_chunks;
    long long rows;  // p_end - p_begin; 0: nothing to launch
    size_t smem;     // dynamic shared memory of pass 1
    bool vec;        // 16-byte pieces of a real u
};

// The checks of both entries in order and their launch geometry.  `args` is the entry's null-pointer check;
// `unrestricted` selects the workspace rule of qs_fock_density_unrestricted and the shared memory of its pass 1: the
// one-read pass for real u and complex densities, else a split pass of real u against a complex density (the packed
// pair) or of complex u.
int fd_geometry(const char* entry, bool args, int64_t n, int64_t p_begin, int64_t p_end, int h_dtype, const void* u,
                int u_dtype, int rho_dtype, int f_dtype, bool unrestricted, const void* workspace,
                int64_t workspace_bytes, FdGeometry* g) {
    QS_REQUIRE(args && n >= 1 && n <= (1 << 20), "%s: bad arguments", entry);
    QS_REQUIRE(0 <= p_begin && p_begin <= p_end && p_end <= n, "%s: bad row range", entry);
    for (int d : {h_dtype, u_dtype, rho_dtype, f_dtype})
        QS_REQUIRE(d == QS_F64 || d == QS_C128, "%s: bad dtype", entry);
    QS_REQUIRE(!(f_dtype == QS_F64 && (h_dtype == QS_C128 || u_dtype == QS_C128 || rho_dtype == QS_C128)),
               "%s: complex u cannot be accumulated into a real Fock matrix", entry);
    g->rows = p_end - p_begin;
    if (g->rows == 0) return QS_OK;
    int64_t need = 0;
    if (unrestricted)
        qs_fock_density_unrestricted_workspace_bytes(n, p_begin, p_end, u_dtype, rho_dtype, &need);
    else
        qs_fock_density_workspace_bytes(n, p_begin, p_end, u_dtype, rho_dtype, &need);
    QS_REQUIRE(u && workspace && workspace_bytes >= need, "%s: workspace too small (%lld < %lld bytes)", entry,
               (long long)workspace_bytes, (long long)need);
    g->n = (int)n;
    g->chunk = (int)fd_chunk(n);
    g->n_chunks = (int)qs_ceil_div(n, g->chunk);
    QS_REQUIRE(g->rows * g->n_chunks < (1LL << 31), "%s: too many planes for one launch", entry);
    const bool real_u = u_dtype == QS_F64;
    if (!unrestricted)
        g->smem = fd_smem_bytes(n, u_dtype, rho_dtype, kCombined);
    else if (real_u && rho_dtype == QS_C128)
        g->smem = fd_smem_bytes(n, u_dtype, rho_dtype, kUnrestricted);
    else
        g->smem = fd_smem_bytes(n, u_dtype, real_u ? QS_C128 : rho_dtype, kSplit);
    QS_REQUIRE(g->smem <= 227 * 1024, "%s: n = %lld needs %zu bytes of shared memory", entry, (long long)n, g->smem);
    // 16-byte loads of a real row need an even row length and a 16-byte aligned plane
    g->vec = real_u && n % 2 == 0 && (reinterpret_cast<uintptr_t>(u) & 15) == 0;
    return QS_OK;
}

template <bool UC, bool RC, int V, int MODE>
int launch_pass1(const void* u, const void* rho, const void* rho_b, const FdGeometry& g, double a_d, double a_x,
                 void* ws, cudaStream_t st) {
    auto kern = fock_density_kernel<UC, RC, V, MODE>;
    QS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smem));
    kern<<<(unsigned)(g.rows * g.n_chunks), kFdThreads, g.smem, st>>>(
        static_cast<const double*>(u), static_cast<const double*>(rho), static_cast<const double*>(rho_b), g.n,
        g.chunk, g.n_chunks, a_d, a_x, static_cast<double*>(ws));
    QS_LAUNCH_CHECK();
    return QS_OK;
}

// Pass 1 of one density for (u complex, rho complex, g.vec) in mode kCombined or kSplit.  Real u is only ever split
// against a complex density, so real u x real rho has no split instantiation.
template <int MODE>
int pass1(const void* u, bool u_c, const void* rho, bool rho_c, const FdGeometry& g, double a_d, double a_x, void* ws,
          cudaStream_t st) {
    if (u_c)
        return rho_c ? launch_pass1<true, true, 1, MODE>(u, rho, nullptr, g, a_d, a_x, ws, st)
                     : launch_pass1<true, false, 1, MODE>(u, rho, nullptr, g, a_d, a_x, ws, st);
    if (rho_c)
        return g.vec ? launch_pass1<false, true, 2, MODE>(u, rho, nullptr, g, a_d, a_x, ws, st)
                     : launch_pass1<false, true, 1, MODE>(u, rho, nullptr, g, a_d, a_x, ws, st);
    if constexpr (MODE == kSplit) {
        qs_set_error("fock_density: no split pass for real u and a real density");
        return QS_ERR_INVALID;
    } else {
        return g.vec ? launch_pass1<false, false, 2, MODE>(u, rho, nullptr, g, a_d, a_x, ws, st)
                     : launch_pass1<false, false, 1, MODE>(u, rho, nullptr, g, a_d, a_x, ws, st);
    }
}

// Bytes of the complex rows pass 1 writes for `rows` planes, `per_chunk` rows of n per (plane, chunk).
int64_t pass1_rows_bytes(int64_t n, int64_t rows, int per_chunk) {
    return rows * qs_ceil_div(n, fd_chunk(n)) * per_chunk * n * 16;
}

}  // namespace

extern "C" int qs_fock_density_workspace_bytes(int64_t n, int64_t p_begin, int64_t p_end, int u_dtype, int rho_dtype,
                                               int64_t* bytes) {
    QS_REQUIRE(bytes && n >= 1 && 0 <= p_begin && p_begin <= p_end && p_end <= n,
               "qs_fock_density_workspace_bytes: bad arguments");
    QS_REQUIRE((u_dtype == QS_F64 || u_dtype == QS_C128) && (rho_dtype == QS_F64 || rho_dtype == QS_C128),
               "qs_fock_density_workspace_bytes: bad dtype");
    const int64_t acc = (u_dtype == QS_C128 || rho_dtype == QS_C128) ? 16 : 8;
    *bytes = (p_end - p_begin) * qs_ceil_div(n, fd_chunk(n)) * n * acc;
    return QS_OK;
}

extern "C" int qs_fock_density(const void* h, int h_dtype, const void* u, int u_dtype, const void* rho, int rho_dtype,
                               int64_t n, double scale_direct, double scale_exchange, void* f, int f_dtype,
                               int64_t p_begin, int64_t p_end, void* workspace, int64_t workspace_bytes,
                               void* stream) {
    FdGeometry g;
    int status = fd_geometry("qs_fock_density", h && rho && f, n, p_begin, p_end, h_dtype, u, u_dtype, rho_dtype,
                             f_dtype, false, workspace, workspace_bytes, &g);
    if (status != QS_OK || g.rows == 0) return status;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    status = pass1<kCombined>(u, u_dtype == QS_C128, rho, rho_dtype == QS_C128, g, scale_direct, scale_exchange,
                              workspace, st);
    if (status != QS_OK) return status;
    fock_density_sum_kernel<<<(unsigned)qs_ceil_div(g.rows * n, 256), 256, 0, st>>>(
        static_cast<const double*>(h), h_dtype == QS_C128, static_cast<const double*>(workspace),
        u_dtype == QS_C128 || rho_dtype == QS_C128, static_cast<double*>(f), f_dtype == QS_C128, g.n, g.n_chunks,
        p_begin, g.rows);
    QS_LAUNCH_CHECK();
    return QS_OK;
}

extern "C" int qs_fock_density_unrestricted_workspace_bytes(int64_t n, int64_t p_begin, int64_t p_end, int u_dtype,
                                                            int rho_dtype, int64_t* bytes) {
    QS_REQUIRE(bytes && n >= 1 && 0 <= p_begin && p_begin <= p_end && p_end <= n,
               "qs_fock_density_unrestricted_workspace_bytes: bad arguments");
    QS_REQUIRE((u_dtype == QS_F64 || u_dtype == QS_C128) && (rho_dtype == QS_F64 || rho_dtype == QS_C128),
               "qs_fock_density_unrestricted_workspace_bytes: bad dtype");
    const int64_t rows = p_end - p_begin;
    if (u_dtype == QS_F64 && rho_dtype == QS_F64)  // one split pass plus the packed density rho_a + i rho_b
        *bytes = pass1_rows_bytes(n, rows, 2) + n * n * 16;
    else if (u_dtype == QS_F64)  // one pass, three rows
        *bytes = pass1_rows_bytes(n, rows, 3);
    else  // one split pass per density
        *bytes = 2 * pass1_rows_bytes(n, rows, 2);
    return QS_OK;
}

extern "C" int qs_fock_density_unrestricted(const void* h, int h_dtype, const void* u, int u_dtype,
                                            const void* rho_alpha, const void* rho_beta, int rho_dtype, int64_t n,
                                            void* f_alpha, void* f_beta, int f_dtype, int64_t p_begin, int64_t p_end,
                                            void* workspace, int64_t workspace_bytes, void* stream) {
    FdGeometry g;
    int status = fd_geometry("qs_fock_density_unrestricted", h && rho_alpha && rho_beta && f_alpha && f_beta, n,
                             p_begin, p_end, h_dtype, u, u_dtype, rho_dtype, f_dtype, true, workspace,
                             workspace_bytes, &g);
    if (status != QS_OK || g.rows == 0) return status;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const bool u_c = u_dtype == QS_C128, rho_c = rho_dtype == QS_C128;
    const int64_t split_bytes = pass1_rows_bytes(n, g.rows, 2);
    char* ws = static_cast<char*>(workspace);
    int layout;
    if (!u_c && !rho_c) {
        layout = kPackedRows;
        cplx* rho_p = reinterpret_cast<cplx*>(ws + split_bytes);
        pack_densities_kernel<<<(unsigned)qs_ceil_div(n * n, 256), 256, 0, st>>>(
            static_cast<const double*>(rho_alpha), static_cast<const double*>(rho_beta), rho_p, n * n);
        QS_LAUNCH_CHECK();
        status = pass1<kSplit>(u, false, rho_p, true, g, 0.0, 0.0, ws, st);
    } else if (!u_c) {
        layout = kOneReadRows;
        status = g.vec ? launch_pass1<false, true, 2, kUnrestricted>(u, rho_alpha, rho_beta, g, 0.0, 0.0, ws, st)
                       : launch_pass1<false, true, 1, kUnrestricted>(u, rho_alpha, rho_beta, g, 0.0, 0.0, ws, st);
    } else {
        layout = kTwoReadRows;
        status = pass1<kSplit>(u, true, rho_alpha, rho_c, g, 0.0, 0.0, ws, st);
        if (status == QS_OK) status = pass1<kSplit>(u, true, rho_beta, rho_c, g, 0.0, 0.0, ws + split_bytes, st);
    }
    if (status != QS_OK) return status;
    fock_density_unrestricted_sum_kernel<<<(unsigned)qs_ceil_div(g.rows * n, 256), 256, 0, st>>>(
        static_cast<const double*>(h), h_dtype == QS_C128, reinterpret_cast<const cplx*>(ws), layout,
        split_bytes / 16, static_cast<double*>(f_alpha), static_cast<double*>(f_beta), f_dtype == QS_C128, g.n,
        g.n_chunks, p_begin, g.rows);
    QS_LAUNCH_CHECK();
    return QS_OK;
}
