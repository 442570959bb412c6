// Coulomb and exchange matrices of a batch of k real densities in one read of a real u:
//
//   J_d[p,q] = sum_{r,s} u[p,r,q,s] rho_d[s,r]        K_d[p,q] = sum_{r,s} u[p,r,s,q] rho_d[s,r]
//
// for p in [p_begin, p_end) and d < k <= QS_COULOMB_EXCHANGE_MAX_BATCH.  For fixed (p, r) the block B = u[p,r,:,:]
// (rows q, columns s) gives J as the product B R and K as B^T R with R[s, d] = rho_d[s, r]: two matrix products on
// the FP64 tensor pipe (DMMA.8x8x4) that differ only in how the A fragment is read from the staged block.
//
// Pass 1: one CTA per (plane p, chunk of r).  The chunk's c n^2 contiguous doubles are streamed through shared
// memory in panels of PR rows of B (cp.async, two stages when they fit), together with R of the current r (two
// buffers, by r parity).  The q rows are dealt to the 8 warps in 8-row tiles (tile t belongs to warp t % 8, slot
// t / 8); a warp keeps the J and K accumulators of its tiles for all k densities in registers over the whole chunk:
//   J: the panel that holds the rows of a tile contracts them over all s (two accumulator sets, even and odd
//      4-column steps, added at the end), so no partial row of B is ever needed;
//   K: every panel contributes its PR rows s to the K columns of all of the warp's tiles.
// The chunk's partial J and K rows go to the workspace.  Pass 2 sums them in chunk order.
//
// No floating-point atomics, and every summation order is fixed by n alone: the chunking (ce_chunk) depends on n,
// the order of the steps within a chunk (r, then s) on nothing else -- not on the panel height or the stage count,
// which the shared-memory budget picks, not on k, and not on the plane range.  A DMMA computes every column of its
// 8 x 8 output from its own column of B, so a density's J and K are bit-identical whatever else is in the batch, at
// whatever position, and a row computed on a shard is bit-identical to the same row of the whole tensor.
#include "common.cuh"

namespace {

constexpr int kCeThreads = 256;
constexpr int kCeWarps = kCeThreads / 32;
constexpr int kCeMaxTiles = 6;  // 8-row tiles per warp: n <= 8 * 8 * 6 = 384

// r per CTA: about 1024 / n, at least 1.  This keeps the partial rows (2 k n per plane and chunk, written and read
// once) below 7 % of the bytes of u for n >= 100 and k <= 16, and gives n * n / c >= 1024 CTAs per full tensor.
inline int64_t ce_chunk(int64_t n) { return qs_ceil_div(1024, n); }

// shared-memory row strides, in doubles: 4 mod 16 keeps both fragment reads (8 rows x 4 columns for J, 4 rows x 8
// columns for K) free of bank conflicts within each half-warp
inline int ce_ld(int64_t n) { return (int)(qs_round_up(n, 16) + 4); }
inline int ce_ldr(int kp) { return kp + 4; }

// panel height and stage count: the first of (64, 2), (32, 2), (64, 1), (32, 1) that fits
struct CeLayout {
    int pr, stages;
    size_t smem;
};

size_t ce_smem(int64_t n, int kp, int pr, int stages) {
    const size_t panel = (size_t)pr * ce_ld(n), rbuf = (size_t)qs_round_up(n, 64) * ce_ldr(kp);
    return 8 * ((size_t)stages * panel + 2 * rbuf);
}

bool ce_layout(int64_t n, int kp, CeLayout* out) {
    const int options[4][2] = {{64, 2}, {32, 2}, {64, 1}, {32, 1}};
    for (const auto& o : options) {
        const size_t b = ce_smem(n, kp, o[0], o[1]);
        if (b <= 227 * 1024) {
            *out = {o[0], o[1], b};
            return true;
        }
    }
    return false;
}

__device__ __forceinline__ void cp_async_16(uint32_t dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_8(uint32_t dst, const void* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// MT: 8-row tiles per warp (ceil(ceil(n / 8) / 8)); NT: 8-density column tiles (k <= 8 NT); V: doubles per copy
// (2: 16-byte copies of an even-length row from a 16-byte aligned u).
template <int MT, int NT, int V>
__global__ void __launch_bounds__(kCeThreads, 1)
    coulomb_exchange_kernel(const double* __restrict__ u, const double* __restrict__ rho, int n, int k, int chunk,
                            int n_chunks, int pr, int stages, double* __restrict__ ws) {
    constexpr int kp = 8 * NT;
    extern __shared__ double ce_smem_d[];
    const int ld = (int)((n + 15) / 16 * 16 + 4), ldr = kp + 4;
    const int n_r = (n + 63) / 64 * 64;
    double* panels = ce_smem_d;                           // [stages][pr][ld]
    double* rbuf = panels + (size_t)stages * pr * ld;     // [2][n_r][ldr]: rbuf[b][s][d] = rho_d[s, r]
    const size_t panel_elems = (size_t)pr * ld, r_elems = (size_t)n_r * ldr;

    const int pl = blockIdx.x / n_chunks;  // plane relative to p_begin
    const int c_idx = blockIdx.x - pl * n_chunks;
    const int r0 = c_idx * chunk;
    const int rc = min(chunk, n - r0);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, t = lane & 3;
    const int n_panels = (n + pr - 1) / pr, items = rc * n_panels;
    const size_t n2 = (size_t)n * n;
    const double* block0 = u + ((size_t)pl * n + r0) * n2;  // u[p, r0]

    // cp.async never writes the padding columns [n, ld) of a panel row, the rows s >= n of R or its columns d >= k:
    // zero them once, a warp per row
    for (int row = warp; row < stages * pr; row += kCeWarps)
        for (int c = n + lane; c < ld; c += 32) panels[row * ld + c] = 0.0;
    for (int row = warp; row < 2 * n_r; row += kCeWarps) {
        const int s = row < n_r ? row : row - n_r;
        for (int d = (s < n ? k : 0) + lane; d < ldr; d += 32) rbuf[row * ldr + d] = 0.0;
    }

    // item i = (rl, j): panel j of u[p, r0 + rl] into stage i % stages, and R of that r with its first panel
    auto issue = [&](int i) {
        const int rl = i / n_panels, j = i - rl * n_panels;
        const int rows = min(pr, n - j * pr);
        const double* src = block0 + (size_t)rl * n2 + (size_t)j * pr * n;
        const uint32_t dst = smem_u32(panels + (size_t)(i % stages) * panel_elems);
        for (int row = warp; row < rows; row += kCeWarps)  // a warp per row: no index division per copy
            for (int col = lane * V; col < n; col += 32 * V) {
                const uint32_t a = dst + 8u * (uint32_t)(row * ld + col);
                if constexpr (V == 2)
                    cp_async_16(a, src + (size_t)row * n + col);
                else
                    cp_async_8(a, src + (size_t)row * n + col);
            }
        if (j == 0) {
            const uint32_t rdst = smem_u32(rbuf + (size_t)(rl & 1) * r_elems);
            const int r = r0 + rl;
            for (int d = warp; d < k; d += kCeWarps)
                for (int s = lane; s < n; s += 32)
                    cp_async_8(rdst + 8u * (uint32_t)(s * ldr + d), rho + (size_t)d * n2 + (size_t)s * n + r);
        }
        cp_async_commit();
    };

    double jacc[MT][NT][2][2], kacc[MT][NT][2];
#pragma unroll
    for (int m = 0; m < MT; ++m)
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            jacc[m][nt][0][0] = jacc[m][nt][0][1] = jacc[m][nt][1][0] = jacc[m][nt][1][1] = 0.0;
            kacc[m][nt][0] = kacc[m][nt][1] = 0.0;
        }

    __syncthreads();  // the zero fill lands before any copy could be mistaken for it
    if (stages == 2) issue(0);
    const int pr_tiles = pr / 8;
    for (int i = 0; i < items; ++i) {
        if (stages == 2) {
            if (i + 1 < items) {
                issue(i + 1);
                cp_async_wait<1>();
            } else {
                cp_async_wait<0>();
            }
        } else {
            issue(i);
            cp_async_wait<0>();
        }
        __syncthreads();
        const int rl = i / n_panels, j = i - rl * n_panels;
        const double* P = panels + (size_t)(i % stages) * panel_elems;
        const double* R = rbuf + (size_t)(rl & 1) * r_elems;
        const int s_base = j * pr, s_rows = min(pr, n - s_base);
#pragma unroll
        for (int m = 0; m < MT; ++m) {
            const int tile = warp + kCeWarps * m;
            if (tile * 8 >= n) continue;
            // J: the tile's rows lie in this panel; contract them over every column s
            if (tile / pr_tiles == j) {
                const double* arow = P + (size_t)(tile * 8 - s_base + g) * ld + t;
                for (int s0 = 0; s0 < n; s0 += 8) {
                    const double a0 = arow[s0], a1 = arow[s0 + 4];
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        const double b0 = R[(s0 + t) * ldr + nt * 8 + g];
                        const double b1 = R[(s0 + 4 + t) * ldr + nt * 8 + g];
                        dmma_8x8x4(jacc[m][nt][0][0], jacc[m][nt][0][1], a0, b0);
                        dmma_8x8x4(jacc[m][nt][1][0], jacc[m][nt][1][1], a1, b1);
                    }
                }
            }
            // K: this panel's rows s into the tile's columns
            const double* acol = P + tile * 8 + g;
            for (int s0 = 0; s0 < s_rows; s0 += 4) {
                const double a = s0 + t < s_rows ? acol[(size_t)(s0 + t) * ld] : 0.0;
#pragma unroll
                for (int nt = 0; nt < NT; ++nt)
                    dmma_8x8x4(kacc[m][nt][0], kacc[m][nt][1], a, R[(s_base + s0 + t) * ldr + nt * 8 + g]);
            }
        }
        __syncthreads();  // the stage and the R buffer are free for the next issue
    }

    // partial rows: ws[pl][c][0 = J, 1 = K][d][q]
    double* out = ws + ((size_t)pl * n_chunks + c_idx) * 2 * k * n;
#pragma unroll
    for (int m = 0; m < MT; ++m) {
        const int q = (warp + kCeWarps * m) * 8 + g;
        if (q >= n) continue;
#pragma unroll
        for (int nt = 0; nt < NT; ++nt)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int d = nt * 8 + 2 * t + e;
                if (d < k) {
                    out[(size_t)d * n + q] = jacc[m][nt][0][e] + jacc[m][nt][1][e];
                    out[((size_t)k + d) * n + q] = kacc[m][nt][e];
                }
            }
    }
}

// J or K of density d, row p_begin + pl: the chunk partials summed in chunk order
__global__ void coulomb_exchange_sum_kernel(const double* __restrict__ ws, double* __restrict__ J,
                                            double* __restrict__ K, int n, int k, int n_chunks, long long p_begin,
                                            long long rows) {
    const long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (e >= 2 * k * rows * n) return;
    const long long q = e % n, rest = e / n;
    const long long pl = rest % rows, wd = rest / rows;  // wd = which * k + d
    double acc = 0.0;
    for (int c = 0; c < n_chunks; ++c) acc += ws[((pl * n_chunks + c) * 2 * k + wd) * n + q];
    const long long which = wd / k, d = wd - which * k;
    (which == 0 ? J : K)[(d * n + p_begin + pl) * n + q] = acc;
}

template <int MT, int NT, int V>
int launch(const void* u, const void* rho, int n, int k, int chunk, int n_chunks, long long rows,
           const CeLayout& lay, void* ws, cudaStream_t st) {
    auto kern = coulomb_exchange_kernel<MT, NT, V>;
    QS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lay.smem));
    kern<<<(unsigned)(rows * n_chunks), kCeThreads, lay.smem, st>>>(
        static_cast<const double*>(u), static_cast<const double*>(rho), n, k, chunk, n_chunks, lay.pr, lay.stages,
        static_cast<double*>(ws));
    QS_LAUNCH_CHECK();
    return QS_OK;
}

template <int NT, int V>
int launch_tiles(int mt, const void* u, const void* rho, int n, int k, int chunk, int n_chunks, long long rows,
                 const CeLayout& lay, void* ws, cudaStream_t st) {
    switch (mt) {
        case 1: return launch<1, NT, V>(u, rho, n, k, chunk, n_chunks, rows, lay, ws, st);
        case 2: return launch<2, NT, V>(u, rho, n, k, chunk, n_chunks, rows, lay, ws, st);
        case 3: return launch<3, NT, V>(u, rho, n, k, chunk, n_chunks, rows, lay, ws, st);
        case 4: return launch<4, NT, V>(u, rho, n, k, chunk, n_chunks, rows, lay, ws, st);
        case 5: return launch<5, NT, V>(u, rho, n, k, chunk, n_chunks, rows, lay, ws, st);
        default: return launch<6, NT, V>(u, rho, n, k, chunk, n_chunks, rows, lay, ws, st);
    }
}

int ce_check_dtypes(const char* entry, int u_dtype, int rho_dtype) {
    for (int d : {u_dtype, rho_dtype}) QS_REQUIRE(d == QS_F64 || d == QS_C128, "%s: bad dtype", entry);
    QS_REQUIRE(u_dtype == QS_F64 && rho_dtype == QS_F64,
               "%s: complex u or densities are not supported (real u and real densities only)", entry);
    return QS_OK;
}

}  // namespace

extern "C" int qs_coulomb_exchange_batch_workspace_bytes(int64_t n, int64_t k, int64_t p_begin, int64_t p_end,
                                                         int u_dtype, int rho_dtype, int64_t* bytes) {
    QS_REQUIRE(bytes && n >= 1 && k >= 1 && k <= QS_COULOMB_EXCHANGE_MAX_BATCH && 0 <= p_begin && p_begin <= p_end &&
                   p_end <= n,
               "qs_coulomb_exchange_batch_workspace_bytes: bad arguments");
    const int status = ce_check_dtypes("qs_coulomb_exchange_batch_workspace_bytes", u_dtype, rho_dtype);
    if (status != QS_OK) return status;
    *bytes = (p_end - p_begin) * qs_ceil_div(n, ce_chunk(n)) * 2 * k * n * 8;
    return QS_OK;
}

extern "C" int qs_coulomb_exchange_batch(const void* u, int u_dtype, const void* rho, int rho_dtype, int64_t n,
                                         int64_t k, void* J, void* K, int64_t p_begin, int64_t p_end,
                                         void* workspace, int64_t workspace_bytes, void* stream) {
    const char* entry = "qs_coulomb_exchange_batch";
    QS_REQUIRE(rho && J && K && n >= 1 && k >= 1, "%s: bad arguments", entry);
    QS_REQUIRE(k <= QS_COULOMB_EXCHANGE_MAX_BATCH, "%s: k = %lld densities, at most %d per launch", entry,
               (long long)k, QS_COULOMB_EXCHANGE_MAX_BATCH);
    QS_REQUIRE(n <= 8 * kCeWarps * kCeMaxTiles, "%s: n = %lld exceeds %d", entry, (long long)n,
               8 * kCeWarps * kCeMaxTiles);
    QS_REQUIRE(0 <= p_begin && p_begin <= p_end && p_end <= n, "%s: bad row range", entry);
    int status = ce_check_dtypes(entry, u_dtype, rho_dtype);
    if (status != QS_OK) return status;
    const long long rows = p_end - p_begin;
    if (rows == 0) return QS_OK;
    int64_t need = 0;
    qs_coulomb_exchange_batch_workspace_bytes(n, k, p_begin, p_end, u_dtype, rho_dtype, &need);
    QS_REQUIRE(u && workspace && workspace_bytes >= need, "%s: workspace too small (%lld < %lld bytes)", entry,
               (long long)workspace_bytes, (long long)need);
    const int chunk = (int)ce_chunk(n), n_chunks = (int)qs_ceil_div(n, chunk);
    QS_REQUIRE(rows * n_chunks < (1LL << 31), "%s: too many planes for one launch", entry);
    const int nt = k <= 8 ? 1 : 2;
    CeLayout lay;
    QS_REQUIRE(ce_layout(n, 8 * nt, &lay), "%s: n = %lld needs more shared memory than a CTA has", entry,
               (long long)n);
    const int mt = (int)qs_ceil_div(qs_ceil_div(n, 8), kCeWarps);
    const bool vec = n % 2 == 0 && (reinterpret_cast<uintptr_t>(u) & 15) == 0;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int ni = (int)n, ki = (int)k;
    if (nt == 1)
        status = vec ? launch_tiles<1, 2>(mt, u, rho, ni, ki, chunk, n_chunks, rows, lay, workspace, st)
                     : launch_tiles<1, 1>(mt, u, rho, ni, ki, chunk, n_chunks, rows, lay, workspace, st);
    else
        status = vec ? launch_tiles<2, 2>(mt, u, rho, ni, ki, chunk, n_chunks, rows, lay, workspace, st)
                     : launch_tiles<2, 1>(mt, u, rho, ni, ki, chunk, n_chunks, rows, lay, workspace, st);
    if (status != QS_OK) return status;
    coulomb_exchange_sum_kernel<<<(unsigned)qs_ceil_div(2 * k * rows * n, 256), 256, 0, st>>>(
        static_cast<const double*>(workspace), static_cast<double*>(J), static_cast<double*>(K), ni, ki, n_chunks,
        p_begin, rows);
    QS_LAUNCH_CHECK();
    return QS_OK;
}
