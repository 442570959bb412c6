// Shared device/host helpers for libqsb200 (sm_100a only).
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/qsb200.h"

// ---------------------------------------------------------------------------------------------
// host-side error plumbing
// ---------------------------------------------------------------------------------------------
void qs_set_error(const char* fmt, ...);

#define QS_CUDA(call)                                                                          \
    do {                                                                                       \
        cudaError_t _e = (call);                                                               \
        if (_e != cudaSuccess) {                                                               \
            qs_set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__,     \
                         __LINE__);                                                            \
            return QS_ERR_CUDA;                                                                \
        }                                                                                      \
    } while (0)

#define QS_REQUIRE(cond, ...)                                                                  \
    do {                                                                                       \
        if (!(cond)) {                                                                         \
            qs_set_error(__VA_ARGS__);                                                         \
            return QS_ERR_INVALID;                                                             \
        }                                                                                      \
    } while (0)

#define QS_LAUNCH_CHECK()                                                                      \
    do {                                                                                       \
        qs_count_launch();                                                                     \
        cudaError_t _e = cudaGetLastError();                                                   \
        if (_e != cudaSuccess) {                                                               \
            qs_set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, \
                         __LINE__);                                                            \
            return QS_ERR_CUDA;                                                                \
        }                                                                                      \
    } while (0)

static inline int64_t qs_round_up(int64_t v, int64_t m) { return (v + m - 1) / m * m; }
static inline int64_t qs_ceil_div(int64_t v, int64_t m) { return (v + m - 1) / m; }
static inline int qs_elem_doubles(int dtype) { return dtype == QS_C128 ? 2 : 1; }

// Instrumentation (core.cu): every kernel launch is counted; when timing is enabled the launch
// sites of a kernel family bracket themselves with CUDA events on the launching stream.
void qs_count_launch();
bool qs_timing_begin(int family, double work, void* stream, int* slot);
void qs_timing_end(int slot, void* stream);

// Number of SMs of the current device, and the device ordinal itself (clamped to [0, kMaxDevices)); both
// caches are per device so that one process may drive several GPUs.
constexpr int kMaxDevices = 64;
int qs_current_device();
int qs_sm_count();

// Shape-dependent index tables (tile lists of masked launches, pair tables of the packed layouts) are the same for
// every call with the same extents.  They are built on the host ONCE per (device, key), uploaded with a blocking
// copy and kept in device memory for the life of the process, so that a steady-state transform issues no
// host-to-device copy at all (a cudaMemcpyAsync from pageable memory synchronises the stream first and drains the
// launch queue).  `key` is any byte string that determines the contents; returns nullptr when the cache is full
// (the caller then stages the table through its workspace as before).
const void* qs_table_cache_get(const void* key, size_t key_bytes);
const void* qs_table_cache_put(const void* key, size_t key_bytes, const void* host_data, size_t bytes);
uint64_t qs_hash_bytes(const void* data, size_t bytes, uint64_t seed);

// Internal (not part of the C ABI): symmetry mask of a quarter transform (see quarter_gemm.cu, tile_wanted) and
// the masked launch used by the symmetry-aware four-index transform (transform.cu).
// Which of the two ordered pairs (r, s), (s, r) the SHARDED symmetry-aware transform computes: the one whose
// cyclic distance d = (s - r) mod m is the shorter (ties, 2 d = m, go to r < s).  Every r then has the same number
// of partners s, so any partition of r over the ranks stays balanced.
#ifdef __CUDACC__
__host__ __device__
#endif
static inline bool qs_cyclic_wanted(long long r, long long s, long long m) {
    const long long d = s >= r ? s - r : s - r + m;
    return d > 0 && (2 * d < m || (2 * d == m && r < s));
}

struct QsTileMask {
    int kind;             // 0 none; 1 column < row_lo; 2 row_hi < row_lo; 3 cyclic pair rule on (column, row_lo):
                          //   wanted iff qs_cyclic_wanted(column, row_lo, ml), or (strict == 0) the same with the
                          //   other member row_lo ^ 1 of the aligned couple (the padded pair lists of the real case)
    int strict;           // 1: "<", 0: "<="
    int64_t dh, mh, dl, ml;  // row_hi(x) = (x / dh) % mh, row_lo(x) = (x / dl) % ml
};
int64_t qs_tile_list_bytes(int64_t X, int64_t K, int64_t W, int a_dtype, int m_dtype);

// Where a quarter transform stores, and which of its tiles it computes.  Output element (x, w), in output elements
// (complex output: complex elements), with x = (x2 * x_mid + x1) * x_inner + x0:
//     (w / w_inner) * sw1 + (w % w_inner) * sw0 + x2 * sx2 + x1 * sx1 + x0 * sx0
// Defaults: one local destination, no middle row split, undealt columns, no tables, every tile; strides are 0.
struct QsQuarterStore {
    void* out = nullptr;                  // the local destination, or:
    void* const* out_table = nullptr;     // scattering store: n_dest destinations, w / w_inner selects one (sw1 unused)
    int64_t n_dest = 0;
    int w_cyclic = 0;                     // scattering: column w goes to destination w % n_dest as its column w / n_dest
    int64_t w_deal = 1;                   // column dealing: logical column j is stored as column (j * w_deal) % W
    int64_t x_inner = 1, x_mid = 0xFFFFFFFFLL, w_inner = 1;  // x_mid 0xFFFFFFFF: x = x1 * x_inner + x0, no sx2
    int64_t sx0 = 0, sx1 = 0, sx2 = 0, sw0 = 0, sw1 = 0;
    // Row tables (device memory), with x = xq * x_inner + xr: row x is at xq_table[xq] + xr_table[xr] in place of
    // xq * sx1 and xr * sx0; a negative xq_table entry drops the rows of that block.
    const long long* xq_table = nullptr;
    const long long* xr_table = nullptr;
    int xq_even = 0;                      // promise: every kept xq_table entry is even
    int xr_paired = 0;                    // promise: xr_table places rows 2k, 2k + 1 adjacently at an even offset
    // Column tables (device memory, W entries each, indexed by the physical column): column w goes to destination
    // out_table[col_dest[w]] at element offset col_off[w], in place of the w / w_inner, w_cyclic and sw0 rules.
    const int32_t* col_dest = nullptr;
    const long long* col_off = nullptr;
    int col_off_even = 0;                 // promise: every col_off entry is even
    // Masked launch: only the tiles the mask, or the host copy of the block table, wants.  list_ws holds
    // qs_tile_list_bytes() bytes of device memory.
    const QsTileMask* mask = nullptr;
    const long long* host_xq_table = nullptr;
    void* list_ws = nullptr;
};
int qs_quarter_launch(const void* A, int a_dtype, int64_t X, int64_t K, int64_t lda, const void* image, int m_dtype,
                      int64_t W, const QsQuarterStore& st, void* stream);

int qs_mirror_fill(void* out, int dtype, int64_t m, int mode, void* stream);

// Internal (not part of the C ABI): coefficient image of the ODQD shielded-Coulomb matrix.
int qs_build_coulomb_image(const double* grid, double alpha, double a, int64_t Gp, void* image, void* stream);

// Internal (not part of the C ABI): planes p in [p_begin, p_end) of qs_transform_two_body_diagonal (structured.cu),
// written to `out`, which points at plane p_begin; the arguments are checked by the exported entries.  A null w2d
// means that the caller has already written the coefficient image of W (w_dtype, as qs_build_coeff_image lays it out
// for A = D) at the start of the workspace: the ODQD build generates it there with qs_build_coulomb_image.
int qs_transform_diagonal_planes(const void* w2d, int w_dtype, const void* C, const void* Ct, int c_dtype, int64_t n,
                                 int64_t m, int64_t p_begin, int64_t p_end, int anti_symmetrize, void* out,
                                 void* workspace, void* stream);

#ifdef __CUDACC__
// ---------------------------------------------------------------------------------------------
// PTX wrappers: mbarrier, TMA (tensor and 1-D bulk), FP64 tensor-core MMA
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}

__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
                 : "memory");
}

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "QS_WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra QS_DONE_%=;\n"
        "bra QS_WAIT_%=;\n"
        "QS_DONE_%=:\n"
        "}\n" ::"r"(bar),
        "r"(parity)
        : "memory");
}

// 2-D tiled TMA load: box at (c0 = fastest coordinate, c1) -> shared, completes on `bar`.
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1,
                                            uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, "
        "{%2, %3}], [%4];" ::"r"(dst),
        "l"(map), "r"(c0), "r"(c1), "r"(bar)
        : "memory");
}

// 1-D bulk copy global -> shared (size multiple of 16 B), completes on `bar`.
__device__ __forceinline__ void bulk_load_1d(uint32_t dst, const void* src, uint32_t bytes,
                                             uint32_t bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
            "r"(dst),
        "l"(src), "r"(bytes), "r"(bar)
        : "memory");
}

__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

// D(8x8) += A(8x4, row) * B(4x8, col) in FP64 on the tensor pipe; SASS: DMMA.8x8x4.
// Lane (g = lane >> 2, t = lane & 3) supplies A[g][t], B[t][g] and owns D[g][2t], D[g][2t+1].
__device__ __forceinline__ void dmma_8x8x4(double& d0, double& d1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(d0), "+d"(d1)
                 : "d"(a), "d"(b));
}

__device__ __forceinline__ void sts_128(uint32_t addr, double a, double b) {
    asm volatile("st.shared.v2.f64 [%0], {%1, %2};" ::"r"(addr), "d"(a), "d"(b) : "memory");
}

// Asynchronous bulk copy shared -> global (16-byte aligned on both sides, size a multiple of 16 B), tracked by the
// issuing thread's bulk async-groups (cp.async.bulk.commit_group / wait_group[.read]).
__device__ __forceinline__ void bulk_store(void* dst, uint32_t src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(bytes)
                 : "memory");
}

__device__ __forceinline__ double2 lds_128(uint32_t addr) {
    double2 v;
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(addr));
    return v;
}
#endif  // __CUDACC__
