// Fock-matrix construction: strided gathers over the occupied index, reduced with warp shuffles.
//
//   qs_fock_general : f = h + sum_i u[p,i,q,i]                 (reference general_orbital_system.py:119-159)
//   qs_fock_spatial : f = h + 2 sum_i u[p,i,q,i] - sum_i u[p,i,i,q]   (reference spatial_orbital_system.py:150-190)
//
// One warp per output element (p, q): lanes stride over the occupied index i, each lane gathers
// u[p,i,q,i] (one 8/16-byte element per 32-byte sector: the pass is sector/latency-bound, not
// bandwidth-bound), then a butterfly __shfl_xor reduction; lane 0 adds h and writes f.
#include "common.cuh"

namespace {

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}

// direct term element (p, i, q) at ud[p*a0 + i*a1 + q*a2], exchange term at ue[p*b0 + i*b1 + q*b2]
struct FockStrides {
    long long a0, a1, a2, b0, b1, b2;
    double scale_d, scale_e;
};

template <bool H_COMPLEX, bool U_COMPLEX, bool EXCHANGE>
__global__ void __launch_bounds__(256) fock_kernel(const double* __restrict__ h, const double* __restrict__ ud,
                                                   const double* __restrict__ ue, double* __restrict__ f, int n,
                                                   int n_occ, long long p_begin, long long p_end, int q_begin,
                                                   int q_count, FockStrides st) {
    const int lane = threadIdx.x & 31;
    const long long warp_global = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    const long long warps_total = ((long long)gridDim.x * blockDim.x) >> 5;
    const long long rows = p_end - p_begin;
    // q runs over the local columns [0, q_count) of the u block; global column = q_begin + q
    for (long long e = warp_global; e < rows * q_count; e += warps_total) {
        const long long pl = e / q_count;  // local row (the u pointers address plane p_begin)
        const int q = (int)(e - pl * q_count);
        double sr = 0.0, si = 0.0;
        for (int i = lane; i < n_occ; i += 32) {
            const long long direct = pl * st.a0 + i * st.a1 + q * st.a2;
            if (U_COMPLEX) {
                const double2 v = reinterpret_cast<const double2*>(ud)[direct];
                sr += st.scale_d * v.x;
                si += st.scale_d * v.y;
            } else {
                sr += st.scale_d * ud[direct];
            }
            if (EXCHANGE) {
                const long long exch = pl * st.b0 + i * st.b1 + q * st.b2;
                if (U_COMPLEX) {
                    const double2 v = reinterpret_cast<const double2*>(ue)[exch];
                    sr += st.scale_e * v.x;
                    si += st.scale_e * v.y;
                } else {
                    sr += st.scale_e * ue[exch];
                }
            }
        }
        sr = warp_sum(sr);
        if (U_COMPLEX) si = warp_sum(si);
        if (lane == 0) {
            const long long o = (p_begin + pl) * n + q_begin + q;
            if (H_COMPLEX) {
                const double2 hv = reinterpret_cast<const double2*>(h)[o];
                reinterpret_cast<double2*>(f)[o] = make_double2(hv.x + sr, hv.y + si);
            } else {
                f[o] = h[o] + sr;
            }
        }
    }
}

int launch_fock(const void* h, int h_dtype, const void* ud, const void* ue, int u_dtype, int64_t n, int64_t n_occ,
                void* f, int64_t p_begin, int64_t p_end, const FockStrides& strides, void* stream,
                int64_t q_begin = 0, int64_t q_count = -1) {
    if (q_count < 0) q_count = n;
    QS_REQUIRE(0 <= n_occ && n_occ <= n, "qs_fock: n_occ out of range");
    // no occupied orbital or an empty row / column range: u is never read, and an empty block may be NULL
    QS_REQUIRE(h && f && n > 0 && (ud || n_occ == 0 || p_begin == p_end || q_count == 0), "qs_fock: bad arguments");
    QS_REQUIRE(0 <= p_begin && p_begin <= p_end && p_end <= n, "qs_fock: bad row range");
    QS_REQUIRE(0 <= q_begin && q_begin + q_count <= n, "qs_fock: bad column range");
    QS_REQUIRE(!(h_dtype == QS_F64 && u_dtype == QS_C128),
               "qs_fock: complex u cannot be accumulated into a real Fock matrix");
    if (p_begin == p_end || q_count == 0) return QS_OK;
    const long long warps = (p_end - p_begin) * q_count;
    long long blocks = qs_ceil_div(warps, 8);
    const long long cap = (long long)qs_sm_count() * 32;
    if (blocks > cap) blocks = cap;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const double* hp = static_cast<const double*>(h);
    const double* dp = static_cast<const double*>(ud);
    const double* ep = static_cast<const double*>(ue);
    double* fp = static_cast<double*>(f);
    const int N = (int)n, NO = (int)n_occ, QB = (int)q_begin, QC = (int)q_count;
#define QS_FOCK_LAUNCH(HC, UC)                                                                                     \
    do {                                                                                                           \
        if (ue)                                                                                                    \
            fock_kernel<HC, UC, true><<<(unsigned)blocks, 256, 0, st>>>(hp, dp, ep, fp, N, NO, p_begin, p_end, QB, QC, strides);  \
        else                                                                                                       \
            fock_kernel<HC, UC, false><<<(unsigned)blocks, 256, 0, st>>>(hp, dp, ep, fp, N, NO, p_begin, p_end, QB, QC, strides); \
    } while (0)
    if (h_dtype == QS_C128 && u_dtype == QS_C128)
        QS_FOCK_LAUNCH(true, true);
    else if (h_dtype == QS_C128)
        QS_FOCK_LAUNCH(true, false);
    else
        QS_FOCK_LAUNCH(false, false);
#undef QS_FOCK_LAUNCH
    QS_LAUNCH_CHECK();
    return QS_OK;
}

}  // namespace

extern "C" int qs_fock_general(const void* h, int h_dtype, const void* u, int u_dtype, int64_t n, int64_t n_occ, void* f,
                               int64_t p_begin, int64_t p_end, void* stream) {
    // u[p,i,q,i]: p*n^3 + i*(n^2 + 1) + q*n
    const FockStrides st = {n * n * n, n * n + 1, n, 0, 0, 0, 1.0, 0.0};
    return launch_fock(h, h_dtype, u, nullptr, u_dtype, n, n_occ, f, p_begin, p_end, st, stream);
}

extern "C" int qs_fock_spatial(const void* h, int h_dtype, const void* u, int u_dtype, int64_t n, int64_t n_occ, void* f,
                               int64_t p_begin, int64_t p_end, void* stream) {
    // 2 u[p,i,q,i] - u[p,i,i,q]: exchange at p*n^3 + i*(n^2 + n) + q
    const FockStrides st = {n * n * n, n * n + 1, n, n * n * n, n * n + n, 1, 2.0, -1.0};
    return launch_fock(h, h_dtype, u, u, u_dtype, n, n_occ, f, p_begin, p_end, st, stream);
}

extern "C" int qs_fock_gathered(const void* h, int h_dtype, const void* direct, const void* exchange, int u_dtype,
                                int64_t n, int64_t n_occ, double scale_direct, double scale_exchange, void* f,
                                void* stream) {
    // direct[i,p,q] = u[p,i,q,i] and exchange[i,p,q] = u[p,i,i,q] gathered by the caller: (n_occ, n, n) blocks
    const FockStrides st = {n, n * n, 1, n, n * n, 1, scale_direct, scale_exchange};
    return launch_fock(h, h_dtype, direct, exchange, u_dtype, n, n_occ, f, 0, n, st, stream);
}

extern "C" int qs_fock_general_cols(const void* h, int h_dtype, const void* u_cols, int u_dtype, int64_t n,
                                    int64_t n_occ, void* f, int64_t q_begin, int64_t q_end, void* stream) {
    // u_cols is the (n, n, q_end - q_begin, n) block u[:, :, q_begin:q_end, :] of a tensor sharded on its
    // third index (the layout a sharded change_basis leaves behind); columns [q_begin, q_end) of f are written.
    QS_REQUIRE(0 <= q_begin && q_begin <= q_end && q_end <= n, "qs_fock_general_cols: bad column range");
    const int64_t qc = q_end - q_begin;
    // u[p,i,q,i]: p*(n*qc*n) + i*(qc*n + 1) + q*n
    const FockStrides st = {n * qc * n, qc * n + 1, n, 0, 0, 0, 1.0, 0.0};
    return launch_fock(h, h_dtype, u_cols, nullptr, u_dtype, n, n_occ, f, 0, n, st, stream, q_begin, qc);
}
