// Four-index transform of a two-body operator that is DIAGONAL in the original basis,
//   u[a,b,c,d] = W[a,b] delta_ac delta_bd        (sinc-DVR storage u_repr = "2d"),
//   u'[p,q,r,s] = sum_ab Ct[p,a] C[a,r] Ct[q,b] C[b,s] W[a,b]      ( - the r <-> s exchange if anti-symmetrised )
// replaces the 5-operand einsum of ODSincDVR.transform_two_body_elements (reference
// sinc_dvr/one_dim/sinc_dvr.py:217-252).  O(m^2 n^2 + m^4 n) instead of the O(n^5) of the dense transform,
// as two chained DMMA GEMMs:
//   D[(p,r), a]   = Ct[p,a] C[a,r]                   (pair products, memory-bound kernel below)
//   Tt[b, (p,r)]  = sum_a D[(p,r), a] W[a,b]         (quarter GEMM, rotated store)
//   u'[p,q,r,s]   = sum_b D[(q,s), b] Tt[b, (p,r)]   (quarter GEMM; the prqs -> pqrs permutation is the store stride)
// The ODQD grid Coulomb build (odqd.cu) is the same transform with W generated from the grid and Ct = C^T, on a
// range of planes p.
#include "common.cuh"

namespace {

// Workspace: the image of W, D, Tt, the image of Tt and the temporary of the anti-symmetrised result, in this order.
// The image of W comes first so that a caller that generates W (the ODQD build) knows where to write it.
struct DiagPlan {
    int d_dtype, t_dtype;
    int64_t pitch, img1_bytes, d_bytes, tt_bytes, img2_bytes, tmp_bytes, total;
};

int make_diag_plan(int64_t n, int64_t m, int w_dtype, int c_dtype, int anti_symmetrize, DiagPlan* plan) {
    plan->d_dtype = c_dtype;
    plan->t_dtype = (w_dtype == QS_C128 || c_dtype == QS_C128) ? QS_C128 : QS_F64;
    plan->pitch = c_dtype == QS_C128 ? n : n + (n & 1);
    const int64_t m2 = m * m;
    plan->d_bytes = qs_round_up(m2 * plan->pitch * 8 * qs_elem_doubles(plan->d_dtype), 1024);
    plan->tt_bytes = qs_round_up(n * m2 * 8 * qs_elem_doubles(plan->t_dtype), 1024);
    int rc = qs_coeff_image_bytes(n, n, plan->d_dtype, w_dtype, &plan->img1_bytes);
    if (rc) return rc;
    rc = qs_coeff_image_bytes(n, m2, plan->d_dtype, plan->t_dtype, &plan->img2_bytes);
    if (rc) return rc;
    plan->img1_bytes = qs_round_up(plan->img1_bytes, 1024);
    plan->img2_bytes = qs_round_up(plan->img2_bytes, 1024);
    plan->tmp_bytes = anti_symmetrize ? qs_round_up(m2 * m2 * 8 * qs_elem_doubles(plan->t_dtype), 1024) : 0;
    plan->total = plan->d_bytes + plan->tt_bytes + plan->img1_bytes + plan->img2_bytes + plan->tmp_bytes;
    return QS_OK;
}

// D[(x * m + y) * pitch + k] = L[x, k] * R[k, y],  L[x, k] = l[x * lsx + k * lsk] (conjugated if l_conj),
// R[k, y] = r[k * m + y].  One CTA: 32 consecutive k (one per lane -> coalesced stores) x XT x-values x YT y-values.
constexpr int kXT = 8, kYT = 64;

template <bool COMPLEX>
__global__ void __launch_bounds__(256) pair_product_kernel(const double* __restrict__ l, long long lsx, long long lsk,
                                                           int l_conj, const double* __restrict__ r,
                                                           double* __restrict__ D, int n, int m, int pitch) {
    constexpr int E = COMPLEX ? 2 : 1;
    __shared__ double ls[kXT][32 * E + 1];
    __shared__ double rs[32][kYT * E + 1];
    const int k0 = blockIdx.x * 32, x0 = blockIdx.y * kXT, y0 = blockIdx.z * kYT;
    for (int i = threadIdx.x; i < kXT * 32; i += blockDim.x) {
        const int xx = i >> 5, kk = i & 31;
        const bool ok = x0 + xx < m && k0 + kk < n;
        const long long src = (long long)(x0 + xx) * lsx + (long long)(k0 + kk) * lsk;
        if (COMPLEX) {
            ls[xx][2 * kk] = ok ? l[2 * src] : 0.0;
            ls[xx][2 * kk + 1] = ok ? (l_conj ? -l[2 * src + 1] : l[2 * src + 1]) : 0.0;
        } else {
            ls[xx][kk] = ok ? l[src] : 0.0;
        }
    }
    for (int i = threadIdx.x; i < 32 * kYT; i += blockDim.x) {
        const int kk = i / kYT, yy = i - kk * kYT;
        const bool ok = k0 + kk < n && y0 + yy < m;
        const long long src = (long long)(k0 + kk) * m + y0 + yy;
        if (COMPLEX) {
            rs[kk][2 * yy] = ok ? r[2 * src] : 0.0;
            rs[kk][2 * yy + 1] = ok ? r[2 * src + 1] : 0.0;
        } else {
            rs[kk][yy] = ok ? r[src] : 0.0;
        }
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int k = k0 + lane;
    if (k >= pitch) return;  // columns n <= k < pitch are written as zeros (the tiles were zero-filled)
    for (int xy = warp; xy < kXT * kYT; xy += nwarps) {
        const int xx = xy / kYT, yy = xy - xx * kYT;
        if (x0 + xx >= m || y0 + yy >= m) continue;
        const long long dst = ((long long)(x0 + xx) * m + y0 + yy) * pitch + k;
        if (COMPLEX) {
            const double ar = ls[xx][2 * lane], ai = ls[xx][2 * lane + 1];
            const double br = rs[lane][2 * yy], bi = rs[lane][2 * yy + 1];
            reinterpret_cast<double2*>(D)[dst] = make_double2(ar * br - ai * bi, ar * bi + ai * br);
        } else {
            D[dst] = ls[xx][lane] * rs[lane][yy];
        }
    }
}

}  // namespace

int qs_transform_diagonal_planes(const void* w2d, int w_dtype, const void* C, const void* Ct, int c_dtype, int64_t n,
                                 int64_t m, int64_t p_begin, int64_t p_end, int anti_symmetrize, void* out,
                                 void* workspace, void* stream) {
    DiagPlan plan;
    int rc = make_diag_plan(n, m, w_dtype, c_dtype, anti_symmetrize, &plan);
    if (rc) return rc;
    char* ws = static_cast<char*>(workspace);
    void* img1 = ws;
    double* D = reinterpret_cast<double*>(ws + plan.img1_bytes);
    void* Tt = ws + plan.img1_bytes + plan.d_bytes;
    void* img2 = static_cast<char*>(Tt) + plan.tt_bytes;
    void* tmp = static_cast<char*>(img2) + plan.img2_bytes;
    cudaStream_t st = static_cast<cudaStream_t>(stream);

    // D[(p,r), a] = Ct[p,a] C[a,r];  Ct = conj(C)^T when absent (reference sinc_dvr.py:225-226).  D is built whole: it
    // is the A operand of the second GEMM for every (q,s).
    const double* lmat = static_cast<const double*>(Ct ? Ct : C);
    const long long lsx = Ct ? n : 1, lsk = Ct ? 1 : m;
    const int l_conj = Ct ? 0 : 1;
    dim3 grid((unsigned)qs_ceil_div(plan.pitch, 32), (unsigned)qs_ceil_div(m, kXT), (unsigned)qs_ceil_div(m, kYT));
    if (c_dtype == QS_C128)
        pair_product_kernel<true><<<grid, 256, 0, st>>>(lmat, lsx, lsk, l_conj, static_cast<const double*>(C), D, (int)n,
                                                        (int)m, (int)plan.pitch);
    else
        pair_product_kernel<false><<<grid, 256, 0, st>>>(lmat, lsx, lsk, l_conj, static_cast<const double*>(C), D,
                                                         (int)n, (int)m, (int)plan.pitch);
    QS_LAUNCH_CHECK();

    const int64_t m2 = m * m;
    const int64_t rows = (p_end - p_begin) * m;  // the rows (p_loc, r) of T these planes need
    // Tt[b, (p_loc,r)]: rows x = (p_loc,r), K = a, new index w = b stored slowest
    if (w2d && (rc = qs_build_coeff_image(w2d, w_dtype, n, 1, 0, n, n, plan.d_dtype, img1, stream))) return rc;
    if ((rc = qs_quarter_transform(D + p_begin * m * plan.pitch * qs_elem_doubles(plan.d_dtype), plan.d_dtype, rows,
                                   n, plan.pitch, img1, w_dtype, n, Tt, rows, 1, 0, 1, 0, rows, stream)))
        return rc;
    // M[k = b, w = (p_loc,r)] = Tt[b * rows + (p_loc,r)]
    if ((rc = qs_build_coeff_image(Tt, plan.t_dtype, rows, 1, 0, n, rows, plan.d_dtype, img2, stream))) return rc;
    // u'[p_loc,q,r,s]: x = (q,s) -> q m^2 + s ; w = (p_loc,r) -> p_loc m^3 + r m
    void* dst = anti_symmetrize ? tmp : out;
    if ((rc = qs_quarter_transform(D, plan.d_dtype, m2, n, plan.pitch, img2, plan.t_dtype, rows, dst, m, 1, m2, m, m,
                                   m2 * m, stream)))
        return rc;
    if (anti_symmetrize) return qs_anti_symmetrize(tmp, plan.t_dtype, m, out, 0, p_end - p_begin, stream);
    return QS_OK;
}

extern "C" int qs_transform_two_body_diagonal_workspace_bytes(int64_t n, int64_t m, int w_dtype, int c_dtype,
                                                              int anti_symmetrize, int64_t* bytes) {
    QS_REQUIRE(n > 0 && m > 0 && bytes, "qs_transform_two_body_diagonal_workspace_bytes: bad arguments");
    DiagPlan plan;
    const int rc = make_diag_plan(n, m, w_dtype, c_dtype, anti_symmetrize, &plan);
    if (rc) return rc;
    *bytes = plan.total;
    return QS_OK;
}

extern "C" int qs_transform_two_body_diagonal(const void* w2d, int w_dtype, const void* C, const void* Ct, int c_dtype,
                                              int64_t n, int64_t m, int anti_symmetrize, void* out, void* workspace,
                                              int64_t workspace_bytes, void* stream) {
    QS_REQUIRE(w2d && C && out && workspace, "qs_transform_two_body_diagonal: null pointer");
    QS_REQUIRE(n > 0 && m > 0 && m <= 4096 && n < (1 << 24), "qs_transform_two_body_diagonal: bad extents");
    QS_REQUIRE((w_dtype == QS_F64 || w_dtype == QS_C128) && (c_dtype == QS_F64 || c_dtype == QS_C128),
               "qs_transform_two_body_diagonal: bad dtype");
    DiagPlan plan;
    int rc = make_diag_plan(n, m, w_dtype, c_dtype, anti_symmetrize, &plan);
    if (rc) return rc;
    QS_REQUIRE(workspace_bytes >= plan.total, "qs_transform_two_body_diagonal: workspace too small (%lld < %lld)",
               (long long)workspace_bytes, (long long)plan.total);
    QS_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 1023) == 0,
               "qs_transform_two_body_diagonal: workspace must be 1 KiB aligned");
    return qs_transform_diagonal_planes(w2d, w_dtype, C, Ct, c_dtype, n, m, 0, m, anti_symmetrize, out, workspace,
                                        stream);
}
