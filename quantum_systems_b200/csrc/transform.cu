// Whole-tensor basis changes built from quarter GEMMs.
//
//   qs_transform_two_body : BasisSet.transform_two_body_elements (reference basis_set.py:336-350)
//   qs_transform_one_body : BasisSet.transform_one_body_elements (reference basis_set.py:329-334)
//
// Four launches of the same kernel "contract the last index, store the new index slowest":
//   u[a,b,c,d] -C-> T1[s,a,b,c] -C-> T2[r,s,a,b] -Ct^T-> T3[q,r,s,a] -Ct^T-> out[p,q,r,s]
// which is the reference's contraction order (s, r, q, p) with every transpose folded into a store.
#include <vector>

#include "common.cuh"

namespace {

// Real tensors with an odd contracted extent cannot be described to TMA directly (row pitch must be a
// multiple of 16 bytes), so every real (X, n) operand uses pitch P = n + (n & 1).  Intermediates are
// written at that pitch by the producing epilogue for free; only the caller's input needs one copy.
struct TwoBodyPlan {
    int t_dtype;  // dtype of every intermediate and of the result
    int64_t pitch_u, pitch_t;
    int64_t pad_bytes, bufA_bytes, bufB_bytes, img_bytes[2], list_bytes, table_bytes, total;
};

int64_t padded_pitch(int64_t n, int dtype) { return dtype == QS_C128 ? n : n + (n & 1); }

int make_plan(int64_t n, int64_t m, int u_dtype, int c_dtype, TwoBodyPlan* plan) {
    plan->t_dtype = (u_dtype == QS_C128 || c_dtype == QS_C128) ? QS_C128 : QS_F64;
    plan->pitch_u = padded_pitch(n, u_dtype);
    plan->pitch_t = padded_pitch(n, plan->t_dtype);
    const int64_t es = 8 * qs_elem_doubles(plan->t_dtype);
    const int64_t P = plan->pitch_t;
    const int64_t t1 = m * n * n * P, t2 = m * m * n * P, t3 = m * m * m * P;
    plan->pad_bytes = plan->pitch_u != n ? qs_round_up(n * n * n * plan->pitch_u * 8, 1024) : 0;
    plan->bufA_bytes = qs_round_up((t1 > t3 ? t1 : t3) * es, 1024);
    plan->bufB_bytes = qs_round_up(t2 * es, 1024);
    // image 0: first step, A has the dtype of u; image 1: later steps, A has t_dtype
    int rc = qs_coeff_image_bytes(n, m, u_dtype, c_dtype, &plan->img_bytes[0]);
    if (rc) return rc;
    rc = qs_coeff_image_bytes(n, m, plan->t_dtype, c_dtype, &plan->img_bytes[1]);
    if (rc) return rc;
    plan->img_bytes[0] = qs_round_up(plan->img_bytes[0], 1024);
    plan->img_bytes[1] = qs_round_up(plan->img_bytes[1], 1024);
    // tile lists of the symmetry-aware variant (steps 2-4), a few hundred KB at most
    int64_t lists = qs_tile_list_bytes(m * n * n, n, m, plan->t_dtype, c_dtype);
    const int64_t l3 = qs_tile_list_bytes(m * m * n, n, m, plan->t_dtype, c_dtype);
    const int64_t l4 = qs_tile_list_bytes(m * m * m, n, m, plan->t_dtype, c_dtype);
    lists = lists > l3 ? lists : l3;
    lists = lists > l4 ? lists : l4;
    plan->list_bytes = qs_round_up(lists, 1024);
    // row-offset tables of the packed pair layout: m^2 entries (step 3 rows -> pair slot) + m(m+1)/2 (pair -> r m + s)
    plan->table_bytes = qs_round_up((m * m + m * (m + 1) / 2 + m) * (int64_t)sizeof(long long), 1024);
    // images: [C for step 1][C for step 2][Ct^T for steps 3, 4]
    plan->total = plan->pad_bytes + plan->bufA_bytes + plan->bufB_bytes + plan->img_bytes[0] + 2 * plan->img_bytes[1] +
                  plan->list_bytes + plan->table_bytes;
    return QS_OK;
}

__global__ void pad_rows_kernel(const double* __restrict__ in, double* __restrict__ out, long long rows, int n,
                                int pitch) {
    const long long total = rows * pitch;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const long long r = i / pitch;
        const int c = (int)(i - r * pitch);
        out[i] = c < n ? in[r * n + c] : 0.0;
    }
}

int pad_rows(const void* in, void* out, int64_t rows, int64_t n, int64_t pitch, void* stream) {
    const long long total = rows * pitch;
    long long blocks = qs_ceil_div(total, 256);
    const long long cap = (long long)qs_sm_count() * 16;
    if (blocks > cap) blocks = cap;
    pad_rows_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const double*>(in), static_cast<double*>(out), rows, (int)n, (int)pitch);
    QS_LAUNCH_CHECK();
    return QS_OK;
}

// Contract the last index of A (rows X, extent K, pitch lda) and store the new index slowest; the
// remaining row index x = (x_hi, x_lo) with x_lo < lo_extent is written at x_hi * lo_pitch + x_lo.
int rotated_quarter(const void* A, int a_dtype, int64_t X, int64_t K, int64_t lda, const void* image, int m_dtype,
                    int64_t W, void* out, int64_t lo_extent, int64_t lo_pitch, void* stream) {
    const int64_t plane = X / lo_extent * lo_pitch;
    return qs_quarter_transform(A, a_dtype, X, K, lda, image, m_dtype, W, out, lo_extent, 1, lo_pitch, 1, 0, plane,
                                stream);
}

int masked_rotated_quarter(const void* A, int a_dtype, int64_t X, int64_t K, int64_t lda, const void* image,
                           int m_dtype, int64_t W, void* out, int64_t lo_extent, int64_t lo_pitch,
                           const QsTileMask* mask, void* list_ws, void* stream) {
    QsQuarterStore s;
    s.out = out;
    s.x_inner = lo_extent;
    s.sx0 = 1;
    s.sx1 = lo_pitch;
    s.sw1 = X / lo_extent * lo_pitch;
    s.mask = mask;
    s.list_ws = list_ws;
    return qs_quarter_launch(A, a_dtype, X, K, lda, image, m_dtype, W, s, stream);
}

// ---------------------------------------------------------------------------------------------
// One-body matrices (n x n, a few hundred KB): out = Ct (h C).  Through the persistent quarter GEMM each of the two
// products is a single 128-row tile -- one or two CTAs, a 25 us latency chain per launch next to 3 us of image
// building -- so small matrices take a plain shared-memory tiled FP64 kernel instead: every 32 x 32 output tile is
// a CTA, the whole chip works on one product for a few microseconds.
//   D[i, j] = sum_k opA(A)[i, k] * B[k, j],   opA(A)[i, k] = A[i * sa_i + k * sa_k], optionally conjugated
// ---------------------------------------------------------------------------------------------
template <bool A_COMPLEX, bool B_COMPLEX>
__global__ void __launch_bounds__(256) small_matmul_kernel(const double* __restrict__ A, long long sa_i, long long sa_k,
                                                           int conj_a, const double* __restrict__ B, int ldb,
                                                           double* __restrict__ D, int ldd, int I, int J, int K) {
    constexpr bool D_COMPLEX = A_COMPLEX || B_COMPLEX;
    __shared__ double ar[32][33], ai[A_COMPLEX ? 32 : 1][33], br[32][33], bi[B_COMPLEX ? 32 : 1][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8 threads, 4 output rows each
    const int i0 = blockIdx.y * 32, j0 = blockIdx.x * 32;
    double dr[4] = {0, 0, 0, 0}, di[4] = {0, 0, 0, 0};
    for (int k0 = 0; k0 < K; k0 += 32) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int row = ty + 8 * r;
            // A tile: element (i0 + row, k0 + tx)
            double vr = 0.0, vi = 0.0;
            if (i0 + row < I && k0 + tx < K) {
                const long long at = (long long)(i0 + row) * sa_i + (long long)(k0 + tx) * sa_k;
                if (A_COMPLEX) {
                    const double2 v = reinterpret_cast<const double2*>(A)[at];
                    vr = v.x;
                    vi = conj_a ? -v.y : v.y;
                } else {
                    vr = A[at];
                }
            }
            ar[row][tx] = vr;
            if (A_COMPLEX) ai[row][tx] = vi;
            // B tile: element (k0 + row, j0 + tx)
            vr = 0.0, vi = 0.0;
            if (k0 + row < K && j0 + tx < J) {
                const long long at = (long long)(k0 + row) * ldb + j0 + tx;
                if (B_COMPLEX) {
                    const double2 v = reinterpret_cast<const double2*>(B)[at];
                    vr = v.x;
                    vi = v.y;
                } else {
                    vr = B[at];
                }
            }
            br[row][tx] = vr;
            if (B_COMPLEX) bi[row][tx] = vi;
        }
        __syncthreads();
#pragma unroll 8
        for (int k = 0; k < 32; ++k) {
            const double b_r = br[k][tx], b_i = B_COMPLEX ? bi[k][tx] : 0.0;
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const double a_r = ar[ty + 8 * r][k], a_i = A_COMPLEX ? ai[ty + 8 * r][k] : 0.0;
                dr[r] = fma(a_r, b_r, dr[r]);
                if (A_COMPLEX && B_COMPLEX) dr[r] = fma(-a_i, b_i, dr[r]);
                if (B_COMPLEX) di[r] = fma(a_r, b_i, di[r]);
                if (A_COMPLEX) di[r] = fma(a_i, b_r, di[r]);
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int i = i0 + ty + 8 * r, j = j0 + tx;
        if (i < I && j < J) {
            if (D_COMPLEX) reinterpret_cast<double2*>(D)[(long long)i * ldd + j] = make_double2(dr[r], di[r]);
            else D[(long long)i * ldd + j] = dr[r];
        }
    }
}

int small_matmul(const void* A, int a_dtype, int64_t sa_i, int64_t sa_k, int conj_a, const void* B, int b_dtype, int64_t ldb,
                 void* D, int64_t ldd, int64_t I, int64_t J, int64_t K, void* stream) {
    const dim3 grid((unsigned)qs_ceil_div(J, 32), (unsigned)qs_ceil_div(I, 32));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const double* a = static_cast<const double*>(A);
    const double* b = static_cast<const double*>(B);
    double* d = static_cast<double*>(D);
    const bool ac = a_dtype == QS_C128, bc = b_dtype == QS_C128;
    if (ac && bc) small_matmul_kernel<true, true><<<grid, 256, 0, st>>>(a, sa_i, sa_k, conj_a, b, (int)ldb, d, (int)ldd, (int)I, (int)J, (int)K);
    else if (ac) small_matmul_kernel<true, false><<<grid, 256, 0, st>>>(a, sa_i, sa_k, conj_a, b, (int)ldb, d, (int)ldd, (int)I, (int)J, (int)K);
    else if (bc) small_matmul_kernel<false, true><<<grid, 256, 0, st>>>(a, sa_i, sa_k, conj_a, b, (int)ldb, d, (int)ldd, (int)I, (int)J, (int)K);
    else small_matmul_kernel<false, false><<<grid, 256, 0, st>>>(a, sa_i, sa_k, conj_a, b, (int)ldb, d, (int)ldd, (int)I, (int)J, (int)K);
    QS_LAUNCH_CHECK();
    return QS_OK;
}

// below this extent a one-body transform takes the small-matrix kernel (two launches, no images)
constexpr int64_t kSmallOneBody = 1024;

}  // namespace

extern "C" int qs_pad_rows(const void* in, void* out, int64_t rows, int64_t n, int64_t pitch, int dtype, void* stream) {
    QS_REQUIRE(in && out && rows > 0 && n > 0 && pitch >= n, "qs_pad_rows: bad arguments");
    const int64_t d = qs_elem_doubles(dtype);  // complex rows are rows of 2n doubles
    return pad_rows(in, out, rows, n * d, pitch * d, stream);
}

extern "C" int qs_transform_two_body_workspace_bytes(int64_t n, int64_t n_new, int u_dtype, int c_dtype,
                                                     int64_t* bytes) {
    QS_REQUIRE(n > 0 && n_new > 0 && bytes, "qs_transform_two_body_workspace_bytes: bad arguments");
    TwoBodyPlan plan;
    int rc = make_plan(n, n_new, u_dtype, c_dtype, &plan);
    if (rc) return rc;
    *bytes = plan.total;
    return QS_OK;
}

namespace {

// Coefficients of the four quarter steps s, r, q, p: steps 1 and 2 contract with the ket matrices C_s and C_r
// (n x m), steps 3 and 4 with the bra matrices Ct_q and Ct_p (m x n); a null bra stands for conj(ket)^T of the
// same index pair (Ct_q: conj(C_s)^T, Ct_p: conj(C_r)^T).
struct StepCoeffs {
    const void *C_s, *C_r, *Ct_q, *Ct_p;
};

// image M[k, w] = Ct[w, k] of a bra step from Ct (m x n row-major), or from conj(C)^T: conj(C[k, w])
int build_bra_image(const void* Ct, const void* C, int c_dtype, int64_t N, int64_t M, int td, void* img, void* stream) {
    if (Ct) return qs_build_coeff_image(Ct, c_dtype, 1, N, 0, N, M, td, img, stream);
    return qs_build_coeff_image(C, c_dtype, M, 1, 1, N, M, td, img, stream);
}

// symmetry = 0: no assumption.  symmetry = 1: u[p,q,r,s] = -u[p,q,s,r]; symmetry = 2: u[p,q,r,s] = u[q,p,s,r] (the
// caller has verified it with qs_two_body_symmetry).  After the two ket contractions T2[r,s,a,b] inherits the
// symmetry in (r,s), so steps 2-4 visit only the tiles that hold a pair r < s (r <= s) and the other half of the
// result is filled in by its mirror image (csrc/symmetry.cu).  That needs one coefficient pair for both kets and one
// for both bras; four different matrices take symmetry = 0.
int two_body_steps(const void* u, int u_dtype, const StepCoeffs& c, int c_dtype, int64_t n, int64_t n_new,
                   int symmetry, void* out, void* workspace, int64_t workspace_bytes, void* stream) {
    QS_REQUIRE(u && c.C_s && c.C_r && out && workspace, "qs_transform_two_body: null pointer");
    QS_REQUIRE(n > 0 && n_new > 0, "qs_transform_two_body: bad extents");
    QS_REQUIRE(symmetry >= 0 && symmetry <= 2, "qs_transform_two_body: unknown symmetry %d", symmetry);
    TwoBodyPlan plan;
    int rc = make_plan(n, n_new, u_dtype, c_dtype, &plan);
    if (rc) return rc;
    QS_REQUIRE(workspace_bytes >= plan.total, "qs_transform_two_body: workspace too small (%lld < %lld)",
               (long long)workspace_bytes, (long long)plan.total);
    QS_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 1023) == 0,
               "qs_transform_two_body: workspace must be 1 KiB aligned");
    const int64_t N = n, M = n_new, P = plan.pitch_t;
    char* ws = static_cast<char*>(workspace);
    void* padded = ws;
    void* bufA = ws + plan.pad_bytes;
    void* bufB = static_cast<char*>(bufA) + plan.bufA_bytes;
    void* img1 = static_cast<char*>(bufB) + plan.bufB_bytes;
    void* img2 = static_cast<char*>(img1) + plan.img_bytes[0];
    void* img3 = static_cast<char*>(img2) + plan.img_bytes[1];
    void* lists = static_cast<char*>(img3) + plan.img_bytes[1];
    long long* tables = reinterpret_cast<long long*>(static_cast<char*>(lists) + plan.list_bytes);
    const int td = plan.t_dtype;

    // step 4 reads a bra image of its own only when its bra differs from step 3's
    const bool bra_p_differs = c.Ct_p != c.Ct_q || (!c.Ct_p && c.C_r != c.C_s);
    QS_REQUIRE(!(symmetry && (bra_p_differs || c.C_r != c.C_s)),
               "qs_transform_two_body: the symmetry-aware steps need one ket and one bra matrix");
    // M[k, w] = C[k, w] (row-major n x m) for steps 1-2
    if ((rc = qs_build_coeff_image(c.C_s, c_dtype, M, 1, 0, N, M, u_dtype, img1, stream))) return rc;
    if ((rc = qs_build_coeff_image(c.C_r, c_dtype, M, 1, 0, N, M, td, img2, stream))) return rc;
    // M[k, w] = Ct[w, k] for step 3 (and step 4 when its bra is the same)
    if ((rc = build_bra_image(c.Ct_q, c.C_s, c_dtype, N, M, td, img3, stream))) return rc;
    const void* a0 = u;
    if (plan.pad_bytes) {
        if ((rc = pad_rows(u, padded, N * N * N, N, plan.pitch_u, stream))) return rc;
        a0 = padded;
    }
    // T1[s,a,b,c] ; T2[r,s,a,b] ; T3[q,r,s,a] (last axis at pitch P) ; out[p,q,r,s] dense
    if ((rc = rotated_quarter(a0, u_dtype, N * N * N, N, plan.pitch_u, img1, c_dtype, M, bufA, N, P, stream))) return rc;
    if (!symmetry) {
        if ((rc = rotated_quarter(bufA, td, M * N * N, N, P, img2, c_dtype, M, bufB, N, P, stream))) return rc;
        if ((rc = rotated_quarter(bufB, td, M * M * N, N, P, img3, c_dtype, M, bufA, N, P, stream))) return rc;
        // step 4's image replaces step 3's in the same slot: the stream orders the rebuild after step 3's reads
        if (bra_p_differs && (rc = build_bra_image(c.Ct_p, c.C_r, c_dtype, N, M, td, img3, stream))) return rc;
        if ((rc = rotated_quarter(bufA, td, M * M * M, N, P, img3, c_dtype, M, out, M, M, stream))) return rc;
        return QS_OK;
    }
    const int strict = symmetry == 1;  // antisymmetry: the diagonal r = s vanishes, only r < s is computed
    // Wanted pairs (r, s), r < s or r <= s, numbered row-major: T3 is kept PACKED by pair, T3p[q, pair, a], so that
    // step 4 is a dense GEMM over m * npairs rows (in the plain layout its 128-row tiles would span the whole
    // range of s and none could be skipped).
    // Real results with an even extent pad every row r of the pair list to whole aligned couples (s even, s + 1): the
    // list of r then starts at the even s at or below its first wanted partner -- one extra element per other r, the
    // diagonal (r, r) or the below-diagonal (r, r - 1), which the mirror fill overwrites afterwards.  Rows 2k and
    // 2k + 1 of step 4 are then neighbours in the result and leave the SM as one 16-byte store (whole 128-byte lines
    // per quarter warp) instead of two scattered 8-byte ones.
    const bool paired = td == QS_F64 && M % 2 == 0;
    auto first_s = [&](int64_t r) {
        const int64_t s0 = strict ? r + 1 : r;
        return paired ? (s0 & ~(int64_t)1) : s0;
    };
    int64_t npairs = 0;
    for (int64_t r = 0; r < M; ++r) npairs += M - first_s(r);
    if (npairs == 0) return qs_mirror_fill(out, td, M, symmetry, stream);  // m = 1, antisymmetric: everything is zero
    // The tables depend on (M, P, strict, paired) only: built once per device and kept in device memory.
    struct { int64_t tag, M, P, strict, paired; } table_key = {0x7ab1e, M, P, strict, paired};
    const long long* dev_tables = static_cast<const long long*>(qs_table_cache_get(&table_key, sizeof(table_key)));
    if (!dev_tables) {
        std::vector<long long> host_tables((size_t)(M * M + npairs));
        long long* slot_of_rs = host_tables.data();          // [r * M + s] -> pair * P, or -1 for an unwanted pair
        long long* rs_of_pair = host_tables.data() + M * M;  // [pair] -> r * M + s
        int64_t pair = 0;
        for (int64_t r = 0; r < M; ++r)
            for (int64_t sI = 0; sI < M; ++sI) {
                const bool wanted = sI >= first_s(r);
                slot_of_rs[r * M + sI] = wanted ? pair * P : -1;
                if (wanted) rs_of_pair[pair++] = r * M + sI;
            }
        dev_tables = static_cast<const long long*>(
            qs_table_cache_put(&table_key, sizeof(table_key), host_tables.data(), host_tables.size() * sizeof(long long)));
        if (!dev_tables) {
            // cache full: stage through the workspace (pageable source: staged by the runtime before the call returns)
            QS_CUDA(cudaMemcpyAsync(tables, host_tables.data(), host_tables.size() * sizeof(long long),
                                    cudaMemcpyHostToDevice, static_cast<cudaStream_t>(stream)));
            dev_tables = tables;
        }
    }
    const long long* dev_slot_of_rs = dev_tables;
    const long long* dev_rs_of_pair = dev_tables + M * M;
    // step 2: rows (s, a, b), new column r -- tiles wanted iff they hold some r < s;  T2[r, s, a, b]
    const QsTileMask m2 = {1, strict, 1, 1, N * N, M};
    if ((rc = masked_rotated_quarter(bufA, td, M * N * N, N, P, img2, c_dtype, M, bufB, N, P, &m2, lists, stream))) return rc;
    // step 3: rows (r, s, a) -- tiles wanted iff they hold some r < s;  packed store T3p[q, pair(r, s), a]
    const QsTileMask m3 = {2, strict, M * N, M, N, M};
    QsQuarterStore s3;
    s3.out = bufA;
    s3.x_inner = N;
    s3.sx0 = 1;
    s3.sw1 = npairs * P;
    s3.xq_table = dev_slot_of_rs;
    s3.xq_even = P % 2 == 0;
    s3.mask = &m3;
    s3.list_ws = lists;
    if ((rc = qs_quarter_launch(bufB, td, M * M * N, N, P, img3, c_dtype, M, s3, stream))) return rc;
    // step 4: dense over rows (q, pair);  out[p, q, r, s] at p M^3 + q M^2 + (r M + s)(pair)
    QsQuarterStore s4;
    s4.out = out;
    s4.x_inner = npairs;
    s4.sx1 = M * M;
    s4.sw1 = M * M * M;
    s4.xr_table = dev_rs_of_pair;
    s4.xr_paired = paired;
    if ((rc = qs_quarter_launch(bufA, td, M * npairs, N, P, img3, c_dtype, M, s4, stream))) return rc;
    return qs_mirror_fill(out, td, M, symmetry, stream);
}

}  // namespace

extern "C" int qs_transform_two_body(const void* u, int u_dtype, const void* C, const void* Ct, int c_dtype, int64_t n,
                                     int64_t n_new, void* out, void* workspace, int64_t workspace_bytes,
                                     void* stream) {
    return qs_transform_two_body_symmetric(u, u_dtype, C, Ct, c_dtype, n, n_new, 0, out, workspace, workspace_bytes,
                                           stream);
}

extern "C" int qs_transform_two_body_symmetric(const void* u, int u_dtype, const void* C, const void* Ct, int c_dtype,
                                               int64_t n, int64_t n_new, int symmetry, void* out, void* workspace,
                                               int64_t workspace_bytes, void* stream) {
    const StepCoeffs c = {C, C, Ct, Ct};
    return two_body_steps(u, u_dtype, c, c_dtype, n, n_new, symmetry, out, workspace, workspace_bytes, stream);
}

// The spin blocks of an unrestricted basis change pair two coefficient matrices: out[p,q,r,s] =
// sum Ct_p[p,a] Ct_q[q,b] u[a,b,c,d] C_r[c,r] C_s[d,s].  Same steps, same workspace, one image per step.
extern "C" int qs_transform_two_body_mixed(const void* u, int u_dtype, const void* C_r, const void* C_s,
                                           const void* Ct_p, const void* Ct_q, int c_dtype, int64_t n, int64_t n_new,
                                           void* out, void* workspace, int64_t workspace_bytes, void* stream) {
    QS_REQUIRE(C_r && C_s, "qs_transform_two_body_mixed: null coefficient matrix");
    const StepCoeffs c = {C_s, C_r, Ct_q, Ct_p};
    return two_body_steps(u, u_dtype, c, c_dtype, n, n_new, 0, out, workspace, workspace_bytes, stream);
}

extern "C" int qs_transform_one_body_workspace_bytes(int64_t n, int64_t n_new, int h_dtype, int c_dtype,
                                                     int64_t* bytes) {
    QS_REQUIRE(n > 0 && n_new > 0 && bytes, "qs_transform_one_body_workspace_bytes: bad arguments");
    const int td = (h_dtype == QS_C128 || c_dtype == QS_C128) ? QS_C128 : QS_F64;
    int64_t img_a, img_b;
    int rc;
    if ((rc = qs_coeff_image_bytes(n, n_new, h_dtype, c_dtype, &img_a))) return rc;
    if ((rc = qs_coeff_image_bytes(n, n_new, td, c_dtype, &img_b))) return rc;
    const int64_t ph = padded_pitch(n, h_dtype), pt = padded_pitch(n, td);
    *bytes = qs_round_up(n * ph * 8, 1024) + qs_round_up(n_new * pt * 8 * qs_elem_doubles(td), 1024) +
             qs_round_up(img_a, 1024) + qs_round_up(img_b, 1024);
    return QS_OK;
}

extern "C" int qs_transform_one_body(const void* h, int h_dtype, const void* C, const void* Ct, int c_dtype, int64_t n,
                                     int64_t n_new, void* out, void* workspace, void* stream) {
    // out[p,q] = sum_ab Ct[p,a] h[a,b] C[b,q] with the same rotated-store kernel:
    //   step 1: T[q, a]   = sum_b h[a, b] C[b, q]     (contract last, new index slowest)
    //   step 2: out[p, q] = sum_a T[q, a] Ct[p, a]    (contract last, new index slowest)
    QS_REQUIRE(h && C && out && workspace, "qs_transform_one_body: null pointer");
    QS_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 1023) == 0,
               "qs_transform_one_body: workspace must be 1 KiB aligned");
    const int td = (h_dtype == QS_C128 || c_dtype == QS_C128) ? QS_C128 : QS_F64;
    int64_t img_a, img_b;
    int rc;
    if (n <= kSmallOneBody && n_new <= kSmallOneBody) {
        // T[a, q] = sum_b h[a, b] C[b, q]  (n x n_new, dtype td) ; out[p, q] = sum_a Ct[p, a] T[a, q]
        void* T = workspace;  // n * n_new elements of td (the workspace of the GEMM path below is larger)
        if ((rc = small_matmul(h, h_dtype, n, 1, 0, C, c_dtype, n_new, T, n_new, n, n_new, n, stream))) return rc;
        if (Ct) return small_matmul(Ct, c_dtype, n, 1, 0, T, td, n_new, out, n_new, n_new, n_new, n, stream);
        // Ct = conj(C)^T: element (p, a) = conj(C[a, p])
        return small_matmul(C, c_dtype, 1, n_new, 1, T, td, n_new, out, n_new, n_new, n_new, n, stream);
    }
    if ((rc = qs_coeff_image_bytes(n, n_new, h_dtype, c_dtype, &img_a))) return rc;
    if ((rc = qs_coeff_image_bytes(n, n_new, td, c_dtype, &img_b))) return rc;
    const int64_t ph = padded_pitch(n, h_dtype), pt = padded_pitch(n, td);
    char* ws = static_cast<char*>(workspace);
    void* hpad = ws;
    void* T = ws + qs_round_up(n * ph * 8, 1024);
    void* img1 = static_cast<char*>(T) + qs_round_up(n_new * pt * 8 * qs_elem_doubles(td), 1024);
    void* img2 = static_cast<char*>(img1) + qs_round_up(img_a, 1024);
    if ((rc = qs_build_coeff_image(C, c_dtype, n_new, 1, 0, n, n_new, h_dtype, img1, stream))) return rc;
    if (Ct) {
        if ((rc = qs_build_coeff_image(Ct, c_dtype, 1, n, 0, n, n_new, td, img2, stream))) return rc;
    } else {
        if ((rc = qs_build_coeff_image(C, c_dtype, n_new, 1, 1, n, n_new, td, img2, stream))) return rc;
    }
    const void* a0 = h;
    if (ph != n) {
        if ((rc = pad_rows(h, hpad, n, n, ph, stream))) return rc;
        a0 = hpad;
    }
    if ((rc = rotated_quarter(a0, h_dtype, n, n, ph, img1, c_dtype, n_new, T, n, pt, stream))) return rc;
    if ((rc = rotated_quarter(T, td, n_new, n, pt, img2, c_dtype, n_new, out, n_new, n_new, stream))) return rc;
    return QS_OK;
}
