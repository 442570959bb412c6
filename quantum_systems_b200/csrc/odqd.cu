// ODQD grid Coulomb build:  u_abcd = sum_pq C_pa C_qb C_pc C_qd W_pq,  W_pq = alpha / sqrt((x_p-x_q)^2 + a^2)
//
// Replaces the 5-operand einsum of ODQD.setup_basis (reference quantum_dots/one_dim/one_dim_qd.py:275-280),
// which numpy contracts as two chained GEMMs.  It is the transform of the diagonal two-body operator W with the grid
// eigenvectors C and Ct = C^T (structured.cu): D[(a,c), p] = C[p,a] C[p,c], Tt = (D W)^T, u = T D^T with the
// acbd -> abcd permutation in the store stride.  W is generated from the grid straight into its coefficient image.
//
// Multi-GPU (SURVEY.md section 8e): the build shards on the leading index a.  A rank computes only the rows
// (a_loc, c) of T and the planes u[a_begin:a_end] -- C and the grid are replicated, D is built whole (it is the
// A operand of the second GEMM for every (b, d)), and there is no communication.
#include "common.cuh"

extern "C" int qs_odqd_coulomb_workspace_bytes(int64_t l, int64_t Gp, int64_t* bytes) {
    QS_REQUIRE(l > 0 && Gp > 0 && bytes, "qs_odqd_coulomb_workspace_bytes: bad arguments");
    return qs_transform_two_body_diagonal_workspace_bytes(Gp, l, QS_F64, QS_F64, 0, bytes);
}

extern "C" int qs_odqd_coulomb(const double* Cmat, const double* grid, double alpha, double a, int64_t l, int64_t Gp,
                               double* u_out, void* workspace, int64_t workspace_bytes, void* stream) {
    return qs_odqd_coulomb_planes(Cmat, grid, alpha, a, l, Gp, u_out, 0, l, workspace, workspace_bytes, stream);
}

extern "C" int qs_odqd_coulomb_planes(const double* Cmat, const double* grid, double alpha, double a, int64_t l,
                                      int64_t Gp, double* u_out, int64_t a_begin, int64_t a_end, void* workspace,
                                      int64_t workspace_bytes, void* stream) {
    QS_REQUIRE(l > 0 && Gp > 0 && l <= 4096, "qs_odqd_coulomb: bad extents");
    QS_REQUIRE(0 <= a_begin && a_begin <= a_end && a_end <= l, "qs_odqd_coulomb: bad plane range");
    if (a_begin == a_end) return QS_OK;  // an empty shard
    QS_REQUIRE(Cmat && grid && u_out && workspace, "qs_odqd_coulomb: null pointer");
    int64_t need;
    int rc = qs_odqd_coulomb_workspace_bytes(l, Gp, &need);
    if (rc) return rc;
    QS_REQUIRE(workspace_bytes >= need, "qs_odqd_coulomb: workspace too small (%lld < %lld)",
               (long long)workspace_bytes, (long long)need);
    QS_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 1023) == 0, "qs_odqd_coulomb: workspace must be 1 KiB aligned");
    if ((rc = qs_build_coulomb_image(grid, alpha, a, Gp, workspace, stream))) return rc;
    return qs_transform_diagonal_planes(nullptr, QS_F64, Cmat, nullptr, QS_F64, Gp, l, a_begin, a_end, 0, u_out,
                                        workspace, stream);
}
