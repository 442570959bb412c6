/*
 * qsb200.h -- C ABI of the B200-native two-body integral pipeline (libqsb200.so).
 *
 * Drop-in boundary for the hot path of HyQD/quantum-systems.  The reference has no FFI of its own
 * (pure Python over numpy); each entry point below replaces the numpy call sites of one reference
 * method, cited as `file:line` relative to /root/reference/quantum_systems/.  A maintainer binds
 * them with ctypes (see INTEGRATION.md); quantum_systems_b200/_native.py is that binding.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name says `host`; the library never allocates
 *     or frees caller-visible memory, scratch is passed in (`workspace`);
 *   - tensors are dense, C-contiguous (row-major); complex128 is interleaved (re, im) doubles;
 *   - `stream` is a cudaStream_t passed as void* (0 = default stream); all work is enqueued
 *     asynchronously on it;
 *   - return value 0 = success, anything else = failure with text in qs_last_error();
 *   - there is no CPU fallback: without a CUDA device every compute entry fails.
 */
#ifndef QSB200_H
#define QSB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QS_F64 0  /* real float64 */
#define QS_C128 1 /* complex128, interleaved */

#define QS_OK 0
#define QS_ERR_INVALID 1
#define QS_ERR_CUDA 2
#define QS_ERR_WORKSPACE 3

/* Library identification and error text (thread-local, valid until the next failing call). */
int qs_version(void);
const char* qs_last_error(void);

/* ---------------------------------------------------------------------------------------------
 * Four-index transform   u'_pqrs = sum_abcd Ct[p,a] Ct[q,b] u[a,b,c,d] C[c,r] C[d,s]
 * replaces BasisSet.transform_two_body_elements (basis_set.py:336-350): four quarter steps in the
 * order s, r, q, p, each an (X x K)*(K x W) FP64 DMMA GEMM whose epilogue stores the new index as
 * the slowest axis, so no separate permutation pass exists.
 *
 *   u      : (n, n, n, n)                dtype u_dtype
 *   C      : (n, n_new)  row-major       dtype c_dtype
 *   Ct     : (n_new, n)  row-major       dtype c_dtype, or NULL for conj(C)^T (basis_set.py:338-339)
 *   out    : (n_new,)*4                  complex128 if either input is complex, else float64
 *   workspace : at least qs_transform_two_body_workspace_bytes() bytes, 1024-byte aligned
 * ------------------------------------------------------------------------------------------- */
int qs_transform_two_body_workspace_bytes(int64_t n, int64_t n_new, int u_dtype, int c_dtype,
                                          int64_t* bytes);
int qs_transform_two_body(const void* u, int u_dtype, const void* C, const void* Ct, int c_dtype,
                          int64_t n, int64_t n_new, void* out, void* workspace,
                          int64_t workspace_bytes, void* stream);

/* Symmetry-aware variant.  Two exact symmetries of u survive the basis change for ANY C, C~ and are visible half
 * way through it (after the two ket contractions T2[r,s,a,b] has them in (r,s)):
 *   bit 0 (1): u[p,q,r,s] = -u[p,q,s,r]   every anti-symmetrised tensor (basis_set.py:776-778)
 *   bit 1 (2): u[p,q,r,s] =  u[q,p,s,r]   particle exchange, every physical interaction (random_basis.py:40-42)
 * qs_two_body_symmetry tests both EXACTLY on the device (one read of u, early exit on the first counter-example;
 * it synchronises the stream to return the flags in *host_flags; device_scratch: 8 bytes; first_match != 0 skips
 * the second test when the first holds and then reports bit 0 only).
 * qs_transform_two_body_symmetric(symmetry = 1 or 2) then runs quarter steps 2-4 only on the tiles that hold a
 * pair r < s (r <= s) -- about 45 % fewer tensor-core flops at n = 128, approaching 3/8 for large n -- and completes
 * the result with its mirror image.  symmetry = 0 is qs_transform_two_body.  Same workspace as the plain call. */
int qs_two_body_symmetry(const void* u, int dtype, int64_t n, int first_match, int* host_flags,
                         void* device_scratch, void* stream);
int qs_transform_two_body_symmetric(const void* u, int u_dtype, const void* C, const void* Ct,
                                    int c_dtype, int64_t n, int64_t n_new, int symmetry, void* out,
                                    void* workspace, int64_t workspace_bytes, void* stream);

/* Four-coefficient transform   out[p,q,r,s] = sum_abcd Ct_p[p,a] Ct_q[q,b] u[a,b,c,d] C_r[c,r] C_s[d,s]
 * the mixed-spin blocks of an unrestricted basis change (see qs_spin_orbital_two_body), whose two ket and two bra
 * indices belong to two different spins.  The same four quarter steps in the order s, r, q, p as qs_transform_two_body, one coefficient image per step.
 *   C_r, C_s   : (n, n_new) row-major     dtype c_dtype
 *   Ct_p, Ct_q : (n_new, n) row-major     dtype c_dtype, or NULL for conj(C_r)^T, conj(C_s)^T respectively
 * u, out and the workspace (qs_transform_two_body_workspace_bytes) as in qs_transform_two_body.  No symmetry is
 * assumed: with two different matrices none survives; equal matrices take qs_transform_two_body_symmetric. */
int qs_transform_two_body_mixed(const void* u, int u_dtype, const void* C_r, const void* C_s,
                                const void* Ct_p, const void* Ct_q, int c_dtype, int64_t n, int64_t n_new,
                                void* out, void* workspace, int64_t workspace_bytes, void* stream);

/* Building blocks of the SHARDED symmetry-aware transform (anti-symmetric u only: its mirror image stays inside a
 * (p, q) plane, i.e. on the rank that owns p).  Of each pair (r, s), (s, r) the rank that owns r computes the one
 * whose cyclic distance (s - r) mod m is the shorter (qs_cyclic_pair_wanted; ties go to r < s), so every r has the
 * same number of partners and the contiguous r-partition stays balanced.
 *   qs_is_antisymmetric_last_pair : exact test on a rank's slab of `planes` leading-index planes (the caller
 *                                   combines the ranks' flags).
 *   qs_cyclic_antisymmetric_fill  : out[p,q,r,s] = -out[p,q,s,r] for the pairs not computed, zero diagonal. */
int qs_is_antisymmetric_last_pair(const void* u, int dtype, int64_t n, int64_t planes, int* host_flag,
                                  void* device_scratch, void* stream);
int qs_cyclic_antisymmetric_fill(void* out, int dtype, int64_t m, int64_t planes, void* stream);
int qs_cyclic_pair_wanted(int64_t r, int64_t s, int64_t m);

/* ---------------------------------------------------------------------------------------------
 * One quarter step, exposed for the sharded (multi-GPU) schedule and for the grid Coulomb build.
 *
 *   out[ (w / w_inner) * sw1 + (w % w_inner) * sw0 + (x / x_inner) * sx1 + (x % x_inner) * sx0 ]
 *       = sum_k A[x, k] * M[k, w]              x < X, k < K, w < W   (element strides of a_dtype/out)
 *
 * A is (X, K) row-major with row pitch `lda` elements.  M is described by (m, m_dtype, m_sk, m_sw,
 * m_conj): M[k, w] = m[k * m_sk + w * m_sw], conjugated if m_conj.  The kernel consumes M through a
 * fragment-ordered "coefficient image" built by qs_build_coeff_image into `image`
 * (qs_coeff_image_bytes() bytes).  Output dtype is complex if A or M is complex.  The store strides
 * are in units of OUTPUT ELEMENTS; the plain rotated store is x_inner = X, sx0 = 1, sx1 = 0,
 * w_inner = 1, sw0 = 0, sw1 = X.
 * ------------------------------------------------------------------------------------------- */
int qs_coeff_image_bytes(int64_t K, int64_t W, int a_dtype, int m_dtype, int64_t* bytes);
int qs_build_coeff_image(const void* m, int m_dtype, int64_t m_sk, int64_t m_sw, int m_conj,
                         int64_t K, int64_t W, int a_dtype, void* image, void* stream);
int qs_quarter_transform(const void* A, int a_dtype, int64_t X, int64_t K, int64_t lda,
                         const void* image, int m_dtype, int64_t W, void* out, int64_t x_inner,
                         int64_t sx0, int64_t sx1, int64_t w_inner, int64_t sw0, int64_t sw1,
                         void* stream);

/* Scattering variant: the fused re-partition of the sharded schedule.  The new index w selects
 * the destination buffer host_out_table[w / w_inner] (n_dest device pointers held in a HOST array;
 * peers' buffers mapped with qs_ipc_open) and is stored at (w % w_inner) * sw0 inside it.  The row
 * index is split three ways, x = (x2 * x_mid + x1) * x_inner + x0, and contributes
 * x2 * sx2 + x1 * sx1 + x0 * sx0, so a shard's planes land between the planes of the other ranks.
 * One launch computes the quarter step AND delivers every tile to the GPU that owns it over
 * NVLink -- the all-to-all of SURVEY.md section 8e without a second pass over memory.
 *
 * Column dealing.  With contiguous column ranges per CTA tile every rank writes to the same one or two
 * peers at any moment (an NVLink ingress hot spot: +29 % on 7 of 8 ranks at n = 400).  `w_deal` > 1
 * (from qs_scatter_deal(W)) makes the j-th column of the tile order the PHYSICAL column (j * w_deal) % W,
 * spreading every tile over all destinations; the image must then come from qs_build_coeff_image_dealt
 * with the same multiplier.  w_deal = 1: columns in natural order (plain qs_build_coeff_image).
 *
 * Cyclic destinations.  `w_cyclic` != 0 replaces the blocks of w_inner columns per destination by a round-robin:
 * column w goes to host_out_table[w % n_dest] and is column w / n_dest there (w_inner is then ignored).  A tile's
 * columns spread over all destinations by themselves (no dealing needed), and the owner of the cyclic columns later
 * writes rows that INTERLEAVE with the other ranks' rows.  That matters: eight ranks that each fill one of eight
 * ADJACENT chunks of a block in a destination's memory at the same time see position-dependent NVLink throughput
 * (the ranks writing the outermost chunks are 30 % slower at n = 192 on 8 B200s -- the slow ranks follow the chunk
 * position, not the physical GPU; profiles/r02h_*, r02i_*). */
int qs_scatter_deal(int64_t W, int64_t* w_deal);
int qs_build_coeff_image_dealt(const void* m, int m_dtype, int64_t m_sk, int64_t m_sw, int m_conj,
                               int64_t K, int64_t W, int a_dtype, int64_t w_deal, void* image,
                               void* stream);
int qs_quarter_transform_scatter(const void* A, int a_dtype, int64_t X, int64_t K, int64_t lda,
                                 const void* image, int m_dtype, int64_t W,
                                 void* const* host_out_table, int64_t n_dest, int64_t x_inner,
                                 int64_t x_mid, int64_t sx0, int64_t sx1, int64_t sx2,
                                 int64_t w_inner, int64_t sw0, int64_t w_deal, int w_cyclic,
                                 void* stream);

/* The scattering store of the anti-symmetric schedule's first exchange: cyclic destinations (column r goes to
 * host_out_table[r % n_dest], column r / n_dest there, stride sw0), restricted to the CTA tiles that hold a pair
 * (r, s) the cyclic pair rule wants -- s = (x / rows_per_s) % W is the row's second index; `padded` != 0 also keeps
 * the other member s ^ 1 of an aligned couple (the padded pair lists of real tensors).  About a third of the tiles
 * of this step, and of its NVLink traffic, go away.  list_ws: qs_quarter_tile_list_bytes() bytes of device memory. */
int qs_quarter_transform_scatter_pairs(const void* A, int a_dtype, int64_t X, int64_t K, int64_t lda,
                                       const void* image, int m_dtype, int64_t W,
                                       void* const* host_out_table, int64_t n_dest, int64_t x_inner,
                                       int64_t x_mid, int64_t sx0, int64_t sx1, int64_t sx2, int64_t sw0,
                                       int64_t rows_per_s, int padded, void* list_ws, int64_t list_ws_bytes,
                                       void* stream);

/* The scattering store with COLUMN TABLES: the physical column w (after dealing) goes to the destination
 * host_out_table[col_dest[w]] (< n_dest <= 16) at element offset col_off[w] inside it; rows are placed as in
 * qs_quarter_transform_scatter (x_inner, x_mid, sx0, sx1, sx2).  col_dest (int32) and col_off (int64) hold W entries
 * each in device memory.  Unlike the blocks of w_inner columns, the tables give every destination any set of
 * columns: the spin-orbital planes of an unrestricted basis, whose owners hold uneven -- possibly empty -- orbital
 * ranges per spin.  `offsets_even` != 0 is the caller's promise that every col_off entry is even (real output then
 * leaves in 16-byte row pairs when the row strides allow it).  Always the register-store epilogue. */
int qs_quarter_transform_scatter_columns(const void* A, int a_dtype, int64_t X, int64_t K, int64_t lda,
                                         const void* image, int m_dtype, int64_t W,
                                         void* const* host_out_table, int64_t n_dest, const int32_t* col_dest,
                                         const int64_t* col_off, int offsets_even, int64_t x_inner,
                                         int64_t x_mid, int64_t sx0, int64_t sx1, int64_t sx2, int64_t w_deal,
                                         void* stream);

/* Epilogue of the quarter GEMM.  Besides storing from registers, a launch can stage each warp's accumulator tile
 * in shared memory ([column][row], 16 real columns at a time, two 4 KiB buffers per warp) and hand every run of rows
 * that is contiguous in the output to the copy engine (cp.async.bulk shared -> global, SASS UBLKCP.G.S), going on
 * to its next tile while the copies drain.  mode 0: register stores everywhere; 1 (default): staged epilogue in the
 * scattering launches, whose stores cross NVLink; 2: wherever the alignment conditions hold (consecutive rows
 * adjacent in the output, every run 16-byte aligned).  Measured on B200s (profiles/r02d_*, r02e_*, r02f_*): for
 * local stores the register epilogue is 1-6 % faster; over NVLink the two are within 1 % of each other -- every
 * store shape reaches the same 712 GB/s (profiles/r02b_peer_store_probe_2gpu.jsonl).  Returns the previous mode.
 * Also settable with QS_BULK=off|scatter|all in the environment (read once). */
int qs_set_bulk_epilogue_mode(int mode);

/* Four-index transform of an operator that is diagonal in the original basis, u[a,b,c,d] = W[a,b] d_ac d_bd
 * (the sinc-DVR storage u_repr = "2d"):
 *   out[p,q,r,s] = sum_ab Ct[p,a] C[a,r] Ct[q,b] C[b,s] W[a,b]   ( - out[p,q,s,r] if anti_symmetrize )
 * replaces the einsum of ODSincDVR.transform_two_body_elements (sinc_dvr/one_dim/sinc_dvr.py:217-252) with
 * two chained DMMA GEMMs, O(m^4 n) instead of O(n^5).
 *   w2d : (n, n) dtype w_dtype;  C : (n, m);  Ct : (m, n) or NULL for conj(C)^T;  out : (m,m,m,m), complex128 if
 *   W or C is complex, else float64.  workspace: qs_transform_two_body_diagonal_workspace_bytes(), 1 KiB aligned. */
int qs_transform_two_body_diagonal_workspace_bytes(int64_t n, int64_t m, int w_dtype, int c_dtype,
                                                   int anti_symmetrize, int64_t* bytes);
int qs_transform_two_body_diagonal(const void* w2d, int w_dtype, const void* C, const void* Ct,
                                   int c_dtype, int64_t n, int64_t m, int anti_symmetrize, void* out,
                                   void* workspace, int64_t workspace_bytes, void* stream);

/* Quarter steps with TABULATED row placement (packed pair layouts of the symmetry-aware transforms).
 * Rows are split x = xq * x_inner + xr.
 *   qs_quarter_transform_rows         : row x is stored at xq_table[xq] + xr * sx0 (+ the column term of
 *       qs_quarter_transform); a NEGATIVE table entry drops the rows of that xq, and CTA tiles without any kept row
 *       are not launched at all (the tile list is derived from host_xq_table, the host copy of the device table
 *       xq_table; list_ws: qs_quarter_tile_list_bytes() bytes of device memory).
 *   qs_quarter_transform_scatter_rows : the scattering store with row x at xq * sx1 + xr_table[xr] inside the
 *       destination buffer chosen by the column (see qs_quarter_transform_scatter).
 * Tables are int64 element offsets in device memory.  `rows_paired` != 0 is the caller's promise that the row table
 * places rows 2k and 2k + 1 next to each other at an even offset (xr_table[2k + 1] = xr_table[2k] + 1, xr_table[2k]
 * even): a real result is then stored in 16-byte pairs forming whole 128-byte lines -- over NVLink that is the
 * difference between 8-byte and full-line writes.  qs_quarter_transform_rows checks its (host) block table itself. */
int qs_quarter_tile_list_bytes(int64_t X, int64_t K, int64_t W, int a_dtype, int m_dtype, int64_t* bytes);
/* Host-only planning of a masked launch (no device is touched): the CTA tiles it would visit, as rows of
 * (first row, last row, first output column, last output column) in host_tiles (capacity rows of 4 int64; may be
 * NULL to only count).  Either a host row table (mask_kind = 0) or the analytic masks of the single-GPU
 * symmetry-aware transform: kind 1 keeps tiles with some column < (<=) row_lo, kind 2 tiles with some row_hi < (<=)
 * row_lo, where row_hi(x) = (x / dh) % mh and row_lo(x) = (x / dl) % ml. */
int qs_quarter_plan_tiles(int64_t X, int64_t K, int64_t W, int a_dtype, int m_dtype, int64_t x_inner,
                          int mask_kind, int strict, int64_t dh, int64_t mh, int64_t dl, int64_t ml,
                          const int64_t* host_xq_table, int64_t* host_tiles, int64_t capacity,
                          int64_t* count);
int qs_quarter_transform_rows(const void* A, int a_dtype, int64_t X, int64_t K, int64_t lda,
                              const void* image, int m_dtype, int64_t W, void* out, int64_t x_inner,
                              int64_t sx0, const int64_t* host_xq_table, const int64_t* xq_table,
                              int64_t w_inner, int64_t sw0, int64_t sw1, void* list_ws,
                              int64_t list_ws_bytes, void* stream);
int qs_quarter_transform_scatter_rows(const void* A, int a_dtype, int64_t X, int64_t K, int64_t lda,
                                      const void* image, int m_dtype, int64_t W,
                                      void* const* host_out_table, int64_t n_dest, int64_t x_inner,
                                      int64_t sx1, const int64_t* xr_table, int64_t w_inner,
                                      int64_t sw0, int64_t w_deal, int rows_paired, void* stream);

/* Copy `rows` rows of n elements into rows of `pitch` >= n elements, zero-filling the tail (real
 * tensors with odd n need an even pitch before they can be described to TMA). */
int qs_pad_rows(const void* in, void* out, int64_t rows, int64_t n, int64_t pitch, int dtype,
                void* stream);

/* Peer-memory plumbing for the scattering store: cudaMalloc + CUDA IPC export / open / close / free.
 * host_handle points at qs_ipc_handle_bytes() bytes of host memory (exchanged between the ranks by
 * the caller, e.g. torch.distributed.all_gather_object). */
int qs_ipc_handle_bytes(void);
int qs_ipc_alloc(int64_t bytes, void** dev_ptr, void* host_handle);
int qs_ipc_open(const void* host_handle, void** dev_ptr);
int qs_ipc_close(void* dev_ptr);
int qs_ipc_free(void* dev_ptr);

/* ---------------------------------------------------------------------------------------------
 * One-body transform  h' = Ct (h C)   replaces BasisSet.transform_one_body_elements
 * (basis_set.py:329-334).  h: (n, n); C: (n, n_new); Ct: (n_new, n) or NULL; out: (n_new, n_new).
 * workspace: qs_transform_one_body_workspace_bytes() bytes, 1024-byte aligned.
 * ------------------------------------------------------------------------------------------- */
int qs_transform_one_body_workspace_bytes(int64_t n, int64_t n_new, int h_dtype, int c_dtype,
                                          int64_t* bytes);
int qs_transform_one_body(const void* h, int h_dtype, const void* C, const void* Ct, int c_dtype,
                          int64_t n, int64_t n_new, void* out, void* workspace, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Spin doubling and anti-symmetrisation (memory-bound passes).
 *
 * qs_add_spin_two_body: U[2p+s1,2q+s2,2r+s3,2s+s4] = u[p,q,r,s] [s1==s3][s2==s4], optionally fused with
 *   U - U.transpose(0,1,3,2).  Replaces BasisSet.add_spin_two_body (basis_set.py:772-774) followed
 *   by BasisSet.anti_symmetrize_u (:776-778).  Only leading-index planes P in [p_begin, p_end) of the
 *   (2l)^4 result are written (to out + 0, i.e. `out` points at the first plane of the shard), which is
 *   the multi-GPU partition.  in_dtype -> out_dtype may widen F64 -> C128 (cast_to_complex, :298-319).
 * qs_anti_symmetrize: out = u - u.transpose(0,1,3,2) on an (n,n,n,n) tensor, planes [p_begin,p_end).
 * qs_add_spin_one_body: kron(h, I2) (:768-770).
 * ------------------------------------------------------------------------------------------- */
int qs_add_spin_two_body(const void* u, int in_dtype, int64_t l, void* out, int out_dtype,
                         int anti_symmetrize, int64_t p_begin, int64_t p_end, void* stream);
int qs_anti_symmetrize(const void* u, int dtype, int64_t n, void* out, int64_t p_begin,
                       int64_t p_end, void* stream);
int qs_add_spin_one_body(const void* h, int in_dtype, int64_t l, void* out, int out_dtype,
                         void* stream);

/* Anti-symmetrised spin-orbital tensor of an unrestricted basis from the spin blocks of the spatial tensor
 *   B_st[i,j,k,l] = sum_abcd conj(C_s[a,i]) conj(C_t[b,j]) u[a,b,c,d] C_s[c,k] C_t[d,l]   (s, t in {alpha, beta})
 *   U[I,J,K,L] = [sI==sK][sJ==sL] B_{sI sJ}[oI,oJ,oK,oL] - [sI==sL][sJ==sK] B_{sI sJ}[oI,oJ,oL,oK]
 * with spin-orbital I = (orbital[I], spin[I]); orbital, spin: int32 device tables of length 2l that together are a
 * bijection onto {0..l-1} x {0, 1} (0 = alpha).  b_aa, b_ab, b_ba, b_bb: (l,l,l,l) of in_dtype; b_ba = NULL derives
 * it from b_ab by particle exchange, B_ba[i,j,k,l] = B_ab[j,i,l,k] (exact when u[a,b,c,d] = u[b,a,d,c]).
 * in_dtype -> out_dtype: F64 -> F64, F64 -> C128 or C128 -> C128.  Planes I in [p_begin, p_end) of the (2l)^4 result
 * are written, to `out` pointing at plane p_begin.  Every output element, zeros included, is written once: reads
 * 4 l^4 input and writes 16 l^4 output elements for the whole tensor. */
int qs_spin_orbital_two_body(const void* b_aa, const void* b_ab, const void* b_ba, const void* b_bb,
                             int in_dtype, int64_t l, const int32_t* orbital, const int32_t* spin,
                             void* out, int out_dtype, int64_t p_begin, int64_t p_end, void* stream);

/* Two-body part of S^2 from the three (n, n) complex128 spin matrices S_x, S_y, S_z:
 *   out[p,q,r,s] = sum_i S_i[p,r] S_i[q,s]  (- sum_i S_i[p,s] S_i[q,r] if anti_symmetrize)
 * replaces the einsum loop of BasisSet.setup_spin_squared_operator (basis_set.py:743-747) and, applied
 * to basis-changed factors C~ S_i C, the second O(n^5) transform of _change_basis_two_body_elements
 * (:379-382).  Planes p in [p_begin, p_end) are written to `out` (complex128). */
int qs_spin_squared_two_body(const void* sx, const void* sy, const void* sz, int64_t n,
                             int anti_symmetrize, void* out, int64_t p_begin, int64_t p_end,
                             void* stream);

/* ---------------------------------------------------------------------------------------------
 * Fock matrices (warp-shuffle reductions over the occupied index).
 *   general : f[p,q] = h[p,q] + sum_{i<n_occ} u[p,i,q,i]                    general_orbital_system.py:119-159
 *   spatial : f[p,q] = h[p,q] + 2 sum_i u[p,i,q,i] - sum_i u[p,i,i,q]       spatial_orbital_system.py:150-190
 * h, f: (n, n) dtype h_dtype (f is overwritten); u: (n,n,n,n) dtype u_dtype (F64 u with C128 h allowed).
 * Rows p in [p_begin, p_end) only; `u` points at plane p_begin of the tensor, h and f at row 0.
 * ------------------------------------------------------------------------------------------- */
int qs_fock_general(const void* h, int h_dtype, const void* u, int u_dtype, int64_t n,
                    int64_t n_occ, void* f, int64_t p_begin, int64_t p_end, void* stream);
int qs_fock_spatial(const void* h, int h_dtype, const void* u, int u_dtype, int64_t n,
                    int64_t n_occ, void* f, int64_t p_begin, int64_t p_end, void* stream);
/* General Fock matrix from a tensor sharded on its THIRD index (what a sharded change_basis leaves):
 * u_cols = u[:, :, q_begin:q_end, :] stored dense as (n, n, q_end-q_begin, n); writes columns
 * [q_begin, q_end) of f (h, f full (n, n) matrices); u_cols may be NULL when the range is empty. */
int qs_fock_general_cols(const void* h, int h_dtype, const void* u_cols, int u_dtype, int64_t n,
                         int64_t n_occ, void* f, int64_t q_begin, int64_t q_end, void* stream);
/* Same reductions on pre-gathered (n_occ, n, n) blocks direct[i,p,q] = u[p,i,q,i] and (optional,
 * may be NULL) exchange[i,p,q] = u[p,i,i,q]:  f = h + scale_direct * sum_i direct + scale_exchange *
 * sum_i exchange.  Used when u lives in host memory and only the needed elements are staged. */
int qs_fock_gathered(const void* h, int h_dtype, const void* direct, const void* exchange,
                     int u_dtype, int64_t n, int64_t n_occ, double scale_direct,
                     double scale_exchange, void* f, void* stream);
/* Fock matrix from a general density matrix rho (n, n), the O(n^4) step of a Hartree-Fock iteration:
 *   f[p,q] = h[p,q] + scale_direct   * sum_{r,s} u[p,r,q,s] rho[s,r]
 *                   + scale_exchange * sum_{r,s} u[p,r,s,q] rho[s,r]          for p in [p_begin, p_end)
 * `u` points at plane p_begin: the (p_end - p_begin, n, n, n) slab u[p_begin:p_end]; h, rho, f are whole (n, n)
 * matrices and rows of f outside [p_begin, p_end) are not touched.  h, u, rho may each be F64 or C128; f_dtype
 * must be C128 when any of them is.  Every element of u is read once.  Deterministic (no atomics): per-(plane,
 * r-chunk) partial rows go to the workspace (qs_fock_density_workspace_bytes) and are summed in a fixed order; the
 * chunking depends on n only, so a row is bit-identical whatever plane range it is computed in. */
int qs_fock_density_workspace_bytes(int64_t n, int64_t p_begin, int64_t p_end, int u_dtype, int rho_dtype,
                                    int64_t* bytes);
int qs_fock_density(const void* h, int h_dtype, const void* u, int u_dtype, const void* rho, int rho_dtype,
                    int64_t n, double scale_direct, double scale_exchange, void* f, int f_dtype,
                    int64_t p_begin, int64_t p_end, void* workspace, int64_t workspace_bytes, void* stream);
/* Unrestricted (UHF) Fock matrices of two spin densities rho_alpha, rho_beta (n, n) of one dtype rho_dtype:
 *   f_s[p,q] = h[p,q] + sum_{r,s} u[p,r,q,s] (rho_alpha + rho_beta)[s,r] - sum_{r,s} u[p,r,s,q] rho_s[s,r]
 * for s in {alpha, beta} and p in [p_begin, p_end); u, h, f_alpha, f_beta and the row range as in qs_fock_density
 * (f_dtype is the dtype of both f).  Real u: u is read once for both spins (real densities through the packed
 * density rho_alpha + i rho_beta, complex ones in one pass over rho_alpha + rho_beta, rho_alpha and rho_beta).
 * Complex u: u is read once per density, i.e. twice.  Deterministic, and a row is bit-identical whatever plane range
 * it is computed in. */
int qs_fock_density_unrestricted_workspace_bytes(int64_t n, int64_t p_begin, int64_t p_end, int u_dtype,
                                                 int rho_dtype, int64_t* bytes);
int qs_fock_density_unrestricted(const void* h, int h_dtype, const void* u, int u_dtype, const void* rho_alpha,
                                 const void* rho_beta, int rho_dtype, int64_t n, void* f_alpha, void* f_beta,
                                 int f_dtype, int64_t p_begin, int64_t p_end, void* workspace,
                                 int64_t workspace_bytes, void* stream);
/* Coulomb and exchange matrices of a batch of k real densities rho (k, n, n) in one read of a real u:
 *   J[d,p,q] = sum_{r,s} u[p,r,q,s] rho[d,s,r]        K[d,p,q] = sum_{r,s} u[p,r,s,q] rho[d,s,r]
 * for d < k <= QS_COULOMB_EXCHANGE_MAX_BATCH and p in [p_begin, p_end), on the FP64 tensor pipe.  `u` points at plane
 * p_begin as in qs_fock_density; J and K are whole (k, n, n) arrays and rows outside [p_begin, p_end) are not
 * touched.  u and rho must be F64 (complex ones are refused); n <= 384.  Deterministic (no atomics), with per-(plane,
 * r-chunk) partial rows in the workspace (qs_coulomb_exchange_batch_workspace_bytes) summed in a fixed order that
 * depends on n only: a density's J and K are bit-identical whatever the other densities of the batch, its position
 * and k, and a row is bit-identical whatever plane range it is computed in. */
#define QS_COULOMB_EXCHANGE_MAX_BATCH 16
int qs_coulomb_exchange_batch_workspace_bytes(int64_t n, int64_t k, int64_t p_begin, int64_t p_end, int u_dtype,
                                              int rho_dtype, int64_t* bytes);
int qs_coulomb_exchange_batch(const void* u, int u_dtype, const void* rho, int rho_dtype, int64_t n, int64_t k,
                              void* J, void* K, int64_t p_begin, int64_t p_end, void* workspace,
                              int64_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * ODQD grid Coulomb build  u_abcd = sum_pq C_pa C_qb C_pc C_qd alpha/sqrt((x_p-x_q)^2 + a^2)
 * replaces the einsum of ODQD.setup_basis (quantum_dots/one_dim/one_dim_qd.py:275-280) with two
 * chained DMMA GEMMs (T = D W, u = T D^T, D[(ac),p] = C_pa C_pc); the acbd -> abcd permutation is
 * fused into the second epilogue and W is generated from the grid, never loaded.
 *   Cmat : (Gp, l) float64, interior-grid eigenvectors;  grid : (Gp,) float64 interior points
 *   u_out: (l,l,l,l) float64 C-contiguous;  workspace >= qs_odqd_coulomb_workspace_bytes()
 * ------------------------------------------------------------------------------------------- */
int qs_odqd_coulomb_workspace_bytes(int64_t l, int64_t Gp, int64_t* bytes);
int qs_odqd_coulomb(const double* Cmat, const double* grid, double alpha, double a, int64_t l,
                    int64_t Gp, double* u_out, void* workspace, int64_t workspace_bytes,
                    void* stream);
/* The same build restricted to planes a in [a_begin, a_end) of u (u_out points at plane a_begin): the
 * multi-GPU partition of SURVEY.md section 8e -- C and the grid replicated, no communication. */
int qs_odqd_coulomb_planes(const double* Cmat, const double* grid, double alpha, double a, int64_t l,
                           int64_t Gp, double* u_out, int64_t a_begin, int64_t a_end, void* workspace,
                           int64_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Two-dimensional harmonic-oscillator Coulomb elements (Anisimovas & Matulis 1998)
 *   u[p,q,r,s] = scale * coulomb_ho(n_p, m_p, n_q, m_q, n_r, m_r, n_s, m_s)
 * replaces coulomb_ho (quantum_dots/two_dim/coulomb_elements.py:6-92) as driven by
 * _get_coulomb_elements (quantum_dots/two_dim/two_dim_helper.py:250-268) and get_coulomb_elements_B
 * (:283-300); `scale` is the sqrt(omega) of TwoDimensionalHarmonicOscillator.setup_basis
 * (quantum_dots/two_dim/two_dim_ho.py:86-88).  The eight nested loops are collapsed analytically
 * to table-driven sums carried in double-double arithmetic (see csrc/tdho.cu).
 *   host_n, host_m : HOST arrays of l radial / angular quantum numbers (n >= 0, n + |m| <= 13)
 *   u_out          : planes [p_begin, p_end) of the (l,l,l,l) float64 tensor, dense
 *   workspace      : qs_tdho_coulomb_workspace_bytes() bytes of device memory (tables)
 * ------------------------------------------------------------------------------------------- */
int qs_tdho_coulomb_workspace_bytes(const int64_t* host_n, const int64_t* host_m, int64_t l,
                                    int64_t* bytes);
int qs_tdho_coulomb(const int64_t* host_n, const int64_t* host_m, int64_t l, double scale,
                    double* u_out, int64_t p_begin, int64_t p_end, void* workspace,
                    int64_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Consumers of the two-body tensor (memory-bound passes on one GPU's leading-index shard).
 *
 * qs_extract_block  : out = u[a0:a1, b0:b1, c0:c1, d0:d1] as a dense tensor -- the u[o,o,v,v]-style
 *                     slicing solvers do with QuantumSystem.o / .v (system.py:47-51).  `u` points at a
 *                     (planes, n, n, n) slab; a0, a1 are relative to its first plane.
 * qs_scale_add      : out = alpha x + beta y over `count` elements (y may be NULL; out may alias x) --
 *                     the sums of QuantumSystem.h_t / u_t (system.py:189-215) and AdiabaticSwitching.u_t
 *                     = f(t) u (time_evolution_operators/operator.py:182-196).  Complex factors need
 *                     a complex tensor.
 * qs_occupied_traces: out6 (DEVICE, 6 doubles) = { tr h[o,o], sum_ij u[i,j,i,j], sum_ij u[i,j,j,i] } as
 *                     (re, im) pairs, i restricted to planes [p_begin, p_end), i, j < n_occ -- the terms of
 *                     compute_reference_energy (general_orbital_system.py:75-117,
 *                     spatial_orbital_system.py:106-148).  `u` points at plane p_begin, h at row 0.
 * ------------------------------------------------------------------------------------------- */
int qs_extract_block(const void* u, int dtype, int64_t n, int64_t planes, int64_t a0, int64_t a1,
                     int64_t b0, int64_t b1, int64_t c0, int64_t c1, int64_t d0, int64_t d1, void* out,
                     void* stream);
int qs_scale_add(const void* x, const void* y, int dtype, int64_t count, double alpha_re,
                 double alpha_im, double beta_re, double beta_im, void* out, void* stream);
int qs_occupied_traces(const void* h, int h_dtype, const void* u, int u_dtype, int64_t n,
                       int64_t n_occ, int64_t p_begin, int64_t p_end, double* out6, void* stream);

/* Instrumentation for the benchmark harness.
 *   qs_launch_count        : kernels launched by this library since it was loaded (process-wide).
 *   qs_kernel_timing_enable: 1 = bracket every launch site of a kernel family with CUDA events on
 *                            the launching stream (cleared on every call); 0 = off (default).
 *   qs_kernel_timing_read  : synchronise and sum the recorded spans of one family: device
 *                            milliseconds, algorithmic work (flops for QS_FAMILY_QUARTER_GEMM, bytes
 *                            for QS_FAMILY_SPIN_PASS) and the number of spans. */
#define QS_FAMILY_QUARTER_GEMM 0
#define QS_FAMILY_SPIN_PASS 1
#define QS_FAMILY_FOCK 2
#define QS_FAMILY_EXCHANGE 3
#define QS_FAMILY_TDHO 4
int64_t qs_launch_count(void);
int qs_kernel_timing_enable(int enable);
int qs_kernel_timing_read(int family, double* host_ms_total, double* host_work_total,
                          int64_t* host_spans);

/* Roofline denominators measured in place: register-resident DMMA.8x8x4 loop (FP64 tensor pipe)
 * and a streaming copy.  Host out-pointers. */
int qs_probe_dmma_tflops(double* host_tflops, void* stream);
int qs_probe_copy_gbs(double* host_gbs, void* scratch, int64_t scratch_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* QSB200_H */
