// Spin doubling and anti-symmetrisation: HBM-bound passes.
//
//   qs_add_spin_two_body : BasisSet.add_spin_two_body (reference basis_set.py:772-774), optionally
//                          fused with BasisSet.anti_symmetrize_u (:776-778) and cast_to_complex (:298-319)
//   qs_anti_symmetrize   : BasisSet.anti_symmetrize_u alone
//   qs_add_spin_one_body : BasisSet.add_spin_one_body (:768-770)
//   qs_spin_orbital_two_body : the anti-symmetrised spin-orbital tensor of an unrestricted basis from the spin
//                          blocks of the spatial tensor (hartree_fock.general_orbital_system)
//
// Fused pass, per output plane (P = 2p+s1, Q = 2q+s2) and 32x32 tile of spatial (r, s):
//   U[P,Q,2r+g,2s+d] = [s1==g][s2==d] A[r,s] - [s1==d][s2==g] A[s,r],   A = u[p,q,:,:]
// The direct tile and the transposed partner tile are both read with coalesced rows and exchanged
// through a padded shared-memory tile; every output element (zeros included) is written exactly once
// with 16-byte vector stores.  Algorithmic traffic: read l^4 + write 16 l^4 elements.
#include "common.cuh"

namespace {

constexpr int kTile = 32;

template <bool IN_COMPLEX>
struct Elem;
template <>
struct Elem<false> {
    double re;
    static __device__ __forceinline__ Elem load(const double* p, long long i) { return {p[i]}; }
    __device__ __forceinline__ double real() const { return re; }
    __device__ __forceinline__ double imag() const { return 0.0; }
};
template <>
struct Elem<true> {
    double re, im;
    static __device__ __forceinline__ Elem load(const double* p, long long i) {
        const double2 v = reinterpret_cast<const double2*>(p)[i];
        return {v.x, v.y};
    }
    __device__ __forceinline__ double real() const { return re; }
    __device__ __forceinline__ double imag() const { return im; }
};

// grid: x = tile index over (r-tile, s-tile), y = q, z = P - p_begin ; block = (32, 8)
template <bool IN_COMPLEX, bool OUT_COMPLEX, bool ANTISYM>
__global__ void __launch_bounds__(256) add_spin_kernel(const double* __restrict__ u, double* __restrict__ out, int l,
                                                        int tiles, long long p_begin) {
    __shared__ double dre[kTile][kTile + 1], ere[kTile][kTile + 1];
    __shared__ double dim_[IN_COMPLEX ? kTile : 1][kTile + 1], eim[IN_COMPLEX ? kTile : 1][kTile + 1];

    const int tr = blockIdx.x / tiles, ts = blockIdx.x % tiles;
    const int q = blockIdx.y;
    const long long P = p_begin + blockIdx.z;
    const int p = (int)(P >> 1), s1 = (int)(P & 1);
    const int r0 = tr * kTile, s0 = ts * kTile;
    const long long n = 2LL * l;
    const double* A = u + ((long long)p * l + q) * l * l * (IN_COMPLEX ? 2 : 1);

    const int tx = threadIdx.x, ty = threadIdx.y;
    // direct tile D[i][j] = A[r0+i, s0+j]; partner tile E[i][j] = A[s0+i, r0+j]
    for (int i = ty; i < kTile; i += 8) {
        if (r0 + i < l && s0 + tx < l) {
            const Elem<IN_COMPLEX> v = Elem<IN_COMPLEX>::load(A, (long long)(r0 + i) * l + s0 + tx);
            dre[i][tx] = v.real();
            if (IN_COMPLEX) dim_[i][tx] = v.imag();
        }
        if (ANTISYM && s0 + i < l && r0 + tx < l) {
            const Elem<IN_COMPLEX> v = Elem<IN_COMPLEX>::load(A, (long long)(s0 + i) * l + r0 + tx);
            ere[i][tx] = v.real();
            if (IN_COMPLEX) eim[i][tx] = v.imag();
        }
    }
    __syncthreads();

    constexpr int OD = OUT_COMPLEX ? 2 : 1;
    if (OUT_COMPLEX) {
        // A spin row holds 64 complex numbers (1 KiB): lane tx writes columns tx and tx + 32 so that each store
        // instruction of the warp covers 512 contiguous bytes (whole sectors, whole lines).
#pragma unroll
        for (int s2 = 0; s2 < 2; ++s2) {
            const long long Q = 2LL * q + s2;
            double* plane = out + (((long long)blockIdx.z * n + Q) * n) * n * OD;
            for (int i = ty; i < kTile; i += 8) {
                const int r = r0 + i;
                if (r >= l) break;
#pragma unroll
                for (int g = 0; g < 2; ++g) {
                    double* row = plane + ((2LL * r + g) * n + 2LL * s0) * OD;
#pragma unroll
                    for (int half = 0; half < 2; ++half) {
                        const int c = tx + 32 * half;  // spin column inside the tile: S = 2 s0 + c
                        const int sl = c >> 1, d = c & 1;
                        if (s0 + sl < l) {
                            const bool direct = (s1 == g) && (s2 == d);
                            const bool exch = ANTISYM && (s1 == d) && (s2 == g);
                            double vr = 0.0, vi = 0.0;
                            if (direct) {
                                vr = dre[i][sl];
                                if (IN_COMPLEX) vi = dim_[i][sl];
                            }
                            if (exch) {
                                vr -= ere[sl][i];
                                if (IN_COMPLEX) vi -= eim[sl][i];
                            }
                            reinterpret_cast<double2*>(row)[c] = make_double2(vr, vi);
                        }
                    }
                }
            }
        }
        return;
    }
    const int s = s0 + tx;
    if (s >= l) return;
#pragma unroll
    for (int s2 = 0; s2 < 2; ++s2) {
        const long long Q = 2LL * q + s2;
        double* plane = out + (((long long)blockIdx.z * n + Q) * n) * n * OD;
        for (int i = ty; i < kTile; i += 8) {
            const int r = r0 + i;
            if (r >= l) break;
            const double ar = dre[i][tx];
            const double br = ANTISYM ? ere[tx][i] : 0.0;
#pragma unroll
            for (int g = 0; g < 2; ++g) {
                // element d of the pair (S = 2s + d): direct if s1==g && s2==d, exchange if s1==d && s2==g
                double vr[2];
#pragma unroll
                for (int d = 0; d < 2; ++d) {
                    const bool direct = (s1 == g) && (s2 == d);
                    const bool exch = ANTISYM && (s1 == d) && (s2 == g);
                    vr[d] = (direct ? ar : 0.0) - (exch ? br : 0.0);
                }
                double* row = plane + ((2LL * r + g) * n + 2LL * s);
                reinterpret_cast<double2*>(row)[0] = make_double2(vr[0], vr[1]);
            }
        }
    }
}

// out[p,q,r,s] = u[p,q,r,s] - u[p,q,s,r].  One block owns the PAIR of 32x32 tiles (R,S) and (S,R), R <= S, of one
// (p,q) plane: every element is read once (T1 = u[R,S], T2 = u[S,R]) and both results are written,
// out[R,S] = T1 - T2^T and out[S,R] = T2 - T1^T -- the algorithmic minimum of one read and one write pass.
// grid: x = tile pair, y = q, z = p - p_begin; block (32, 8)
template <bool COMPLEX>
__global__ void __launch_bounds__(256) antisym_kernel(const double* __restrict__ u, double* __restrict__ out, int n,
                                                       int tiles, long long p_begin) {
    constexpr int ED = COMPLEX ? 2 : 1;
    __shared__ double t1[ED][kTile][kTile + 1];
    __shared__ double t2[ED][kTile][kTile + 1];
    // linear pair index -> (tr <= ts): row tr starts at tr * tiles - tr (tr - 1) / 2
    int tr = 0, rem = blockIdx.x;
    while (rem >= tiles - tr) {
        rem -= tiles - tr;
        ++tr;
    }
    const int ts = tr + rem;
    const int r0 = tr * kTile, s0 = ts * kTile;
    const long long plane = (((long long)(p_begin + blockIdx.z) * n + blockIdx.y) * n) * n;
    const long long oplane = (((long long)blockIdx.z * n + blockIdx.y) * n) * n;
    const int tx = threadIdx.x, ty = threadIdx.y;
    for (int i = ty; i < kTile; i += 8) {
        if (r0 + i < n && s0 + tx < n) {
            const long long idx = plane + (long long)(r0 + i) * n + s0 + tx;
            if (COMPLEX) {
                const double2 v = reinterpret_cast<const double2*>(u)[idx];
                t1[0][i][tx] = v.x;
                t1[ED - 1][i][tx] = v.y;
            } else {
                t1[0][i][tx] = u[idx];
            }
        }
        if (tr != ts && s0 + i < n && r0 + tx < n) {
            const long long idx = plane + (long long)(s0 + i) * n + r0 + tx;
            if (COMPLEX) {
                const double2 v = reinterpret_cast<const double2*>(u)[idx];
                t2[0][i][tx] = v.x;
                t2[ED - 1][i][tx] = v.y;
            } else {
                t2[0][i][tx] = u[idx];
            }
        }
    }
    __syncthreads();
    double(*other)[kTile][kTile + 1] = (tr == ts) ? t1 : t2;  // a diagonal tile is its own partner
    for (int i = ty; i < kTile; i += 8) {
        if (r0 + i < n && s0 + tx < n) {
            const long long oidx = oplane + (long long)(r0 + i) * n + s0 + tx;
            if (COMPLEX)
                reinterpret_cast<double2*>(out)[oidx] =
                    make_double2(t1[0][i][tx] - other[0][tx][i], t1[ED - 1][i][tx] - other[ED - 1][tx][i]);
            else
                out[oidx] = t1[0][i][tx] - other[0][tx][i];
        }
        if (tr != ts && s0 + i < n && r0 + tx < n) {
            const long long oidx = oplane + (long long)(s0 + i) * n + r0 + tx;
            if (COMPLEX)
                reinterpret_cast<double2*>(out)[oidx] =
                    make_double2(t2[0][i][tx] - t1[0][tx][i], t2[ED - 1][i][tx] - t1[ED - 1][tx][i]);
            else
                out[oidx] = t2[0][i][tx] - t1[0][tx][i];
        }
    }
}

// Spin-orbital tensor of an unrestricted basis from its spin blocks.  Output plane (I, J) needs one spatial plane,
// A = B_{sI sJ}[oI, oJ], and its transpose:
//   U[I,J,K,L] = [sK==sI][sL==sJ] A[oK,oL] - [sL==sI][sK==sJ] A[oL,oK]
// A derived B_ba plane is B_ab[oJ, oI] transposed, so there the two tiles swap roles.  The tile scheme is
// add_spin_kernel's: one block owns the direct tile D[i][j] = A[r0+i, s0+j] and its partner E[i][j] = A[s0+i, r0+j],
// both read with coalesced rows, and writes the four spin-orbital elements (K(r, g), L(s, d)) of every spatial
// (r, s) of the tile -- each output element, zeros included, exactly once.  K and L come from the inverse of the
// index tables, built by each block for its 32 + 32 orbitals.  Unlike add_spin_kernel's fixed order, a spin pair
// (s, 0), (s, 1) is one 16-byte store only where the tables put it on an aligned couple of real outputs.
// grid: x = tile index over (r-tile, s-tile), y = J, z = I - p_begin ; block = (32, 8)
template <bool IN_COMPLEX, bool OUT_COMPLEX>
__global__ void __launch_bounds__(256) spin_orbital_kernel(const double* __restrict__ b_aa,
                                                            const double* __restrict__ b_ab,
                                                            const double* __restrict__ b_ba,
                                                            const double* __restrict__ b_bb,
                                                            const int* __restrict__ orbital,
                                                            const int* __restrict__ spin, double* __restrict__ out,
                                                            int l, int tiles, long long p_begin) {
    __shared__ double dre[kTile][kTile + 1], ere[kTile][kTile + 1];
    __shared__ double dim_[IN_COMPLEX ? kTile : 1][kTile + 1], eim[IN_COMPLEX ? kTile : 1][kTile + 1];
    __shared__ int row_of[2][kTile], col_of[2][kTile];  // [spin][orbital - r0 (s0)] -> spin-orbital index

    const int tr = blockIdx.x / tiles, ts = blockIdx.x % tiles;
    const int J = blockIdx.y;
    const long long I = p_begin + blockIdx.z;
    const int r0 = tr * kTile, s0 = ts * kTile;
    const long long n = 2LL * l;
    const int oI = orbital[I], sI = spin[I], oJ = orbital[J], sJ = spin[J];
    const bool derived = sI == 1 && sJ == 0 && b_ba == nullptr;
    const double* blk = sI == 0 ? (sJ == 0 ? b_aa : b_ab) : (sJ == 0 ? (derived ? b_ab : b_ba) : b_bb);
    const long long src_plane = derived ? (long long)oJ * l + oI : (long long)oI * l + oJ;
    const double* A = blk + src_plane * l * l * (IN_COMPLEX ? 2 : 1);

    const int tx = threadIdx.x, ty = threadIdx.y;
    for (int t = ty * 32 + tx; t < n; t += 256) {
        const int o = orbital[t], sp = spin[t];
        if (o >= r0 && o < r0 + kTile) row_of[sp][o - r0] = t;
        if (o >= s0 && o < s0 + kTile) col_of[sp][o - s0] = t;
    }
    for (int i = ty; i < kTile; i += 8) {
        if (r0 + i < l && s0 + tx < l) {
            const Elem<IN_COMPLEX> v = Elem<IN_COMPLEX>::load(A, (long long)(r0 + i) * l + s0 + tx);
            dre[i][tx] = v.real();
            if (IN_COMPLEX) dim_[i][tx] = v.imag();
        }
        if (s0 + i < l && r0 + tx < l) {
            const Elem<IN_COMPLEX> v = Elem<IN_COMPLEX>::load(A, (long long)(s0 + i) * l + r0 + tx);
            ere[i][tx] = v.real();
            if (IN_COMPLEX) eim[i][tx] = v.imag();
        }
    }
    __syncthreads();

    constexpr int OD = OUT_COMPLEX ? 2 : 1;
    double* plane = out + ((long long)blockIdx.z * n + J) * n * n * OD;
    if (OUT_COMPLEX) {
        // lane tx writes spin columns tx and tx + 32 of the tile, (s, d) = (s0 + c / 2, c % 2): in the usual orders
        // (spin fastest within runs of orbitals) each store instruction of the warp covers 512 contiguous bytes
#pragma unroll
        for (int g = 0; g < 2; ++g) {
            for (int i = ty; i < kTile; i += 8) {
                if (r0 + i >= l) break;
                double* row = plane + (long long)row_of[g][i] * n * OD;
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    const int c = tx + 32 * half;
                    const int sl = c >> 1, d = c & 1;
                    if (s0 + sl < l) {
                        const bool direct = (g == sI) && (d == sJ);
                        const bool exch = (d == sI) && (g == sJ);
                        double ar = dre[i][sl], br = ere[sl][i];
                        double ai = IN_COMPLEX ? dim_[i][sl] : 0.0, bi = IN_COMPLEX ? eim[sl][i] : 0.0;
                        if (derived) {
                            const double cr = ar, ci = ai;
                            ar = br, ai = bi, br = cr, bi = ci;
                        }
                        double vr = 0.0, vi = 0.0;
                        if (direct) vr = ar, vi = ai;
                        if (exch) vr -= br, vi -= bi;
                        reinterpret_cast<double2*>(row)[col_of[d][sl]] = make_double2(vr, vi);
                    }
                }
            }
        }
        return;
    }
    const int sl = tx;
    if (s0 + sl >= l) return;
    const int L0 = col_of[0][sl], L1 = col_of[1][sl];
#pragma unroll
    for (int g = 0; g < 2; ++g) {
        for (int i = ty; i < kTile; i += 8) {
            if (r0 + i >= l) break;
            double a = dre[i][sl], b = ere[sl][i];
            if (derived) {
                const double t = a;
                a = b, b = t;
            }
            double v[2];
#pragma unroll
            for (int d = 0; d < 2; ++d) {
                v[d] = 0.0;
                if ((g == sI) && (d == sJ)) v[d] = a;
                if ((d == sI) && (g == sJ)) v[d] -= b;
            }
            double* row = plane + (long long)row_of[g][i] * n;
            if (L1 == L0 + 1 && !(L0 & 1)) {
                *reinterpret_cast<double2*>(row + L0) = make_double2(v[0], v[1]);
            } else if (L0 == L1 + 1 && !(L1 & 1)) {
                *reinterpret_cast<double2*>(row + L1) = make_double2(v[1], v[0]);
            } else {
                row[L0] = v[0];
                row[L1] = v[1];
            }
        }
    }
}

template <bool IN_COMPLEX, bool OUT_COMPLEX>
__global__ void add_spin_one_body_kernel(const double* __restrict__ h, double* __restrict__ out, int l) {
    const long long n = 2LL * l;
    const long long total = n * n;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const int P = (int)(i / n), Q = (int)(i % n);
        double re = 0.0, im = 0.0;
        if ((P & 1) == (Q & 1)) {
            const long long src = (long long)(P >> 1) * l + (Q >> 1);
            re = IN_COMPLEX ? h[2 * src] : h[src];
            im = IN_COMPLEX ? h[2 * src + 1] : 0.0;
        }
        if (OUT_COMPLEX) {
            out[2 * i] = re;
            out[2 * i + 1] = im;
        } else {
            out[i] = re;
        }
    }
}

// spin_2_tb[p,q,r,s] = sum_i S_i[p,r] S_i[q,s]  (- sum_i S_i[p,s] S_i[q,r] when anti-symmetrised), i in {x,y,z}
// (reference basis_set.py:743-747 and :523-526).  One block per (p, q): the six needed rows live in
// shared memory, the (r, s) plane is written with coalesced 16-byte stores.  Write-bound: 16 n^4 bytes.
__global__ void __launch_bounds__(256) spin2_tb_kernel(const double2* __restrict__ sx, const double2* __restrict__ sy,
                                                       const double2* __restrict__ sz, double2* __restrict__ out, int n,
                                                       int antisym, long long p_begin) {
    extern __shared__ double2 rows[];  // [6][n]: S_i[p,:] for i = x,y,z then S_i[q,:]
    const long long pq = blockIdx.x;
    const int p = (int)(p_begin + pq / n), q = (int)(pq % n);
    const double2* mats[3] = {sx, sy, sz};
    for (int j = threadIdx.x; j < 3 * n; j += blockDim.x) {
        const int i = j / n, c = j - i * n;
        rows[i * n + c] = mats[i][(long long)p * n + c];
        rows[(3 + i) * n + c] = mats[i][(long long)q * n + c];
    }
    __syncthreads();
    double2* plane = out + pq * (long long)n * n;
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
        const int r = e / n, s = e - r * n;
        double re = 0.0, im = 0.0;
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const double2 a = rows[i * n + r], b = rows[(3 + i) * n + s];
            re += a.x * b.x - a.y * b.y;
            im += a.x * b.y + a.y * b.x;
            if (antisym) {
                const double2 c = rows[i * n + s], d = rows[(3 + i) * n + r];
                re -= c.x * d.x - c.y * d.y;
                im -= c.x * d.y + c.y * d.x;
            }
        }
        plane[e] = make_double2(re, im);
    }
}

}  // namespace

extern "C" int qs_add_spin_two_body(const void* u, int in_dtype, int64_t l, void* out, int out_dtype, int anti_symmetrize,
                                    int64_t p_begin, int64_t p_end, void* stream) {
    QS_REQUIRE(l > 0 && 0 <= p_begin && p_begin <= p_end && p_end <= 2 * l, "qs_add_spin_two_body: bad plane range");
    QS_REQUIRE(!(in_dtype == QS_C128 && out_dtype == QS_F64), "qs_add_spin_two_body: cannot narrow complex to real");
    if (p_begin == p_end) return QS_OK;  // an empty shard (trailing rank of a block partition)
    QS_REQUIRE(u && out, "qs_add_spin_two_body: bad arguments");
    QS_REQUIRE(l <= 32767, "qs_add_spin_two_body: l too large");
    if (p_begin == p_end) return QS_OK;
    const int tiles = (int)qs_ceil_div(l, kTile);
    const int64_t planes = p_end - p_begin;
    const dim3 block(32, 8);
    const double* in = static_cast<const double*>(u);
    double* o = static_cast<double*>(out);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int span = -1;
    {
        // algorithmic bytes: the spatial planes read once + every output element written once
        const double n4 = (double)planes * 8.0 * l * l * l;  // output elements
        qs_timing_begin(QS_FAMILY_SPIN_PASS,
                        n4 / 16.0 * 8.0 * qs_elem_doubles(in_dtype) + n4 * 8.0 * qs_elem_doubles(out_dtype), stream,
                        &span);
    }
    // gridDim.z is limited to 65535 and gridDim.y too: l <= 32767 covers y; chunk z
    for (int64_t z0 = 0; z0 < planes; z0 += 65535) {
        const int64_t nz = planes - z0 < 65535 ? planes - z0 : 65535;
        const dim3 grid((unsigned)(tiles * tiles), (unsigned)l, (unsigned)nz);
        const int64_t n = 2 * l;
        double* oz = o + z0 * n * n * n * qs_elem_doubles(out_dtype);
        const long long pb = p_begin + z0;
#define QS_SPIN_LAUNCH(IC, OC)                                                                  \
    do {                                                                                        \
        if (anti_symmetrize)                                                                    \
            add_spin_kernel<IC, OC, true><<<grid, block, 0, st>>>(in, oz, (int)l, tiles, pb);   \
        else                                                                                    \
            add_spin_kernel<IC, OC, false><<<grid, block, 0, st>>>(in, oz, (int)l, tiles, pb);  \
    } while (0)
        if (in_dtype == QS_C128)
            QS_SPIN_LAUNCH(true, true);
        else if (out_dtype == QS_C128)
            QS_SPIN_LAUNCH(false, true);
        else
            QS_SPIN_LAUNCH(false, false);
#undef QS_SPIN_LAUNCH
        QS_LAUNCH_CHECK();
    }
    qs_timing_end(span, stream);
    return QS_OK;
}

extern "C" int qs_spin_orbital_two_body(const void* b_aa, const void* b_ab, const void* b_ba, const void* b_bb,
                                        int in_dtype, int64_t l, const int32_t* orbital, const int32_t* spin,
                                        void* out, int out_dtype, int64_t p_begin, int64_t p_end, void* stream) {
    QS_REQUIRE(l > 0 && 0 <= p_begin && p_begin <= p_end && p_end <= 2 * l,
               "qs_spin_orbital_two_body: bad plane range");
    QS_REQUIRE((in_dtype == QS_F64 || in_dtype == QS_C128) && (out_dtype == QS_F64 || out_dtype == QS_C128),
               "qs_spin_orbital_two_body: unknown dtype");
    QS_REQUIRE(!(in_dtype == QS_C128 && out_dtype == QS_F64),
               "qs_spin_orbital_two_body: cannot narrow complex to real");
    if (p_begin == p_end) return QS_OK;  // an empty shard
    QS_REQUIRE(b_aa && b_ab && b_bb && orbital && spin && out, "qs_spin_orbital_two_body: bad arguments");
    QS_REQUIRE(l <= 32767, "qs_spin_orbital_two_body: l too large");
    const int tiles = (int)qs_ceil_div(l, kTile);
    const int64_t planes = p_end - p_begin;
    const int64_t n = 2 * l;
    const dim3 block(32, 8);
    const double *aa = static_cast<const double*>(b_aa), *ab = static_cast<const double*>(b_ab),
                 *ba = static_cast<const double*>(b_ba), *bb = static_cast<const double*>(b_bb);
    double* o = static_cast<double*>(out);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int span = -1;
    // algorithmic bytes: one spatial plane per output plane (I, J) + every output element written once
    qs_timing_begin(QS_FAMILY_SPIN_PASS,
                    (double)planes * n * l * l * 8.0 * qs_elem_doubles(in_dtype) +
                        (double)planes * n * n * n * 8.0 * qs_elem_doubles(out_dtype),
                    stream, &span);
    for (int64_t z0 = 0; z0 < planes; z0 += 65535) {
        const int64_t nz = planes - z0 < 65535 ? planes - z0 : 65535;
        const dim3 grid((unsigned)(tiles * tiles), (unsigned)n, (unsigned)nz);
        double* oz = o + z0 * n * n * n * qs_elem_doubles(out_dtype);
        const long long pb = p_begin + z0;
        if (in_dtype == QS_C128)
            spin_orbital_kernel<true, true><<<grid, block, 0, st>>>(aa, ab, ba, bb, orbital, spin, oz, (int)l, tiles, pb);
        else if (out_dtype == QS_C128)
            spin_orbital_kernel<false, true><<<grid, block, 0, st>>>(aa, ab, ba, bb, orbital, spin, oz, (int)l, tiles, pb);
        else
            spin_orbital_kernel<false, false><<<grid, block, 0, st>>>(aa, ab, ba, bb, orbital, spin, oz, (int)l, tiles, pb);
        QS_LAUNCH_CHECK();
    }
    qs_timing_end(span, stream);
    return QS_OK;
}

extern "C" int qs_anti_symmetrize(const void* u, int dtype, int64_t n, void* out, int64_t p_begin, int64_t p_end,
                                  void* stream) {
    QS_REQUIRE(n > 0 && 0 <= p_begin && p_begin <= p_end && p_end <= n, "qs_anti_symmetrize: bad plane range");
    if (p_begin == p_end) return QS_OK;  // an empty shard
    QS_REQUIRE(u && out && u != out, "qs_anti_symmetrize: bad arguments (in-place is not supported)");
    QS_REQUIRE(n <= 65535, "qs_anti_symmetrize: n too large");
    if (p_begin == p_end) return QS_OK;
    const int tiles = (int)qs_ceil_div(n, kTile);
    const dim3 block(32, 8);
    const dim3 grid((unsigned)(tiles * (tiles + 1) / 2), (unsigned)n, (unsigned)(p_end - p_begin));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int span = -1;
    qs_timing_begin(QS_FAMILY_SPIN_PASS, 2.0 * (double)(p_end - p_begin) * n * n * n * 8.0 * qs_elem_doubles(dtype),
                    stream, &span);
    if (dtype == QS_C128)
        antisym_kernel<true><<<grid, block, 0, st>>>(static_cast<const double*>(u), static_cast<double*>(out), (int)n,
                                                     tiles, p_begin);
    else
        antisym_kernel<false><<<grid, block, 0, st>>>(static_cast<const double*>(u), static_cast<double*>(out), (int)n,
                                                      tiles, p_begin);
    QS_LAUNCH_CHECK();
    qs_timing_end(span, stream);
    return QS_OK;
}

extern "C" int qs_add_spin_one_body(const void* h, int in_dtype, int64_t l, void* out, int out_dtype, void* stream) {
    QS_REQUIRE(h && out && l > 0, "qs_add_spin_one_body: bad arguments");
    QS_REQUIRE(!(in_dtype == QS_C128 && out_dtype == QS_F64), "qs_add_spin_one_body: cannot narrow complex to real");
    const long long total = 4LL * l * l;
    long long blocks = qs_ceil_div(total, 256);
    if (blocks > 148 * 8) blocks = 148 * 8;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const double* in = static_cast<const double*>(h);
    double* o = static_cast<double*>(out);
    if (in_dtype == QS_C128)
        add_spin_one_body_kernel<true, true><<<(unsigned)blocks, 256, 0, st>>>(in, o, (int)l);
    else if (out_dtype == QS_C128)
        add_spin_one_body_kernel<false, true><<<(unsigned)blocks, 256, 0, st>>>(in, o, (int)l);
    else
        add_spin_one_body_kernel<false, false><<<(unsigned)blocks, 256, 0, st>>>(in, o, (int)l);
    QS_LAUNCH_CHECK();
    return QS_OK;
}

extern "C" int qs_spin_squared_two_body(const void* sx, const void* sy, const void* sz, int64_t n, int anti_symmetrize,
                                        void* out, int64_t p_begin, int64_t p_end, void* stream) {
    QS_REQUIRE(n > 0 && 0 <= p_begin && p_begin <= p_end && p_end <= n, "qs_spin_squared_two_body: bad plane range");
    if (p_begin == p_end) return QS_OK;  // an empty shard
    QS_REQUIRE(sx && sy && sz && out, "qs_spin_squared_two_body: bad arguments");
    if (p_begin == p_end) return QS_OK;
    const int smem = 6 * (int)n * 16;
    QS_REQUIRE(smem <= 200 * 1024, "qs_spin_squared_two_body: n too large");
    if (smem > 48 * 1024)
        QS_CUDA(cudaFuncSetAttribute(spin2_tb_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    const long long blocks = (p_end - p_begin) * n;
    QS_REQUIRE(blocks < (1LL << 31), "qs_spin_squared_two_body: grid too large");
    spin2_tb_kernel<<<(unsigned)blocks, 256, smem, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const double2*>(sx), static_cast<const double2*>(sy), static_cast<const double2*>(sz),
        static_cast<double2*>(out), (int)n, anti_symmetrize, p_begin);
    QS_LAUNCH_CHECK();
    return QS_OK;
}
