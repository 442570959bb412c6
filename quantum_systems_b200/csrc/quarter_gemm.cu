// Quarter transform: one index contraction of the four-index transform as an FP64 tensor-core GEMM.
//
//   out[w-major rotated store] = sum_k A[x, k] * M[k, w]
//
// Replaces one np.tensordot (+ transpose) of BasisSet.transform_two_body_elements
// (reference quantum_systems/basis_set.py:342-348).  Design (DESIGN.md, "quarter GEMM"):
//   * every dtype combination is lowered to ONE real GEMM:  a complex A row is 2K real numbers
//     (interleaved storage IS the [re, im] K-doubling), and the coefficient matrix is expanded to a
//     real (K', W') "image" [[Mr, Mi], [-Mi, Mr]] (4M complex product, no extra passes);
//   * A tiles (128 rows x 16 k') arrive by TMA with the 128-byte swizzle; the coefficient image
//     is pre-arranged in MMA fragment order, so it arrives by one 1-D bulk copy per stage;
//   * one persistent CTA per SM, 12 warps: two MMA groups of 4 warps (one warp per SM sub-partition, a
//     32 x (8*NT) accumulator tile each in registers) issue mma.sync m8n8k4 f64 (SASS DMMA.8x8x4; measured
//     16 clk issue interval per sub-partition, 26 clk latency) on alternate tiles, each fed by its own TMA
//     producer warp over its own full/empty mbarrier stage ring; the producer warp group donates registers
//     (setmaxnreg 40 / 232); tile starts are ordered so one group's epilogue overlaps the other's main loop
//     (details above quarter_gemm_kernel);
//   * the epilogue writes the new index as the slowest axis (or any 2-level strided address).
#include <stdlib.h>

#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "common.cuh"

namespace {

constexpr int kBlockX = 128;    // rows of A per CTA tile
constexpr int kChunkK = 16;     // k' per pipeline stage (= one 128-byte swizzled row)
constexpr int kGroups = 2;      // MMA warp groups that ping-pong on the tensor pipe
constexpr int kGroupWarps = 4;  // one warp per SM sub-partition
constexpr int kMmaWarps = kGroups * kGroupWarps;
constexpr int kThreads = (kMmaWarps + 4) * 32;  // + the producer warp group (register donor, one lane issues TMA)
// Register split (setmaxnreg, whole warp groups): the kernel launches with 168 registers per thread
// (65536 / 384); the producer group shrinks to 40 and each MMA group grows to 232 (2 x 128 x 232 + 128 x 40 <= 384 x 168).
// At 24 the producer's tile loop spills to local memory; 232 still holds every NT = 8 instantiation without spills.
constexpr int kRegsProducer = 40;
constexpr int kRegsMma = 232;
constexpr int kATileBytes = kBlockX * kChunkK * 8;  // 16 KiB

constexpr int kMaxDest = 16;    // destination buffers of a scattering store (ranks of one NVSwitch domain)

// Unsigned division by a launch constant d >= 1 of numerators below 2^31 as a multiply and a shift: with
// l = ceil(log2 d), shift = 31 + l and mul = ceil(2^shift / d) < 2^32, the error e = mul d - 2^shift < d makes
// x e < 2^31 2^l = 2^shift, so (x mul) >> shift == x / d exactly (make_divisor on the host).
struct Divisor {
    uint32_t mul, shift;
};

__device__ __forceinline__ uint32_t divide(uint32_t x, Divisor d) {
    return (uint32_t)(((unsigned long long)x * d.mul) >> d.shift);
}

struct QuarterParams {
    const double* image;      // [tiles_w][nchunks][2][NT][32][2] doubles (this launch's tile group)
    double* out;
    // Scattering store (fused re-partition): when ndest > 0 the new index w selects the destination
    // buffer outs[w / w_inner] -- a peer GPU's memory mapped over NVLink -- and sw1 is unused.
    double* outs[kMaxDest];
    int ndest;
    uint32_t X;               // rows of A
    uint32_t Wp;              // real columns actually valid (W or 2W)
    uint32_t w_first;         // first real column of this launch's tile group
    uint32_t tiles_x;         // ceil(X / 128)
    int nchunks;              // ceil(K'/16)
    int last_halves;          // 8-k' halves of the last chunk that hold data (1 or 2)
    int tiles_w;              // column tiles in this group, each 8*NT wide
    // store address = (w/w_inner)*sw1 + (w%w_inner)*sw0 + x2*sx2 + x1*sx1 + x0*sx0 with
    // x = (x2 * x_mid + x1) * x_inner + x0, in OUTPUT ELEMENTS (w = w' for real output, w'/2 for complex)
    uint32_t x_inner, x_mid, w_inner;
    Divisor x_inner_div, tiles_w_div;
    long long sx0, sx1, sx2, sw0, sw1;
    int vec2;                 // real output: row pairs (x, x + 1), x even, are adjacent and 16-byte aligned
    // Column dealing (scattering store): logical output column j of the tile order is the physical column
    // (j * deal_mul) % deal_mod, so every CTA tile's columns are spread over ALL destinations and the NVLink
    // traffic of a launch is uniform in time (contiguous column ranges make every rank write to the same one or
    // two peers at once: measured +29 % on 7 of 8 ranks at n = 400).  deal_mul == 1: identity.
    uint32_t deal_mul, deal_mod;
    // Cyclic destinations (scattering store): column w belongs to destination w % ndest and is column w / ndest there
    // (instead of blocks of w_inner columns per destination).  Consecutive columns then go to different
    // destinations by themselves, and a rank that owns the cyclic columns writes rows INTERLEAVED with the other
    // ranks' rows later on, never one of W adjacent chunks of a block (see sharded.py, "where the tiles land").
    int w_cyclic;
    // Optional tile list (symmetry-aware transforms): when non-null the launch visits only the n_listed linear
    // tile ids (row_tile * tiles_w + col_tile, ascending) stored there instead of all tiles_x * tiles_w tiles.
    const uint32_t* tile_list;
    uint32_t n_listed;
    // Optional row-offset tables (packed pair layouts of the symmetry-aware transform): with x = xq * x_inner + xr
    // the row contributes xq_table[xq] instead of xq * sx1 (a negative entry drops the row: nothing is stored) and
    // xr_table[xr] instead of xr * sx0.  Element offsets.
    const long long* xq_table;
    const long long* xr_table;
    // Column tables (kernels instantiated with COLS only): physical column w goes to outs[col_dest[w]] at element
    // offset col_off[w] -- uneven, caller-defined column ranges per destination.  Rows are placed as above.
    const int* col_dest;
    const long long* col_off;
};

__device__ __forceinline__ uint32_t dealt_column(uint32_t w, uint32_t mul, uint32_t mod) {
    return mul == 1 ? w : (uint32_t)(((unsigned long long)w * mul) % mod);
}

// Store addressing of the strided, staged and split epilogues (the rotated one has its own, see quarter_gemm_kernel).
// Base of output column wl (before dealing) for output elements of ES bytes: the dealt column w goes to destination
// w % ndest as its column w / ndest (cyclic) or to block w / w_inner as its column w % w_inner.  `plain`
// (w_inner == 1 and no destination table, evaluated once per tile) stores column w at w * sw1.  COLS: the column
// tables place the dealt column instead.
template <int ES, bool COLS = false>
__device__ __forceinline__ double* column_base(const QuarterParams& p, bool plain, uint32_t wl) {
    const uint32_t w = dealt_column(wl, p.deal_mul, p.deal_mod);
    if constexpr (COLS) return p.outs[p.col_dest[w]] + (ES / 8) * p.col_off[w];
    if (plain) return p.out + (ES / 8) * ((long long)w * p.sw1);
    const uint32_t wq = p.w_cyclic ? w % (uint32_t)p.ndest : w / p.w_inner;
    const uint32_t wr = p.w_cyclic ? w / (uint32_t)p.ndest : w - wq * p.w_inner;
    return (p.ndest ? p.outs[wq] : p.out) + (ES / 8) * ((long long)wq * p.sw1 + (long long)wr * p.sw0);
}

// Offset of row block xq (rows xq * x_inner + xr): through x_mid, the block table or sx1.  `kept` enters as "the row
// is in range" and leaves false for a block the table drops (a row the symmetry does not need).
__device__ __forceinline__ long long block_offset(const QuarterParams& p, uint32_t xq, bool& kept) {
    if (p.x_mid != 0xFFFFFFFFu) {
        const uint32_t x2 = xq / p.x_mid;
        const uint32_t x1 = xq - x2 * p.x_mid;
        return (long long)x2 * p.sx2 + (long long)x1 * p.sx1;
    }
    if (p.xq_table && kept) {
        const long long tq = p.xq_table[xq];
        if (tq < 0) kept = false;
        return tq;
    }
    return (long long)xq * p.sx1;
}

// Offset of row x and whether anything is stored for it: the in-block part from the row table or xr * sx0, plus
// the block's offset.
__device__ __forceinline__ bool row_offset(const QuarterParams& p, uint32_t x, long long& off) {
    bool kept = x < p.X;
    const uint32_t xq = divide(x, p.x_inner_div);
    const uint32_t xr = x - xq * p.x_inner;
    off = (p.xr_table && kept) ? p.xr_table[xr] : (long long)xr * p.sx0;
    off += block_offset(p, xq, kept);
    return kept;
}

// The k-th tile of this launch: through the optional list.
__device__ __forceinline__ uint32_t tile_at(const QuarterParams& p, uint32_t k) {
    return p.tile_list ? p.tile_list[k] : k;
}

#ifdef QS_DBG_NOWAIT
#define QS_FULL_WAIT(bar, par) ((void)0)
#else
#define QS_FULL_WAIT(bar, par) mbar_wait(bar, par)
#endif

#ifdef QS_DBG_PHASE_CLOCKS
// Development switch (tools/qgemm_bench.cu): every MMA warp of quarter_gemm_kernel stamps clock64() at tile start, at
// the start of the main loop (after the ordered-start wait), at the end of the main loop and at the end of the
// epilogue (which includes the wait for the next tile's first chunk and its fragment loads), and adds the three phase
// lengths to histograms of kPhaseBinClk-clock bins.  Not part of a default build.
constexpr int kPhaseBins = 256, kPhaseBinClk = 256;
__device__ unsigned long long g_phase_hist[3][kPhaseBins];
__device__ unsigned long long g_phase_sum[3];
__device__ unsigned long long g_phase_count;
__device__ __forceinline__ void phase_record(int lane, const long long (&t)[4]) {
    if (lane != 0) return;
    for (int ph = 0; ph < 3; ++ph) {
        const unsigned long long d = (unsigned long long)(t[ph + 1] - t[ph]);
        const unsigned long long bin = d / kPhaseBinClk;
        atomicAdd(&g_phase_hist[ph][bin < kPhaseBins ? bin : kPhaseBins - 1], 1ull);
        atomicAdd(&g_phase_sum[ph], d);
    }
    atomicAdd(&g_phase_count, 1ull);
}
#define QS_PHASE_STAMP(i) (phase_t[i] = clock64())
#else
#define QS_PHASE_STAMP(i) ((void)0)
#endif

// Row ownership inside a warp's 32 x 8NT tile: MMA row g of m-tile mt is tile row
//     row_base(g) + (mt & 1) + 16 * (mt >> 1),      row_base = {0, 4, 2, 6, 8, 12, 10, 14}[g].
// (a) the two row groups of a quarter-warp (g = 2q, 2q + 1) differ in bit 2, so the TMA-swizzled LDS.128 fragment
//     loads are conflict-free; (b) a thread owns PAIRS of adjacent rows (mt = 0,1 and mt = 2,3) and the 8 lanes of a
//     column own 16 consecutive rows, so the epilogue writes whole 128-byte lines with 16-byte stores.
__device__ __forceinline__ int row_base(int g) { return 2 * ((g >> 1) & 1) + 4 * (g & 1) + 8 * (g >> 2); }

// Staged epilogue (BULK kernels): every MMA warp owns two 4 KiB staging buffers in shared memory.
constexpr int kStagingPerWarp = 2 * 4096;
constexpr int kStagingBytes = kMmaWarps * kStagingPerWarp;  // 64 KiB

// One stage ring per MMA group: as many stages (an A tile and a B tile of B_TILE_BYTES) as fit, at most 6.  The
// generic kernel's B tile is 16 k' x 8*NT w' doubles, NT KiB: 4 stages at NT = 8; with the staging buffers of the
// BULK epilogue 3 at NT >= 5, else 4.
template <int B_TILE_BYTES, bool BULK = false>
struct RingConfig {
    static constexpr int kBTileBytes = B_TILE_BYTES;
    // stages stay 1 KiB aligned: the 128-byte TMA swizzle of the A tile is a function of the address bits
    static constexpr int kStageBytes = kATileBytes + (kBTileBytes + 1023) / 1024 * 1024;
    static constexpr int kGroupBudget = BULK ? (227 * 1024 - kStagingBytes - 3 * 1024) / kGroups : 110 * 1024;
    static constexpr int kFit = kGroupBudget / kStageBytes;
    static constexpr int kStages = kFit < 6 ? kFit : 6;
    static constexpr int kRingBytes = kStages * kStageBytes;
    static constexpr int kBarrierBytes = (kGroups * 2 * kStages + 2) * 8;
    // rings | barriers (padded to 128 B) | staging buffers ; + 1 KiB slack for the 1 KiB alignment of the rings
    static constexpr int kStagingOffset = kGroups * kRingBytes + (kBarrierBytes + 127) / 128 * 128;
    static constexpr int kSmemBytes = kStagingOffset + (BULK ? kStagingBytes : 0) + 1024;
};

// The CTA frame of both kernels.  The barriers sit behind the two rings: group g has full[s] at bar_base + 16 g S + 8 s,
// empty[s] S slots further, then order[g] at bar_base + 16 G S + 8 g.  The producer warp group gives its registers
// to the MMA groups (setmaxnreg) and one lane of warp 8 + g fills group g's ring: chunk j of the group's tiles (in
// order) goes to stage j % S.  Returns true on the MMA warps, which then hold kRegsMma registers.
template <class Ring>
__device__ __forceinline__ bool cta_frame(const CUtensorMap& map_a, const QuarterParams& p, uint32_t smem_base,
                                          uint32_t my_tiles) {
    constexpr int kStages = Ring::kStages;
    const uint32_t bar_base = smem_base + kGroups * Ring::kRingBytes;
    const uint32_t bar_order = bar_base + kGroups * 2 * kStages * 8;
    if (threadIdx.x == 0) {
        for (int gs = 0; gs < kGroups * kStages; ++gs) {
            const uint32_t base = bar_base + (gs / kStages) * 16 * kStages + (gs % kStages) * 8;
            mbar_init(base, 1);
            mbar_init(base + 8 * kStages, kGroupWarps);
        }
        mbar_init(bar_order, kGroupWarps);
        mbar_init(bar_order + 8, kGroupWarps);
        mbar_fence_init();
        prefetch_tensormap(&map_a);
    }
    __syncthreads();

    const int warp = threadIdx.x >> 5;
    if (warp >= kMmaWarps) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kRegsProducer));
        const int pg = warp - kMmaWarps;  // producer of group pg
        if (pg >= kGroups) return false;
        if ((threadIdx.x & 31) == 0) {
            const uint32_t ring = smem_base + pg * Ring::kRingBytes;
            const uint32_t bar_full = bar_base + pg * 16 * kStages;
            const uint32_t bar_empty = bar_full + 8 * kStages;
            uint32_t j = 0;
            for (uint32_t i = pg; i < my_tiles; i += kGroups) {
                const uint32_t tile = tile_at(p, blockIdx.x + i * gridDim.x);
                const uint32_t tx = divide(tile, p.tiles_w_div);
                const uint32_t tw = tile - tx * (uint32_t)p.tiles_w;
                const int px0 = (int)(tx * kBlockX);
                const double* img = p.image + (size_t)tw * p.nchunks * (Ring::kBTileBytes / 8);
                for (int c = 0; c < p.nchunks; ++c, ++j) {
                    const uint32_t s = j % kStages;
                    if (j >= (uint32_t)kStages) mbar_wait(bar_empty + 8 * s, ((j / kStages) - 1) & 1);
                    const uint32_t full = bar_full + 8 * s;
#ifdef QS_DBG_NOLOAD
                    mbar_arrive(full);
                    (void)px0; (void)img; (void)ring;
#else
                    mbar_expect_tx(full, kATileBytes + Ring::kBTileBytes);
                    const uint32_t dst = ring + s * Ring::kStageBytes;
                    tma_load_2d(dst, &map_a, c * kChunkK, px0, full);
                    bulk_load_1d(dst + kATileBytes, img + (size_t)c * (Ring::kBTileBytes / 8), Ring::kBTileBytes,
                                 full);
#endif
                }
            }
        }
        return false;
    }
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kRegsMma));
    return true;
}

// One persistent CTA per SM, 12 warps:
//   warps 0-3     MMA group 0, one warp per SM sub-partition, a 32 x 8NT accumulator tile each in registers;
//   warps 4-7     MMA group 1, same sub-partitions; the groups work on alternate tiles of the CTA;
//   warps 8, 9    TMA producers, one per group, each running its own full/empty stage ring (one elected lane);
//   warps 10, 11  idle; the producer warp group exists to donate its registers to the MMA groups (setmaxnreg).
// Tile starts are ORDERED: a group may start tile i only after the other group has passed the midpoint of the
// main loop of tile i - 1.  In steady state both groups are in their main loops half a tile apart (two warps per
// sub-partition hide each other's fragment-load and barrier latencies), and each group's epilogue falls into the
// middle of the other's main loop.  Without the ordering (two independent CTAs per SM) the epilogues drift into
// phase -- the group that is behind runs at full speed while the one ahead stores -- and nothing hides them
// (measured 81 % of the DMMA peak); with strict alternation (one group at a time) a lone warp per sub-partition
// cannot hide its own LDS/scoreboard stalls (measured 86 %).
// BULK: the epilogue does not store from registers.  Each warp drops its 32 x 8NT accumulator tile, 16 real columns
// at a time, into a shared-memory staging buffer laid out [column][row] and hands every run of rows that is
// contiguous in the output (256 bytes for a real, 512 bytes for a complex column) to the copy engine with
// cp.async.bulk shared -> global.  The warp goes on to its next tile while the copies drain: the stores -- over
// NVLink in the scattering launches -- no longer hold the tensor pipe through the depth of the store queue.
// ROTATED: the local rotated store of the dense transforms (one destination, no dealing, no row tables, x_mid
// unused, sx0 = 1, 16-byte row pairs for real output), element (x, w) at w sw1 + (x / x_inner) sx1 + x % x_inner.  It
// carries none of the other addressing modes, so the kernel the headline transform runs is small and keeps no
// per-launch branches in its epilogue.
// Cross-tile pipelining: after its main loop a warp waits for the first chunk of its NEXT tile and loads that chunk's
// first A and B fragments (registers that are dead in the epilogue) before it stores the current tile, so its DMMA
// stream restarts right behind the stores.
// COLUMNS: the strided register epilogue with the column tables (col_dest, col_off) choosing each column's
// destination and offset; a kernel of its own, so the other epilogues keep no table branch.
enum Epilogue { kEpiStrided = 0, kEpiBulk = 1, kEpiRotated = 2, kEpiColumns = 3 };

template <int NT, bool COMPLEX_OUT, int EPI>
__global__ void __launch_bounds__(kThreads, 1)
quarter_gemm_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ QuarterParams p) {
    constexpr bool BULK = EPI == kEpiBulk;
    using Ring = RingConfig<NT * 1024, BULK>;
    constexpr int kStageBytes = Ring::kStageBytes;
    constexpr int kStages = Ring::kStages;

    extern __shared__ unsigned char smem_raw[];
    uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    asm volatile("" : "+r"(smem_base));  // keep it in a register: ptxas otherwise re-derives it inside the main loop
    const uint32_t bar_base = smem_base + kGroups * Ring::kRingBytes;  // barrier layout: see cta_frame
    const uint32_t bar_order = bar_base + kGroups * 2 * kStages * 8;

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t total_tiles = p.tile_list ? p.n_listed : p.tiles_x * (uint32_t)p.tiles_w;
    const uint32_t my_tiles = blockIdx.x < total_tiles ? (total_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    if (!cta_frame<Ring>(map_a, p, smem_base, my_tiles)) return;

    // ===== MMA groups: warp wg of group `group` owns rows [32 wg, 32 wg + 32) x all 8*NT columns of its tile =====
    const int group = warp >> 2;
    const int wg = warp & 3;
    const uint32_t ring = smem_base + group * Ring::kRingBytes;
    const uint32_t bar_full = bar_base + group * 16 * kStages;
    const uint32_t bar_empty = bar_full + 8 * kStages;
    const int g = lane >> 2;
    const int t = lane & 3;
    const int rbase = row_base(g);

    // A fragment address inside a stage: row r = 32*wg + rbase + (mt & 1) + 16*(mt >> 1) (128 B per row), logical
    // 16-byte chunk (4h + t) stored at chunk ^ (r & 7) by the TMA 128-byte swizzle; r & 7 == (rbase & 7) | (mt & 1).
    const uint32_t a_row_off = (uint32_t)(32 * wg + rbase) * 128u;
    const uint32_t b_lane_off = kATileBytes + (uint32_t)lane * 16u;
    auto a_frag_off = [&](int mt, int h) {
        return a_row_off + (uint32_t)((mt & 1) * 128 + (mt >> 1) * 2048) +
               (uint32_t)(((4 * h + t) ^ ((rbase & 7) | (mt & 1))) << 4);
    };

    // fragment loads and the two k-steps (4 k' each) of one half chunk.  Loop order nt-outer / mt-inner: b[nt] dies
    // progressively during the second k-step and is re-loaded for the NEXT half right behind its last use, and
    // the A fragments are double-buffered (a0 / a1), so one warp per sub-partition keeps the DMMA pipe fed
    // across half and chunk boundaries (no second warp is there to fill a bubble during a group's turn).
#ifdef QS_DBG_NOLDS
    auto load_a = [&](double2(&a)[4], uint32_t stage, int h) {
#pragma unroll
        for (int mt = 0; mt < 4; ++mt) a[mt] = make_double2(1.0 + lane + mt, 0.5 + h);
    };
    auto load_b = [&](uint32_t stage, int h, int nt) { return make_double2(2.0 + lane + nt, 0.25 + h); };
#else
    auto load_a = [&](double2(&a)[4], uint32_t stage, int h) {
#pragma unroll
        for (int mt = 0; mt < 4; ++mt) a[mt] = lds_128(stage + a_frag_off(mt, h));
    };
    auto load_b = [&](uint32_t stage, int h, int nt) {
        return lds_128(stage + b_lane_off + (uint32_t)(h * NT + nt) * 512u);
    };
#endif

    uint32_t bulk_pass = 0;  // BULK: staging passes done so far (selects the buffer, bounds the pending copy groups)
#ifdef QS_DBG_PHASE_CLOCKS
    long long phase_t[4];
#endif
    // The group's tiles take consecutive chunks of its ring: chunk j sits in stage s = j % kStages, phase parity
    // par = (j / kStages) & 1.  a0 and b hold the first fragments of the chunk about to start.
    uint32_t s = 0, par = 0;
    uint32_t stage = ring;
    double2 a0[4], a1[4], b[NT];
    auto load_first = [&]() {
        QS_FULL_WAIT(bar_full + 8 * s, par);
        load_a(a0, stage, 0);
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) b[nt] = load_b(stage, 0, nt);
    };
    if ((uint32_t)group < my_tiles) load_first();
    for (uint32_t i = group; i < my_tiles; i += kGroups) {
        QS_PHASE_STAMP(0);
        const uint32_t tile = tile_at(p, blockIdx.x + i * gridDim.x);

        double acc[4][NT][2];
#pragma unroll
        for (int mt = 0; mt < 4; ++mt)
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) acc[mt][nt][0] = acc[mt][nt][1] = 0.0;

        // k-step on the .x halves of the fragments.  `tail_*`: the last B fragment of this half is still to be
        // fetched (the reloads trail their last reader by one column group, so the LDS never waits for a DMMA
        // that has not read its operands yet).
        auto step_x = [&](const double2(&a)[4], double2(&b)[NT], bool tail, uint32_t tail_stage, int tail_h) {
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
#pragma unroll
                for (int mt = 0; mt < 4; ++mt) dmma_8x8x4(acc[mt][nt][0], acc[mt][nt][1], a[mt].x, b[nt].x);
                if (nt == 0 && NT > 1 && tail) b[NT - 1] = load_b(tail_stage, tail_h, NT - 1);
            }
        };
        auto step_y = [&](const double2(&a)[4], const double2(&b)[NT]) {
#pragma unroll
            for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                for (int mt = 0; mt < 4; ++mt) dmma_8x8x4(acc[mt][nt][0], acc[mt][nt][1], a[mt].y, b[nt].y);
        };
        // k-step on the .y halves; b[nt - 1] is re-loaded for the NEXT half behind column group nt
        // (b[NT - 1] follows in the next step_x)
        auto step_y_reload = [&](const double2(&a)[4], double2(&b)[NT], uint32_t next_stage, int next_h) {
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
#pragma unroll
                for (int mt = 0; mt < 4; ++mt) dmma_8x8x4(acc[mt][nt][0], acc[mt][nt][1], a[mt].y, b[nt].y);
                if (NT == 1) b[0] = load_b(next_stage, next_h, 0);
                else if (nt >= 1) b[nt - 1] = load_b(next_stage, next_h, nt - 1);
            }
        };

        // ordered start: the other group has passed the signal point (midpoint) of the main loop of tile i - 1
        const uint32_t k = i >> 1;
        if (i > 0) mbar_wait(bar_order + 8 * group, (group == 0 ? k - 1 : k) & 1);
        const int signal_chunk = (p.nchunks - 1) >> 1;
        QS_PHASE_STAMP(1);

        bool tail = false;  // b[NT - 1] of the half about to start is still to be fetched
        for (int c = 0; c + 1 < p.nchunks; ++c) {
            step_x(a0, b, tail, stage, 0);
            load_a(a1, stage, 1);
            step_y_reload(a0, b, stage, 1);
            step_x(a1, b, true, stage, 1);
            const uint32_t s_done = s;
            if (++s == (uint32_t)kStages) {
                s = 0;
                par ^= 1;
            }
            const uint32_t next_stage = ring + s * kStageBytes;
            QS_FULL_WAIT(bar_full + 8 * s, par);
            load_a(a0, next_stage, 0);
            step_y_reload(a1, b, next_stage, 0);
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(bar_empty + 8 * s_done);
                if (c == signal_chunk) mbar_arrive(bar_order + 8 * (group ^ 1));
            }
            stage = next_stage;
            tail = true;
        }
        // last chunk: it may hold <= 8 valid k', then its all-zero second half is skipped
        step_x(a0, b, tail, stage, 0);
        if (p.last_halves == 2) {
            load_a(a1, stage, 1);
            step_y_reload(a0, b, stage, 1);
            step_x(a1, b, true, stage, 1);
            step_y(a1, b);
        } else {
            step_y(a0, b);
        }
        __syncwarp();
        if (lane == 0) {
            mbar_arrive(bar_empty + 8 * s);
            if (signal_chunk == p.nchunks - 1) mbar_arrive(bar_order + 8 * (group ^ 1));
        }
        QS_PHASE_STAMP(2);
        // the next tile's first chunk follows in the ring; its fragments load while this tile is stored
        if (++s == (uint32_t)kStages) {
            s = 0;
            par ^= 1;
        }
        stage = ring + s * kStageBytes;
        if (i + kGroups < my_tiles) load_first();

        // ===== epilogue: rotated / strided / scattering store straight from the accumulators =====
#ifdef QS_DBG_NOSTORE
        {
            double sum = 0.0;
#pragma unroll
            for (int mt = 0; mt < 4; ++mt)
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) sum += acc[mt][nt][0] + acc[mt][nt][1];
            if (sum == 1.2345e-300) p.out[0] = sum;
#ifdef QS_DBG_PHASE_CLOCKS
            QS_PHASE_STAMP(3);
            phase_record(lane, phase_t);
#endif
            continue;
        }
#endif
        const uint32_t tile_x = divide(tile, p.tiles_w_div);
        const uint32_t tile_w = tile - tile_x * (uint32_t)p.tiles_w;
        const uint32_t x0 = tile_x * kBlockX;
        const uint32_t wbase = p.w_first + tile_w * (8 * NT);
        const bool plain_w = p.w_inner == 1 && p.ndest == 0;
        if constexpr (BULK) {
            constexpr int ES = COMPLEX_OUT ? 16 : 8;         // bytes per output element
            constexpr int CPP = COMPLEX_OUT ? 8 : 16;        // output columns per pass (16 real accumulator columns)
            constexpr int COL_BYTES = 32 * ES;               // one staged column: this warp's 32 rows
            constexpr int PASSES = (NT + 1) / 2;
            const uint32_t stage0 = smem_base + Ring::kStagingOffset + (uint32_t)warp * kStagingPerWarp;
            // this warp's rows [xw0, xw0 + nrow) fall into blocks xq of x_inner rows; consecutive rows of a block
            // are adjacent in the output (sx0 = 1): one run per block
            const uint32_t xw0 = x0 + 32 * wg;
            const uint32_t nrow = xw0 < p.X ? (p.X - xw0 < 32u ? p.X - xw0 : 32u) : 0u;
            const uint32_t xq0 = divide(xw0, p.x_inner_div);
            const uint32_t xr0 = xw0 - xq0 * p.x_inner;
            const uint32_t nruns = nrow ? (xr0 + nrow + p.x_inner - 1) / p.x_inner : 0u;
            const uint32_t items = CPP * nruns;              // (column, run) pairs per pass
#pragma unroll
            for (int pass = 0; pass < PASSES; ++pass) {
                const uint32_t buf = stage0 + (uint32_t)((bulk_pass + pass) & 1) * 4096u;
                // the copies issued from this buffer two passes ago have read it (at most one group may be pending)
                if (bulk_pass + pass >= 2) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
                __syncwarp();
#pragma unroll
                for (int ntl = 0; ntl < 2; ++ntl) {
                    const int nt = 2 * pass + ntl;
                    if (nt < NT) {
                        if (COMPLEX_OUT) {
                            // complex column 4 ntl + t of the pass, element (re, im) = acc[mt][nt][0..1]
                            const uint32_t col = buf + (uint32_t)(4 * ntl + t) * COL_BYTES;
#pragma unroll
                            for (int mt = 0; mt < 4; ++mt)
                                sts_128(col + (uint32_t)(rbase + (mt & 1) + 16 * (mt >> 1)) * 16u, acc[mt][nt][0],
                                        acc[mt][nt][1]);
                        } else {
#pragma unroll
                            for (int e = 0; e < 2; ++e) {
                                const uint32_t col = buf + (uint32_t)(8 * ntl + 2 * t + e) * COL_BYTES;
                                sts_128(col + (uint32_t)rbase * 8u, acc[0][nt][e], acc[1][nt][e]);
                                sts_128(col + (uint32_t)(rbase + 16) * 8u, acc[2][nt][e], acc[3][nt][e]);
                            }
                        }
                    }
                }
                // generic-proxy writes -> async-proxy reads of the copy engine
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                for (uint32_t it = lane; it < items; it += 32) {
                    const uint32_t c = it % CPP, run = it / CPP;
                    const uint32_t wl = (COMPLEX_OUT ? (wbase >> 1) : wbase) + (uint32_t)(CPP * pass) + c;  // output column
                    // padding columns of the last column tile, and the absent second column group of an odd NT
                    if (wl >= (COMPLEX_OUT ? (p.Wp >> 1) : p.Wp) || 2 * pass + (int)(c / (CPP / 2)) >= NT) continue;
                    double* colp = column_base<ES>(p, plain_w, wl);
                    // run `run`: rows [rs, rs + len) of the warp's 32, block xq0 + run, first row of the block xr
                    const uint32_t rs = run ? run * p.x_inner - xr0 : 0u;
                    const uint32_t xr = run ? 0u : xr0;
                    uint32_t len = p.x_inner - xr;
                    if (len > nrow - rs) len = nrow - rs;
                    bool kept = true;
                    const long long off = xr + block_offset(p, xq0 + run, kept);
                    if (!kept) continue;
                    bulk_store(colp + (ES / 8) * off, buf + c * COL_BYTES + rs * ES, len * ES);
                }
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
            bulk_pass += PASSES;
        } else if constexpr (EPI == kEpiRotated) {
            // rows x = xt + (mt & 1) + 16 (mt >> 1) of this thread; for real output the row pairs (xt, xt + 1) and
            // (xt + 16, xt + 17) share a block (xt and x_inner are even) and leave as one 16-byte store each
            const uint32_t xt = x0 + 32 * wg + rbase;
            constexpr int NX = COMPLEX_OUT ? 4 : 2;
            long long xoff[NX];
            bool xok[NX];
#pragma unroll
            for (int r = 0; r < NX; ++r) {
                const uint32_t x = COMPLEX_OUT ? xt + (r & 1) + 16 * (r >> 1) : xt + 16 * r;
                const uint32_t xq = divide(x, p.x_inner_div);
                xok[r] = x < p.X;
                xoff[r] = (long long)xq * p.sx1 + (long long)(x - xq * p.x_inner);
            }
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                const uint32_t wp = wbase + 8 * nt + 2 * t;  // real column of acc[..][nt][0]; wp + 1 for [1]
                if (COMPLEX_OUT) {
                    if (wp < p.Wp) {
                        double* col = p.out + 2 * ((long long)(wp >> 1) * p.sw1);
#pragma unroll
                        for (int mt = 0; mt < 4; ++mt)
                            if (xok[mt])
                                *reinterpret_cast<double2*>(col + 2 * xoff[mt]) = make_double2(acc[mt][nt][0], acc[mt][nt][1]);
                    }
                } else {
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        if (wp + e < p.Wp) {
                            double* col = p.out + (long long)(wp + e) * p.sw1;
#pragma unroll
                            for (int r = 0; r < 2; ++r)
                                if (xok[r])
                                    *reinterpret_cast<double2*>(col + xoff[r]) =
                                        make_double2(acc[2 * r][nt][e], acc[2 * r + 1][nt][e]);
                        }
                    }
                }
            }
        } else {
        long long xoff[4];
        bool xok[4];
#pragma unroll
        for (int mt = 0; mt < 4; ++mt) xok[mt] = row_offset(p, x0 + 32 * wg + rbase + (mt & 1) + 16 * (mt >> 1), xoff[mt]);
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            const uint32_t wp = wbase + 8 * nt + 2 * t;  // real column of acc[..][nt][0]; wp + 1 for [1]
            if (COMPLEX_OUT) {
                if (wp < p.Wp) {
                    double* col = column_base<16, EPI == kEpiColumns>(p, plain_w, wp >> 1);
#pragma unroll
                    for (int mt = 0; mt < 4; ++mt)
                        if (xok[mt])
                            *reinterpret_cast<double2*>(col + 2 * xoff[mt]) = make_double2(acc[mt][nt][0], acc[mt][nt][1]);
                }
            } else {
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    if (wp + e < p.Wp) {
                        double* col = column_base<8, EPI == kEpiColumns>(p, plain_w, wp + e);
                        if (p.vec2) {
                            // rows (mt = 0, 1) and (mt = 2, 3) are adjacent and 16-byte aligned in the output
                            if (xok[0]) *reinterpret_cast<double2*>(col + xoff[0]) = make_double2(acc[0][nt][e], acc[1][nt][e]);
                            if (xok[2]) *reinterpret_cast<double2*>(col + xoff[2]) = make_double2(acc[2][nt][e], acc[3][nt][e]);
                        } else {
#pragma unroll
                            for (int mt = 0; mt < 4; ++mt)
                                if (xok[mt]) col[xoff[mt]] = acc[mt][nt][e];
                        }
                    }
                }
            }
        }
        }  // register-store epilogue
#ifdef QS_DBG_PHASE_CLOCKS
        QS_PHASE_STAMP(3);
        phase_record(lane, phase_t);
#endif
    }
    // the staging buffers must outlive the copies that read them; completion also orders the stores before the exit
    if constexpr (BULK) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}


// ---------------------------------------------------------------------------------------------
// Split variant: complex A times REAL M ("2M").  Z = (Ar + i Ai) M = Ar M + i Ai M is two real products with
// the SAME coefficient fragments; lowering it to the generic kernel through the real image [[M, 0], [0, M]]
// would issue twice the DMMAs, half of them on zeros.  Here a lane's A fragment double2 is (re, im) of one
// complex k (interleaved storage, as in the generic kernel): the .x halves feed the accumulators of the real
// parts, the .y halves those of the imaginary parts, both against one B fragment per (k, column) taken from an
// image that stores M once:  image[tile][chunk][ntc][lane][h] = M[8 chunk + 4h + t][w_first + 8 NTC tile + 8 ntc + g].
// Same CTA organisation as quarter_gemm_kernel (two ordered MMA groups, per-group TMA producer and ring,
// setmaxnreg split); a CTA tile is 128 rows x 8 NTC complex columns (NTC <= 4).
// ---------------------------------------------------------------------------------------------
template <int NTC>
using SplitRing = RingConfig<NTC * 512>;  // B tile: 8 complex k x 8*NTC columns, one double each

template <int NTC, bool COLS = false>
__global__ void __launch_bounds__(kThreads, 1)
quarter_gemm_split_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ QuarterParams p) {
    using Ring = SplitRing<NTC>;
    constexpr int kStageBytes = Ring::kStageBytes;
    constexpr int kStages = Ring::kStages;

    extern __shared__ unsigned char smem_raw[];
    uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    asm volatile("" : "+r"(smem_base));
    const uint32_t bar_base = smem_base + kGroups * Ring::kRingBytes;
    const uint32_t bar_order = bar_base + kGroups * 2 * kStages * 8;

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t total_tiles = p.tile_list ? p.n_listed : p.tiles_x * (uint32_t)p.tiles_w;
    const uint32_t my_tiles = blockIdx.x < total_tiles ? (total_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    if (!cta_frame<Ring>(map_a, p, smem_base, my_tiles)) return;

    const int group = warp >> 2;
    const int wg = warp & 3;
    const uint32_t ring = smem_base + group * Ring::kRingBytes;
    const uint32_t bar_full = bar_base + group * 16 * kStages;
    const uint32_t bar_empty = bar_full + 8 * kStages;
    const int g = lane >> 2;
    const int t = lane & 3;
    const int rbase = row_base(g);
    const uint32_t a_row_off = (uint32_t)(32 * wg + rbase) * 128u;
    const uint32_t b_lane_off = kATileBytes + (uint32_t)lane * 16u;
    auto a_frag_off = [&](int mt, int h) {
        return a_row_off + (uint32_t)((mt & 1) * 128 + (mt >> 1) * 2048) +
               (uint32_t)(((4 * h + t) ^ ((rbase & 7) | (mt & 1))) << 4);
    };
    auto load_a = [&](double2(&a)[4], uint32_t stage, int h) {
#pragma unroll
        for (int mt = 0; mt < 4; ++mt) a[mt] = lds_128(stage + a_frag_off(mt, h));
    };
    auto load_b = [&](double2(&b)[NTC], uint32_t stage) {
#pragma unroll
        for (int ntc = 0; ntc < NTC; ++ntc) b[ntc] = lds_128(stage + b_lane_off + (uint32_t)ntc * 512u);
    };

    for (uint32_t i = group; i < my_tiles; i += kGroups) {
        const uint32_t tile = tile_at(p, blockIdx.x + i * gridDim.x);

        double re[4][NTC][2], im[4][NTC][2];
#pragma unroll
        for (int mt = 0; mt < 4; ++mt)
#pragma unroll
            for (int ntc = 0; ntc < NTC; ++ntc) re[mt][ntc][0] = re[mt][ntc][1] = im[mt][ntc][0] = im[mt][ntc][1] = 0.0;

        // one half chunk (4 complex k): real parts of A against b, then imaginary parts against the same b
        auto half_step = [&](const double2(&a)[4], const double2(&b)[NTC], bool second) {
#pragma unroll
            for (int ntc = 0; ntc < NTC; ++ntc)
#pragma unroll
                for (int mt = 0; mt < 4; ++mt)
                    dmma_8x8x4(re[mt][ntc][0], re[mt][ntc][1], a[mt].x, second ? b[ntc].y : b[ntc].x);
#pragma unroll
            for (int ntc = 0; ntc < NTC; ++ntc)
#pragma unroll
                for (int mt = 0; mt < 4; ++mt)
                    dmma_8x8x4(im[mt][ntc][0], im[mt][ntc][1], a[mt].y, second ? b[ntc].y : b[ntc].x);
        };

        const uint32_t j = (i >> 1) * (uint32_t)p.nchunks;
        uint32_t s = j % kStages, par = (j / kStages) & 1;
        uint32_t stage = ring + s * kStageBytes;
        double2 a0[4], a1[4], b0[NTC], b1[NTC];
        mbar_wait(bar_full + 8 * s, par);
        load_a(a0, stage, 0);
        load_b(b0, stage);

        const uint32_t k = i >> 1;
        if (i > 0) mbar_wait(bar_order + 8 * group, (group == 0 ? k - 1 : k) & 1);
        const int signal_chunk = (p.nchunks - 1) >> 1;

        // chunks are processed in pairs of register sets (a0/b0 <-> a1's successor) without copies: the loop
        // body is written once for "current = (a0, b0)" and the fragments of the next chunk land in (a0, b1) ...
        for (int c = 0; c + 1 < p.nchunks; ++c) {
            load_a(a1, stage, 1);           // second half of this chunk, in flight during the first half's DMMAs
            half_step(a0, b0, false);
            const uint32_t s_done = s;
            if (++s == (uint32_t)kStages) {
                s = 0;
                par ^= 1;
            }
            const uint32_t next_stage = ring + s * kStageBytes;
            mbar_wait(bar_full + 8 * s, par);
            load_a(a0, next_stage, 0);      // first half of the next chunk, in flight during the second half
            load_b(b1, next_stage);
            half_step(a1, b0, true);
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(bar_empty + 8 * s_done);
                if (c == signal_chunk) mbar_arrive(bar_order + 8 * (group ^ 1));
            }
#pragma unroll
            for (int ntc = 0; ntc < NTC; ++ntc) b0[ntc] = b1[ntc];
            stage = next_stage;
        }
        // last chunk: it may hold <= 4 valid complex k, then its all-zero second half is skipped
        if (p.last_halves == 2) load_a(a1, stage, 1);
        half_step(a0, b0, false);
        if (p.last_halves == 2) half_step(a1, b0, true);
        __syncwarp();
        if (lane == 0) {
            mbar_arrive(bar_empty + 8 * s);
            if (signal_chunk == p.nchunks - 1) mbar_arrive(bar_order + 8 * (group ^ 1));
        }

        // ===== epilogue: complex128 (re, im) pairs, rotated / strided / scattering store =====
        const uint32_t tile_x = divide(tile, p.tiles_w_div);
        const uint32_t tile_w = tile - tile_x * (uint32_t)p.tiles_w;
        const uint32_t x0 = tile_x * kBlockX;
        long long xoff[4];
        bool xok[4];
#pragma unroll
        for (int mt = 0; mt < 4; ++mt) xok[mt] = row_offset(p, x0 + 32 * wg + rbase + (mt & 1) + 16 * (mt >> 1), xoff[mt]);
        const uint32_t wbase = p.w_first + tile_w * (8 * NTC);  // complex columns
        const bool plain_w = p.w_inner == 1 && p.ndest == 0;
#pragma unroll
        for (int ntc = 0; ntc < NTC; ++ntc) {
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const uint32_t wl = wbase + 8 * ntc + 2 * t + e;
                if (wl >= p.Wp) continue;  // Wp = number of complex columns in this mode
                double* col = column_base<16, COLS>(p, plain_w, wl);
#pragma unroll
                for (int mt = 0; mt < 4; ++mt)
                    if (xok[mt])
                        *reinterpret_cast<double2*>(col + 2 * xoff[mt]) = make_double2(re[mt][ntc][e], im[mt][ntc][e]);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// coefficient image: real (K', W') expansion of M laid out in MMA fragment order, per tile group
//   image[tile][chunk][h][nt][lane][e] = M'[16*chunk + 8h + 2t + e][w_first + 8*NT*tile + 8nt + g]
// ---------------------------------------------------------------------------------------------
struct ImageParams {
    const double* m;
    long long sk, sw;  // element strides of M[k, w]
    int m_complex, a_complex, conj;
    int Kp, Wp;        // real extents: K * (a_complex ? 2 : 1), W * (out_complex ? 2 : 1)
    int NT, nchunks, tiles_w, w_first;
    int coulomb;       // 1: M[k, w] = alpha / sqrt((m[k] - m[w])^2 + a^2), m = grid (ODQD interaction)
    double alpha, a2;
    unsigned deal_mul, deal_mod;  // image column j holds M[:, (j * deal_mul) % deal_mod] (see QuarterParams)
    int split;         // 1: complex A x real M, image of quarter_gemm_split_kernel (NT holds NTC, Wp complex columns)
    int K;             // split: complex k extent
};

__device__ __forceinline__ double image_value(const ImageParams& q, int kp, int wp) {
    if (kp >= q.Kp || wp >= q.Wp) return 0.0;
    if (q.coulomb) {
        // reference quantum_dots/one_dim/one_dim_qd.py:29-32 (_shielded_coulomb)
        const double dx = q.m[kp] - q.m[wp];
        return q.alpha / sqrt(dx * dx + q.a2);
    }
    const bool out_complex = q.m_complex || q.a_complex;
    const int k = q.a_complex ? (kp >> 1) : kp;
    const int ka = q.a_complex ? (kp & 1) : 0;  // 0: real part of A column, 1: imaginary part
    int w = out_complex ? (wp >> 1) : wp;
    const int wb = out_complex ? (wp & 1) : 0;  // 0: real part of output, 1: imaginary part
    if (q.deal_mul > 1) w = (int)(((unsigned long long)w * q.deal_mul) % q.deal_mod);
    const long long idx = (long long)k * q.sk + (long long)w * q.sw;
    double mr, mi = 0.0;
    if (q.m_complex) {
        mr = q.m[2 * idx];
        mi = q.m[2 * idx + 1];
        if (q.conj) mi = -mi;
    } else {
        mr = q.m[idx];
    }
    // (ar + i ai)(mr + i mi): re = ar mr - ai mi ; im = ar mi + ai mr
    if (ka == 0) return wb == 0 ? mr : mi;
    return wb == 0 ? -mi : mr;
}

// image[tile][chunk][ntc][lane][h] = M[8 chunk + 4h + t][w_first + 8 NTC tile + 8 ntc + g]   (split variant)
__global__ void build_split_image_kernel(ImageParams q, double* __restrict__ image) {
    const long long per_chunk = 64LL * q.NT;
    const long long total = (long long)q.tiles_w * q.nchunks * per_chunk;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        long long r = i;
        const int h = r & 1; r >>= 1;
        const int lane = r & 31; r >>= 5;
        const int ntc = r % q.NT; r /= q.NT;
        const int chunk = r % q.nchunks;
        const int tw = r / q.nchunks;
        const int g = lane >> 2, t = lane & 3;
        const int k = 8 * chunk + 4 * h + t;
        int w = q.w_first + 8 * q.NT * tw + 8 * ntc + g;
        double v = 0.0;
        if (k < q.K && w < q.Wp) {
            if (q.deal_mul > 1) w = (int)(((unsigned long long)w * q.deal_mul) % q.deal_mod);
            v = q.m[(long long)k * q.sk + (long long)w * q.sw];
        }
        image[i] = v;
    }
}

__global__ void build_image_kernel(ImageParams q, double* __restrict__ image) {
    const long long per_chunk = 128LL * q.NT;
    const long long total = (long long)q.tiles_w * q.nchunks * per_chunk;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        long long r = i;
        const int e = r & 1; r >>= 1;
        const int lane = r & 31; r >>= 5;
        const int nt = r % q.NT; r /= q.NT;
        const int h = r & 1; r >>= 1;
        const int chunk = r % q.nchunks;
        const int tw = r / q.nchunks;
        const int g = lane >> 2, t = lane & 3;
        const int kp = 16 * chunk + 8 * h + 2 * t + e;
        const int wp = q.w_first + 8 * q.NT * tw + 8 * nt + g;
        image[i] = image_value(q, kp, wp);
    }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
// The W' real columns are cut into 8-wide MMA column tiles; those are dealt to CTA tiles of NT <= 8
// column tiles each, in at most two groups whose NT differ by one (e.g. W' = 400 -> 6 x NT=7 + 1 x NT=8),
// so no CTA tile carries more than 7 padding columns.  Each group is one persistent launch.
// Which launches use the staged asynchronous epilogue (QS_BULK = off | scatter | all; default scatter).  Measured on
// a B200 (profiles/r02d_perf_bulk_vs_register_epilogue.jsonl): for LOCAL stores the register epilogue is 1-6 %
// faster (one more ring stage, no lane-serialised copy issue), so only the scattering launches -- whose stores
// cross NVLink and otherwise hold the warp through the depth of the store queue -- stage their tiles.
int g_bulk_mode = -1;
int bulk_mode() {
    if (g_bulk_mode < 0) {
        const char* v = getenv("QS_BULK");
        g_bulk_mode = !v ? 1 : !strcmp(v, "off") ? 0 : !strcmp(v, "all") ? 2 : 1;
    }
    return g_bulk_mode;
}

struct TileGroup {
    int NT, tiles_w, w_first;
    int64_t image_offset;  // doubles
};

struct Tiling {
    int split;  // complex A x real M: quarter_gemm_split_kernel, TileGroup::NT holds NTC (complex column tiles)
    int Kp, Wp, nchunks, last_halves, ngroups;
    TileGroup group[2];
    int64_t image_doubles;
};

Tiling make_tiling(int64_t K, int64_t W, int a_dtype, int m_dtype) {
    Tiling tl;
    const bool out_complex = a_dtype == QS_C128 || m_dtype == QS_C128;
    tl.split = (a_dtype == QS_C128 && m_dtype == QS_F64) ? 1 : 0;
    tl.Kp = (int)(K * (a_dtype == QS_C128 ? 2 : 1));
    tl.Wp = (int)(tl.split ? W : W * (out_complex ? 2 : 1));  // split: complex columns, 8 per column tile
    tl.nchunks = (int)qs_ceil_div(tl.Kp, kChunkK);
    tl.last_halves = (tl.Kp - (tl.nchunks - 1) * kChunkK) <= 8 ? 1 : 2;
    const int max_nt = tl.split ? 4 : 8;                       // column tiles per CTA tile
    const int per_tile_chunk = tl.split ? 64 : 128;            // image doubles per column tile and chunk
    const int col_tiles = (int)qs_ceil_div(tl.Wp, 8);
    const int cta_tiles = (int)qs_ceil_div(col_tiles, max_nt);
    const int base = col_tiles / cta_tiles, extra = col_tiles % cta_tiles;
    tl.ngroups = 0;
    int64_t off = 0;
    int w = 0;
    if (extra > 0) {
        tl.group[tl.ngroups++] = {base + 1, extra, w, off};
        off += (int64_t)extra * tl.nchunks * per_tile_chunk * (base + 1);
        w += extra * (base + 1) * 8;
    }
    tl.group[tl.ngroups++] = {base, cta_tiles - extra, w, off};
    off += (int64_t)(cta_tiles - extra) * tl.nchunks * per_tile_chunk * base;
    tl.image_doubles = off;
    return tl;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(ptr);
    }
    return fn;
}

// One persistent CTA per SM (at most one per tile) of KERNEL with SMEM bytes of dynamic shared memory.
template <auto KERNEL, int SMEM>
int launch_variant(const CUtensorMap& map, const QuarterParams& p, cudaStream_t st) {
    static_assert(SMEM <= 227 * 1024, "shared memory budget of one CTA per SM");
    static bool configured[kMaxDevices] = {false};  // the attribute belongs to the device's context
    const int dev = qs_current_device();
    if (!configured[dev]) {
        QS_CUDA(cudaFuncSetAttribute(KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
        configured[dev] = true;
    }
    const int64_t total = p.tile_list ? (int64_t)p.n_listed : (int64_t)p.tiles_x * p.tiles_w;
    const int64_t resident = qs_sm_count();
    const int64_t grid = total < resident ? total : resident;
    KERNEL<<<(unsigned)grid, kThreads, SMEM, st>>>(map, p);
    QS_LAUNCH_CHECK();
    return QS_OK;
}

template <bool CO, int EPI>
int launch_nt(int NT, const CUtensorMap& map, const QuarterParams& p, cudaStream_t st) {
    constexpr bool B = EPI == kEpiBulk;
    switch (NT) {
        case 1: return launch_variant<quarter_gemm_kernel<1, CO, EPI>, RingConfig<1 * 1024, B>::kSmemBytes>(map, p, st);
        case 2: return launch_variant<quarter_gemm_kernel<2, CO, EPI>, RingConfig<2 * 1024, B>::kSmemBytes>(map, p, st);
        case 3: return launch_variant<quarter_gemm_kernel<3, CO, EPI>, RingConfig<3 * 1024, B>::kSmemBytes>(map, p, st);
        case 4: return launch_variant<quarter_gemm_kernel<4, CO, EPI>, RingConfig<4 * 1024, B>::kSmemBytes>(map, p, st);
        case 5: return launch_variant<quarter_gemm_kernel<5, CO, EPI>, RingConfig<5 * 1024, B>::kSmemBytes>(map, p, st);
        case 6: return launch_variant<quarter_gemm_kernel<6, CO, EPI>, RingConfig<6 * 1024, B>::kSmemBytes>(map, p, st);
        case 7: return launch_variant<quarter_gemm_kernel<7, CO, EPI>, RingConfig<7 * 1024, B>::kSmemBytes>(map, p, st);
        case 8: return launch_variant<quarter_gemm_kernel<8, CO, EPI>, RingConfig<8 * 1024, B>::kSmemBytes>(map, p, st);
    }
    qs_set_error("internal: NT=%d out of range", NT);
    return QS_ERR_INVALID;
}

template <bool CO>
int launch_epilogue(int epi, int NT, const CUtensorMap& map, const QuarterParams& p, cudaStream_t st) {
    switch (epi) {
        case kEpiStrided: return launch_nt<CO, kEpiStrided>(NT, map, p, st);
        case kEpiBulk: return launch_nt<CO, kEpiBulk>(NT, map, p, st);
        case kEpiColumns: return launch_nt<CO, kEpiColumns>(NT, map, p, st);
        default: return launch_nt<CO, kEpiRotated>(NT, map, p, st);
    }
}

// Divisor of d (1 <= d < 2^32) for numerators below 2^31 (see Divisor).
Divisor make_divisor(uint64_t d) {
    uint32_t l = 0;
    while ((1ull << l) < d) ++l;
    const uint32_t shift = 31 + l;
    return {(uint32_t)(((1ull << shift) + d - 1) / d), shift};
}

template <bool COLS>
int launch_split_ntc(int NTC, const CUtensorMap& map, const QuarterParams& p, cudaStream_t st) {
    switch (NTC) {
        case 1: return launch_variant<quarter_gemm_split_kernel<1, COLS>, SplitRing<1>::kSmemBytes>(map, p, st);
        case 2: return launch_variant<quarter_gemm_split_kernel<2, COLS>, SplitRing<2>::kSmemBytes>(map, p, st);
        case 3: return launch_variant<quarter_gemm_split_kernel<3, COLS>, SplitRing<3>::kSmemBytes>(map, p, st);
        case 4: return launch_variant<quarter_gemm_split_kernel<4, COLS>, SplitRing<4>::kSmemBytes>(map, p, st);
    }
    qs_set_error("internal: NTC=%d out of range", NTC);
    return QS_ERR_INVALID;
}

int launch_split(bool cols, int NTC, const CUtensorMap& map, const QuarterParams& p, cudaStream_t st) {
    return cols ? launch_split_ntc<true>(NTC, map, p, st) : launch_split_ntc<false>(NTC, map, p, st);
}

int build_image(ImageParams q, const Tiling& tl, void* image, void* stream) {
    q.Kp = tl.Kp;
    q.Wp = tl.Wp;
    q.nchunks = tl.nchunks;
    q.split = tl.split;
    q.K = tl.Kp / 2;
    QS_REQUIRE(!(tl.split && q.coulomb), "internal: the Coulomb image has no split form");
    for (int gi = 0; gi < tl.ngroups; ++gi) {
        const TileGroup& gr = tl.group[gi];
        q.NT = gr.NT;
        q.tiles_w = gr.tiles_w;
        q.w_first = gr.w_first;
        const long long total = (long long)gr.tiles_w * tl.nchunks * (tl.split ? 64 : 128) * gr.NT;
        long long blocks = qs_ceil_div(total, 256);
        const long long cap = (long long)qs_sm_count() * 16;
        if (blocks > cap) blocks = cap;
        double* dst = static_cast<double*>(image) + gr.image_offset;
        if (tl.split)
            build_split_image_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(q, dst);
        else
            build_image_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(q, dst);
        QS_LAUNCH_CHECK();
    }
    return QS_OK;
}

}  // namespace

// 0: register stores everywhere; 1: staged asynchronous epilogue in the scattering launches (default); 2: wherever
// the alignment conditions hold.  Returns the previous mode.  Development / test switch (also QS_BULK in the
// environment, read once).
extern "C" int qs_set_bulk_epilogue_mode(int mode) {
    const int previous = bulk_mode();
    if (mode >= 0 && mode <= 2) g_bulk_mode = mode;
    return previous;
}

#ifdef QS_DBG_PHASE_CLOCKS
// Copies out the phase histograms (3 x kPhaseBins), the summed phase lengths (3) and the number of warp tiles recorded
// since the last reset; `reset` zeroes them afterwards.
extern "C" int qs_dbg_phase_clocks(unsigned long long* hist, unsigned long long* sum, unsigned long long* count,
                                   int reset) {
    if (hist) QS_CUDA(cudaMemcpyFromSymbol(hist, g_phase_hist, sizeof(g_phase_hist)));
    if (sum) QS_CUDA(cudaMemcpyFromSymbol(sum, g_phase_sum, sizeof(g_phase_sum)));
    if (count) QS_CUDA(cudaMemcpyFromSymbol(count, g_phase_count, sizeof(g_phase_count)));
    if (reset) {
        static const unsigned long long zeros[3 * kPhaseBins] = {};
        QS_CUDA(cudaMemcpyToSymbol(g_phase_hist, zeros, sizeof(g_phase_hist)));
        QS_CUDA(cudaMemcpyToSymbol(g_phase_sum, zeros, sizeof(g_phase_sum)));
        QS_CUDA(cudaMemcpyToSymbol(g_phase_count, zeros, sizeof(g_phase_count)));
    }
    return QS_OK;
}
#endif

extern "C" int qs_coeff_image_bytes(int64_t K, int64_t W, int a_dtype, int m_dtype, int64_t* bytes) {
    QS_REQUIRE(K > 0 && W > 0 && bytes, "qs_coeff_image_bytes: bad arguments");
    QS_REQUIRE(K < (1 << 24) && W < (1 << 24), "qs_coeff_image_bytes: K or W too large");
    const Tiling tl = make_tiling(K, W, a_dtype, m_dtype);
    *bytes = tl.image_doubles * 8;
    return QS_OK;
}

namespace {
int64_t gcd64(int64_t a, int64_t b) {
    while (b) {
        const int64_t t = a % b;
        a = b;
        b = t;
    }
    return a;
}
}  // namespace

// Multiplier of the column dealing for W output columns: the integer nearest to W / golden ratio that is
// coprime to W (consecutive multiples are then a low-discrepancy sequence mod W).  1 = no dealing.
extern "C" int qs_scatter_deal(int64_t W, int64_t* w_deal) {
    QS_REQUIRE(W > 0 && w_deal, "qs_scatter_deal: bad arguments");
    *w_deal = 1;
    if (W < 16) return QS_OK;
    int64_t s = (int64_t)((double)W * 0.6180339887498949 + 0.5);
    while (s < W && gcd64(s, W) != 1) ++s;
    if (s > 1 && s < W) *w_deal = s;
    return QS_OK;
}

extern "C" int qs_build_coeff_image_dealt(const void* m, int m_dtype, int64_t m_sk, int64_t m_sw, int m_conj,
                                          int64_t K, int64_t W, int a_dtype, int64_t w_deal, void* image,
                                          void* stream) {
    QS_REQUIRE(m && image && K > 0 && W > 0, "qs_build_coeff_image: bad arguments");
    QS_REQUIRE(w_deal >= 1 && w_deal < (W > 1 ? W : 2) && gcd64(w_deal, W) == 1,
               "qs_build_coeff_image: the dealing multiplier %lld is not coprime to W = %lld", (long long)w_deal,
               (long long)W);
    const Tiling tl = make_tiling(K, W, a_dtype, m_dtype);
    ImageParams q;
    memset(&q, 0, sizeof(q));
    q.m = static_cast<const double*>(m);
    q.sk = m_sk;
    q.sw = m_sw;
    q.m_complex = m_dtype == QS_C128;
    q.a_complex = a_dtype == QS_C128;
    q.conj = m_conj;
    q.deal_mul = (unsigned)w_deal;
    q.deal_mod = (unsigned)W;
    return build_image(q, tl, image, stream);
}

extern "C" int qs_build_coeff_image(const void* m, int m_dtype, int64_t m_sk, int64_t m_sw, int m_conj, int64_t K,
                                    int64_t W, int a_dtype, void* image, void* stream) {
    return qs_build_coeff_image_dealt(m, m_dtype, m_sk, m_sw, m_conj, K, W, a_dtype, 1, image, stream);
}

// Coefficient image of the shielded-Coulomb matrix W[p, q] on `grid` (real, Gp x Gp), never
// materialised as a dense matrix.  Internal entry used by qs_odqd_coulomb_planes, which hands the image to the
// diagonal two-body transform as its W.
int qs_build_coulomb_image(const double* grid, double alpha, double a, int64_t Gp, void* image, void* stream) {
    QS_REQUIRE(grid && image && Gp > 0, "qs_build_coulomb_image: bad arguments");
    const Tiling tl = make_tiling(Gp, Gp, QS_F64, QS_F64);
    ImageParams q;
    memset(&q, 0, sizeof(q));
    q.m = grid;
    q.coulomb = 1;
    q.alpha = alpha;
    q.a2 = a * a;
    return build_image(q, tl, image, stream);
}

namespace {

// Is any (row, column) of the CTA tile (rows [x0, x1], output columns [w0, w1]) wanted by the mask?
//   kind 1: wanted iff column < row_lo (strict) or <= (not strict),  row_lo(x) = (x / dl) % ml
//   kind 2: wanted iff row_hi < row_lo (or <=),  row_hi(x) = (x / dh) % mh,  dl divides dh
// Conservative (never drops a wanted tile); exact when a tile does not straddle a block of the coarser index.
bool tile_wanted(const QsTileMask& m, int64_t x0, int64_t x1, int64_t w0, int64_t w1) {
    const int64_t l0 = x0 / m.dl, l1 = x1 / m.dl;
    if (m.kind == 3) {
        // every (row_lo, column) of the tile against the cyclic pair rule; a tile holds one or two values of row_lo
        // (128 rows) and at most 64 columns, so brute force is cheap -- and exact
        const int64_t blocks = l1 - l0 + 1 < m.ml ? l1 - l0 + 1 : m.ml;
        for (int64_t b = 0; b < blocks; ++b) {
            const int64_t s = (l0 + b) % m.ml;
            for (int64_t r = w0; r <= w1 && r < m.ml; ++r)
                if (qs_cyclic_wanted(r, s, m.ml) || (!m.strict && qs_cyclic_wanted(r, s ^ 1, m.ml))) return true;
        }
        return false;
    }
    int64_t lo_max;  // the largest row_lo inside the tile
    if (l1 - l0 >= m.ml - 1 || (l1 % m.ml) < (l0 % m.ml)) lo_max = m.ml - 1;  // covers a whole period or wraps
    else lo_max = l1 % m.ml;
    if (m.kind == 1) return m.strict ? w0 < lo_max : w0 <= lo_max;
    const int64_t h0 = x0 / m.dh, h1 = x1 / m.dh;
    if (h1 > h0 + 1) return true;  // spans several values of the coarser index: keep
    if (h1 == h0 + 1) {
        // two blocks: the first runs to the end of its row_lo range, the second starts at row_lo = 0
        const int64_t hi0 = h0 % m.mh, hi1 = h1 % m.mh, lo1 = l1 % m.ml;
        const bool first = m.strict ? hi0 < m.ml - 1 : hi0 <= m.ml - 1;
        const bool second = m.strict ? hi1 < lo1 : hi1 <= lo1;
        return first || second;
    }
    const int64_t hi = h0 % m.mh;
    return m.strict ? hi < lo_max : hi <= lo_max;
}

// Per tile group, the ascending list of the linear tile ids (row_tile * tiles_w + col_tile) a masked launch visits:
// by the row table (a tile is wanted iff one of its rows is kept) or by the analytic mask.  Returns the kept share.
double plan_tile_lists(const Tiling& tl, int64_t X, int64_t x_inner, bool out_complex, const QsTileMask* mask,
                       const long long* host_xq_table, std::vector<uint32_t> (&lists)[2]) {
    const int64_t tiles_x = qs_ceil_div(X, kBlockX);
    const int cols_per_elem = (out_complex && !tl.split) ? 2 : 1;  // real columns per output element
    int64_t all = 0, kept = 0;
    for (int gi = 0; gi < tl.ngroups; ++gi) {
        const TileGroup& gr = tl.group[gi];
        for (int64_t rt = 0; rt < tiles_x; ++rt) {
            const int64_t x0 = rt * kBlockX, x1 = (x0 + kBlockX < X ? x0 + kBlockX : X) - 1;
            for (int ct = 0; ct < gr.tiles_w; ++ct) {
                const int64_t c0 = gr.w_first + (int64_t)ct * 8 * gr.NT;
                int64_t c1 = c0 + 8 * gr.NT - 1;
                if (c1 > tl.Wp - 1) c1 = tl.Wp - 1;
                ++all;
                bool wanted;
                if (host_xq_table) {
                    wanted = false;
                    for (int64_t xq = x0 / x_inner; xq <= x1 / x_inner && !wanted; ++xq) wanted = host_xq_table[xq] >= 0;
                } else {
                    wanted = tile_wanted(*mask, x0, x1, c0 / cols_per_elem, c1 / cols_per_elem);
                }
                if (wanted) {
                    lists[gi].push_back((uint32_t)(rt * gr.tiles_w + ct));
                    ++kept;
                }
            }
        }
    }
    return all ? (double)kept / (double)all : 1.0;
}

// The tile lists of a masked launch depend on the extents and the mask only, never on the data: they are planned on
// the host once per (device, shape, mask), uploaded once and reused from device memory by every later call
// (qs_table_cache_*), so a steady-state masked launch issues no host-to-device copy.
struct PlannedLists {
    const uint32_t* dev[2];
    uint32_t count[2];
    double fraction;
};

struct ListKey {
    int tag, a_dtype, m_dtype, out_complex, kind, strict, device, pad;
    int64_t X, x_inner, K, W, dh, mh, dl, ml, table_len;
    uint64_t table_hash;
};

std::mutex g_lists_mutex;
std::unordered_map<std::string, PlannedLists>* g_lists = nullptr;

// Returns false when the device-side cache is full; the caller then stages `lists` through its workspace.
bool planned_lists(const Tiling& tl, int a_dtype, int m_dtype, int64_t X, int64_t x_inner, int64_t K, int64_t W,
                   bool out_complex, const QsTileMask* mask, const long long* host_xq_table, PlannedLists* out,
                   std::vector<uint32_t> (&lists)[2]) {
    ListKey key;
    memset(&key, 0, sizeof(key));
    key.tag = 0x715;
    key.a_dtype = a_dtype;
    key.m_dtype = m_dtype;
    key.out_complex = out_complex;
    key.device = qs_current_device();
    key.X = X;
    key.x_inner = x_inner;
    key.K = K;
    key.W = W;
    if (host_xq_table) {
        key.table_len = qs_ceil_div(X, x_inner);
        key.table_hash = qs_hash_bytes(host_xq_table, (size_t)key.table_len * sizeof(long long), 17);
    } else {
        key.kind = mask->kind;
        key.strict = mask->strict;
        key.dh = mask->dh;
        key.mh = mask->mh;
        key.dl = mask->dl;
        key.ml = mask->ml;
    }
    const std::string k(reinterpret_cast<const char*>(&key), sizeof(key));
    {
        std::lock_guard<std::mutex> lock(g_lists_mutex);
        if (g_lists) {
            auto it = g_lists->find(k);
            if (it != g_lists->end()) {
                *out = it->second;
                return true;
            }
        }
    }
    PlannedLists pl;
    memset(&pl, 0, sizeof(pl));
    pl.fraction = plan_tile_lists(tl, X, x_inner, out_complex, mask, host_xq_table, lists);
    for (int gi = 0; gi < tl.ngroups; ++gi) {
        pl.count[gi] = (uint32_t)lists[gi].size();
        if (lists[gi].empty()) continue;
        ListKey gk = key;
        gk.pad = gi + 1;
        pl.dev[gi] = static_cast<const uint32_t*>(
            qs_table_cache_put(&gk, sizeof(gk), lists[gi].data(), lists[gi].size() * sizeof(uint32_t)));
        if (!pl.dev[gi]) {
            out->fraction = pl.fraction;
            return false;
        }
    }
    std::lock_guard<std::mutex> lock(g_lists_mutex);
    if (!g_lists) g_lists = new std::unordered_map<std::string, PlannedLists>();
    (*g_lists)[k] = pl;
    *out = pl;
    return true;
}

}  // namespace

// Internal (common.cuh): one quarter transform, stored as `s` describes.
int qs_quarter_launch(const void* A, int a_dtype, int64_t X, int64_t K, int64_t lda, const void* image, int m_dtype,
                      int64_t W, const QsQuarterStore& s, void* stream) {
    QS_REQUIRE(A && image && (s.out || s.out_table), "qs_quarter_transform: null pointer");
    QS_REQUIRE(s.w_deal >= 1 && s.w_deal < (W > 1 ? W : 2) && gcd64(s.w_deal, W) == 1,
               "qs_quarter_transform_scatter: the dealing multiplier %lld is not coprime to W = %lld",
               (long long)s.w_deal, (long long)W);
    QS_REQUIRE(X > 0 && K > 0 && W > 0 && lda >= K, "qs_quarter_transform: bad extents");
    QS_REQUIRE(X < (1LL << 31) - kBlockX, "qs_quarter_transform: X=%lld exceeds 2^31", (long long)X);
    QS_REQUIRE(s.x_inner > 0 && s.w_inner > 0 && s.x_inner < (1LL << 32) && s.w_inner < (1LL << 31) && s.x_mid > 0 &&
                   s.x_mid < (1LL << 32),
               "qs_quarter_transform: bad inner extents");
    const int64_t n_dest = s.n_dest;
    QS_REQUIRE(n_dest >= 0 && n_dest <= kMaxDest, "qs_quarter_transform_scatter: at most %d destinations", kMaxDest);
    const bool columns = s.col_off != nullptr;
    QS_REQUIRE(n_dest == 0 || s.w_cyclic || columns || qs_ceil_div(W, s.w_inner) <= n_dest,
               "qs_quarter_transform_scatter: W=%lld needs more than %lld destinations of %lld", (long long)W,
               (long long)n_dest, (long long)s.w_inner);
    QS_REQUIRE(!s.w_cyclic || n_dest > 0, "qs_quarter_transform_scatter: cyclic columns need a destination table");
    QS_REQUIRE(!columns || (s.col_dest && n_dest > 0 && !s.w_cyclic && !s.xq_table && !s.xr_table && !s.mask &&
                            !s.host_xq_table),
               "qs_quarter_transform_scatter_columns: column tables need a destination table and no row tables");
    const Tiling tl = make_tiling(K, W, a_dtype, m_dtype);
    const bool out_complex = a_dtype == QS_C128 || m_dtype == QS_C128;
    const int64_t pitch_bytes = lda * 8 * qs_elem_doubles(a_dtype);
    QS_REQUIRE(pitch_bytes % 16 == 0,
               "qs_quarter_transform: row pitch of A must be a multiple of 16 bytes (pad odd real K)");
    // A and the image are TMA / bulk-copy sources (16 bytes); the epilogue stores whole elements
    const uintptr_t out_mask = out_complex ? 15 : 7;
    QS_REQUIRE((reinterpret_cast<uintptr_t>(A) & 15) == 0 && (reinterpret_cast<uintptr_t>(image) & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(s.out) & out_mask) == 0,
               "qs_quarter_transform: A and image must be 16-byte aligned, out element-aligned");
    for (int64_t d = 0; d < n_dest; ++d)
        QS_REQUIRE(s.out_table[d] && (reinterpret_cast<uintptr_t>(s.out_table[d]) & out_mask) == 0,
                   "qs_quarter_transform_scatter: destination %lld is null or misaligned", (long long)d);

    EncodeTiledFn encode = get_encode_fn();
    QS_REQUIRE(encode, "cuTensorMapEncodeTiled unavailable (no CUDA driver?)");
    CUtensorMap map;
    const cuuint64_t gdim[2] = {(cuuint64_t)tl.Kp, (cuuint64_t)X};
    const cuuint64_t gstride[1] = {(cuuint64_t)pitch_bytes};
    const cuuint32_t box[2] = {kChunkK, kBlockX};
    const cuuint32_t estr[2] = {1, 1};
    CUresult cr = encode(&map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<void*>(A), gdim, gstride, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) {
        qs_set_error("cuTensorMapEncodeTiled failed with CUresult %d (X=%lld K'=%d pitch=%lld)", (int)cr, (long long)X,
                     tl.Kp, (long long)pitch_bytes);
        return QS_ERR_CUDA;
    }

    int xq_even = s.xq_even;
    if (s.host_xq_table) {  // the caller's own table: every kept entry must be even for 16-byte aligned real runs
        xq_even = 1;
        for (int64_t q = 0, nq = qs_ceil_div(X, s.x_inner); q < nq && xq_even; ++q)
            xq_even = s.host_xq_table[q] < 0 || s.host_xq_table[q] % 2 == 0;
    }
    // Real rows leave in 16-byte pieces (row pairs of the register epilogue, runs of the staged one) when all extents,
    // strides and bases are even and every destination is 16-byte aligned.  With tabulated offsets that is the
    // table's business: block offsets (xq_table) must be even.
    // Column tables: the caller's promise that every column offset is even stands in for an even sw0.
    bool even16 = s.x_inner % 2 == 0 && X % 2 == 0 && s.sx1 % 2 == 0 && s.sx2 % 2 == 0 &&
                  (columns ? s.col_off_even != 0 : s.sw0 % 2 == 0) &&
                  (n_dest > 0 || s.sw1 % 2 == 0) && (reinterpret_cast<uintptr_t>(s.out) & 15) == 0 &&
                  (!s.xq_table || xq_even);
    for (int64_t d = 0; d < n_dest; ++d) even16 = even16 && (reinterpret_cast<uintptr_t>(s.out_table[d]) & 15) == 0;
    // Row-pair stores of the real register epilogue also need rows 2k, 2k + 1 adjacent: sx0 = 1, or a per-row table
    // (xr_table) that places them so (`xr_paired`, the caller's promise).
    const bool rows_adjacent = s.xr_table ? s.xr_paired != 0 : s.sx0 == 1;
    const int vec2 = !out_complex && rows_adjacent && even16;
    // Staged asynchronous epilogue: consecutive rows of a block are adjacent in the output (sx0 = 1) and every run of
    // rows handed to cp.async.bulk starts 16-byte aligned: always for complex output (16-byte elements), for real
    // output under the conditions above.  Rows placed one by one (xr_table) and columns placed by the column tables
    // keep the register stores.
    const bool bulk = (bulk_mode() == 2 || (bulk_mode() == 1 && n_dest > 1)) && s.sx0 == 1 && !s.xr_table &&
                      !columns && !tl.split && (out_complex || even16);
    // The rotated epilogue: one local destination, undealt columns, no row tables, the two-level row split with
    // adjacent rows, and 16-byte row pairs for real output.
    const bool rotated = n_dest == 0 && s.w_deal == 1 && !s.xq_table && !s.xr_table && s.x_mid == 0xFFFFFFFFLL &&
                         s.w_inner == 1 && s.sx0 == 1 && (out_complex || vec2);
    const int epi = columns ? kEpiColumns : bulk ? kEpiBulk : rotated ? kEpiRotated : kEpiStrided;

    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // symmetry mask: per tile group, the ascending list of wanted linear tile ids, staged into list_ws
    std::vector<uint32_t> lists[2];
    double wanted_fraction = 1.0;
    QS_REQUIRE(!(s.xq_table || s.xr_table) || s.x_mid == 0xFFFFFFFFLL,
               "qs_quarter_transform: row-offset tables need the two-level row split");
    const bool masked = (s.mask && s.mask->kind) || s.host_xq_table;
    PlannedLists cached;
    memset(&cached, 0, sizeof(cached));
    bool lists_cached = false;
    if (masked) {
        QS_REQUIRE(s.list_ws && s.w_deal == 1, "qs_quarter_transform: a masked launch needs list space and undealt columns");
        lists_cached = planned_lists(tl, a_dtype, m_dtype, X, s.x_inner, K, W, out_complex, s.mask, s.host_xq_table,
                                     &cached, lists);
        wanted_fraction = cached.fraction;
    }
    int span = -1;
    // issued flops; the split variant's Wp counts complex columns, each fed by Kp real multiply-adds per row
    qs_timing_begin(QS_FAMILY_QUARTER_GEMM, 2.0 * (double)X * tl.Kp * tl.Wp * wanted_fraction, stream, &span);
    uint32_t* list_dev = static_cast<uint32_t*>(s.list_ws);
    for (int gi = 0; gi < tl.ngroups; ++gi) {
        const TileGroup& gr = tl.group[gi];
        QuarterParams p;
        memset(&p, 0, sizeof(p));
        if (masked && lists_cached) {
            if (cached.count[gi] == 0) continue;
            p.tile_list = cached.dev[gi];
            p.n_listed = cached.count[gi];
        } else if (masked) {
            // table cache full: stage this call's list through the workspace (pageable source: the runtime
            // stages the bytes before returning)
            if (lists[gi].empty()) continue;
            QS_CUDA(cudaMemcpyAsync(list_dev, lists[gi].data(), lists[gi].size() * sizeof(uint32_t),
                                    cudaMemcpyHostToDevice, st));
            p.tile_list = list_dev;
            p.n_listed = (uint32_t)lists[gi].size();
            list_dev += (lists[gi].size() + 3) / 4 * 4;
        }
        p.image = static_cast<const double*>(image) + gr.image_offset;
        p.out = static_cast<double*>(s.out);
        p.ndest = (int)n_dest;
        for (int64_t d = 0; d < n_dest; ++d) p.outs[d] = static_cast<double*>(s.out_table[d]);
        p.X = (uint32_t)X;
        p.Wp = (uint32_t)tl.Wp;
        p.w_first = (uint32_t)gr.w_first;
        p.tiles_x = (uint32_t)qs_ceil_div(X, kBlockX);
        p.nchunks = tl.nchunks;
        p.last_halves = tl.last_halves;
        p.tiles_w = gr.tiles_w;
        p.x_inner = (uint32_t)s.x_inner;
        p.x_inner_div = make_divisor((uint64_t)s.x_inner);
        p.tiles_w_div = make_divisor((uint64_t)gr.tiles_w);
        p.x_mid = (uint32_t)s.x_mid;
        p.w_inner = (uint32_t)s.w_inner;
        p.sx0 = s.sx0;
        p.sx1 = s.sx1;
        p.sx2 = s.sx2;
        p.sw0 = s.sw0;
        p.sw1 = n_dest ? 0 : s.sw1;
        p.vec2 = vec2;
        p.deal_mul = (uint32_t)s.w_deal;
        p.deal_mod = (uint32_t)W;
        p.w_cyclic = s.w_cyclic;
        p.xq_table = s.xq_table;
        p.xr_table = s.xr_table;
        p.col_dest = s.col_dest;
        p.col_off = s.col_off;
        QS_REQUIRE((int64_t)p.tiles_x * p.tiles_w < (1LL << 31), "qs_quarter_transform: too many tiles");
        const int rc = tl.split      ? launch_split(columns, gr.NT, map, p, st)
                       : out_complex ? launch_epilogue<true>(epi, gr.NT, map, p, st)
                                     : launch_epilogue<false>(epi, gr.NT, map, p, st);
        if (rc) return rc;
    }
    qs_timing_end(span, stream);
    return QS_OK;
}

// Internal (common.cuh): device memory a masked quarter transform needs for its tile lists (QsQuarterStore::list_ws).
int64_t qs_tile_list_bytes(int64_t X, int64_t K, int64_t W, int a_dtype, int m_dtype) {
    const Tiling tl = make_tiling(K, W, a_dtype, m_dtype);
    int64_t tiles = 0;
    for (int gi = 0; gi < tl.ngroups; ++gi) tiles += qs_ceil_div(X, kBlockX) * tl.group[gi].tiles_w + 4;
    return tiles * (int64_t)sizeof(uint32_t);
}

// Host-only: the tiles a masked quarter transform would launch, as rows of (first row, last row, first output
// column, last output column) -- for inspection and for CPU tests of the masks (no device is touched).
// mask_kind 0 with a host_xq_table plans by the table; otherwise the analytic mask (kind, strict, dh, mh, dl, ml).
extern "C" int qs_quarter_plan_tiles(int64_t X, int64_t K, int64_t W, int a_dtype, int m_dtype, int64_t x_inner,
                                     int mask_kind, int strict, int64_t dh, int64_t mh, int64_t dl, int64_t ml,
                                     const int64_t* host_xq_table, int64_t* host_tiles, int64_t capacity,
                                     int64_t* count) {
    QS_REQUIRE(X > 0 && K > 0 && W > 0 && x_inner > 0 && count, "qs_quarter_plan_tiles: bad arguments");
    QS_REQUIRE(mask_kind || host_xq_table, "qs_quarter_plan_tiles: neither a mask nor a row table");
    const Tiling tl = make_tiling(K, W, a_dtype, m_dtype);
    const bool out_complex = a_dtype == QS_C128 || m_dtype == QS_C128;
    const QsTileMask mask = {mask_kind, strict, dh, mh, dl, ml};
    std::vector<uint32_t> lists[2];
    plan_tile_lists(tl, X, x_inner, out_complex, &mask, reinterpret_cast<const long long*>(host_xq_table), lists);
    const int cols_per_elem = (out_complex && !tl.split) ? 2 : 1;
    int64_t n = 0;
    for (int gi = 0; gi < tl.ngroups; ++gi) {
        const TileGroup& gr = tl.group[gi];
        for (uint32_t id : lists[gi]) {
            if (host_tiles && n < capacity) {
                const int64_t rt = id / gr.tiles_w, ct = id % gr.tiles_w;
                const int64_t c0 = gr.w_first + ct * 8 * gr.NT;
                int64_t c1 = c0 + 8 * gr.NT - 1;
                if (c1 > tl.Wp - 1) c1 = tl.Wp - 1;
                host_tiles[4 * n + 0] = rt * kBlockX;
                host_tiles[4 * n + 1] = (rt * kBlockX + kBlockX < X ? rt * kBlockX + kBlockX : X) - 1;
                host_tiles[4 * n + 2] = c0 / cols_per_elem;
                host_tiles[4 * n + 3] = c1 / cols_per_elem;
            }
            ++n;
        }
    }
    *count = n;
    return QS_OK;
}

extern "C" int qs_quarter_tile_list_bytes(int64_t X, int64_t K, int64_t W, int a_dtype, int m_dtype, int64_t* bytes) {
    QS_REQUIRE(X > 0 && K > 0 && W > 0 && bytes, "qs_quarter_tile_list_bytes: bad arguments");
    *bytes = qs_tile_list_bytes(X, K, W, a_dtype, m_dtype);
    return QS_OK;
}

extern "C" int qs_quarter_transform_rows(const void* A, int a_dtype, int64_t X, int64_t K, int64_t lda,
                                         const void* image, int m_dtype, int64_t W, void* out, int64_t x_inner,
                                         int64_t sx0, const int64_t* host_xq_table, const int64_t* xq_table,
                                         int64_t w_inner, int64_t sw0, int64_t sw1, void* list_ws,
                                         int64_t list_ws_bytes, void* stream) {
    QS_REQUIRE(host_xq_table && xq_table && list_ws, "qs_quarter_transform_rows: null pointer");
    QS_REQUIRE(X > 0 && K > 0 && W > 0 && list_ws_bytes >= qs_tile_list_bytes(X, K, W, a_dtype, m_dtype),
               "qs_quarter_transform_rows: tile-list space too small");
    QsQuarterStore s;
    s.out = out;
    s.x_inner = x_inner;
    s.sx0 = sx0;
    s.xq_table = reinterpret_cast<const long long*>(xq_table);
    s.host_xq_table = reinterpret_cast<const long long*>(host_xq_table);
    s.w_inner = w_inner;
    s.sw0 = sw0;
    s.sw1 = sw1;
    s.list_ws = list_ws;
    return qs_quarter_launch(A, a_dtype, X, K, lda, image, m_dtype, W, s, stream);
}

extern "C" int qs_quarter_transform_scatter_rows(const void* A, int a_dtype, int64_t X, int64_t K, int64_t lda,
                                                 const void* image, int m_dtype, int64_t W,
                                                 void* const* host_out_table, int64_t n_dest, int64_t x_inner,
                                                 int64_t sx1, const int64_t* xr_table, int64_t w_inner, int64_t sw0,
                                                 int64_t w_deal, int rows_paired, void* stream) {
    QS_REQUIRE(host_out_table && n_dest > 0 && xr_table, "qs_quarter_transform_scatter_rows: null pointer");
    QsQuarterStore s;
    s.out_table = host_out_table;
    s.n_dest = n_dest;
    s.x_inner = x_inner;
    s.sx1 = sx1;
    s.xr_table = reinterpret_cast<const long long*>(xr_table);
    s.xr_paired = rows_paired;
    s.w_inner = w_inner;
    s.sw0 = sw0;
    s.w_deal = w_deal;
    return qs_quarter_launch(A, a_dtype, X, K, lda, image, m_dtype, W, s, stream);
}

// The scattering store restricted to the CTA tiles that hold a pair (column r, row index s) the cyclic pair rule of
// the anti-symmetric schedule wants (mask kind 3: s = (x / rows_per_s) % W; `padded` != 0 also keeps the other member
// s ^ 1 of an aligned couple, matching the padded pair lists of the real case).  Columns are undealt (cyclic
// destinations).  list_ws: qs_quarter_tile_list_bytes() bytes of device memory (used only if the table cache is full).
extern "C" int qs_quarter_transform_scatter_pairs(const void* A, int a_dtype, int64_t X, int64_t K, int64_t lda,
                                                  const void* image, int m_dtype, int64_t W,
                                                  void* const* host_out_table, int64_t n_dest, int64_t x_inner,
                                                  int64_t x_mid, int64_t sx0, int64_t sx1, int64_t sx2, int64_t sw0,
                                                  int64_t rows_per_s, int padded, void* list_ws,
                                                  int64_t list_ws_bytes, void* stream) {
    QS_REQUIRE(host_out_table && n_dest > 0 && list_ws, "qs_quarter_transform_scatter_pairs: null pointer");
    QS_REQUIRE(X > 0 && K > 0 && W > 0 && rows_per_s > 0 &&
                   list_ws_bytes >= qs_tile_list_bytes(X, K, W, a_dtype, m_dtype),
               "qs_quarter_transform_scatter_pairs: bad extents or tile-list space too small");
    const QsTileMask mask = {3, padded ? 0 : 1, 1, 1, rows_per_s, W};
    QsQuarterStore s;
    s.out_table = host_out_table;
    s.n_dest = n_dest;
    s.w_cyclic = 1;
    s.x_inner = x_inner;
    s.x_mid = x_mid;
    s.sx0 = sx0;
    s.sx1 = sx1;
    s.sx2 = sx2;
    s.sw0 = sw0;
    s.mask = &mask;
    s.list_ws = list_ws;
    return qs_quarter_launch(A, a_dtype, X, K, lda, image, m_dtype, W, s, stream);
}

extern "C" int qs_quarter_transform(const void* A, int a_dtype, int64_t X, int64_t K, int64_t lda, const void* image,
                                    int m_dtype, int64_t W, void* out, int64_t x_inner, int64_t sx0, int64_t sx1,
                                    int64_t w_inner, int64_t sw0, int64_t sw1, void* stream) {
    QsQuarterStore s;
    s.out = out;
    s.x_inner = x_inner;
    s.sx0 = sx0;
    s.sx1 = sx1;
    s.w_inner = w_inner;
    s.sw0 = sw0;
    s.sw1 = sw1;
    return qs_quarter_launch(A, a_dtype, X, K, lda, image, m_dtype, W, s, stream);
}

extern "C" int qs_quarter_transform_scatter(const void* A, int a_dtype, int64_t X, int64_t K, int64_t lda,
                                            const void* image, int m_dtype, int64_t W, void* const* host_out_table,
                                            int64_t n_dest, int64_t x_inner, int64_t x_mid, int64_t sx0, int64_t sx1,
                                            int64_t sx2, int64_t w_inner, int64_t sw0, int64_t w_deal,
                                            int w_cyclic, void* stream) {
    QS_REQUIRE(host_out_table && n_dest > 0, "qs_quarter_transform_scatter: empty destination table");
    QsQuarterStore s;
    s.out_table = host_out_table;
    s.n_dest = n_dest;
    s.w_cyclic = w_cyclic;
    s.w_deal = w_deal;
    s.x_inner = x_inner;
    s.x_mid = x_mid;
    s.sx0 = sx0;
    s.sx1 = sx1;
    s.sx2 = sx2;
    s.w_inner = w_inner;
    s.sw0 = sw0;
    return qs_quarter_launch(A, a_dtype, X, K, lda, image, m_dtype, W, s, stream);
}

// The scattering store with column tables: physical column w goes to host_out_table[col_dest[w]] at element offset
// col_off[w] (device tables of W entries).  Rows as in qs_quarter_transform_scatter.
extern "C" int qs_quarter_transform_scatter_columns(const void* A, int a_dtype, int64_t X, int64_t K, int64_t lda,
                                                    const void* image, int m_dtype, int64_t W,
                                                    void* const* host_out_table, int64_t n_dest,
                                                    const int32_t* col_dest, const int64_t* col_off,
                                                    int offsets_even, int64_t x_inner, int64_t x_mid, int64_t sx0,
                                                    int64_t sx1, int64_t sx2, int64_t w_deal, void* stream) {
    QS_REQUIRE(host_out_table && n_dest > 0 && col_dest && col_off,
               "qs_quarter_transform_scatter_columns: null pointer or empty destination table");
    QsQuarterStore s;
    s.out_table = host_out_table;
    s.n_dest = n_dest;
    s.col_dest = col_dest;
    s.col_off = reinterpret_cast<const long long*>(col_off);
    s.col_off_even = offsets_even;
    s.w_deal = w_deal;
    s.x_inner = x_inner;
    s.x_mid = x_mid;
    s.sx0 = sx0;
    s.sx1 = sx1;
    s.sx2 = sx2;
    return qs_quarter_launch(A, a_dtype, X, K, lda, image, m_dtype, W, s, stream);
}
