// First Linear of the SOCIAL grid embedding on tcgen05, CTA-pair kernel (round 2).
//
//   hidden1[p, :] = relu(b1 + sum_{winning (cell, j) of p} W1[:, cell-slab] . lat_j)
//   (reference: GridBasedPooling.social + the first Linear of two_layer,
//    trajnetbaselines/lstm/gridbased_pooling.py:145-170,227-305,316-323)
//
// Orientation (the transpose of round 1's sparse_layer1_tc_kernel): D[p, col] with the pedestrians on
// the M side -- 128 TMEM lanes per CTA, one pedestrian per lane -- and the output columns on the N
// side.  Per grid cell c one K = 16 product
//     D[p, col] += L_c[p, 0:16] . W_c[col, 0:16]
// where L_c[p, :] is the latent vector of p's winning neighbour in cell c, or zero.
//   * Two CTAs (one TPC) run tcgen05.mma.cta_group::2 with M = 256: each CTA owns 128 pedestrians (its own
//     A operand) and HALF of the weight columns of the tile (B is shared by the pair), so every weight byte
//     fetched from L2 serves 256 pedestrians and each SM's shared memory holds only half of B.
//   * The A operand lives in tensor memory, in a ring of stages behind the accumulators.  Builder warps, one
//     thread per pedestrian row (= TMEM lane), write every row of every cell (no re-zeroing, no buckets): the
//     thread reads "which neighbour of mine sits in cell c" from the per-row cell map pool_prepare leaves in
//     global memory (16 cells per 16-byte load, prefetched), copies the neighbour's split latent vector from a
//     per-tile table in shared memory and stores it with one tcgen05.st per cell.  Shared memory carries only
//     the weights, which buys a deep weight ring.
//   * The weight slabs W_c are stored pre-swizzled (SWIZZLE_32B image) in global memory, so one
//     plain bulk copy (cp.async.bulk) of any multiple of 16 rows lands the tile the UMMA
//     descriptor expects.
//   * Work decomposition: the (pedestrian tile, 32-column block) space is linearised and cut into
//     equal contiguous ranges, one per CTA pair; a range is processed in rounds of at most two
//     contexts (tile, column range) with at most 288 accumulator columns, so a range that straddles a
//     tile boundary still keeps all SMs equally loaded (5120 pedestrians x 1024 columns on 74 pairs:
//     8.65 blocks each, against 128 of 148 SMs busy in round 1).
//   * Pipeline item = 4 grid cells (K = 64) of the round's tile, or of both tiles of a two-tile round (2 cells
//     when the round has more than 256 accumulator columns): one barrier round trip builders -> MMA issuers ->
//     tcgen05.commit per item.
//   * Precision: 3-pass bf16 (hi, lo) split, fp32 accumulation in TMEM, like the other kernels;
//     results are bit-identical to sparse_layer1_tc_kernel (same products, same order per column).
//   Measurements and the designs this one replaced: DESIGN.md section 4.1.
//
// Warp roles (512 threads): 0 = weight producer, 1 / 2 = MMA issuers (leader CTA only; 1 also owns the TMEM
// allocation), 3 = weight relay, 4..7 / 8..11 = builders (one-tile round: even / odd items; two-tile round:
// one tile each); all 16 warps run the epilogue (4 per TMEM lane quarter).
#include <cuda.h>
#include <cuda_bf16.h>
#include <algorithm>
#include <mutex>
#include <vector>

#include "common.cuh"

namespace tb2 {

constexpr int kSpThreads = 512;
constexpr int kSpSA = 3;                 // ring of A stages (built on the fly, short turn-around)
constexpr int kSpSBMax = 8;              // ring of weight stages (bulk copies from L2: ~1500 cycles from request to landing):
                                         // 5 x 4 cells (one tile) / 8 x 2 cells (two tiles)
constexpr int kSpMaxBlocks = 9;          // 32-column blocks per round (288 accumulator columns)
constexpr int kSpDCols = kSpMaxBlocks * 32;
constexpr int kSpMaxCells = 256;
constexpr int kSpLatRows = 256;          // local latent table (rows of the scenes a 128-row tile touches) + 1
constexpr uint32_t kSpBCell = (uint32_t)(kSpDCols / 2) * 64u;          // bytes of weights per cell and CTA of a pair (288 columns)
// dynamic shared memory behind the 1024-byte alignment: [weight ring | latent table 1 | latent table 0] (the second
// latent table is the one of a two-tile round)
constexpr size_t kSpDynBytes = 220 * 1024;
static_assert((size_t)5 * 4 * kSpBCell <= kSpDynBytes - (size_t)kSpLatRows * 64, "one-tile weight ring");
static_assert((size_t)8 * 2 * kSpBCell <= kSpDynBytes - (size_t)2 * kSpLatRows * 64, "two-tile weight ring");
static_assert(1024 + kSpDynBytes + 64 <= 227 * 1024 - 1024, "shared memory budget");

// TMEM: accumulators in columns [0, 288), the A ring behind them: 3 stages x 64 columns (one-tile item: 4 cells x
// (hi 8 | lo 8) columns; two-tile item of 2 cells: 2 cells x 2 tiles x 16 columns)
constexpr uint32_t kSpACol0 = 320;
constexpr uint32_t kSpAStageCols = 64;
static_assert(kSpDCols <= (int)kSpACol0 && kSpACol0 + kSpSA * kSpAStageCols <= 512, "TMEM budget");

__device__ __forceinline__ uint32_t sp_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void sp_mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void sp_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// arrive on a barrier of the leader CTA (cluster address).  Default semantics (.release.cta) like CUTLASS'
// ClusterBarrier::arrive: a .release.cluster arrive per builder warp and item cost ~2000 cycles of serial
// latency per item (measured), and the data this signal publishes is read by THIS SM's tensor core, behind
// the tcgen05.fence each builder thread executed.
__device__ __forceinline__ void sp_mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void sp_mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "SP_WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra SP_WAIT_DONE;\n"
        "bra SP_WAIT_LOOP;\n"
        "SP_WAIT_DONE:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}
// the leader's "A and B of this item are ready" barrier (also arrived on from the peer CTA)
__device__ __forceinline__ void sp_mbar_wait_cluster(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "SPC_WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra SPC_WAIT_DONE;\n"
        "bra SPC_WAIT_LOOP;\n"
        "SPC_WAIT_DONE:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void sp_bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// completion of all earlier tcgen05.mma of this thread -> arrive on `bar` in both CTAs of the pair
__device__ __forceinline__ void sp_commit(uint32_t bar) {
    const uint16_t mask = 3;
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"(mask) : "memory");
}


// One round of a unit: `n0` 32-column blocks of pedestrian tile `tile` starting at block `blk0`, then (n1 > 0) the
// first `n1` blocks of tile + 1.  Planned on the host (plan_rounds) so that no piece is narrower than 3 blocks.
struct SpRound { int tile, blk0, n0, n1; };

__device__ __forceinline__ void sp_tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}

struct SpParams {
    const int* scene_off;
    const int* row_scene;
    const unsigned char* cell_row;   // [M, cells]: scene-local index of the winning neighbour (0xFF none, 0xFE NaN-padded slot)
    const float* lat;                // [M, 16] fp32
    const float* benc;               // [16]
    const float* base;               // [OUT]
    const unsigned char* w;          // bf16 [cells][OUT / 8][hi: 8 rows x 16 | lo: 8 rows x 16], 16-byte chunks swizzled by ((col >> 2) & 1)
    float* out;                      // fp32 [M, OUT] or null
    __nv_bfloat16* out_hi;           // bf16 split [M, OUT] or null
    __nv_bfloat16* out_lo;
    const SpRound* rounds;           // [units * rounds_per_unit] (plan_rounds)
    int M, OUT, cells, rounds_per_unit;
    float constant;
};

// MMA with A = 128 lanes x 8 TMEM columns (16 bf16 of K per lane) of each CTA, B from shared memory (64-bit
// descriptor kept in registers: the issuing thread is a single thread, every instruction between two MMAs counts)
__device__ __forceinline__ void sp_umma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
// one pedestrian row (lane) of one cell: hi (8 columns) | lo (8 columns)
__device__ __forceinline__ void sp_tmem_st16(uint32_t taddr, const uint4& h0, const uint4& h1, const uint4& l0, const uint4& l1) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
                 ::"r"(taddr), "r"(h0.x), "r"(h0.y), "r"(h0.z), "r"(h0.w), "r"(h1.x), "r"(h1.y), "r"(h1.z), "r"(h1.w),
                   "r"(l0.x), "r"(l0.y), "r"(l0.z), "r"(l0.w), "r"(l1.x), "r"(l1.y), "r"(l1.z), "r"(l1.w) : "memory");
}

// Builder body for one pipeline item of KC cells: the row's (hi | lo) vectors of the item's cells go to the lane's
// 16 TMEM columns per cell; `bytes` holds the KC cell-map bytes of this row (LSB first).
template <int KC>
__device__ __forceinline__ void sp_build_item(uint32_t a_item, uint32_t cell_cols, uint32_t bytes, int off_r, int nlat,
                                              const uint4* lh, const uint4* ll) {
#pragma unroll
    for (int kc = 0; kc < KC; ++kc) {
        const uint32_t j = (bytes >> (8 * kc)) & 0xffu;
        uint4 h0 = make_uint4(0u, 0u, 0u, 0u), h1 = h0, l0 = h0, l1 = h0;
        if (j != 0xffu) {
            const int li = j == 0xfeu ? nlat : (int)j + off_r;
            h0 = lh[li * 2]; h1 = lh[li * 2 + 1];
            l0 = ll[li * 2]; l1 = ll[li * 2 + 1];
        }
        sp_tmem_st16(a_item + (uint32_t)kc * cell_cols, h0, h1, l0, l1);
    }
}

// Builder role of one warp for one round: thread = pedestrian row; `cr` = the row's cell map (16 cells per uint4) or
// null for rows past the end.  One-tile round: the two builder groups (warps 4..7 / 8..11) take the even / odd items
// (KC = 4).  Two-tile round (kTwo): group bg builds the A operand of pedestrian tile bg inside EVERY item.
template <int KC, bool kTwo>
__device__ __forceinline__ void sp_builder(const uint4* cr, int groups, uint32_t a_tmem, int bg, int off_r, int nlat,
                                           const uint4* lh, const uint4* ll, uint64_t* empty_a,
                                           const uint32_t (&full_remote)[kSpSA], int lane,
                                           uint32_t SA, uint32_t stage_cols) {
    static_assert(kTwo || KC == 4, "one-tile rounds use 4-cell items");
    const uint4 none = make_uint4(~0u, ~0u, ~0u, ~0u);
    constexpr int ipg = 16 / KC;                       // items per 16-cell load of the row's cell map
    constexpr int step = kTwo ? 1 : 2;
    uint4 cur = cr ? __ldg(cr) : none;
    for (int g16 = 0; g16 < groups; ++g16) {
        const uint4 next = (cr && g16 + 1 < groups) ? __ldg(cr + g16 + 1) : none;     // prefetched one group ahead
#pragma unroll
        for (int jj = 0; jj < ipg / step; ++jj) {
            uint32_t g, bytes;                          // item index inside the round, its KC cell-map bytes
            if (kTwo) {
                g = (uint32_t)(g16 * ipg + jj);
                const int c = jj * KC;                  // first cell of the item inside the 16-cell load (compile time)
                const uint32_t w = (c >> 2) == 0 ? cur.x : (c >> 2) == 1 ? cur.y : (c >> 2) == 2 ? cur.z : cur.w;
                bytes = KC == 4 ? w : (w >> (8 * (c & 3))) & ((1u << (8 * (KC & 3))) - 1u);
            } else {
                g = (uint32_t)(g16 * ipg + 2 * jj + bg);
                bytes = jj == 0 ? (bg ? cur.y : cur.x) : (bg ? cur.w : cur.z);
            }
            const uint32_t sa = g % SA, pa = (g / SA) & 1u;
            sp_mbar_wait(sp_smem_u32(&empty_a[sa]), pa ^ 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            sp_build_item<KC>(a_tmem + sa * stage_cols, kTwo ? 32u : 16u, bytes, off_r, nlat, lh, ll);
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) sp_mbar_arrive_cluster(full_remote[sa]);
        }
        cur = next;
    }
}

__global__ void __launch_bounds__(kSpThreads, 1) sparse_layer1_pair_kernel(SpParams p) {
    constexpr int R = 256;                                // pedestrian rows per tile: 128 per CTA of the pair
    extern __shared__ __align__(1024) unsigned char smem_sp[];
    __shared__ __align__(8) uint64_t full_a[kSpSA];       // leader: A (both CTAs) built AND weights (both CTAs) landed
    __shared__ __align__(8) uint64_t empty_a[kSpSA];      // MMAs that read the A stage done
    __shared__ __align__(8) uint64_t full_b[kSpSBMax];    // local weight slabs landed
    __shared__ __align__(8) uint64_t empty_b[kSpSBMax];   // MMAs that read the weight stage done
    __shared__ __align__(8) uint64_t acc_full_bar;
    __shared__ uint32_t tmem_base_slot;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint32_t rank;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
    const int unit = (int)(blockIdx.x >> 1);

    const uint32_t ring = (sp_smem_u32(smem_sp) + 1023u) & ~1023u;          // weight ring
    unsigned char* ring_ptr = smem_sp + (ring - sp_smem_u32(smem_sp));
    uint4* latH[2];
    uint4* latL[2];
    latH[0] = reinterpret_cast<uint4*>(ring_ptr + kSpDynBytes - (size_t)kSpLatRows * 64);
    latL[0] = latH[0] + kSpLatRows * 2;
    latH[1] = reinterpret_cast<uint4*>(ring_ptr + kSpDynBytes - (size_t)2 * kSpLatRows * 64);
    latL[1] = latH[1] + kSpLatRows * 2;

    // ---- prologue: TMEM (the barriers are initialised per round) ----------------------------------
    if (warp == 1) {
        uint32_t ncols = 512;
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"(sp_smem_u32(&tmem_base_slot)), "r"(ncols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = tmem_base_slot;

    // leader's full barrier as seen from this CTA (cluster address space)
    uint32_t full_remote[kSpSA];
#pragma unroll
    for (int s = 0; s < kSpSA; ++s) {
        uint32_t local = sp_smem_u32(&full_a[s]);
        asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(full_remote[s]) : "r"(local), "r"(0));
    }

    uint32_t round_idx = 0;
    for (int ri = 0; ri < p.rounds_per_unit; ++ri) {
        const SpRound rd = p.rounds[(size_t)unit * p.rounds_per_unit + ri];
        if (rd.n0 == 0) continue;                         // padding round (uniform for the whole cluster)
        const int nsub = rd.n1 > 0 ? 2 : 1;
        // pipeline shape of the round (the barriers are re-initialised for it)
        // two-tile round of <= 256 accumulator columns: items of 4 cells of both tiles (one barrier round trip per
        // 4 cells instead of 2: the issuers of a two-tile round barely run ahead of the tensor pipe), 2 A stages of 128 TMEM
        // columns at [256, 512)
        const bool wide_items = nsub == 2 && (rd.n0 + rd.n1) * 32 <= 256;
        const uint32_t SA = wide_items ? 2u : (uint32_t)kSpSA;
        const uint32_t a_col0 = wide_items ? 256u : kSpACol0, a_stage_cols = wide_items ? 128u : kSpAStageCols;
        const int KC = nsub == 2 && !wide_items ? 2 : 4;     // grid cells per pipeline item
        const uint32_t SB = nsub == 2 && !wide_items ? 8u : 5u;   // weight stages
        const int n_items = p.cells / KC;                    // cells is a multiple of 16
        const uint32_t n_issuers = 2u;
        if (tid == 0) {
            for (int s2 = 0; s2 < kSpSA; ++s2) {
                if (round_idx > 0) {
                    asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(sp_smem_u32(&full_a[s2])) : "memory");
                    asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(sp_smem_u32(&empty_a[s2])) : "memory");
                }
                // builders per item and CTA: one group of 4 warps (one tile) or both groups (two tiles)
                sp_mbar_init(sp_smem_u32(&full_a[s2]), ((nsub == 2 ? 8 : 4) + 1) * 2);        // + the weight relay
                sp_mbar_init(sp_smem_u32(&empty_a[s2]), n_issuers);      // one tcgen05.commit per active MMA issuer
            }
            for (int s2 = 0; s2 < kSpSBMax; ++s2) {
                if (round_idx > 0) {
                    asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(sp_smem_u32(&full_b[s2])) : "memory");
                    asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(sp_smem_u32(&empty_b[s2])) : "memory");
                }
                sp_mbar_init(sp_smem_u32(&full_b[s2]), 1);
                sp_mbar_init(sp_smem_u32(&empty_b[s2]), n_issuers);
            }
            if (round_idx > 0) asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(sp_smem_u32(&acc_full_bar)) : "memory");
            sp_mbar_init(sp_smem_u32(&acc_full_bar), n_issuers);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        // piece x: columns [col0[x], col0[x] + ncols[x]) of tile[x]; accumulators of piece 1 behind those of piece 0
        const int tile[2] = {rd.tile, rd.tile + 1};
        const int col0[2] = {rd.blk0 * 32, 0};
        const uint32_t ncols[2] = {(uint32_t)rd.n0 * 32u, (uint32_t)rd.n1 * 32u};
        const uint32_t nr[2] = {ncols[0] / 2, ncols[1] / 2};                // rows of each piece's slab held by this CTA
        const uint32_t b_cell = 64u * (nr[0] + nr[1]);                       // weight bytes per cell: piece 0 rows | piece 1 rows
        const uint32_t b_stage = (uint32_t)KC * b_cell;
        // weights of item `it` of this round -> stage it % SB (the producer thread; the stage must be free)
        auto load_item = [&](int it) {
            const uint32_t sb = (uint32_t)it % SB;
            const uint32_t bar = sp_smem_u32(&full_b[sb]);
            const uint32_t st = ring + sb * b_stage;
            sp_mbar_expect_tx(bar, b_stage);
            for (int kc = 0; kc < KC; ++kc) {
                const size_t cellsrc = (size_t)(it * KC + kc) * p.OUT;
                sp_bulk_load(st + kc * b_cell, p.w + (cellsrc + col0[0] + rank * nr[0]) * 64, nr[0] * 64u, bar);
                if (nsub == 2)
                    sp_bulk_load(st + kc * b_cell + nr[0] * 64u, p.w + (cellsrc + col0[1] + rank * nr[1]) * 64, nr[1] * 64u, bar);
            }
        };
        // The weights depend on nothing the previous kernel writes: the producer thread (which has just initialised
        // the barriers) requests the first SB items before the round's setup -- in the first round before the wait
        // for the previous kernel, so they land while pool_prepare is still running.
        const int n_pre = n_items < (int)SB ? n_items : (int)SB;
        if (tid == 0)
            for (int it = 0; it < n_pre; ++it) load_item(it);
        if (round_idx == 0) {
            grid_dep_wait();          // cell map / latent vectors come from pool_prepare
            grid_dep_launch();
        }
        // ---- round setup (all warps): split latent tables of the one / two tiles ---------------------
        int rbase[2], nrows[2], lbase[2], nlat[2];
#pragma unroll
        for (int x = 0; x < 2; ++x) {
            rbase[x] = tile[x] * R + (int)rank * 128;
            int nrw = p.M - rbase[x];
            nrw = nrw < 0 ? 0 : (nrw > 128 ? 128 : nrw);
            if (x >= nsub) nrw = 0;
            nrows[x] = nrw;
            lbase[x] = 0; nlat[x] = 0;
            if (nrw > 0) {
                const int s_lo = p.row_scene[rbase[x]], s_hi = p.row_scene[rbase[x] + nrw - 1];
                lbase[x] = p.scene_off[s_lo];
                nlat[x] = p.scene_off[s_hi + 1] - lbase[x];
            }
        }
#pragma unroll
        for (int x = 0; x < 2; ++x) {
            if (nrows[x] == 0) continue;
            for (int idx = tid; idx < (nlat[x] + 1) * 8; idx += kSpThreads) {       // 2 values per thread
                const int r = idx >> 3, k = (idx & 7) * 2;
                const float* src = r < nlat[x] ? p.lat + (size_t)(lbase[x] + r) * 16 : p.benc;
                const float v0 = src[k] - p.constant, v1 = src[k + 1] - p.constant;
                const __nv_bfloat16 h0 = __float2bfloat16_rn(v0), h1 = __float2bfloat16_rn(v1);
                const __nv_bfloat16 l0 = __float2bfloat16_rn(v0 - __bfloat162float(h0));
                const __nv_bfloat16 l1 = __float2bfloat16_rn(v1 - __bfloat162float(h1));
                reinterpret_cast<uint32_t*>(latH[x])[idx] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
                reinterpret_cast<uint32_t*>(latL[x])[idx] = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
            }
        }
        __syncthreads();
        // the peer's barriers must be initialised before the first remote arrive / multicast commit
        asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
        asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");

        // MMA groups of a one-tile round: a 9-block piece is issued as N = 160 + 128 over the same A operand
        const bool split = ncols[0] > 256u;

        if (warp == 0) {
            // ===== weight producer: one bulk copy per cell and piece, up to SB items ahead =====
            if (lane == 0) {
                for (int it = n_pre; it < n_items; ++it) {
                    const uint32_t sb = (uint32_t)it % SB, pb = ((uint32_t)it / SB) & 1u;
                    sp_mbar_wait(sp_smem_u32(&empty_b[sb]), pb ^ 1u);
                    load_item(it);
                }
            }
            __syncwarp();
        } else if (warp == 1 || warp == 2) {
            // ===== MMA issuers (leader CTA of a pair), one thread each; everything that does not change per cell is
            // hoisted (a single thread retires ~1 instruction per 4 cycles, ~80 cycles per MMA all in all).  The
            // tensor core must see two independent accumulator chains interleaved: a chain of dependent MMAs
            // narrower than ~200 columns runs at the ~100-cycle accumulate latency, not at N / 2 cycles.  (Measured
            // alternatives: one thread issuing both chains in turn 87 cycles per MMA = issue-bound; two threads on
            // DIFFERENT items did not interleave, 800 cycles per cell instead of 432.) =====
            if (lane == 0 && rank == 0) {
                const int gq = warp - 1;
                const uint32_t b_desc_hi = (uint32_t)(512 >> 4) | (1u << 14) | (6u << 29);    // row groups alternate hi / lo
                const uint64_t b_base = ((uint64_t)b_desc_hi << 32) | (uint64_t)((ring & 0x3FFFFu) >> 4);
                const uint64_t bcell16 = b_cell >> 4;
                const uint32_t idesc_base = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(R >> 4) << 24);
                // MMA group of this issuer.  One tile: a 9-block piece is issued as N = 160 + 128 over the same A
                // operand by the two issuers, anything narrower by issuer 0 alone.  Two tiles: issuer gq owns piece gq
                // (its own A columns inside the stage).  Both issuers wake on the same barrier and issue the same
                // number of MMAs per item, so their two accumulator chains interleave in the tensor core's queue.
                uint32_t gn, d;
                uint64_t b_off16;
                if (nsub == 2) {
                    gn = ncols[gq];
                    d = tmem_base + (gq ? ncols[0] : 0u);
                    b_off16 = gq ? (uint64_t)(nr[0] * 4u) : 0u;                      // piece 1's rows behind piece 0's
                } else {
                    gn = split ? (gq == 0 ? 160u : ncols[0] - 160u) : (gq == 0 ? ncols[0] : 0u);
                    d = tmem_base + ((split && gq == 1) ? 160u : 0u);
                    b_off16 = (split && gq == 1) ? (uint64_t)((160u / 2) * 4u) : 0u;    // the group's rows inside a cell
                }
                const bool have = gn > 0;
                const uint32_t idesc = idesc_base | ((gn >> 3) << 17);
                for (int it = 0; it < n_items; ++it) {
                    const uint32_t sa = (uint32_t)it % SA, pa = ((uint32_t)it / SA) & 1u;
                    const uint32_t sb = (uint32_t)it % SB;
                    sp_mbar_wait_cluster(sp_smem_u32(&full_a[sa]), pa);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    if (have) {
                        // A from tensor memory: stage sa, (two tiles: the issuer's own tile inside every cell)
                        uint32_t at = tmem_base + a_col0 + sa * a_stage_cols + (nsub == 2 ? (uint32_t)gq * 16u : 0u);
                        const uint32_t at_cell = nsub == 2 ? 32u : 16u;
                        uint64_t bd = b_base + (uint64_t)(sb * (b_stage >> 4)) + b_off16;
                        sp_umma_ts(d, at, bd, idesc, it > 0 ? 1u : 0u);                  // hi . hi
                        sp_umma_ts(d, at + 8u, bd, idesc, 1u);                           // lo . hi
                        sp_umma_ts(d, at, bd + (256u >> 4), idesc, 1u);                  // hi . lo
#pragma unroll 3
                        for (int kc = 1; kc < KC; ++kc) {
                            at += at_cell; bd += bcell16;
                            sp_umma_ts(d, at, bd, idesc, 1u);
                            sp_umma_ts(d, at + 8u, bd, idesc, 1u);
                            sp_umma_ts(d, at, bd + (256u >> 4), idesc, 1u);
                        }
                    }
                    sp_commit(sp_smem_u32(&empty_a[sa]));
                    sp_commit(sp_smem_u32(&empty_b[sb]));
                }
                sp_commit(sp_smem_u32(&acc_full_bar));
            }
            __syncwarp();
        } else if (warp == 3) {
            // ===== weight relay (one thread per CTA): "the weights of item `it` have landed in THIS CTA" joins the
            // builders' arrivals on the leader's full barrier of the item's A stage, so that the MMA issuers wait on one
            // barrier per item and the builders never wait for the weights (they are the critical warps of a two-tile
            // round).  The A stage's previous phase must have completed before this phase's arrival. =====
            if (lane == 0) {
                for (int it = 0; it < n_items; ++it) {
                    const uint32_t sa = (uint32_t)it % SA, pa = ((uint32_t)it / SA) & 1u;
                    const uint32_t sb = (uint32_t)it % SB, pb = ((uint32_t)it / SB) & 1u;
                    sp_mbar_wait(sp_smem_u32(&empty_a[sa]), pa ^ 1u);
                    sp_mbar_wait(sp_smem_u32(&full_b[sb]), pb);
                    sp_mbar_arrive_cluster(full_remote[sa]);
                }
            }
            __syncwarp();
        } else if (warp >= 4 && warp < 12) {
            // ===== A builders: thread = pedestrian row; every row of every cell's (hi, lo) vector is written =====
            const int bg = (warp - 4) >> 2;
            const uint32_t r = (uint32_t)((warp & 3) * 32 + lane);
            const int x = nsub == 2 ? bg : 0;                       // two tiles: builder group bg owns tile bg
            const int row = rbase[x] + (int)r;
            const bool row_ok = (int)r < nrows[x];
            const uint4* cr = row_ok ? reinterpret_cast<const uint4*>(p.cell_row + (size_t)row * p.cells) : nullptr;
            const int off_r = row_ok ? p.scene_off[p.row_scene[row]] - lbase[x] : 0;
            // this warp's TMEM lane quarter, first column of the A ring (two tiles: [cell][tile][hi | lo])
            const uint32_t a_tmem = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + a_col0 + (nsub == 2 ? (uint32_t)bg * 16u : 0u);
#define TB2_SP_BUILD(KCV, TWO)                                                                                          \
    sp_builder<KCV, TWO>(cr, p.cells >> 4, a_tmem, bg, off_r, nlat[x], latH[x], latL[x], empty_a, full_remote, lane,    \
                         SA, a_stage_cols)
            if (nsub == 2) { if (wide_items) TB2_SP_BUILD(4, true); else TB2_SP_BUILD(2, true); }
            else TB2_SP_BUILD(4, false);
#undef TB2_SP_BUILD
        }
        {
            // ===== epilogue (all 16 warps, 4 per TMEM lane quarter): thread = pedestrian row, 16 columns per tcgen05.ld =====
            const int q = warp & 3, sub = warp >> 2;
            sp_mbar_wait(sp_smem_u32(&acc_full_bar), 0u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
            // accumulator column d of an MMA group = row (d mod n/2) of the slab of CTA (d div n/2): 16-column
            // chunks never straddle the two halves (n/2 is a multiple of 16)
            const int nchunk0 = (int)ncols[0] >> 4, nchunk = (int)(ncols[0] + ncols[1]) >> 4;
            auto chunk_col = [&](int ch, int& x) {           // first global hidden1 column of 16-column chunk ch, its piece
                x = ch >= nchunk0 ? 1 : 0;
                int dx = (x ? ch - nchunk0 : ch) * 16;                           // column inside the piece's accumulators
                const int nrx = (int)ncols[x] / 2;                               // rows per CTA of the piece
                int gn = (int)ncols[x], goff = 0;                                // MMA group of this column
                if (split) {
                    if (dx >= 160) { dx -= 160; gn = (int)ncols[0] - 160; goff = 160 / 2; }
                    else gn = 160;
                }
                const int half = gn / 2;                                         // rows per CTA of the group
                const int hsel = dx >= half ? 1 : 0;                             // which CTA's rows
                return col0[x] + hsel * nrx + goff + (dx - hsel * half);
            };
            for (int ch = sub; ch < nchunk; ch += 4) {
                int x;
                const int col = chunk_col(ch, x);
                const int row = tile[x] * R + (int)rank * 128 + q * 32 + lane;
                uint32_t v[16];
                sp_tmem_ld16(trow + (uint32_t)(ch * 16), v);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (row < p.M) {
                    const size_t o = (size_t)row * p.OUT + col;
                    float bias[16];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.base + col) + i);
                        bias[4 * i] = b4.x; bias[4 * i + 1] = b4.y; bias[4 * i + 2] = b4.z; bias[4 * i + 3] = b4.w;
                    }
                    if (p.out_hi) {
                        uint32_t ph[8], pl[8];
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const float x0 = fmaxf(__uint_as_float(v[2 * i]) + bias[2 * i], 0.f);
                            const float x1 = fmaxf(__uint_as_float(v[2 * i + 1]) + bias[2 * i + 1], 0.f);
                            const __nv_bfloat16 h0 = __float2bfloat16_rn(x0), h1 = __float2bfloat16_rn(x1);
                            const __nv_bfloat16 l0 = __float2bfloat16_rn(x0 - __bfloat162float(h0));
                            const __nv_bfloat16 l1 = __float2bfloat16_rn(x1 - __bfloat162float(h1));
                            ph[i] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
                            pl[i] = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
                        }
                        uint4* dh = reinterpret_cast<uint4*>(p.out_hi + o);
                        uint4* dl = reinterpret_cast<uint4*>(p.out_lo + o);
                        dh[0] = make_uint4(ph[0], ph[1], ph[2], ph[3]); dh[1] = make_uint4(ph[4], ph[5], ph[6], ph[7]);
                        dl[0] = make_uint4(pl[0], pl[1], pl[2], pl[3]); dl[1] = make_uint4(pl[4], pl[5], pl[6], pl[7]);
                    } else {
                        float4* d4 = reinterpret_cast<float4*>(p.out + o);
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            float4 y;
                            y.x = fmaxf(__uint_as_float(v[4 * i]) + bias[4 * i], 0.f);
                            y.y = fmaxf(__uint_as_float(v[4 * i + 1]) + bias[4 * i + 1], 0.f);
                            y.z = fmaxf(__uint_as_float(v[4 * i + 2]) + bias[4 * i + 2], 0.f);
                            y.w = fmaxf(__uint_as_float(v[4 * i + 3]) + bias[4 * i + 3], 0.f);
                            d4[i] = y;
                        }
                    }
                }
            }
        }
        ++round_idx;
        // the next round overwrites the latent tables, the TMEM accumulators and the peer's accumulators
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
        asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    }
    if (warp == 1) {
        uint32_t ncols = 512;
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(ncols) : "memory");
    }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
bool sparse_pair_supported(const tb2_lstm* m, const tb2_layout* l) {
    if (m->cfg.pool_type != TB2_POOL_SOCIAL || m->C != 16 || m->Wt1_sw_hi == nullptr) return false;
    if (m->mlp_dims[1] % 32 != 0 || m->mlp_dims[1] / 32 < kSpMaxBlocks) return false;
    if (m->cells > kSpMaxCells || m->cells % 16 != 0) return false;
    // local latent table of a 128-row tile: the scenes it touches, <= 128 + 2 (n_max - 1) rows, + 1;
    // cell-map bytes hold scene-local indices (0xFE / 0xFF reserved)
    return 128 + 2 * (l->n_max - 1) + 1 <= kSpLatRows - 1 && l->n_max <= 0xFD;
}

// Cut the linearised (tile, 32-column block) space [0, tiles * nb) into n_rounds consecutive rounds of 1..cap
// blocks, such that a round lies inside one tile or straddles exactly one tile boundary with both pieces at
// least `minpiece` blocks (a 32- or 64-column MMA costs ~50 cycles, not 16 / 32), at most 8, and at most cap2
// together.  Reachability
// DP over (round, end position) inside a window around the even split.
static bool plan_rounds_dp(long long total, int nb, int n_rounds, int cap, int cap2, int minpiece, std::vector<SpRound>& out) {
    const int W = 24;                                      // positions considered: even split +- W
    std::vector<std::vector<signed char>> from((size_t)n_rounds + 1, std::vector<signed char>(2 * W + 1, -1));
    auto base = [&](int k) { return (long long)k * total / n_rounds; };
    from[0][W] = 0;
    for (int k = 0; k < n_rounds; ++k) {
        for (int o = 0; o <= 2 * W; ++o) {
            if (from[k][o] < 0) continue;
            const long long pos = base(k) + o - W;
            for (int sz = 1; sz <= cap; ++sz) {
                const long long end = pos + sz;
                if (end > total) break;
                const long long t0 = pos / nb, t1 = (end - 1) / nb;
                if (t1 > t0 + 1) continue;
                if (t1 == t0 + 1) {
                    const long long a = (t0 + 1) * nb - pos, b = end - (t0 + 1) * nb;
                    if (a < minpiece || b < minpiece || a > 8 || b > 8 || sz > cap2) continue;
                }
                const long long off = end - base(k + 1) + W;
                if (off < 0 || off > 2 * W) continue;
                if (from[k + 1][(size_t)off] < 0) from[k + 1][(size_t)off] = (signed char)sz;
            }
        }
    }
    const long long off_end = total - base(n_rounds) + W;
    if (off_end < 0 || off_end > 2 * W || from[n_rounds][(size_t)off_end] < 0) return false;
    out.assign((size_t)n_rounds, SpRound{0, 0, 0, 0});
    long long end = total;
    for (int k = n_rounds; k > 0; --k) {
        const int sz = from[k][(size_t)(end - base(k) + W)];
        const long long pos = end - sz;
        const long long t0 = pos / nb;
        const long long in0 = std::min<long long>(sz, (t0 + 1) * nb - pos);
        out[(size_t)k - 1] = SpRound{(int)t0, (int)(pos - t0 * nb), (int)in0, (int)(sz - in0)};
        end = pos;
    }
    return end == 0;
}

// the round table of a (layout, OUT, units) combination lives with the layout (device memory of its device)
static int get_plan(const tb2_layout* l, int OUT, int units_max, const tb2_layout::PairPlan** out, cudaStream_t st) {
    static std::mutex mu;
    std::lock_guard<std::mutex> lock(mu);
    tb2_layout* lm = const_cast<tb2_layout*>(l);
    for (const auto& e : lm->pair_plans)
        if (e.OUT == OUT && e.units_max == units_max) { *out = &e; return TB2_OK; }
    const int R = 256, nb = OUT / 32;                     // 256-row tiles (128 per CTA of a pair) x 32-column blocks
    const long long tiles = (l->M + R - 1) / R, total = tiles * nb;
    int units = units_max;
    if ((long long)units > total) units = (int)total;
    const int rpu = (int)((total + (long long)units * kSpMaxBlocks - 1) / ((long long)units * kSpMaxBlocks));
    const int n_rounds = units * rpu;
    std::vector<SpRound> rounds;
    bool ok = false;       // smallest maximum round first (the kernel's time is the largest round), then the widest narrow piece
    // a two-tile round feeds two narrower accumulator chains and is slower per block than a one-tile round
    // (DESIGN.md section 4.1): it gets one block less than the cap when the split allows it
    for (int cap = (int)((total + n_rounds - 1) / n_rounds); cap <= kSpMaxBlocks && !ok; ++cap)
        for (int relax = 0; relax < 2 && !ok; ++relax)
            for (int minpiece = 3; minpiece >= 1 && !ok; --minpiece)
                ok = plan_rounds_dp(total, nb, n_rounds, cap, relax ? cap : std::max(cap - 1, 1), minpiece, rounds);
    if (!ok) { set_error("sparse_layer1_pair: no round plan (internal)"); return TB2_ERR_INVALID; }
    SpRound* dev = nullptr;
    TB2_CHECK_CUDA(cudaMalloc(&dev, rounds.size() * sizeof(SpRound)));
    lm->owned.push_back(dev);
    TB2_CHECK_CUDA(cudaMemcpyAsync(dev, rounds.data(), rounds.size() * sizeof(SpRound), cudaMemcpyHostToDevice, st));
    TB2_CHECK_CUDA(cudaStreamSynchronize(st));       // one-time (per layout): the host vector is a temporary
    tb2_layout::PairPlan e;
    e.OUT = OUT; e.units_max = units_max; e.units = units; e.rounds_per_unit = rpu; e.dev = dev;
    lm->pair_plans.push_back(e);
    *out = &lm->pair_plans.back();
    return TB2_OK;
}

int launch_sparse_pair(const tb2_lstm* m, const tb2_layout* l, Workspace* ws, float* out, void* out_hi, void* out_lo,
                       cudaStream_t st) {
    static int sm_count[64] = {0};
    int dev = 0;
    TB2_CHECK_CUDA(cudaGetDevice(&dev));
    if (sm_count[dev & 63] == 0)
        TB2_CHECK_CUDA(cudaDeviceGetAttribute(&sm_count[dev & 63], cudaDevAttrMultiProcessorCount, dev));
    const int d1 = m->mlp_dims[1];
    const int units_max = sm_count[dev & 63] / 2;
    SpParams p;
    const tb2_layout::PairPlan* plan = nullptr;
    int rc;
    if ((rc = get_plan(l, d1, units_max, &plan, st))) return rc;
    const int units = plan->units;
    p.rounds = (const SpRound*)plan->dev;
    p.rounds_per_unit = plan->rounds_per_unit;
    p.scene_off = l->scene_off;
    p.row_scene = l->row_scene;
    p.cell_row = ws->cell_row;
    p.lat = ws->lat;
    p.benc = m->benc;
    p.base = m->base1;
    p.w = (const unsigned char*)m->Wt1_sw_hi;
    p.out = out;
    p.out_hi = (__nv_bfloat16*)out_hi;
    p.out_lo = (__nv_bfloat16*)out_lo;
    p.M = l->M;
    p.OUT = d1;
    p.cells = m->cells;
    p.constant = m->cfg.constant;
    const size_t smem = 1024 + kSpDynBytes + 64;
    static_assert(1024 + kSpDynBytes + 64 <= 227 * 1024 - 512, "shared memory budget");
    static DynSmemConfig configured;
    TB2_CHECK_CUDA(configured.ensure(sparse_layer1_pair_kernel, smem));
    {
        KernelTimer kt("sparse_layer1_pair_ts", st);
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(2 * units);
        cfg.blockDim = dim3(kSpThreads);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = st;
        cudaLaunchAttribute attr[2];
        int na = 0;
        if (pdl_enabled()) {
            attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            attr[na].val.programmaticStreamSerializationAllowed = 1;
            ++na;
        }
        attr[na].id = cudaLaunchAttributeClusterDimension;
        attr[na].val.clusterDim.x = 2;
        attr[na].val.clusterDim.y = 1;
        attr[na].val.clusterDim.z = 1;
        ++na;
        cfg.attrs = attr;
        cfg.numAttrs = na;
        TB2_CHECK_CUDA(cudaLaunchKernelEx(&cfg, sparse_layer1_pair_kernel, p));
    }
    TB2_LAUNCH_CHECK();
    return TB2_OK;
}

// weight repack: W1[o][c * cells + cell] -> bf16 [cell][o / 8][hi | lo][o % 8][16] with the two 16-byte halves
// of a row exchanged where ((o >> 2) & 1): the SWIZZLE_32B shared-memory image (8-row atoms of 256 bytes,
// hi and lo atoms alternating, SBO = 512) of any slab whose first row is a multiple of 8, so ONE plain bulk
// copy per cell lands both operand tiles the UMMA descriptors expect
__global__ void repack_layer1_sw_kernel(const float* __restrict__ W1, __nv_bfloat16* __restrict__ dst, int OUT, int cells) {
    size_t total = (size_t)cells * OUT * 16;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (size_t)gridDim.x * blockDim.x) {
        const int c = (int)(idx & 15);
        const size_t co = idx >> 4;
        const int o = (int)(co % OUT), cell = (int)(co / OUT);
        const float v = W1[(size_t)o * 16 * cells + (size_t)c * cells + cell];
        const __nv_bfloat16 h = __float2bfloat16_rn(v);
        const int chunk = (c >> 3) ^ ((o >> 2) & 1);
        const size_t atom = ((size_t)cell * OUT + (size_t)(o & ~7)) * 32;          // bf16 elements: 8 rows x (hi 16 + lo 16)
        const size_t e = atom + (size_t)(o & 7) * 16 + (size_t)(chunk * 8 + (c & 7));
        dst[e] = h;
        dst[e + 128] = __float2bfloat16_rn(v - __bfloat162float(h));
    }
}

int launch_repack_layer1_sw(const float* W1, void* hi, void* lo, int OUT, int cells, cudaStream_t st) {
    (void)lo;     // one interleaved image of 2 x cells x OUT x 16 bf16 behind `hi`
    repack_layer1_sw_kernel<<<1024, 256, 0, st>>>(W1, (__nv_bfloat16*)hi, OUT, cells);
    TB2_LAUNCH_CHECK();
    return TB2_OK;
}

}  // namespace tb2
