// First Linear of the SOCIAL grid embedding on tcgen05 (5th-gen tensor cores, TMEM accumulators).
//
//   hidden1[p, :] = relu(b1 + sum_{winning (cell, j) of p} W1[:, cell-slab] . lat_j)
//   (reference: GridBasedPooling.social + the first Linear of two_layer,
//    trajnetbaselines/lstm/gridbased_pooling.py:145-170,227-305,316-323)
//
// Formulation: for one scene group (<= 160 pedestrians) and one 256-column chunk of the output,
//     D^T[col, p] = sum over cells c of  W_c^T[col, 0:16] . L_c[0:16, p]
// where L_c[:, p] is the latent vector of p's winning neighbour in cell c, or zero.  Per cell this
// is one tcgen05.mma with M = 128 output columns (x2 blocks), N = pedestrians of the group,
// K = 16, and the fp32 accumulator never leaves TMEM until all cells are done -- no scatter, no
// shared-memory accumulators, no atomics.  The weight slab W_c arrives by TMA (32-byte swizzle);
// L_c is built in shared memory by one warp from the per-cell buckets of winner pairs (rows of the
// previous use of the stage are re-zeroed, so the tile is dense-zero except <= ~10 rows).
// Precision: 3-pass bf16 (hi, lo) split like the other tensor-core kernels.
//
// Why not the warp-level mma.sync kernel (sparse_layer1_mma_kernel): measured on B200 it is bound
// by the legacy HMMA issue rate (~32 cycles per m16n8k16 per SM sub-partition); tcgen05 runs the
// zero-padded product ~2x faster end to end even though it multiplies the zeros.
//
// Warp roles (384 threads): 0 = TMA producer, 1 = TMEM alloc + MMA issuer, 2 = L-tile builder,
// 4..11 = epilogue (lane quarter = warp % 4, column block = (warp - 4) / 4), 3, 12, 13 = more builders.
#include <cuda.h>
#include <cuda_bf16.h>

#include "common.cuh"

namespace tb2 {

constexpr int kScThreads = 448;          // 14 warps: TMA, MMA, 4 builders (2, 3, 12, 13), 8 epilogue (4..11)
constexpr int kScBuilders = 4;
constexpr int kScCols = 256;            // output columns per CTA (2 blocks of M = 128)
constexpr int kScStages = 7;
constexpr int kScMaxN = 160;            // pedestrians per group (MMA N, multiple of 16)
constexpr uint32_t kScABytes = 128 * 32;                 // one (block, part) weight tile: 128 cols x 16 k bf16
constexpr uint32_t kScBBytes = kScMaxN * 32;             // one part of L_c: N rows x 16 k bf16
constexpr uint32_t kScStageBytes = 4 * kScABytes + 2 * kScBBytes;   // 16 KB + 10 KB

__device__ __forceinline__ uint32_t sc_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void sc_mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void sc_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void sc_mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void sc_mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "SC_WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra SC_WAIT_DONE;\n"
        "bra SC_WAIT_LOOP;\n"
        "SC_WAIT_DONE:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void sc_tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
// K-major operand with 32-byte rows, SWIZZLE_32B: 8-row atoms of 256 bytes, SBO = 256
__device__ __forceinline__ uint64_t sc_umma_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)(256 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)6 << 61;          // SWIZZLE_32B
    return d;
}
__device__ __forceinline__ void sc_umma(uint32_t tmem_d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "l"(a), "l"(b), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void sc_umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void sc_tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}

struct ScParams {
    const int* group_off;
    const int* scene_off;
    const int* win_count;
    const uint32_t* win_ent;
    const float* lat;            // [M, 16] fp32
    const float* benc;           // [16]
    const float* base;           // [OUT]
    float* out;                  // fp32 [M, OUT] or null
    __nv_bfloat16* out_hi;       // bf16 split [M, OUT] or null
    __nv_bfloat16* out_lo;
    int OUT, cells, nm1, cap;
    float constant;
};

// byte offset of (row r, 16-byte chunk c) inside a SWIZZLE_32B K-major tile
__device__ __forceinline__ uint32_t sw32(uint32_t r, uint32_t c) { return r * 32u + ((c ^ ((r >> 2) & 1u)) << 4); }

__global__ void __launch_bounds__(kScThreads, 1)
sparse_layer1_tc_kernel(const __grid_constant__ CUtensorMap map_w_hi, const __grid_constant__ CUtensorMap map_w_lo,
                        ScParams p) {
    extern __shared__ __align__(1024) unsigned char smem_sc[];
    __shared__ __align__(8) uint64_t full_a[kScStages];
    __shared__ __align__(8) uint64_t full_b[kScStages];
    __shared__ __align__(8) uint64_t empty_bar[kScStages];
    __shared__ __align__(8) uint64_t acc_full_bar;
    __shared__ uint32_t tmem_base_slot;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int s0 = p.group_off[blockIdx.x], s1 = p.group_off[blockIdx.x + 1];
    const int row0 = p.scene_off[s0];
    const int P = p.scene_off[s1] - row0;
    const int Npad = (P + 15) & ~15;
    const int chunk0 = blockIdx.y * kScCols;

    const uint32_t ring = (sc_smem_u32(smem_sc) + 1023u) & ~1023u;
    unsigned char* ring_ptr = smem_sc + (ring - sc_smem_u32(smem_sc));
    unsigned char* tail = ring_ptr + (size_t)kScStages * kScStageBytes;
    int* start = reinterpret_cast<int*>(tail);                            // [cells + 1]
    int* cursor = start + p.cells + 1;                                    // [cells]
    uint32_t* ent = reinterpret_cast<uint32_t*>(cursor + p.cells);        // [cap * nm1]: lat row << 16 | ped row
    int* cnt_s = reinterpret_cast<int*>(ent + (size_t)p.cap * p.nm1);     // [cap]
    int* sbase = cnt_s + p.cap;                                           // [cap]
    uint16_t* item_cell = reinterpret_cast<uint16_t*>(sbase + p.cap);     // [cells] non-empty cells, ascending
    // latent vectors of the group, already split: [cap + 1][16] bf16 x 2 (row cap = NaN-padded slot, b_enc)
    uint4* latH = reinterpret_cast<uint4*>((reinterpret_cast<uintptr_t>(item_cell + p.cells) + 15) & ~(uintptr_t)15);
    uint4* latL = latH + (size_t)(p.cap + 1) * 2;

    // ---- phase 0 (all warps): barriers + TMEM, so the TMA producer can start streaming at once -----
    if (warp == 0 && lane == 0) {
        for (int s = 0; s < kScStages; ++s) {
            sc_mbar_init(sc_smem_u32(&full_a[s]), 1);
            sc_mbar_init(sc_smem_u32(&full_b[s]), 1);
            sc_mbar_init(sc_smem_u32(&empty_bar[s]), 1);
        }
        sc_mbar_init(sc_smem_u32(&acc_full_bar), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        uint32_t ncols = 512;
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"(sc_smem_u32(&tmem_base_slot)), "r"(ncols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = tmem_base_slot;
    const int n_items = p.cells;          // every cell is one pipeline item (empty buckets multiply zeros)
    grid_dep_wait();          // winners / latent vectors (and, after a weight update, the slabs) come from earlier kernels
    grid_dep_launch();

    // ---- phase 1 (warps 1..13, 416 threads): zeroed L tiles, split latent vectors, per-cell buckets,
    //      while warp 0 already streams the first weight slabs -------------------------------------------
    constexpr int kSetupThreads = kScThreads - 32;
    auto setup_sync = [] { asm volatile("bar.sync 1, %0;" ::"n"(kSetupThreads) : "memory"); };
    if (warp != 0) {
        const int t2 = tid - 32;
        for (int s = 0; s < kScStages; ++s) {        // L tiles start as all-zero
            uint4* b = reinterpret_cast<uint4*>(ring_ptr + (size_t)s * kScStageBytes + 4 * kScABytes);
            for (int i = t2; i < (int)(2 * kScBBytes / 16); i += kSetupThreads) b[i] = make_uint4(0u, 0u, 0u, 0u);
        }
        for (int c = t2; c < p.cells; c += kSetupThreads) cursor[c] = 0;
        for (int idx = t2; idx < (P + 1) * 8; idx += kSetupThreads) {       // 2 values per thread
            const int r = idx >> 3, k = (idx & 7) * 2;
            const float* src = r < P ? p.lat + (size_t)(row0 + r) * 16 : p.benc;
            const float v0 = src[k] - p.constant, v1 = src[k + 1] - p.constant;
            const __nv_bfloat16 h0 = __float2bfloat16_rn(v0), h1 = __float2bfloat16_rn(v1);
            const __nv_bfloat16 l0 = __float2bfloat16_rn(v0 - __bfloat162float(h0));
            const __nv_bfloat16 l1 = __float2bfloat16_rn(v1 - __bfloat162float(h1));
            const int dst = (r < P ? r : p.cap) * 8 + (k >> 1);           // 32-bit words, 8 per row
            reinterpret_cast<uint32_t*>(latH)[dst] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
            reinterpret_cast<uint32_t*>(latL)[dst] = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
        }
        for (int r = t2; r < P; r += kSetupThreads) cnt_s[r] = p.win_count[row0 + r];
        for (int sb = s0 + (warp - 1); sb < s1; sb += kSetupThreads / 32) {
            const int a = p.scene_off[sb] - row0, b2 = p.scene_off[sb + 1] - row0;
            for (int r = a + lane; r < b2; r += 32) sbase[r] = a;
        }
        setup_sync();
        const int total = P * p.nm1;
        const uint32_t* raw = p.win_ent + (size_t)row0 * p.nm1;    // rows of a group are contiguous
        for (int idx = t2; idx < total; idx += kSetupThreads) {
            int r = idx / p.nm1, k = idx - r * p.nm1;
            if (k < cnt_s[r]) atomicAdd(&cursor[raw[idx] >> 16], 1);
        }
        setup_sync();
        if (t2 < 32) {
            int per = (p.cells + 31) / 32;
            int lo = t2 * per, hi = min(lo + per, p.cells);
            int sum = 0;
            for (int c = lo; c < hi; ++c) sum += cursor[c];
            int incl = sum;
            for (int d = 1; d < 32; d <<= 1) {
                int v = __shfl_up_sync(0xffffffffu, incl, d);
                if (t2 >= d) incl += v;
            }
            int run = incl - sum;
            for (int c = lo; c < hi; ++c) {
                int cnt = cursor[c];
                start[c] = run;
                cursor[c] = run;
                run += cnt;
            }
            if (t2 == 31) start[p.cells] = incl;
        }
        setup_sync();
        for (int idx = t2; idx < total; idx += kSetupThreads) {
            int r = idx / p.nm1, k = idx - r * p.nm1;
            if (k < cnt_s[r]) {
                const uint32_t e = raw[idx];
                const int pos = atomicAdd(&cursor[e >> 16], 1);
                const int j = (int)(e & 0xffff);
                const uint32_t lrow = (uint32_t)(j == 0xffff ? p.cap : sbase[r] + j);
                ent[pos] = (lrow << 16) | (uint32_t)r;
            }
        }
        // generic-proxy writes (zeroed tiles) must be visible to the tensor core's async-proxy reads
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        setup_sync();
    }

    if (warp == 0) {
        // ===== TMA producer: weight slabs of the non-empty cells =====
        if (lane == 0) {
            for (int it = 0; it < n_items; ++it) {
                const int s = it % kScStages;
                const uint32_t ph = (it / kScStages) & 1;
                sc_mbar_wait(sc_smem_u32(&empty_bar[s]), ph ^ 1);
                const uint32_t bar = sc_smem_u32(&full_a[s]);
                const uint32_t base = ring + s * kScStageBytes;
                const int wrow = it * p.OUT + chunk0;
                sc_mbar_expect_tx(bar, 4 * kScABytes);
                sc_tma_load_2d(base + 0 * kScABytes, &map_w_hi, bar, 0, wrow);
                sc_tma_load_2d(base + 1 * kScABytes, &map_w_hi, bar, 0, wrow + 128);
                sc_tma_load_2d(base + 2 * kScABytes, &map_w_lo, bar, 0, wrow);
                sc_tma_load_2d(base + 3 * kScABytes, &map_w_lo, bar, 0, wrow + 128);
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (lane == 0) {
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(Npad >> 3) << 17) | (8u << 24);
            for (int it = 0; it < n_items; ++it) {
                const int s = it % kScStages;
                const uint32_t ph = (it / kScStages) & 1;
                sc_mbar_wait(sc_smem_u32(&full_a[s]), ph);
                sc_mbar_wait(sc_smem_u32(&full_b[s]), ph);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t base = ring + s * kScStageBytes;
                const uint64_t b_hi = sc_umma_desc(base + 4 * kScABytes);
                const uint64_t b_lo = sc_umma_desc(base + 4 * kScABytes + kScBBytes);
#pragma unroll
                for (int blk = 0; blk < 2; ++blk) {
                    const uint64_t a_hi = sc_umma_desc(base + blk * kScABytes);
                    const uint64_t a_lo = sc_umma_desc(base + (2 + blk) * kScABytes);
                    const uint32_t d = tmem_base + (uint32_t)(blk * 256);
                    sc_umma(d, a_hi, b_hi, idesc, it > 0 ? 1u : 0u);
                    sc_umma(d, a_hi, b_lo, idesc, 1u);
                    sc_umma(d, a_lo, b_hi, idesc, 1u);
                }
                sc_umma_commit(sc_smem_u32(&empty_bar[s]));
            }
            sc_umma_commit(sc_smem_u32(&acc_full_bar));
        }
        __syncwarp();
    } else if (warp == 2 || warp == 3 || warp >= 12) {
        // ===== L-tile builders (4 warps, items round-robin).  Stateless: the rows written by the
        // previous user of a stage (item it - kScStages) are re-derived from its bucket and zeroed,
        // then the rows of this item's bucket are written. =====
        const int bidx = warp < 4 ? warp - 2 : warp - 10;          // 0..3
        for (int it = bidx; it < n_items; it += kScBuilders) {
            const int s = it % kScStages;
            const uint32_t ph = (it / kScStages) & 1;
            sc_mbar_wait(sc_smem_u32(&empty_bar[s]), ph ^ 1);
            unsigned char* bh = ring_ptr + (size_t)s * kScStageBytes + 4 * kScABytes;
            unsigned char* bl = bh + kScBBytes;
            if (it >= kScStages) {
                const int pc = it - kScStages;
                for (int e = start[pc] + lane; e < start[pc + 1]; e += 32) {
                    const uint32_t r = ent[e] & 0xffffu;
                    *reinterpret_cast<uint4*>(bh + sw32(r, 0)) = make_uint4(0u, 0u, 0u, 0u);
                    *reinterpret_cast<uint4*>(bh + sw32(r, 1)) = make_uint4(0u, 0u, 0u, 0u);
                    *reinterpret_cast<uint4*>(bl + sw32(r, 0)) = make_uint4(0u, 0u, 0u, 0u);
                    *reinterpret_cast<uint4*>(bl + sw32(r, 1)) = make_uint4(0u, 0u, 0u, 0u);
                }
                __syncwarp();
            }
            const int cell = it;
            for (int e = start[cell] + lane; e < start[cell + 1]; e += 32) {
                const uint32_t en = ent[e];
                const uint32_t r = en & 0xffffu, lr = en >> 16;
                *reinterpret_cast<uint4*>(bh + sw32(r, 0)) = latH[lr * 2];
                *reinterpret_cast<uint4*>(bh + sw32(r, 1)) = latH[lr * 2 + 1];
                *reinterpret_cast<uint4*>(bl + sw32(r, 0)) = latL[lr * 2];
                *reinterpret_cast<uint4*>(bl + sw32(r, 1)) = latL[lr * 2 + 1];
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) sc_mbar_arrive(sc_smem_u32(&full_b[s]));
        }
    } else if (warp >= 4 && warp < 12) {
        // ===== epilogue: TMEM lane = output column, TMEM column = pedestrian =====
        const int q = warp & 3, blk = (warp - 4) >> 2;
        const int col = chunk0 + blk * 128 + q * 32 + lane;
        sc_mbar_wait(sc_smem_u32(&acc_full_bar), 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const float b = col < p.OUT ? p.base[col] : 0.f;
        const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(blk * 256);
        for (int p0 = 0; p0 < Npad; p0 += 16) {
            uint32_t v[16];
            if (n_items > 0) {
                sc_tmem_ld16(trow + (uint32_t)p0, v);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            } else {
#pragma unroll
                for (int i = 0; i < 16; ++i) v[i] = 0u;
            }
            if (col < p.OUT) {
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const int pr = p0 + i;
                    if (pr < P) {
                        const float x = fmaxf(__uint_as_float(v[i]) + b, 0.f);
                        const size_t o = (size_t)(row0 + pr) * p.OUT + col;
                        if (p.out_hi) {
                            const __nv_bfloat16 h = __float2bfloat16_rn(x);
                            p.out_hi[o] = h;
                            p.out_lo[o] = __float2bfloat16_rn(x - __bfloat162float(h));
                        } else {
                            p.out[o] = x;
                        }
                    }
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        uint32_t ncols = 512;
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(ncols) : "memory");
    }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
typedef CUresult (*ScEncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int make_slab_map(CUtensorMap* map, const void* base, size_t rows) {
    static ScEncodeTiledFn fn = nullptr;
    if (!fn) {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (ScEncodeTiledFn)ptr;
    }
    if (!fn) { set_error("cuTensorMapEncodeTiled unavailable"); return TB2_ERR_CUDA; }
    cuuint64_t dims[2] = {16, (cuuint64_t)rows};
    cuuint64_t strides[1] = {32};
    cuuint32_t box[2] = {16, 128};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(slab) failed (" + std::to_string((int)r) + ")"); return TB2_ERR_CUDA; }
    return TB2_OK;
}

size_t sparse_tc_smem_bytes(int cap, int cells, int nm1) {
    size_t b = 1024 + (size_t)kScStages * kScStageBytes;
    b += (size_t)(2 * cells + 1) * sizeof(int);
    b += (size_t)cap * nm1 * sizeof(uint32_t);
    b += (size_t)cap * 2 * sizeof(int);
    b += (size_t)cells * sizeof(uint16_t);
    b += (size_t)(cap + 1) * 64 + 16;                     // split latent vectors
    return b + 64;
}

bool sparse_tc_supported(const tb2_lstm* m, const tb2_layout* l, int gsel) {
    if (m->cfg.pool_type != TB2_POOL_SOCIAL || m->C != 16 || m->Wt1_nat_hi == nullptr) return false;
    if (m->mlp_dims[1] % kScCols != 0) return false;
    if (l->group_cap[gsel] > kScMaxN) return false;
    const int nm1 = l->n_max > 1 ? l->n_max - 1 : 1;
    return sparse_tc_smem_bytes(l->group_cap[gsel], m->cells, nm1) <= 227 * 1024;
}

int launch_sparse_tc(const tb2_lstm* m, const tb2_layout* l, int gsel, Workspace* ws, float* out, void* out_hi,
                     void* out_lo, cudaStream_t st) {
    const int nm1 = l->n_max > 1 ? l->n_max - 1 : 1;
    const int d1 = m->mlp_dims[1];
    CUtensorMap mh, ml;
    int rc;
    if ((rc = make_slab_map(&mh, m->Wt1_nat_hi, (size_t)m->cells * d1))) return rc;
    if ((rc = make_slab_map(&ml, m->Wt1_nat_lo, (size_t)m->cells * d1))) return rc;
    ScParams p;
    p.group_off = l->group_off[gsel];
    p.scene_off = l->scene_off;
    p.win_count = ws->win_count;
    p.win_ent = ws->win_ent;
    p.lat = ws->lat;
    p.benc = m->benc;
    p.base = m->base1;
    p.out = out;
    p.out_hi = (__nv_bfloat16*)out_hi;
    p.out_lo = (__nv_bfloat16*)out_lo;
    p.OUT = d1;
    p.cells = m->cells;
    p.nm1 = nm1;
    p.cap = l->group_cap[gsel];
    p.constant = m->cfg.constant;
    const size_t smem = sparse_tc_smem_bytes(p.cap, m->cells, nm1);
    static DynSmemConfig configured;
    TB2_CHECK_CUDA(configured.ensure(sparse_layer1_tc_kernel, smem));
    dim3 grid(l->num_groups[gsel], d1 / kScCols);
    {
        KernelTimer kt("sparse_layer1_tc", st);
        launch_pdl(sparse_layer1_tc_kernel, grid, dim3(kScThreads), smem, st, mh, ml, p);
    }
    TB2_LAUNCH_CHECK();
    return TB2_OK;
}

// weight repack: W1[o][c * cells + cell] -> (hi, lo)[cell][o][c] bf16, natural k order (TMA source)
__global__ void repack_layer1_nat_kernel(const float* __restrict__ W1, __nv_bfloat16* __restrict__ hi,
                                         __nv_bfloat16* __restrict__ lo, int OUT, int cells) {
    size_t total = (size_t)cells * OUT * 16;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (size_t)gridDim.x * blockDim.x) {
        const int c = (int)(idx & 15);
        const size_t co = idx >> 4;
        const int o = (int)(co % OUT), cell = (int)(co / OUT);
        const float v = W1[(size_t)o * 16 * cells + (size_t)c * cells + cell];
        const __nv_bfloat16 h = __float2bfloat16_rn(v);
        hi[idx] = h;
        lo[idx] = __float2bfloat16_rn(v - __bfloat162float(h));
    }
}

int launch_repack_layer1_nat(const float* W1, void* hi, void* lo, int OUT, int cells, cudaStream_t st) {
    repack_layer1_nat_kernel<<<1024, 256, 0, st>>>(W1, (__nv_bfloat16*)hi, (__nv_bfloat16*)lo, OUT, cells);
    TB2_LAUNCH_CHECK();
    return TB2_OK;
}

}  // namespace tb2
