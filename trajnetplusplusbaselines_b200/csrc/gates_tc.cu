// Fused recurrence step on the tensor cores: LSTMCell gate GEMM (tcgen05 + TMEM + TMA) with the
// cell update, the Gaussian head and the position feedback in the epilogue.
//
// Same contract as lstm_gates_kernel (csrc/lstm_step.cu; reference LSTM.step lstm.py:118-168,
// torch.nn.LSTMCell, Hidden2Normal modules.py:56-64), specialised for E = 64, H = 128,
// pool_to_input: gates[M, 512] = [emb | pooled | h][M, K] . [W_ih | W_hh]^T, K = 64 + P + 128.
//
// All three K segments arrive as bf16 (hi, lo) pairs written by their producers (embed_split,
// the grid-embedding layer's epilogue, the previous step's epilogue) and the product is the
// 3-pass split  A_hi.W_hi + A_hi.W_lo + A_lo.W_hi  accumulated in fp32 in TMEM.
//
// Grid: (2, ceil(M / 128)) with __cluster_dims__(2, 1, 1).  The two CTAs of a cluster share a
// 128-row tile and each owns 64 hidden units x 4 gates (256 TMEM columns; W rows are permuted at
// repack so a CTA's tile holds complete i/f/g/o quadruples).  Warp roles as in gemm_tc.cu.  The
// epilogue thread of a row reads its gates from TMEM, updates c / h (fp32 state + bf16 split for
// the next step) and accumulates its half of the 5-wide Hidden2Normal dot products; rank 1 ships
// its partial sums to rank 0 through distributed shared memory and rank 0 finishes mu / sigma /
// rho and the fed-back position.
#include <cuda.h>
#include <cuda_bf16.h>
#include <math_constants.h>

#include "common.cuh"

namespace tb2 {

constexpr int kGtBM = 128;
constexpr int kGtBN = 256;          // 64 units x 4 gates
constexpr int kGtBK = 64;
constexpr int kGtStages = 2;
constexpr int kGtThreads = 576;        // TMA warp, MMA warp, 16 epilogue warps (4 per TMEM lane quarter)
constexpr int kGtEpiThreads = 512;
constexpr int kGtH = 128;
constexpr uint32_t kGtABytes = kGtBM * kGtBK * 2;      // 16 KB
constexpr uint32_t kGtBBytes = kGtBN * kGtBK * 2;      // 32 KB
constexpr uint32_t kGtStageBytes = 2 * kGtABytes + 2 * kGtBBytes;   // 96 KB
constexpr uint32_t kGtTmemCols = 256;

__device__ __forceinline__ uint32_t g_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void g_mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void g_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void g_mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "G_WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra G_WAIT_DONE;\n"
        "bra G_WAIT_LOOP;\n"
        "G_WAIT_DONE:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void g_tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ uint64_t g_umma_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
__device__ __forceinline__ void g_umma(uint32_t tmem_d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "l"(a), "l"(b), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void g_umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void g_tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
// Gate non-linearities on the SFU (ex2.approx, ~2 ulp) -- the epilogue was bound by the ~200
// instructions per hidden unit of the libm-accurate expf / tanhf.  Absolute error ~1e-7 per
// activation, the same order as fp32 summation-order noise; parity is re-measured in the tests.
__device__ __forceinline__ float g_sigmoid(float x) { return __fdividef(1.f, 1.f + __expf(-x)); }
__device__ __forceinline__ float g_tanh(float x) { return 1.f - __fdividef(2.f, __expf(2.f * x) + 1.f); }

struct GateTcParams {
    const float2* obs1;
    const float2* obs2;
    const float* h_in;          // [M, 128] fp32 state before the step
    const float* c_in;
    float* h_out;
    float* c_out;
    const __nv_bfloat16* hs_in_hi;   // split of h_in (read through TMA; here only for masked copy-through)
    const __nv_bfloat16* hs_in_lo;
    __nv_bfloat16* hs_out_hi;   // [M, 128] split of h_out for the next step
    __nv_bfloat16* hs_out_lo;
    float* normal_out;          // [M, 5]
    float2* pos_out;            // [M] or null
    const float* bg;            // [512] b_ih + b_hh, original gate order
    const float* Wn;            // [5, 128]
    const float* bn;            // [5]
    int M, P;
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kGtThreads, 1)
lstm_gates_tc_kernel(const __grid_constant__ CUtensorMap map_emb_hi, const __grid_constant__ CUtensorMap map_emb_lo,
                     const __grid_constant__ CUtensorMap map_pool_hi, const __grid_constant__ CUtensorMap map_pool_lo,
                     const __grid_constant__ CUtensorMap map_h_hi, const __grid_constant__ CUtensorMap map_h_lo,
                     const __grid_constant__ CUtensorMap map_w_hi, const __grid_constant__ CUtensorMap map_w_lo,
                     GateTcParams p) {
    extern __shared__ __align__(1024) unsigned char smem_gt[];
    __shared__ __align__(8) uint64_t full_bar[kGtStages];
    __shared__ __align__(8) uint64_t empty_bar[kGtStages];
    __shared__ __align__(8) uint64_t tmem_full_bar;
    __shared__ uint32_t tmem_base_slot;
    __shared__ float wn_s[5][64];          // Hidden2Normal weights of this CTA's 64 units
    __shared__ float bg_s[4][64];          // fused gate bias of this CTA's units
    __shared__ float peer_part[kGtBM][5];  // rank 0: partial head sums received from rank 1
    __shared__ float part_s[4][kGtBM][5];  // per unit-group partial head sums of this CTA

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int rank = blockIdx.x;           // cluster rank == n-tile: units [64 rank, 64 rank + 64)
    const int m0 = blockIdx.y * kGtBM;
    const int kb_pool = p.P / kGtBK;       // k-blocks: [emb | pooled x kb_pool | h x 2]
    const int num_kb = 1 + kb_pool + 2;
    const uint32_t ring = (g_smem_u32(smem_gt) + 1023u) & ~1023u;

    for (int i = threadIdx.x; i < 5 * 64; i += kGtThreads) wn_s[i / 64][i % 64] = p.Wn[(i / 64) * kGtH + rank * 64 + (i % 64)];
    for (int i = threadIdx.x; i < 4 * 64; i += kGtThreads) bg_s[i / 64][i % 64] = p.bg[(i / 64) * kGtH + rank * 64 + (i % 64)];

    if (warp == 0 && lane == 0) {
        for (int s = 0; s < kGtStages; ++s) {
            g_mbar_init(g_smem_u32(&full_bar[s]), 1);
            g_mbar_init(g_smem_u32(&empty_bar[s]), 1);
        }
        g_mbar_init(g_smem_u32(&tmem_full_bar), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"(g_smem_u32(&tmem_base_slot)), "r"(kGtTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = tmem_base_slot;
    grid_dep_wait();          // embedding / pooled / state operands come from the previous kernels
    grid_dep_launch();
    // cluster barrier phase 1 (arrive now, wait before the first DSMEM access): a CTA may only
    // touch its peer's shared memory once the peer is known to be resident
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    bool waited_phase1 = false;

    float part[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
    bool row_valid = false, row_masked = true;
    int row = 0;

    if (warp == 0) {
        if (lane == 0) {
            for (int kb = 0; kb < num_kb; ++kb) {
                const int s = kb % kGtStages;
                const uint32_t phase = (kb / kGtStages) & 1;
                g_mbar_wait(g_smem_u32(&empty_bar[s]), phase ^ 1);
                const uint32_t bar = g_smem_u32(&full_bar[s]);
                const uint32_t base = ring + s * kGtStageBytes;
                g_mbar_expect_tx(bar, kGtStageBytes);
                const CUtensorMap *ahi, *alo;
                int ka;
                if (kb == 0) { ahi = &map_emb_hi; alo = &map_emb_lo; ka = 0; }
                else if (kb <= kb_pool) { ahi = &map_pool_hi; alo = &map_pool_lo; ka = (kb - 1) * kGtBK; }
                else { ahi = &map_h_hi; alo = &map_h_lo; ka = (kb - 1 - kb_pool) * kGtBK; }
                g_tma_load_2d(base, ahi, bar, ka, m0);
                g_tma_load_2d(base + kGtABytes, alo, bar, ka, m0);
                g_tma_load_2d(base + 2 * kGtABytes, &map_w_hi, bar, kb * kGtBK, rank * kGtBN);
                g_tma_load_2d(base + 2 * kGtABytes + kGtBBytes, &map_w_lo, bar, kb * kGtBK, rank * kGtBN);
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(kGtBN >> 3) << 17) |
                                   ((uint32_t)(kGtBM >> 4) << 24);
            for (int kb = 0; kb < num_kb; ++kb) {
                const int s = kb % kGtStages;
                const uint32_t phase = (kb / kGtStages) & 1;
                g_mbar_wait(g_smem_u32(&full_bar[s]), phase);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t base = ring + s * kGtStageBytes;
                const uint64_t a_hi = g_umma_desc(base);
                const uint64_t a_lo = g_umma_desc(base + kGtABytes);
                const uint64_t b_hi = g_umma_desc(base + 2 * kGtABytes);
                const uint64_t b_lo = g_umma_desc(base + 2 * kGtABytes + kGtBBytes);
#pragma unroll
                for (int k = 0; k < kGtBK / 16; ++k) {
                    const uint64_t adv = (uint64_t)((k * 16 * 2) >> 4);
                    g_umma(tmem_base, a_hi + adv, b_hi + adv, idesc, (kb | k) != 0);
                    g_umma(tmem_base, a_hi + adv, b_lo + adv, idesc, 1u);
                    g_umma(tmem_base, a_lo + adv, b_hi + adv, idesc, 1u);
                }
                g_umma_commit(g_smem_u32(&empty_bar[s]));
            }
            g_umma_commit(g_smem_u32(&tmem_full_bar));
        }
        __syncwarp();
    } else {
        const int q = warp & 3;              // TMEM lane quarter this warp may read
        const int ug = (warp - 2) >> 2;      // 16-unit slice of the CTA's 64 hidden units
        row = m0 + q * 32 + lane;
        row_valid = row < p.M;
        float2 o1 = make_float2(CUDART_NAN_F, CUDART_NAN_F), o2 = o1;
        if (row_valid) { o1 = p.obs1[row]; o2 = p.obs2[row]; }
        row_masked = isnan(o1.x) || isnan(o2.x);                             // lstm.py:118
        g_mbar_wait(g_smem_u32(&tmem_full_bar), 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
        // All MMAs have retired, so the operand ring is free: each epilogue warp stages its
        // [32 rows x 16 units] tiles of c and h there, so that global loads / stores run with
        // lanes along the unit dimension (8 rows x 64 B per instruction) instead of one row per lane.
        float* tile_h = reinterpret_cast<float*>(smem_gt + (ring - g_smem_u32(smem_gt))) + (size_t)(warp - 2) * (2 * 32 * 17);
        float* tile_c = tile_h + 32 * 17;
        const int rsub = lane >> 2, c4 = (lane & 3) * 4;
        const size_t col0 = (size_t)rank * 64 + ug * 16 + c4;
#pragma unroll
        for (int ps = 0; ps < 4; ++ps) {
            const int rl = ps * 8 + rsub;
            const int gr = m0 + q * 32 + rl;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (gr < p.M) v = *reinterpret_cast<const float4*>(p.c_in + (size_t)gr * kGtH + col0);
            float* t = tile_c + rl * 17 + c4;
            t[0] = v.x; t[1] = v.y; t[2] = v.z; t[3] = v.w;
        }
        __syncwarp();
        {
            const int u0 = ug * 16;
            uint32_t gi[16], gf[16], gg[16], go[16];
            g_tmem_ld16(trow + 0 * 64 + u0, gi);
            g_tmem_ld16(trow + 1 * 64 + u0, gf);
            g_tmem_ld16(trow + 2 * 64 + u0, gg);
            g_tmem_ld16(trow + 3 * 64 + u0, go);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            float* th = tile_h + lane * 17;
            float* tc = tile_c + lane * 17;
            if (row_valid && !row_masked) {
#pragma unroll
                for (int v = 0; v < 16; ++v) {
                    const int u = u0 + v;
                    const float ig = g_sigmoid(__uint_as_float(gi[v]) + bg_s[0][u]);
                    const float fg = g_sigmoid(__uint_as_float(gf[v]) + bg_s[1][u]);
                    const float gt = g_tanh(__uint_as_float(gg[v]) + bg_s[2][u]);
                    const float og = g_sigmoid(__uint_as_float(go[v]) + bg_s[3][u]);
                    const float cn = fg * tc[v] + ig * gt;
                    const float hn = og * g_tanh(cn);
                    tc[v] = cn;
                    th[v] = hn;
#pragma unroll
                    for (int o = 0; o < 5; ++o) part[o] = fmaf(hn, wn_s[o][u], part[o]);
                }
            } else if (row_valid) {
                // absent track: state copied through unchanged (lstm.py:158-166); tile_c already holds c_in
                const float* hin = p.h_in + (size_t)row * kGtH + rank * 64 + u0;
#pragma unroll
                for (int v = 0; v < 16; ++v) th[v] = hin[v];
            }
        }
        __syncwarp();
#pragma unroll
        for (int ps = 0; ps < 4; ++ps) {
            const int rl = ps * 8 + rsub;
            const int gr = m0 + q * 32 + rl;
            if (gr < p.M) {
                const float* sh = tile_h + rl * 17 + c4;
                const float* sc = tile_c + rl * 17 + c4;
                const float hv[4] = {sh[0], sh[1], sh[2], sh[3]};
                const size_t o = (size_t)gr * kGtH + col0;
                *reinterpret_cast<float4*>(p.h_out + o) = make_float4(hv[0], hv[1], hv[2], hv[3]);
                *reinterpret_cast<float4*>(p.c_out + o) = make_float4(sc[0], sc[1], sc[2], sc[3]);
                unsigned short hh[4], hl[4];
#pragma unroll
                for (int w = 0; w < 4; ++w) {
                    const __nv_bfloat16 h = __float2bfloat16_rn(hv[w]);
                    hh[w] = __bfloat16_as_ushort(h);
                    hl[w] = __bfloat16_as_ushort(__float2bfloat16_rn(hv[w] - __bfloat162float(h)));
                }
                *reinterpret_cast<uint2*>(p.hs_out_hi + o) =
                    make_uint2((uint32_t)hh[0] | ((uint32_t)hh[1] << 16), (uint32_t)hh[2] | ((uint32_t)hh[3] << 16));
                *reinterpret_cast<uint2*>(p.hs_out_lo + o) =
                    make_uint2((uint32_t)hl[0] | ((uint32_t)hl[1] << 16), (uint32_t)hl[2] | ((uint32_t)hl[3] << 16));
            }
        }
        // combine the four unit-groups of a row (fixed order: deterministic)
        {
            const int rl = q * 32 + lane;
#pragma unroll
            for (int o = 0; o < 5; ++o) part_s[ug][rl][o] = part[o];
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kGtEpiThreads) : "memory");
        if (ug == 0) {
            const int rl = q * 32 + lane;
#pragma unroll
            for (int o = 0; o < 5; ++o) part[o] = ((part_s[0][rl][o] + part_s[1][rl][o]) + part_s[2][rl][o]) + part_s[3][rl][o];
        }
        if (rank == 1 && ug == 0) {
            asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");     // phase 1: peer is resident
            waited_phase1 = true;
            // ship this half's head sums to rank 0 through distributed shared memory
            const int rl = q * 32 + lane;
            const uint32_t local = g_smem_u32(&peer_part[rl][0]);
            uint32_t remote;
            asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(local), "r"(0));
#pragma unroll
            for (int o = 0; o < 5; ++o)
                asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(remote + 4 * o), "f"(part[o]) : "memory");
        }
    }
    // cluster barrier phase 2: rank 1's partial sums are visible in rank 0's shared memory afterwards
    if (!waited_phase1) asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
    if (warp >= 2 && warp < 6 && rank == 0 && row_valid) {
        const int rl = (warp & 3) * 32 + lane;
        float* no = p.normal_out + (size_t)row * 5;
        if (row_masked) {
#pragma unroll
            for (int o = 0; o < 5; ++o) no[o] = CUDART_NAN_F;
            if (p.pos_out) p.pos_out[row] = make_float2(CUDART_NAN_F, CUDART_NAN_F);
        } else {
            float s[5];
#pragma unroll
            for (int o = 0; o < 5; ++o) s[o] = part[o] + peer_part[rl][o] + p.bn[o];
            const float n0 = s[0], n1 = s[1];
            no[0] = n0;
            no[1] = n1;
            no[2] = 0.01f + 0.2f * g_sigmoid(s[2]);                           // modules.py:60-62
            no[3] = 0.01f + 0.2f * g_sigmoid(s[3]);
            no[4] = 0.7f * g_sigmoid(s[4]);
            if (p.pos_out) {
                const float2 o2 = p.obs2[row];
                p.pos_out[row] = make_float2(o2.x + n0, o2.y + n1);          // lstm.py:232,255
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kGtTmemCols) : "memory");
    }
}

// ------------------------------------------------------------------------------------------
// producers of the split operands
// ------------------------------------------------------------------------------------------
// emb[M, 64] = cat(relu(W_e . (4 v) + b_e), 0, 0) as bf16 (hi, lo)   (modules.py:24-30)
__global__ void embed_split_kernel(const float2* __restrict__ obs1, const float2* __restrict__ obs2,
                                   const float* __restrict__ We, const float* __restrict__ be,
                                   __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo, int M, int E) {
    grid_dep_wait();
    grid_dep_launch();
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= M * E) return;
    const int m = idx / E, k = idx - m * E;
    const float2 a = obs1[m], b = obs2[m];
    float v = 0.f;
    if (k < E - 2 && !(isnan(a.x) || isnan(b.x))) {
        const float vx = (b.x - a.x) * 4.0f, vy = (b.y - a.y) * 4.0f;
        v = fmaxf(fmaf(We[2 * k + 1], vy, fmaf(We[2 * k], vx, be[k])), 0.f);
    }
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    hi[idx] = h;
    lo[idx] = __float2bfloat16_rn(v - __bfloat162float(h));
}

__global__ void split_rows_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ hi,
                                  __nv_bfloat16* __restrict__ lo, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const float v = src[i];
        const __nv_bfloat16 h = __float2bfloat16_rn(v);
        hi[i] = h;
        lo[i] = __float2bfloat16_rn(v - __bfloat162float(h));
    }
}

// W_cat[n][k] = [W_ih | W_hh] with rows permuted to (rank, gate, unit) order, as bf16 (hi, lo)
__global__ void repack_gates_tc_kernel(const float* __restrict__ w_ih, const float* __restrict__ w_hh,
                                       __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo,
                                       int in_dim, int H) {
    const int K = in_dim + H;
    size_t total = (size_t)4 * H * K;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (size_t)gridDim.x * blockDim.x) {
        const int k = (int)(idx % K);
        const int n = (int)(idx / K);                 // permuted row: rank * 256 + gate * 64 + ul
        const int rank = n / 256, gate = (n % 256) / 64, ul = n % 64;
        const int src = gate * H + rank * 64 + ul;    // original gate column
        const float v = k < in_dim ? w_ih[(size_t)src * in_dim + k] : w_hh[(size_t)src * H + (k - in_dim)];
        const __nv_bfloat16 h = __float2bfloat16_rn(v);
        hi[idx] = h;
        lo[idx] = __float2bfloat16_rn(v - __bfloat162float(h));
    }
}

int make_bf16_tile_map(CUtensorMap* map, const void* base, int rows, int cols, int box_rows);

bool gates_tc_supported(const tb2_lstm* m) {
    if (m->H != kGtH || m->E != 64) return false;
    if (m->cfg.pool_type != TB2_POOL_NONE && !m->cfg.pool_to_input) return false;
    if (m->P % kGtBK != 0) return false;
    return true;
}

int launch_repack_gates_tc(const float* w_ih, const float* w_hh, void* hi, void* lo, int in_dim, int H,
                           cudaStream_t st) {
    repack_gates_tc_kernel<<<512, 256, 0, st>>>(w_ih, w_hh, (__nv_bfloat16*)hi, (__nv_bfloat16*)lo, in_dim, H);
    TB2_LAUNCH_CHECK();
    return TB2_OK;
}

int launch_embed_split(const tb2_lstm* m, int M, const float* obs1, const float* obs2, void* hi, void* lo,
                       cudaStream_t st) {
    const int total = M * m->E;
    {
        KernelTimer kt("embed_split", st);
        launch_pdl(embed_split_kernel, dim3((total + 255) / 256), dim3(256), 0, st, (const float2*)obs1,
                   (const float2*)obs2, (const float*)m->We, (const float*)m->be, (__nv_bfloat16*)hi,
                   (__nv_bfloat16*)lo, M, m->E);
    }
    TB2_LAUNCH_CHECK();
    return TB2_OK;
}

int launch_split_rows(const float* src, void* hi, void* lo, size_t n, cudaStream_t st) {
    split_rows_kernel<<<256, 256, 0, st>>>(src, (__nv_bfloat16*)hi, (__nv_bfloat16*)lo, n);
    TB2_LAUNCH_CHECK();
    return TB2_OK;
}

int launch_gates_tc(const tb2_lstm* m, const tb2_layout* l, int phase, const float* obs1, const float* obs2,
                    const void* emb_hi, const void* emb_lo, const void* pool_hi, const void* pool_lo,
                    const void* hs_in_hi, const void* hs_in_lo, void* hs_out_hi, void* hs_out_lo,
                    const float* h_in, const float* c_in, float* h_out, float* c_out, float* normal_out,
                    float* pos_out, cudaStream_t st) {
    const int M = l->M;
    CUtensorMap me_hi, me_lo, mp_hi, mp_lo, mh_hi, mh_lo, mw_hi, mw_lo;
    int rc;
    if ((rc = make_bf16_tile_map(&me_hi, emb_hi, M, 64, kGtBM))) return rc;
    if ((rc = make_bf16_tile_map(&me_lo, emb_lo, M, 64, kGtBM))) return rc;
    if (m->P > 0) {
        if ((rc = make_bf16_tile_map(&mp_hi, pool_hi, M, m->P, kGtBM))) return rc;
        if ((rc = make_bf16_tile_map(&mp_lo, pool_lo, M, m->P, kGtBM))) return rc;
    } else {
        mp_hi = me_hi;
        mp_lo = me_lo;
    }
    if ((rc = make_bf16_tile_map(&mh_hi, hs_in_hi, M, kGtH, kGtBM))) return rc;
    if ((rc = make_bf16_tile_map(&mh_lo, hs_in_lo, M, kGtH, kGtBM))) return rc;
    if ((rc = make_bf16_tile_map(&mw_hi, m->Wg_hi[phase], 4 * kGtH, m->K_gate, kGtBN))) return rc;
    if ((rc = make_bf16_tile_map(&mw_lo, m->Wg_lo[phase], 4 * kGtH, m->K_gate, kGtBN))) return rc;
    GateTcParams p;
    p.obs1 = (const float2*)obs1;
    p.obs2 = (const float2*)obs2;
    p.h_in = h_in; p.c_in = c_in; p.h_out = h_out; p.c_out = c_out;
    p.hs_in_hi = (const __nv_bfloat16*)hs_in_hi; p.hs_in_lo = (const __nv_bfloat16*)hs_in_lo;
    p.hs_out_hi = (__nv_bfloat16*)hs_out_hi; p.hs_out_lo = (__nv_bfloat16*)hs_out_lo;
    p.normal_out = normal_out;
    p.pos_out = (float2*)pos_out;
    p.bg = m->bg[phase];
    p.Wn = m->Wn;
    p.bn = m->bn;
    p.M = M;
    p.P = m->P;
    const size_t smem = (size_t)kGtStages * kGtStageBytes + 1024;
    static DynSmemConfig configured;
    TB2_CHECK_CUDA(configured.ensure(lstm_gates_tc_kernel, smem));
    dim3 grid(2, (M + kGtBM - 1) / kGtBM);
    {
        KernelTimer kt("lstm_gates_tc", st);
        launch_pdl(lstm_gates_tc_kernel, grid, dim3(kGtThreads), smem, st, me_hi, me_lo, mp_hi, mp_lo, mh_hi, mh_lo,
                   mw_hi, mw_lo, p);
    }
    TB2_LAUNCH_CHECK();
    return TB2_OK;
}

}  // namespace tb2
