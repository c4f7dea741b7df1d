// Grid pooling: neighbour binning, last-writer-wins scatter, sparse grid-embedding layer.
//
// Replaces GridBasedPooling.{occupancies,directional,social,occupancy} and the first Linear of
// the grid embedding (reference: trajnetbaselines/lstm/gridbased_pooling.py:112-170,227-305,
// 308-335).  The reference materialises a dense [B*N, C, n, n] grid (84 MB per step for
// Social-LSTM at B=256) of which <= N-1 cells per pedestrian are non-constant; here the grid
// never exists: pool_prepare_kernel resolves the scatter-overwrite into a per-pedestrian list
// of winning (cell, neighbour) pairs, and sparse_layer1_kernel applies the first Linear as
//     out[i, :] = base + sum_{winning (cell, j) of i} (val(i, j) - constant) . W1[:, cell-slab]
// streaming the cell-major weight slabs once per scene group.
#include <cuda_bf16.h>
#include <math_constants.h>
#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "common.cuh"

namespace tb2 {

// ------------------------------------------------------------------------------------------
// resolve_obs: decoder input rule (lstm.py:240-250) -- rows of the scene primaries come from
// the previous predictions, everything else from the teacher-forcing / observed frame.
// ------------------------------------------------------------------------------------------
__global__ void resolve_obs_kernel(const float2* __restrict__ base, const float2* __restrict__ pred,
                                   const int* __restrict__ row_scene,
                                   const int* __restrict__ scene_off, float2* __restrict__ out, int M) {
    grid_dep_wait();
    grid_dep_launch();
    int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= M) return;
    bool primary = (scene_off[row_scene[m]] == m);
    out[m] = primary ? pred[m] : base[m];
}

int launch_resolve_obs(const tb2_layout* l, const float* base, const float* pred, float* out,
                       cudaStream_t st) {
    int threads = 256, blocks = (l->M + threads - 1) / threads;
    {
        KernelTimer kt("resolve_obs", st);
        launch_pdl(resolve_obs_kernel, dim3(blocks), dim3(threads), 0, st, (const float2*)base, (const float2*)pred,
                   (const int*)l->row_scene, (const int*)l->scene_off, (float2*)out, l->M);
    }
    TB2_LAUNCH_CHECK();
    return TB2_OK;
}

// ------------------------------------------------------------------------------------------
// pool_prepare: one CTA per scene.
//   * positions: NaN -> -500 (gridbased_pooling.py:248-249)
//   * social: lat[j] = W_enc . nan_to_num(h_j) + b_enc (:160-167; computed once per j, the
//     reference recomputes it for each of the N-1 observers)
//   * every ordered pair (i, jj): cell index with fp32 true division (:276), range test
//     (:278-279), out-of-range -> cell 0 (:281)
//   * scatter-overwrite in ascending j (:293) resolved to "is this pair the last writer of its
//     cell"; padded slots (scene smaller than the batch maximum) are trailing out-of-range
//     writers of cell 0 exactly like the reference's NaN padding (lstm.py:31-40).
// ------------------------------------------------------------------------------------------
// One warp per pedestrian of the scene (latent projection, then the row of winners), between 8 and 20 warps: two CTAs
// of 640 threads per SM need <= 51 registers per thread.  (The kernel is instruction-issue bound: ncu round 2 showed
// 1800 instructions per warp at 8 cycles each with 8 warps per scene.)
constexpr int kPrepMaxThreads = 640;
static int prep_threads(int n_max) { return 32 * std::min(std::max(n_max, 8), kPrepMaxThreads / 32); }
constexpr int kMaxSceneForPrep = 256;   // per-warp cell row buffer

struct PrepParams {
    const float2* obs1;
    const float2* obs2;
    const float* hidden;      // [M, H] or null
    const int* scene_off;
    const float* WencT;       // [H, C]
    const float* benc;
    float* lat;               // [M, C]
    int* win_count;
    uint32_t* win_ent;
    float* win_val;
    int* pair_cell;
    uint8_t* pair_flag;
    uint8_t* cell_row;        // [M, n * n] per-row cell map for sparse_layer1_pair (or null)
    const float* We;          // input embedding (fused producer of the gate kernel's emb operand)
    const float* be;
    __nv_bfloat16* emb_hi;    // [M, E] bf16 split or null
    __nv_bfloat16* emb_lo;
    int E;
    int n_max, H, C, n, pool_type, front, skip_masked, write_pairs, pad_to_max;
    float side, width;
};

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

__device__ __forceinline__ float nan_to_num_f(float x) {
    if (isnan(x)) return 0.f;
    if (isinf(x)) return x > 0 ? 3.402823466e+38f : -3.402823466e+38f;
    return x;
}

__global__ void __launch_bounds__(kPrepMaxThreads, 2) pool_prepare_kernel(PrepParams p) {
    const int kPrepThreads = (int)blockDim.x, kPrepWarps = kPrepThreads >> 5;
    extern __shared__ __align__(16) float smem_prep[];
    const int scene = blockIdx.x;
    const int row0 = p.scene_off[scene];
    const int n_s = p.scene_off[scene + 1] - row0;
    const int nm1 = p.n_max - 1;
    float2* pos = reinterpret_cast<float2*>(smem_prep);                 // [n_s] obs2 with -500
    float2* vel = pos + n_s;                                            // [n_s] obs2 - obs1 (may be NaN)
    int* cellrow = reinterpret_cast<int*>(vel + n_s);                   // [kPrepWarps][nm1]
    float* Ws = reinterpret_cast<float*>(cellrow + ((kPrepWarps * (nm1 > 0 ? nm1 : 1) + 3) & ~3));   // 16-byte aligned (social)
    float* hs = Ws + (p.H + 8) * p.C;                                   // [n_s][H] (social); Ws: see the two layouts below
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // social, 16 latent channels of a 128-wide state (the BASELINE configuration): lat on a (4 channels x 16 k) register
    // tile per lane, weights [k][c] staged once (they do not depend on the previous kernel: requested before the wait)
    const bool social = p.pool_type == TB2_POOL_SOCIAL;
    const bool fast_lat = social && p.C == 16 && p.H == 128;
    if (fast_lat) {
        // Ws: 8 blocks of 16 k rows x 16 channels, block stride 272 floats (staggers the banks of the 8 k-slices)
        for (int idx = tid; idx < 128 * 4; idx += kPrepThreads) {
            const int k = idx >> 2, q4 = idx & 3;
            cp_async16(Ws + (k >> 4) * 272 + (k & 15) * 16 + q4 * 4, p.WencT + k * 16 + q4 * 4);
        }
    } else if (social) {
        // W_enc in [C][H] order (k contiguous) so the dot products below run on float4 pairs
        for (int idx = tid; idx < p.H * p.C; idx += kPrepThreads) {
            const int k = idx / p.C, c = idx - k * p.C;          // WencT is [H][C]: coalesced read
            Ws[c * (p.H + 4) + k] = p.WencT[idx];                // row stride H + 4: 2-way instead of 16-way conflicts
        }
    }
    grid_dep_wait();          // obs / hidden state come from the previous kernels of the stream
    grid_dep_launch();

    if (fast_lat) {           // raw rows (nan_to_num is applied where they are read), asynchronously
        const float* hsrc = p.hidden + (size_t)row0 * 128;
        for (int idx = tid; idx < n_s * 32; idx += kPrepThreads) cp_async16(hs + idx * 4, hsrc + idx * 4);
    }
    cp_async_commit();
    for (int j = tid; j < n_s; j += kPrepThreads) {
        float2 a = p.obs1[row0 + j], b = p.obs2[row0 + j];
        vel[j] = make_float2(b.x - a.x, b.y - a.y);
        if (isnan(b.x) || isnan(b.y)) b = make_float2(-500.f, -500.f);
        pos[j] = b;
    }
    if (social && !fast_lat) {
        // stage nan_to_num(h) of the scene in shared memory (coalesced float4 loads)
        const float4* hsrc = reinterpret_cast<const float4*>(p.hidden + (size_t)row0 * p.H);
        float4* hdst = reinterpret_cast<float4*>(hs);
        for (int idx = tid; idx < n_s * p.H / 4; idx += kPrepThreads) {
            float4 v = hsrc[idx];
            v.x = nan_to_num_f(v.x); v.y = nan_to_num_f(v.y); v.z = nan_to_num_f(v.z); v.w = nan_to_num_f(v.w);
            hdst[idx] = v;
        }
    }
    cp_async_wait_all();
    __syncthreads();
    if (p.emb_hi != nullptr) {
        // emb = cat(relu(W_e . (4 v) + b_e), 0, 0) (modules.py:24-30) as bf16 (hi, lo) for the gate GEMM
        const int e_shift = (p.E & (p.E - 1)) == 0 ? 31 - __clz(p.E) : -1;       // E = 64: no integer division per element
        for (int idx = tid; idx < n_s * p.E; idx += kPrepThreads) {
            const int j = e_shift >= 0 ? idx >> e_shift : idx / p.E, k = idx - j * p.E;
            const float2 v = vel[j];
            float e = 0.f;
            if (k < p.E - 2 && !isnan(v.x))
                e = fmaxf(fmaf(p.We[2 * k + 1], v.y * 4.0f, fmaf(p.We[2 * k], v.x * 4.0f, p.be[k])), 0.f);
            const __nv_bfloat16 h = __float2bfloat16_rn(e);
            p.emb_hi[(size_t)(row0 + j) * p.E + k] = h;
            p.emb_lo[(size_t)(row0 + j) * p.E + k] = __float2bfloat16_rn(e - __bfloat162float(h));
        }
    }
    if (fast_lat) {
        // lat[j][c] = sum_k nan_to_num(h[j][k]) * WencT[k][c] + benc[c]: one warp per pedestrian, lane = (4 channels,
        // 16-wide k slice); the slice sums are added across the 8 slices by an xor tree (fixed order)
        const int c4 = lane & 3, kq = lane >> 2;
        const float4* wp = reinterpret_cast<const float4*>(Ws + kq * 272) + c4;
        const float4 bc = *reinterpret_cast<const float4*>(p.benc + c4 * 4);
        for (int j = warp; j < n_s; j += kPrepWarps) {
            const float4* hp = reinterpret_cast<const float4*>(hs + j * 128 + kq * 16);
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                float4 hv = hp[q];
                // nan_to_num only where a value is not finite (exponent all ones): one test per four values
                const uint32_t m = max(max(__float_as_uint(hv.x) & 0x7fffffffu, __float_as_uint(hv.y) & 0x7fffffffu),
                                       max(__float_as_uint(hv.z) & 0x7fffffffu, __float_as_uint(hv.w) & 0x7fffffffu));
                if (m >= 0x7f800000u) {
                    hv.x = nan_to_num_f(hv.x); hv.y = nan_to_num_f(hv.y); hv.z = nan_to_num_f(hv.z); hv.w = nan_to_num_f(hv.w);
                }
                const float hk[4] = {hv.x, hv.y, hv.z, hv.w};
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float4 w = wp[(4 * q + i) * 4];
                    acc.x = fmaf(hk[i], w.x, acc.x); acc.y = fmaf(hk[i], w.y, acc.y);
                    acc.z = fmaf(hk[i], w.z, acc.z); acc.w = fmaf(hk[i], w.w, acc.w);
                }
            }
#pragma unroll
            for (int off = 4; off < 32; off <<= 1) {
                acc.x += __shfl_xor_sync(0xffffffffu, acc.x, off); acc.y += __shfl_xor_sync(0xffffffffu, acc.y, off);
                acc.z += __shfl_xor_sync(0xffffffffu, acc.z, off); acc.w += __shfl_xor_sync(0xffffffffu, acc.w, off);
            }
            if (kq == 0)
                *reinterpret_cast<float4*>(p.lat + (size_t)(row0 + j) * 16 + c4 * 4) =
                    make_float4(acc.x + bc.x, acc.y + bc.y, acc.z + bc.z, acc.w + bc.w);
        }
    } else if (social) {
        // lat[j][c] = sum_k nan_to_num(h[j][k]) * WencT[k][c] + benc[c]
        const int total = n_s * p.C;
        for (int idx = tid; idx < total; idx += kPrepThreads) {
            int j = idx / p.C, c = idx - j * p.C;
            const float4* hrow = reinterpret_cast<const float4*>(hs + j * p.H);
            const float4* wrow = reinterpret_cast<const float4*>(Ws + c * (p.H + 4));
            float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;      // 4 independent chains (sum order fixed)
#pragma unroll 4
            for (int k4 = 0; k4 < p.H / 4; ++k4) {
                const float4 hv = hrow[k4], wv = wrow[k4];
                a0 = fmaf(hv.x, wv.x, a0); a1 = fmaf(hv.y, wv.y, a1);
                a2 = fmaf(hv.z, wv.z, a2); a3 = fmaf(hv.w, wv.w, a3);
            }
            p.lat[(size_t)(row0 + j) * p.C + c] = ((a0 + a1) + (a2 + a3)) + p.benc[c];
        }
    }
    if (nm1 <= 0) {   // single-pedestrian batch: constant grid (gridbased_pooling.py:252-253)
        for (int i = tid; i < n_s; i += kPrepThreads) p.win_count[row0 + i] = 0;
        if (p.cell_row)
            for (int idx = tid; idx < n_s * p.n * p.n; idx += kPrepThreads) p.cell_row[(size_t)row0 * p.n * p.n + idx] = 0xffu;
        return;
    }

    const float offx = p.width * 0.5f;
    const float offy = p.front ? 0.f : p.width * 0.5f;
    int* myrow = cellrow + warp * nm1;

    for (int i = warp; i < n_s; i += kPrepWarps) {
        const size_t gi = (size_t)(row0 + i) * nm1;
        const float2 pi = pos[i];
        const float2 vi = vel[i];
        // pass 1: cell index of every neighbour slot (padded slots are out of range)
        for (int jj = lane; jj < nm1; jj += 32) {
            int j = jj + (jj >= i);
            int cell = 0, inr = 0;
            if (!p.pad_to_max && j >= n_s) {      // per-scene semantics: the slot does not exist at all
                myrow[jj] = -100;
                if (p.write_pairs) {
                    p.pair_cell[gi + jj] = 0;
                    p.pair_flag[gi + jj] = 0;
                }
                continue;
            }
            {
                // padded slots (j >= n_s) are NaN rows in the reference's padded batch -> -500
                const float2 pj = (j < n_s) ? pos[j] : make_float2(-500.f, -500.f);
                float rx = pj.x - pi.x, ry = pj.y - pi.y;
                float ox = __fadd_rn(__fdiv_rn(rx, p.side), offx);      // fp32 true division, :276
                float oy = __fadd_rn(__fdiv_rn(ry, p.side), offy);
                bool viol = (ox < 0.f) || (ox >= p.width) || (oy < 0.f) || (oy >= p.width);
                if (!viol) {
                    inr = 1;
                    cell = (int)ox * p.n + (int)oy;                     // :284-287
                }
            }
            myrow[jj] = inr ? cell : -1;
            if (p.write_pairs) {      // debug export (tb2_grid_indices) only
                p.pair_cell[gi + jj] = cell;
                p.pair_flag[gi + jj] = (uint8_t)inr;
            }
        }
        __syncwarp();
        // pass 2: winners, compacted in ascending jj
        const bool masked = isnan(vi.x);      // obs2 - obs1 is NaN iff the track is absent at either frame
        int count = 0;
        uint8_t* crow = p.cell_row ? p.cell_row + (size_t)(row0 + i) * (p.n * p.n) : nullptr;
        if (crow) {       // all cells empty, winners marked below (same warp: ordered by the __syncwarp)
            for (int c = lane * 4; c < p.n * p.n; c += 128) *reinterpret_cast<uint32_t*>(crow + c) = 0xffffffffu;
            __syncwarp();
        }
        if (!(p.skip_masked && masked)) {
            for (int base = 0; base < nm1; base += 32) {
                int jj = base + lane;
                bool win = false;
                int cell = 0;
                // a later in-range writer of the same cell, or (for cell 0) any later out-of-range
                // writer incl. padding, overrides this pair.  Within the 32-slot chunk this is one
                // warp match; only scenes with more than 33 pedestrians need the loop over later chunks.
                cell = (jj < nm1) ? myrow[jj] : -2 - lane;                 // inactive lanes: unique keys
                const unsigned same = __match_any_sync(0xffffffffu, cell);
                const unsigned oor = __ballot_sync(0xffffffffu, jj < nm1 && cell == -1);
                const unsigned later = lane == 31 ? 0u : (0xffffffffu << (lane + 1));
                win = jj < nm1 && cell >= 0 && (same & later) == 0u && !(cell == 0 && (oor & later) != 0u);
                for (int k = base + 32; win && k < nm1; ++k) {
                    int ck = myrow[k];
                    if (ck == cell || (cell == 0 && ck == -1)) win = false;
                }
                unsigned ball = __ballot_sync(0xffffffffu, win);
                if (win) {
                    int slot = count + __popc(ball & ((1u << lane) - 1u));
                    int j = jj + (jj >= i);
                    // a padded slot can only win in the (discarded) row of an absent pedestrian
                    p.win_ent[gi + slot] = ((uint32_t)cell << 16) | (uint32_t)(j < n_s ? j : 0xffff);
                    if (crow) crow[cell] = (uint8_t)(j < n_s ? j : 0xfe);
                    if (p.pool_type == TB2_POOL_DIRECTIONAL) {
                        const float2 vj = (j < n_s) ? vel[j] : make_float2(CUDART_NAN_F, CUDART_NAN_F);
                        p.win_val[(gi + slot) * 2 + 0] = nan_to_num_f(vj.x - vi.x);      // :131-140
                        p.win_val[(gi + slot) * 2 + 1] = nan_to_num_f(vj.y - vi.y);
                    } else if (p.pool_type == TB2_POOL_OCCUPANCY) {
                        p.win_val[(gi + slot) * 2 + 0] = 1.f;                             // :266-267
                    }
                }
                count += __popc(ball);
            }
        }
        if (lane == 0) p.win_count[row0 + i] = count;
        __syncwarp();
    }
}

int launch_pool_prepare(const tb2_lstm* m, const tb2_layout* l, const float* hidden,
                        const float* obs1, const float* obs2, int skip_masked, int write_pairs,
                        int write_emb, Workspace* ws, cudaStream_t st) {
    TB2_REQUIRE(l->n_max <= kMaxSceneForPrep, "scene larger than 256 pedestrians");
    PrepParams p;
    p.obs1 = (const float2*)obs1;
    p.obs2 = (const float2*)obs2;
    p.hidden = hidden;
    p.scene_off = l->scene_off;
    p.WencT = m->WencT;
    p.benc = m->benc;
    p.lat = ws->lat;
    p.win_count = ws->win_count;
    p.win_ent = ws->win_ent;
    p.win_val = ws->win_val;
    p.pair_cell = ws->pair_cell;
    p.pair_flag = ws->pair_flag;
    // the cell map is written as 32-bit words: n * n must be a multiple of 4 (the pair kernel asks for 16)
    p.cell_row = (m->cfg.pool_type == TB2_POOL_SOCIAL && (m->cfg.n * m->cfg.n) % 16 == 0 && l->n_max <= 0xFD) ? ws->cell_row : nullptr;
    p.n_max = l->n_max;
    p.H = m->H;
    p.C = m->C;
    p.n = m->cfg.n;
    p.pool_type = m->cfg.pool_type;
    p.front = m->cfg.front;
    p.skip_masked = skip_masked;
    p.pad_to_max = l->pad_to_max;
    p.write_pairs = write_pairs;
    p.We = m->We;
    p.be = m->be;
    p.E = m->E;
    p.emb_hi = write_emb ? (__nv_bfloat16*)ws->emb_hi : nullptr;
    p.emb_lo = write_emb ? (__nv_bfloat16*)ws->emb_lo : nullptr;
    p.side = m->cfg.cell_side;        // pool_size == 1
    p.width = (float)m->cfg.n;
    int nm1 = l->n_max > 1 ? l->n_max - 1 : 1;
    const int nthreads = prep_threads(l->n_max);
    size_t smem = (size_t)l->n_max * 2 * sizeof(float2) + (size_t)(((nthreads / 32) * nm1 + 3) & ~3) * sizeof(int);
    if (m->cfg.pool_type == TB2_POOL_SOCIAL) smem += ((size_t)(m->H + 8) * m->C + (size_t)l->n_max * m->H) * sizeof(float);
    smem = (smem + 15) & ~(size_t)15;
    static DynSmemConfig configured;
    TB2_REQUIRE(smem <= 227 * 1024, "scene too large for pool_prepare shared memory");
    TB2_CHECK_CUDA(configured.ensure(pool_prepare_kernel, smem, 48 * 1024));
    {
        KernelTimer kt("pool_prepare", st);
        launch_pdl(pool_prepare_kernel, dim3(l->B), dim3(nthreads), smem, st, p);
    }
    TB2_LAUNCH_CHECK();
    return TB2_OK;
}

// Debug export (tb2_grid_indices): copy of the pair tables.
__global__ void copy_pairs_kernel(const int* __restrict__ cell, const uint8_t* __restrict__ flag,
                                  int32_t* __restrict__ cell_out, uint8_t* __restrict__ flag_out,
                                  size_t total) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < total) {
        cell_out[i] = cell[i];
        flag_out[i] = flag[i];
    }
}

int launch_grid_indices_copy(const tb2_layout* l, const Workspace* ws, int32_t* cell_out,
                             uint8_t* flag_out, cudaStream_t st) {
    size_t total = (size_t)l->M * (size_t)(l->n_max - 1);
    if (total == 0) return TB2_OK;
    int threads = 256;
    unsigned blocks = (unsigned)((total + threads - 1) / threads);
    copy_pairs_kernel<<<blocks, threads, 0, st>>>(ws->pair_cell, ws->pair_flag, cell_out, flag_out, total);
    TB2_LAUNCH_CHECK();
    return TB2_OK;
}

// ------------------------------------------------------------------------------------------
// dense grid writer (embedding_arch == 'None'): [M, C*cells], channel-major like
// gridbased_pooling.py:294-295,107.  One CTA per pedestrian.
// ------------------------------------------------------------------------------------------
__global__ void dense_grid_kernel(const int* __restrict__ win_count, const uint32_t* __restrict__ win_ent,
                                  const float* __restrict__ win_val, const float* __restrict__ lat,
                                  const int* __restrict__ row_scene, const int* __restrict__ scene_off,
                                  const float* __restrict__ benc, float* __restrict__ out, int C,
                                  int cells, int nm1, float constant, int pool_type) {
    const int m = blockIdx.x;
    float* row = out + (size_t)m * C * cells;
    for (int k = threadIdx.x; k < C * cells; k += blockDim.x) row[k] = constant;
    __syncthreads();
    const int cnt = win_count[m];
    const int row0 = scene_off[row_scene[m]];
    for (int idx = threadIdx.x; idx < cnt * C; idx += blockDim.x) {
        int e = idx / C, c = idx - e * C;
        uint32_t ent = win_ent[(size_t)m * nm1 + e];
        int cell = ent >> 16, j = ent & 0xffff;
        float v;
        if (pool_type == TB2_POOL_SOCIAL) v = (j == 0xffff) ? benc[c] : lat[(size_t)(row0 + j) * C + c];
        else v = win_val[((size_t)m * nm1 + e) * 2 + c];
        row[c * cells + cell] = v;
    }
}

// ------------------------------------------------------------------------------------------
// sparse_layer1: first Linear of the grid embedding on the winner lists.
//   grid  = (scene groups, OUT / 256 column chunks), 512 threads: thread = (half, column)
//   smem  = acc[P][256] | lat[P][C] (social) | bucket tables | entries sorted by cell
//   The CTA walks the cells in ascending order; the C x 256 weight slab of the next cell is
//   prefetched into registers while the pairs binned in the current cell are applied.  Pairs are
//   binned by (cell, parity of the pedestrian row): half h of the CTA only ever updates
//   accumulator rows of parity h, so the two halves need no synchronisation while they drift
//   apart across cells, every row is accumulated in ascending cell order by one thread per
//   column, and the result is deterministic.
// ------------------------------------------------------------------------------------------
constexpr int kL1Cols = 256;
constexpr int kL1Threads = 512;

struct L1Params {
    const int* group_off;     // [G+1] scene indices
    const int* scene_off;
    const int* win_count;
    const uint32_t* win_ent;
    const float* win_val;
    const float* lat;
    const float* benc;        // [C] (social): lat of a NaN-padded slot
    const float* Wt;          // [cells, C, OUT]
    const float* base;        // [OUT]
    float* out;               // [M, OUT] fp32, or null when the split outputs below are used
    __nv_bfloat16* out_hi;    // [M, OUT] bf16 (hi, lo) split for the tensor-core layer that follows
    __nv_bfloat16* out_lo;
    int OUT, cells, nm1, cap, relu;
    float constant;
};

template <int C, bool SOCIAL>
__global__ void __launch_bounds__(kL1Threads, 1) sparse_layer1_kernel(L1Params p) {
    extern __shared__ __align__(16) unsigned char smem_l1[];
    const int tid = threadIdx.x;
    const int colc = tid & (kL1Cols - 1);
    const int half = tid >> 8;
    const int col = blockIdx.y * kL1Cols + colc;
    const bool col_ok = col < p.OUT;
    const int s0 = p.group_off[blockIdx.x], s1 = p.group_off[blockIdx.x + 1];
    const int row0 = p.scene_off[s0];
    const int P = p.scene_off[s1] - row0;

    float* acc = reinterpret_cast<float*>(smem_l1);                       // [cap][256]
    float* latS = acc + (size_t)p.cap * kL1Cols;                          // [cap + 1][C] (social)
    const int bins = 2 * p.cells;                                         // bin = cell * 2 + (row & 1)
    int* start = reinterpret_cast<int*>(latS + (SOCIAL ? (size_t)(p.cap + 1) * C : 0));   // [bins+1]
    int* cursor = start + bins + 1;                                       // [bins]
    uint16_t* entP = reinterpret_cast<uint16_t*>(cursor + bins);          // [cap*nm1]
    uint16_t* entS = entP + (size_t)p.cap * p.nm1;                        // [cap*nm1] (social)
    float* entV = reinterpret_cast<float*>(                               // [cap*nm1][C] (non-social)
        reinterpret_cast<unsigned char*>(entP) +
        (((size_t)p.cap * p.nm1 * 2 * sizeof(uint16_t) + 15) & ~(size_t)15));
    uint32_t* raw = reinterpret_cast<uint32_t*>(entV + (SOCIAL ? 0 : (size_t)p.cap * p.nm1 * C));   // [cap*nm1]
    int* cnt_s = reinterpret_cast<int*>(raw + (size_t)p.cap * p.nm1);    // [cap]
    int* sbase = cnt_s + p.cap;                                           // [cap]

    for (int c = tid; c < bins; c += kL1Threads) cursor[c] = 0;
    // one coalesced pass over the group's winner lists (rows of a group are contiguous in memory)
    for (int r = tid; r < P; r += kL1Threads) cnt_s[r] = p.win_count[row0 + r];
    {
        const uint32_t* src = p.win_ent + (size_t)row0 * p.nm1;
        for (int idx = tid; idx < P * p.nm1; idx += kL1Threads) raw[idx] = src[idx];
    }
    for (int sb = s0 + (tid >> 5); sb < s1; sb += kL1Threads / 32) {
        const int a = p.scene_off[sb] - row0, b2 = p.scene_off[sb + 1] - row0;
        for (int r = a + (tid & 31); r < b2; r += 32) sbase[r] = a;
    }
    if (SOCIAL) {
        for (int idx = tid; idx < P * C; idx += kL1Threads) latS[idx] = p.lat[(size_t)row0 * C + idx] - p.constant;
        if (tid < C) latS[(size_t)p.cap * C + tid] = p.benc[tid] - p.constant;   // row `cap`: padded slot
    }
    const float b = col_ok ? p.base[col] : 0.f;
    for (int r = half; r < P; r += 2) acc[r * kL1Cols + colc] = b;
    __syncthreads();
    // histogram of winners per cell
    const int total = P * p.nm1;
    for (int idx = tid; idx < total; idx += kL1Threads) {
        int r = idx / p.nm1, k = idx - r * p.nm1;
        if (k < cnt_s[r]) atomicAdd(&cursor[(raw[idx] >> 16) * 2 + (r & 1)], 1);
    }
    __syncthreads();
    if (tid < 32) {   // exclusive scan of the histogram by one warp
        int per = (bins + 31) / 32;
        int lo = tid * per, hi = min(lo + per, bins);
        int sum = 0;
        for (int c = lo; c < hi; ++c) sum += cursor[c];
        int incl = sum;
        for (int d = 1; d < 32; d <<= 1) {
            int v = __shfl_up_sync(0xffffffffu, incl, d);
            if (tid >= d) incl += v;
        }
        int run = incl - sum;
        for (int c = lo; c < hi; ++c) {
            int cnt = cursor[c];
            start[c] = run;
            cursor[c] = run;
            run += cnt;
        }
        if (tid == 31) start[bins] = incl;
    }
    __syncthreads();
    for (int idx = tid; idx < total; idx += kL1Threads) {
        int r = idx / p.nm1, k = idx - r * p.nm1;
        if (k < cnt_s[r]) {
            size_t g = (size_t)(row0 + r) * p.nm1 + k;
            uint32_t ent = raw[idx];
            int pos = atomicAdd(&cursor[(ent >> 16) * 2 + (r & 1)], 1);
            entP[pos] = (uint16_t)r;
            if (SOCIAL) {
                const int j = (int)(ent & 0xffff);      // scene-local j -> group-local row
                entS[pos] = (uint16_t)(j == 0xffff ? p.cap : sbase[r] + j);
            } else {
#pragma unroll
                for (int c = 0; c < C; ++c) entV[(size_t)pos * C + c] = p.win_val[g * 2 + c] - p.constant;
            }
        }
    }
    __syncthreads();

    float w[C], wn[C];
    const float* wcol = p.Wt + col;
#pragma unroll
    for (int c = 0; c < C; ++c) w[c] = col_ok ? wcol[(size_t)c * p.OUT] : 0.f;
    for (int cell = 0; cell < p.cells; ++cell) {
        if (cell + 1 < p.cells) {
#pragma unroll
            for (int c = 0; c < C; ++c)
                wn[c] = col_ok ? wcol[((size_t)(cell + 1) * C + c) * p.OUT] : 0.f;
        }
        const int e0 = start[cell * 2 + half], e1 = start[cell * 2 + half + 1];
        for (int e = e0; e < e1; ++e) {
            const int r = entP[e];
            float a = acc[r * kL1Cols + colc];
            if (SOCIAL) {
                const float4* lv = reinterpret_cast<const float4*>(latS + (size_t)entS[e] * C);
#pragma unroll
                for (int c4 = 0; c4 < C / 4; ++c4) {
                    float4 v = lv[c4];
                    a = fmaf(v.x, w[c4 * 4 + 0], a);
                    a = fmaf(v.y, w[c4 * 4 + 1], a);
                    a = fmaf(v.z, w[c4 * 4 + 2], a);
                    a = fmaf(v.w, w[c4 * 4 + 3], a);
                }
            } else {
#pragma unroll
                for (int c = 0; c < C; ++c) a = fmaf(entV[(size_t)e * C + c], w[c], a);
            }
            acc[r * kL1Cols + colc] = a;
        }
#pragma unroll
        for (int c = 0; c < C; ++c) w[c] = wn[c];
    }
    __syncthreads();
    if (col_ok) {
        for (int r = half; r < P; r += 2) {
            float v = acc[r * kL1Cols + colc];
            if (p.relu) v = fmaxf(v, 0.f);
            const size_t o = (size_t)(row0 + r) * p.OUT + col;
            if (p.out_hi) {
                const __nv_bfloat16 h = __float2bfloat16_rn(v);
                p.out_hi[o] = h;
                p.out_lo[o] = __float2bfloat16_rn(v - __bfloat162float(h));
            } else {
                p.out[o] = v;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// sparse_layer1_mma: the social grid (C = 16 latent channels) on the tensor cores.
//   For one cell the pairs binned there form A [pairs x 16] (latent vectors of the winning
//   neighbours) and the cell's weight slab is B [16 x 256]; pairs-per-cell is ~10, far below the
//   64/128-row minimum of tcgen05.mma, so this irregular piece uses warp-level
//   mma.sync.m16n8k16 (bf16 inputs, fp32 accumulate) with the same 3-pass (hi, lo) split as the
//   dense layers.  Warp w owns output columns [32w, 32w+32) of the chunk for ALL pedestrians of
//   the scene group, so accumulator rows are never shared between warps: no atomics, no
//   barriers inside the cell loop, deterministic ascending-cell summation.
//   smem: acc[P][264] fp32 | lat_hi, lat_lo [P+1][16] bf16 (k-permuted) | buckets | entries
//   Weights: Wt_hi / Wt_lo [cell][OUT][16] bf16, k permuted so a lane's B fragment is one 8-byte
//   load (position 4t..4t+3 = k {2t, 2t+1, 2t+8, 2t+9}); next cell's fragments are prefetched.
// ------------------------------------------------------------------------------------------
constexpr int kMmaAccStride = kL1Cols + 8;

__device__ __forceinline__ void mma_bf16_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
        "{%0, %1, %2, %3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__device__ __forceinline__ int kperm16(int k) { return 4 * ((k & 7) >> 1) + 2 * (k >> 3) + (k & 1); }

struct L1MmaParams {
    const int* group_off;
    const int* scene_off;
    const int* win_count;
    const uint32_t* win_ent;
    const float* lat;
    const float* benc;
    const __nv_bfloat16* Wt_hi;   // [cells, OUT, 4 (t), 8]: per (column, t) the 4 hi then the 4 lo values
    const __nv_bfloat16* Wt_lo;   //   of k = {2t, 2t+1, 2t+8, 2t+9} -> one 16-byte load per lane and n-tile (Wt_lo unused)
    const float* base;
    float* out;
    __nv_bfloat16* out_hi;
    __nv_bfloat16* out_lo;
    int OUT, cells, nm1, cap, relu;
    float constant;
};

constexpr int kMmaThreads = 256;          // 8 warps x 32 output columns

__global__ void __launch_bounds__(kMmaThreads, 1) sparse_layer1_mma_kernel(L1MmaParams p) {
    extern __shared__ __align__(16) unsigned char smem_l1m[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const int s0 = p.group_off[blockIdx.x], s1 = p.group_off[blockIdx.x + 1];
    const int row0 = p.scene_off[s0];
    const int P = p.scene_off[s1] - row0;
    const int chunk0 = blockIdx.y * kL1Cols;

    // acc rows [0, cap) real, [cap, cap + 16) dummies absorbing the padding rows of an MMA tile;
    // lat rows [0, cap) real, cap = NaN-padded slot (b_enc), cap + 1 = zeros (padding rows)
    float* acc = reinterpret_cast<float*>(smem_l1m);                                       // [cap+16][264]
    __nv_bfloat16* latH = reinterpret_cast<__nv_bfloat16*>(acc + (size_t)(p.cap + 16) * kMmaAccStride);   // [cap+2][16]
    __nv_bfloat16* latL = latH + (size_t)(p.cap + 2) * 16;
    int* start = reinterpret_cast<int*>(latL + (size_t)(p.cap + 2) * 16);                  // [cells+1]
    int* cursor = start + p.cells + 1;                                                     // [cells]
    uint32_t* ent = reinterpret_cast<uint32_t*>(cursor + p.cells);                         // [cap*nm1 + 16]: lat row << 16 | acc row
    uint32_t* raw = ent + (size_t)p.cap * p.nm1 + 16;                                      // [cap*nm1] winner lists as written by pool_prepare
    int* cnt_s = reinterpret_cast<int*>(raw + (size_t)p.cap * p.nm1);                      // [cap] winners per row
    int* sbase = cnt_s + p.cap;                                                            // [cap] first group-local row of the row's scene

    for (int c = tid; c < p.cells; c += kMmaThreads) cursor[c] = 0;
    // one coalesced pass over the group's winner lists (rows of a group are contiguous in memory)
    for (int r = tid; r < P; r += kMmaThreads) cnt_s[r] = p.win_count[row0 + r];
    {
        const uint32_t* src = p.win_ent + (size_t)row0 * p.nm1;
        for (int idx = tid; idx < P * p.nm1; idx += kMmaThreads) raw[idx] = src[idx];
    }
    for (int sb = s0 + warp; sb < s1; sb += kMmaThreads / 32) {
        const int a = p.scene_off[sb] - row0, b = p.scene_off[sb + 1] - row0;
        for (int r = a + lane; r < b; r += 32) sbase[r] = a;
    }
    for (int idx = tid; idx < (P + 2) * 16; idx += kMmaThreads) {
        const int r = idx >> 4, k = idx & 15;
        float v = 0.f;
        if (r < P) v = p.lat[(size_t)(row0 + r) * 16 + k] - p.constant;
        else if (r == P) v = p.benc[k] - p.constant;
        const __nv_bfloat16 h = __float2bfloat16_rn(v);
        const int dst = (r < P ? r : p.cap + (r - P)) * 16 + kperm16(k);
        latH[dst] = h;
        latL[dst] = __float2bfloat16_rn(v - __bfloat162float(h));
    }
    {
        const int col = chunk0 + tid;                     // 256 threads = 256 columns of the chunk
        const float b = col < p.OUT ? p.base[col] : 0.f;
        for (int r = 0; r < P; ++r) acc[r * kMmaAccStride + tid] = b;
    }
    __syncthreads();
    const int total = P * p.nm1;
    for (int idx = tid; idx < total; idx += kMmaThreads) {
        int r = idx / p.nm1, k = idx - r * p.nm1;
        if (k < cnt_s[r]) atomicAdd(&cursor[raw[idx] >> 16], 1);
    }
    __syncthreads();
    if (tid < 32) {
        int per = (p.cells + 31) / 32;
        int lo = tid * per, hi = min(lo + per, p.cells);
        int sum = 0;
        for (int c = lo; c < hi; ++c) sum += cursor[c];
        int incl = sum;
        for (int d = 1; d < 32; d <<= 1) {
            int v = __shfl_up_sync(0xffffffffu, incl, d);
            if (tid >= d) incl += v;
        }
        int run = incl - sum;
        for (int c = lo; c < hi; ++c) {
            int cnt = cursor[c];
            start[c] = run;
            cursor[c] = run;
            run += cnt;
        }
        if (tid == 31) start[p.cells] = incl;
    }
    __syncthreads();
    for (int idx = tid; idx < total; idx += kMmaThreads) {
        int r = idx / p.nm1, k = idx - r * p.nm1;
        if (k < cnt_s[r]) {
            const uint32_t e = raw[idx];
            const int pos = atomicAdd(&cursor[e >> 16], 1);
            const int j = (int)(e & 0xffff);
            const uint32_t lrow = (uint32_t)(j == 0xffff ? p.cap : sbase[r] + j);
            ent[pos] = (lrow << 16) | (uint32_t)r;
        }
    }
    __syncthreads();

    // padding rows of a tile: zero latent row, per-lane dummy accumulator rows
    const uint32_t dummy0 = ((uint32_t)(p.cap + 1) << 16) | (uint32_t)(p.cap + g);
    const uint32_t dummy1 = ((uint32_t)(p.cap + 1) << 16) | (uint32_t)(p.cap + 8 + g);
    // this lane loads, for n-tile j (j = 0..3), column chunk0 + 32 warp + 8 j + g
    const int ncol0 = chunk0 + warp * 32 + g;
    const size_t cell_stride = (size_t)p.OUT * 32;       // bf16 elements per cell (hi + lo interleaved)
    const __nv_bfloat16* wh = p.Wt_hi + (size_t)ncol0 * 32 + 8 * t;
    bool okc[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) okc[j] = ncol0 + 8 * j < p.OUT;
    struct BFrag { uint2 h[4], l[4]; };
    auto load_b = [&](int cell) -> BFrag {
        BFrag f;
        const size_t o = (size_t)cell * cell_stride;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            // one 16-byte L2 load per n-tile: (hi.x, hi.y, lo.x, lo.y) fragments of column ncol0 + 8 j
            const uint4 v = okc[j] ? __ldcg(reinterpret_cast<const uint4*>(wh + o + (size_t)j * 8 * 32))
                                   : make_uint4(0u, 0u, 0u, 0u);
            f.h[j] = make_uint2(v.x, v.y);
            f.l[j] = make_uint2(v.z, v.w);
        }
        return f;
    };
    float* accw = acc + warp * 32 + 2 * t;
    const uint32_t* latHw = reinterpret_cast<const uint32_t*>(latH) + 2 * t;   // 32-bit words: row stride 8
    const uint32_t* latLw = reinterpret_cast<const uint32_t*>(latL) + 2 * t;
    auto process = [&](int e0, int e1, const BFrag& b) {
        for (int eb = e0; eb < e1; eb += 16) {
            const int i0 = eb + g, i1 = i0 + 8;
            const uint32_t en0 = i0 < e1 ? ent[i0] : dummy0;
            const uint32_t en1 = i1 < e1 ? ent[i1] : dummy1;
            const uint32_t l0 = (en0 >> 16) * 8, l1 = (en1 >> 16) * 8;
            uint32_t ah[4], al[4];
            ah[0] = latHw[l0]; ah[1] = latHw[l1]; ah[2] = latHw[l0 + 1]; ah[3] = latHw[l1 + 1];
            al[0] = latLw[l0]; al[1] = latLw[l1]; al[2] = latLw[l0 + 1]; al[3] = latLw[l1 + 1];
            float* a0 = accw + (en0 & 0xffffu) * kMmaAccStride;
            float* a1 = accw + (en1 & 0xffffu) * kMmaAccStride;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float d[4] = {0.f, 0.f, 0.f, 0.f};
                mma_bf16_16816(d, ah, b.h[j].x, b.h[j].y);
                mma_bf16_16816(d, ah, b.l[j].x, b.l[j].y);
                mma_bf16_16816(d, al, b.h[j].x, b.h[j].y);
                float2* q0 = reinterpret_cast<float2*>(a0 + 8 * j);
                float2* q1 = reinterpret_cast<float2*>(a1 + 8 * j);
                float2 u0 = *q0, u1 = *q1;
                u0.x += d[0]; u0.y += d[1]; u1.x += d[2]; u1.y += d[3];
                *q0 = u0; *q1 = u1;
            }
        }
    };
    // register ring of 4 fragment sets: the slab of cell c+4 is requested right after cell c is
    // consumed, i.e. three cell-times ahead of its use
    const int nc = p.cells;
    auto phys = [&](int i) { return i; };
    BFrag b0 = load_b(phys(0));
    BFrag b1 = load_b(phys(min(1, nc - 1)));
    BFrag b2 = load_b(phys(min(2, nc - 1)));
    BFrag b3 = load_b(phys(min(3, nc - 1)));
    for (int cell = 0; cell < nc; cell += 4) {
        int c = phys(cell);
        process(start[c], start[c + 1], b0);
        if (cell + 4 < nc) b0 = load_b(phys(cell + 4));
        if (cell + 1 < nc) {
            c = phys(cell + 1);
            process(start[c], start[c + 1], b1);
            if (cell + 5 < nc) b1 = load_b(phys(cell + 5));
        }
        if (cell + 2 < nc) {
            c = phys(cell + 2);
            process(start[c], start[c + 1], b2);
            if (cell + 6 < nc) b2 = load_b(phys(cell + 6));
        }
        if (cell + 3 < nc) {
            c = phys(cell + 3);
            process(start[c], start[c + 1], b3);
            if (cell + 7 < nc) b3 = load_b(phys(cell + 7));
        }
    }
    __syncthreads();
    {
        const int col = chunk0 + tid;
        if (col < p.OUT) {
            for (int r = 0; r < P; ++r) {
                float v = acc[r * kMmaAccStride + tid];
                if (p.relu) v = fmaxf(v, 0.f);
                const size_t o = (size_t)(row0 + r) * p.OUT + col;
                if (p.out_hi) {
                    const __nv_bfloat16 h = __float2bfloat16_rn(v);
                    p.out_hi[o] = h;
                    p.out_lo[o] = __float2bfloat16_rn(v - __bfloat162float(h));
                } else {
                    p.out[o] = v;
                }
            }
        }
    }
}

static size_t l1_mma_smem_bytes(int cap, int cells, int nm1) {
    size_t b = (size_t)(cap + 16) * kMmaAccStride * sizeof(float);
    b += (size_t)(cap + 2) * 16 * 2 * sizeof(__nv_bfloat16);
    b += (size_t)(2 * cells + 1) * sizeof(int);
    b += ((size_t)cap * nm1 + 16) * sizeof(uint32_t);     // sorted entries
    b += (size_t)cap * nm1 * sizeof(uint32_t);            // raw winner lists
    b += (size_t)cap * 2 * sizeof(int);                   // winners per row, scene base per row
    return b + 16;
}

// weight repack for the mma path: W1[o][c * cells + cell] -> (hi, lo)[cell][o][kperm(c)]
__global__ void repack_layer1_mma_kernel(const float* __restrict__ W1, __nv_bfloat16* __restrict__ hi,
                                         __nv_bfloat16* __restrict__ lo, int OUT, int cells) {
    size_t total = (size_t)cells * OUT * 16;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (size_t)gridDim.x * blockDim.x) {
        const int c = (int)(idx & 15);
        const size_t co = idx >> 4;
        const int o = (int)(co % OUT), cell = (int)(co / OUT);
        const float v = W1[(size_t)o * 16 * cells + (size_t)c * cells + cell];
        const __nv_bfloat16 h = __float2bfloat16_rn(v);
        const int kp = kperm16(c);                      // = 4 t + i
        const size_t dst = (co << 5) + (size_t)(kp >> 2) * 8 + (kp & 3);
        hi[dst] = h;                                    // `hi` holds the interleaved (hi | lo) slabs
        hi[dst + 4] = __float2bfloat16_rn(v - __bfloat162float(h));
        (void)lo;
    }
}

int launch_repack_layer1_mma(const float* W1, void* hi, void* lo, int OUT, int cells, cudaStream_t st) {
    repack_layer1_mma_kernel<<<1024, 256, 0, st>>>(W1, (__nv_bfloat16*)hi, (__nv_bfloat16*)lo, OUT, cells);
    TB2_LAUNCH_CHECK();
    return TB2_OK;
}

static size_t l1_smem_bytes(int cap, int C, bool social, int cells, int nm1) {
    size_t b = (size_t)cap * kL1Cols * sizeof(float);
    if (social) b += (size_t)(cap + 1) * C * sizeof(float);
    b += (size_t)(4 * cells + 1) * sizeof(int);
    size_t ents = ((size_t)cap * nm1 * 2 * sizeof(uint16_t) + 15) & ~(size_t)15;
    b += ents;
    if (!social) b += (size_t)cap * nm1 * C * sizeof(float);
    b += (size_t)cap * nm1 * sizeof(uint32_t) + (size_t)cap * 2 * sizeof(int);    // raw winner lists, per-row tables
    return b + 16;
}

// ------------------------------------------------------------------------------------------
// dense_layer: Y = act(X . W^T + b), X [M, K], WT [K, N] (transposed at repack).  fp32 FFMA,
// 64 x 64 x 16 tiles, 4 x 4 micro-tiles.  (Layers >= 2 of the grid embedding.)
// ------------------------------------------------------------------------------------------
constexpr int kDT = 64, kDK = 16;

__global__ void __launch_bounds__(256) dense_layer_kernel(const float* __restrict__ X,
                                                          const float* __restrict__ WT,
                                                          const float* __restrict__ bias,
                                                          float* __restrict__ Y, int M, int K, int N,
                                                          int relu) {
    __shared__ float As[kDK][kDT + 4];
    __shared__ float Bs[kDK][kDT];
    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;
    const int m0 = blockIdx.y * kDT, n0 = blockIdx.x * kDT;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    for (int k0 = 0; k0 < K; k0 += kDK) {
        // A tile: 64 rows x 16 k  (thread loads 4 consecutive k of one row)
        {
            int r = tid >> 2, kq = (tid & 3) * 4;
            int m = m0 + r;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                int k = k0 + kq + q;
                As[kq + q][r] = (m < M && k < K) ? X[(size_t)m * K + k] : 0.f;
            }
        }
        // B tile: 16 k x 64 cols
        {
            int kk = tid >> 4, cq = (tid & 15) * 4;
            int k = k0 + kk;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                int n = n0 + cq + q;
                Bs[kk][cq + q] = (k < K && n < N) ? WT[(size_t)k * N + n] : 0.f;
            }
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < kDK; ++kk) {
            float a[4], bb[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = As[kk][ty * 4 + i];
#pragma unroll
            for (int j = 0; j < 4; ++j) bb[j] = Bs[kk][tx * 4 + j];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        int m = m0 + ty * 4 + i;
        if (m >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            int n = n0 + tx * 4 + j;
            if (n >= N) continue;
            float v = acc[i][j] + bias[n];
            if (relu) v = fmaxf(v, 0.f);
            Y[(size_t)m * N + n] = v;
        }
    }
}

static int launch_dense(const float* X, const float* WT, const float* b, float* Y, int M, int K, int N,
                        int relu, cudaStream_t st) {
    dim3 grid((N + kDT - 1) / kDT, (M + kDT - 1) / kDT);
    {
        KernelTimer kt("dense_layer", st);
        dense_layer_kernel<<<grid, 256, 0, st>>>(X, WT, b, Y, M, K, N, relu);
    }
    TB2_LAUNCH_CHECK();
    return TB2_OK;
}

// ------------------------------------------------------------------------------------------
// First Linear for occupancy / directional grids (C <= 2 payload channels): the whole weight
// chunk [cells * C][CH output columns] fits in shared memory, so a CTA loads it once and then
// walks its rows; each row is base + sum over its <= N-1 winners of C weight rows (a few dozen
// FMAs per output).  grid = (row groups, column chunks), sized to one wave of the SMs.
// ------------------------------------------------------------------------------------------
struct RowsParams {
    const int* win_count;
    const uint32_t* win_ent;
    const float* win_val;
    const float* Wt;          // [cells, C, OUT]
    const float* base;        // [OUT]
    float* out;               // [M, OUT] fp32 or null
    __nv_bfloat16* out_hi;    // [M, OUT] bf16 (hi, lo) split or null
    __nv_bfloat16* out_lo;
    int M, OUT, cells, C, nm1, CH, rows_per_cta, relu;
    float constant;
};

constexpr int kRowsThreads = 1024;

__global__ void __launch_bounds__(kRowsThreads, 1) pool_rows_kernel(RowsParams p) {
    extern __shared__ __align__(16) unsigned char smem_rows[];
    float* Ws = reinterpret_cast<float*>(smem_rows);                            // [cells * C][CH]
    const int KW = p.cells * p.C;
    int* cnt_s = reinterpret_cast<int*>(Ws + (size_t)KW * p.CH);                // [rows_per_cta]
    uint32_t* ent_s = reinterpret_cast<uint32_t*>(cnt_s + p.rows_per_cta);      // [rows_per_cta][nm1]
    float* val_s = reinterpret_cast<float*>(ent_s + (size_t)p.rows_per_cta * p.nm1);   // [rows_per_cta][nm1][2]
    const int tid = threadIdx.x;
    grid_dep_wait();
    grid_dep_launch();
    const int col0 = blockIdx.y * p.CH;
    const int r0 = blockIdx.x * p.rows_per_cta;
    const int nrows = min(p.rows_per_cta, p.M - r0);
    if (nrows <= 0) return;
    // weight chunk: rows of CH floats at stride OUT (CH is a multiple of 4, OUT too when vectorised)
    const int cw = min(p.CH, p.OUT - col0);
    if ((p.OUT & 3) == 0 && (cw & 3) == 0) {
        const int q = cw >> 2;
        for (int idx = tid; idx < KW * q; idx += kRowsThreads) {
            const int k = idx / q, c4 = idx - k * q;
            *reinterpret_cast<float4*>(Ws + (size_t)k * p.CH + c4 * 4) =
                *reinterpret_cast<const float4*>(p.Wt + (size_t)k * p.OUT + col0 + c4 * 4);
        }
    } else {
        for (int idx = tid; idx < KW * cw; idx += kRowsThreads) {
            const int k = idx / cw, c = idx - k * cw;
            Ws[(size_t)k * p.CH + c] = p.Wt[(size_t)k * p.OUT + col0 + c];
        }
    }
    for (int r = tid; r < nrows; r += kRowsThreads) cnt_s[r] = p.win_count[r0 + r];
    {
        const uint32_t* esrc = p.win_ent + (size_t)r0 * p.nm1;
        for (int idx = tid; idx < nrows * p.nm1; idx += kRowsThreads) ent_s[idx] = esrc[idx];
        const float* vsrc = p.win_val + (size_t)r0 * p.nm1 * 2;
        for (int idx = tid; idx < nrows * p.nm1 * 2; idx += kRowsThreads) val_s[idx] = vsrc[idx] - p.constant;
    }
    __syncthreads();
    const int lanes = kRowsThreads / p.CH;          // row lanes (CH = 256 -> 1, 128 -> 2, 64 -> 4, 32 -> 8)
    const int colc = tid % p.CH, lane = tid / p.CH;
    const int col = col0 + colc;
    if (col >= p.OUT) return;
    const float b = p.base[col];
    for (int r = lane; r < nrows; r += lanes) {
        float acc = b;
        const int cnt = cnt_s[r];
        const uint32_t* er = ent_s + (size_t)r * p.nm1;
        const float* vr = val_s + (size_t)r * p.nm1 * 2;
        for (int e = 0; e < cnt; ++e) {
            const float* w = Ws + (size_t)(er[e] >> 16) * p.C * p.CH + colc;
            acc = fmaf(w[0], vr[2 * e], acc);
            if (p.C == 2) acc = fmaf(w[p.CH], vr[2 * e + 1], acc);
        }
        if (p.relu) acc = fmaxf(acc, 0.f);
        const size_t o = (size_t)(r0 + r) * p.OUT + col;
        if (p.out_hi) {
            const __nv_bfloat16 h = __float2bfloat16_rn(acc);
            p.out_hi[o] = h;
            p.out_lo[o] = __float2bfloat16_rn(acc - __bfloat162float(h));
        }
        if (p.out) p.out[o] = acc;
    }
}

// returns the column chunk width the row kernel can use for this model (0 = does not fit)
static int pool_rows_chunk(const tb2_lstm* m, int OUT) {
    if (m->cfg.pool_type == TB2_POOL_SOCIAL || m->C > 2) return 0;
    const size_t KW = (size_t)m->cells * m->C;
    for (int ch = 256; ch >= 32; ch >>= 1) {
        if (ch > 32 && ch / 2 >= OUT) continue;          // do not pad tiny layers
        if (KW * ch * sizeof(float) <= 160 * 1024) return ch;
    }
    return 0;
}

static int launch_pool_rows(const tb2_lstm* m, const tb2_layout* l, const Workspace* ws, int OUT, int nm1,
                            float* out, __nv_bfloat16* out_hi, __nv_bfloat16* out_lo, cudaStream_t st) {
    RowsParams p;
    p.win_count = ws->win_count; p.win_ent = ws->win_ent; p.win_val = ws->win_val;
    p.Wt = m->Wt1; p.base = m->base1; p.out = out; p.out_hi = out_hi; p.out_lo = out_lo;
    p.M = l->M; p.OUT = OUT; p.cells = m->cells; p.C = m->C; p.nm1 = nm1; p.relu = 1;
    p.constant = m->cfg.constant;
    p.CH = pool_rows_chunk(m, OUT);
    const int chunks = (OUT + p.CH - 1) / p.CH;
    // one wave: ~148 CTAs in total, winner lists of a CTA's rows must fit next to the weights
    int groups = (148 + chunks - 1) / chunks;
    int rows = (l->M + groups - 1) / groups;
    const size_t wbytes = (size_t)m->cells * m->C * p.CH * sizeof(float);
    const size_t per_row = sizeof(int) + (size_t)nm1 * (sizeof(uint32_t) + 2 * sizeof(float));
    const int max_rows = (int)((220 * 1024 - wbytes) / per_row);
    if (rows > max_rows) rows = max_rows;
    if (rows < 1) rows = 1;
    groups = (l->M + rows - 1) / rows;
    p.rows_per_cta = rows;
    const size_t smem = wbytes + (size_t)rows * per_row;
    static DynSmemConfig configured;
    TB2_CHECK_CUDA(configured.ensure(pool_rows_kernel, smem));
    {
        KernelTimer kt("pool_rows", st);
        launch_pdl(pool_rows_kernel, dim3(groups, chunks), dim3(kRowsThreads), smem, st, p);
    }
    TB2_LAUNCH_CHECK();
    return TB2_OK;
}

template <int C, bool SOCIAL>
static int launch_l1_t(const L1Params& p, int groups, size_t smem, cudaStream_t st) {
    static DynSmemConfig configured;
    TB2_CHECK_CUDA(configured.ensure(sparse_layer1_kernel<C, SOCIAL>, smem));
    dim3 grid(groups, (p.OUT + kL1Cols - 1) / kL1Cols);
    {
        KernelTimer kt("sparse_layer1", st);
        sparse_layer1_kernel<C, SOCIAL><<<grid, kL1Threads, smem, st>>>(p);
    }
    TB2_LAUNCH_CHECK();
    return TB2_OK;
}

// Grid -> pooled vector (GridBasedPooling.forward after the grid is known, :106-110).
int launch_pool_mlp(const tb2_lstm* m, const tb2_layout* l, Workspace* ws, float* pooled_out,
                    void* pool_hi, void* pool_lo, cudaStream_t st) {
    const int nm1 = l->n_max > 1 ? l->n_max - 1 : 1;
    // producers that cannot write the bf16 split themselves go through fp32 scratch + split_rows
    const bool want_split = pool_hi != nullptr;
    const bool last_is_l1 = m->n_mlp == 1;
    const bool last_is_tc = m->n_mlp == 2 && m->W_hi[1] != nullptr;
    const bool direct_split = want_split && (last_is_l1 || last_is_tc);
    if (want_split && !direct_split && pooled_out == nullptr) pooled_out = ws->pooled;
    int rc_all = TB2_OK;
    if (m->n_mlp == 0) {
        dense_grid_kernel<<<l->M, 128, 0, st>>>(ws->win_count, ws->win_ent, ws->win_val, ws->lat,
                                                l->row_scene, l->scene_off, m->benc, pooled_out, m->C,
                                                m->cells, nm1, m->cfg.constant, m->cfg.pool_type);
        TB2_LAUNCH_CHECK();
        if (want_split) rc_all = launch_split_rows(pooled_out, pool_hi, pool_lo, (size_t)l->M * m->pool_out, st);
        return rc_all;
    }
    const int d1 = m->mlp_dims[1];
    const bool social = m->cfg.pool_type == TB2_POOL_SOCIAL;
    // few column chunks -> small scene groups so the grid still covers the SMs
    const int chunks = (d1 + kL1Cols - 1) / kL1Cols;
    int gsel = chunks >= 4 ? 0 : 1;
    size_t smem = l1_smem_bytes(l->group_cap[gsel], m->C, social, m->cells, nm1);
    if (smem > 227 * 1024 && gsel == 0) {
        gsel = 1;
        smem = l1_smem_bytes(l->group_cap[gsel], m->C, social, m->cells, nm1);
    }
    TB2_REQUIRE(smem <= 227 * 1024, "scene group does not fit in shared memory (scene too large)");
    L1Params p;
    p.group_off = l->group_off[gsel];
    p.scene_off = l->scene_off;
    p.win_count = ws->win_count;
    p.win_ent = ws->win_ent;
    p.win_val = ws->win_val;
    p.lat = ws->lat;
    p.benc = m->benc;
    p.Wt = m->Wt1;
    p.base = m->base1;
    p.OUT = d1;
    p.cells = m->cells;
    p.nm1 = nm1;
    p.cap = l->group_cap[gsel];
    p.relu = 1;
    p.constant = m->cfg.constant;
    float* l1_out = (m->n_mlp == 1) ? pooled_out : ws->act[0];
    // second Linear on the tensor cores: layer 1 hands its activations over as bf16 (hi, lo)
    const bool tc2 = m->n_mlp >= 2 && m->W_hi[1] != nullptr;
    p.out = tc2 ? nullptr : l1_out;
    p.out_hi = tc2 ? reinterpret_cast<__nv_bfloat16*>(ws->act[0]) : nullptr;
    p.out_lo = tc2 ? reinterpret_cast<__nv_bfloat16*>(ws->act[1]) : nullptr;
    if (last_is_l1 && direct_split) {      // one_layer embedding feeding the tensor-core gates
        p.out = pooled_out;                // may be null
        p.out_hi = reinterpret_cast<__nv_bfloat16*>(pool_hi);
        p.out_lo = reinterpret_cast<__nv_bfloat16*>(pool_lo);
    }
    int rc;
    // TB2_SPARSE (A/B and debug knob) forces round 1's kernels: "tc" and "bucket" skip the pair kernel, "mma" also
    // sparse_layer1_tc, "bucket" also pool_rows
    enum { kL1Default, kL1Tc, kL1Mma, kL1Bucket } force = kL1Default;
    if (const char* e = getenv("TB2_SPARSE")) {
        if (!strcmp(e, "tc")) force = kL1Tc;
        else if (!strcmp(e, "mma")) force = kL1Mma;
        else if (!strcmp(e, "bucket")) force = kL1Bucket;
        else if (e[0]) { set_error("TB2_SPARSE must be tc, mma or bucket"); return TB2_ERR_INVALID; }
    }
    if (force != kL1Bucket && pool_rows_chunk(m, d1) > 0) {   // occupancy / directional: weights resident in smem
        rc = launch_pool_rows(m, l, ws, d1, nm1, p.out, p.out_hi, p.out_lo, st);
    } else
    if (force == kL1Default && ws->cell_row && sparse_pair_supported(m, l)) {   // social, 16 latent channels: CTA-pair tcgen05 kernel
        rc = launch_sparse_pair(m, l, ws, p.out, p.out_hi, p.out_lo, st);
    } else
    if (force != kL1Mma && sparse_tc_supported(m, l, 0)) {  // social, 16 latent channels: tcgen05 path
        rc = launch_sparse_tc(m, l, 0, ws, p.out, p.out_hi, p.out_lo, st);
    } else
    if (m->Wt1_hi != nullptr) {      // social, 16 latent channels: warp-level tensor-core path
        int gm = 0;
        size_t sm = l1_mma_smem_bytes(l->group_cap[gm], m->cells, nm1);
        if (sm > 227 * 1024) { gm = 1; sm = l1_mma_smem_bytes(l->group_cap[gm], m->cells, nm1); }
        TB2_REQUIRE(sm <= 227 * 1024, "scene group does not fit in shared memory (scene too large)");
        L1MmaParams q;
        q.group_off = l->group_off[gm]; q.scene_off = l->scene_off; q.win_count = ws->win_count;
        q.win_ent = ws->win_ent; q.lat = ws->lat; q.benc = m->benc;
        q.Wt_hi = (const __nv_bfloat16*)m->Wt1_hi; q.Wt_lo = (const __nv_bfloat16*)m->Wt1_lo;
        q.base = m->base1; q.out = p.out; q.out_hi = p.out_hi; q.out_lo = p.out_lo;
        q.OUT = d1; q.cells = m->cells; q.nm1 = nm1; q.cap = l->group_cap[gm]; q.relu = 1;
        q.constant = m->cfg.constant;
        static DynSmemConfig configured;
        TB2_CHECK_CUDA(configured.ensure(sparse_layer1_mma_kernel, sm));
        dim3 grid(l->num_groups[gm], (d1 + kL1Cols - 1) / kL1Cols);
        {
            KernelTimer kt("sparse_layer1_mma", st);
            sparse_layer1_mma_kernel<<<grid, kMmaThreads, sm, st>>>(q);
        }
        TB2_LAUNCH_CHECK();
        rc = TB2_OK;
    } else
    switch (m->cfg.pool_type) {
        case TB2_POOL_OCCUPANCY: rc = launch_l1_t<1, false>(p, l->num_groups[gsel], smem, st); break;
        case TB2_POOL_DIRECTIONAL: rc = launch_l1_t<2, false>(p, l->num_groups[gsel], smem, st); break;
        case TB2_POOL_SOCIAL:
            if (m->C == 16) rc = launch_l1_t<16, true>(p, l->num_groups[gsel], smem, st);
            else if (m->C == 8) rc = launch_l1_t<8, true>(p, l->num_groups[gsel], smem, st);
            else if (m->C == 4) rc = launch_l1_t<4, true>(p, l->num_groups[gsel], smem, st);
            else if (m->C == 32) rc = launch_l1_t<32, true>(p, l->num_groups[gsel], smem, st);
            else { set_error("social latent_dim must be 4, 8, 16 or 32"); return TB2_ERR_UNSUPPORTED; }
            break;
        default: set_error("bad pool type"); return TB2_ERR_INVALID;
    }
    if (rc != TB2_OK) return rc;
    const float* x = l1_out;
    for (int layer = 1; layer < m->n_mlp; ++layer) {
        float* y = (layer == m->n_mlp - 1) ? pooled_out : ws->act[layer & 1];
        if (layer == 1 && tc2) {
            // act[0] / act[1] hold the split input; a third layer (if any) reads fp32 from ws->pooled-sized scratch
            if (m->n_mlp > 2) y = ws->act2;
            const bool last = (m->n_mlp == 2);
            rc = launch_dense_tc(ws->act[0], ws->act[1], m->W_hi[1], m->W_lo[1], m->bl[1],
                                 (last && direct_split) ? pooled_out : y,
                                 (last && direct_split) ? pool_hi : nullptr, (last && direct_split) ? pool_lo : nullptr,
                                 l->M, m->mlp_dims[1], m->mlp_dims[2], 1, st);
        } else
        rc = launch_dense(x, m->WT[layer], m->bl[layer], y, l->M, m->mlp_dims[layer], m->mlp_dims[layer + 1], 1, st);
        if (rc != TB2_OK) return rc;
        x = y;
    }
    if (want_split && !direct_split) return launch_split_rows(pooled_out, pool_hi, pool_lo, (size_t)l->M * m->pool_out, st);
    return TB2_OK;
}

}  // namespace tb2
