// Backward of the recurrence (BPTT) for training -- reference: what autograd does for
// Trainer.train_batch (trajnetbaselines/lstm/trainer.py:229-269) through LSTM.forward
// (lstm/lstm.py:170-264).
//
// Gradient structure exploited (SURVEY.md 8a/A12, probe-verified on the reference): fed-back
// positions are detached (lstm.py:242-250), and for vanilla / occupancy / directional pooling the
// pooled vector does not depend on any hidden state, so a track's gradient never leaves its own
// LSTM chain.  The caller passes the list of ACTIVE rows (tracks that receive a non-zero upstream
// gradient: the scene primaries for PredictionLoss, loss.py:57,67) and the whole backward runs
// on those R rows only, in phases:
//   (A) per step: winners (pool_prepare) and the gather of X = [emb | pooled | h_prev], the pooled
//       rows recomputed from the winner list, plus the dense grid row of each active track;
//   (B) gate pre-activations of all steps in one GEMM per cell (encoder / decoder weights);
//   (C) the sequential chain, ONE kernel per step: cell + head backward with the recurrent
//       dgates(s+1) . W_hh mat-vec fused in;
//   (D) input gradients of all steps in one GEMM;  (E) every parameter gradient as one reduction
//       over all S * R (step, row) records, rows split over CTAs with the partial sums added in a
//       fixed order.  No floating-point atomics: results are bit-identical from run to run.
// Social pooling couples the tracks of a scene through lat_j = W_enc h_j: every track receives
// gradient, so social_backward (further down) runs the same phases on all M rows and adds the
// backward of the grid MLP and of the hidden-state scatter to the chain.
#include <cublas_v2.h>
#include <dlfcn.h>
#include <mutex>
#include <cuda_bf16.h>
#include <math_constants.h>

#include "common.cuh"

namespace tb2 {

constexpr int kBH = 128;

__device__ __forceinline__ float sigm(float x) { return 1.f / (1.f + expf(-x)); }

// X[r] = [emb(vel) | pooled | h_prev] for the active rows (one CTA per row).  The pooled part is
// recomputed from the step's winner list: pooled = relu(base + sum_winners Wt1[cell, c, :] * val)
// (one_layer embedding, constant = 0) -- R rows instead of re-running the first Linear on all M.
__global__ void __launch_bounds__(256) bwd_gather_kernel(
    const int* __restrict__ rows, int R, const float2* __restrict__ obs1, const float2* __restrict__ obs2,
    const float* __restrict__ We, const float* __restrict__ be, const float* __restrict__ h_prev,
    const int* __restrict__ win_count, const uint32_t* __restrict__ win_ent, const float* __restrict__ win_val,
    const float* __restrict__ Wt1, const float* __restrict__ base1, int nm1, int C, int cells,
    const float* __restrict__ pooled_src, float* __restrict__ X, float* __restrict__ G, float* __restrict__ vel,
    int* __restrict__ masked, int E, int P, int K) {
    __shared__ uint32_t ent_s[64];
    __shared__ float val_s[64][2];
    const int r = blockIdx.x;
    if (r >= R) return;
    const int m = rows[r];
    const float2 a = obs1[m], b = obs2[m];
    const bool msk = isnan(a.x) || isnan(b.x);
    const float vx = msk ? 0.f : (b.x - a.x) * 4.0f, vy = msk ? 0.f : (b.y - a.y) * 4.0f;
    if (threadIdx.x == 0) {
        masked[r] = msk ? 1 : 0;
        vel[2 * r] = vx;
        vel[2 * r + 1] = vy;
    }
    float* x = X + (size_t)r * K;
    float* grow = G ? G + (size_t)r * C * cells : nullptr;     // the reference's grid row [C * n * n]
    if (grow)
        for (int k = threadIdx.x; k < C * cells; k += blockDim.x) grow[k] = 0.f;
    if (msk) {
        for (int k = threadIdx.x; k < K; k += blockDim.x) x[k] = 0.f;
        return;
    }
    for (int k = threadIdx.x; k < E; k += blockDim.x)
        x[k] = k < E - 2 ? fmaxf(fmaf(We[2 * k + 1], vy, fmaf(We[2 * k], vx, be[k])), 0.f) : 0.f;
    for (int k = threadIdx.x; k < kBH; k += blockDim.x)
        x[E + P + k] = h_prev ? h_prev[(size_t)m * kBH + k] : 0.f;
    if (pooled_src) {      // pooled vector of this row as the forward kernels produced it
        for (int o = threadIdx.x; o < P; o += blockDim.x) x[E + o] = pooled_src[(size_t)m * P + o];
    } else if (P > 0) {
        const int cnt = win_count[m];
        float acc[4];     // up to 4 output columns per thread (P <= 1024)
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int o = threadIdx.x + q * blockDim.x;
            acc[q] = o < P ? base1[o] : 0.f;
        }
        for (int e0 = 0; e0 < cnt; e0 += 64) {
            const int n = min(64, cnt - e0);
            __syncthreads();
            if (threadIdx.x < n) {
                const size_t g = (size_t)m * nm1 + e0 + threadIdx.x;
                ent_s[threadIdx.x] = win_ent[g];
                val_s[threadIdx.x][0] = win_val[g * 2];
                val_s[threadIdx.x][1] = win_val[g * 2 + 1];
            }
            __syncthreads();
            if (threadIdx.x < n)      // a cell has one winner per row: plain stores (after the zero fill above)
                for (int c = 0; c < C; ++c)
                    grow[c * cells + (ent_s[threadIdx.x] >> 16)] = val_s[threadIdx.x][c];
            for (int e = 0; e < n; ++e) {
                const int cell = ent_s[e] >> 16;
                for (int c = 0; c < C; ++c) {
                    const float v = val_s[e][c];
                    const float* wrow = Wt1 + ((size_t)cell * C + c) * P;
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int o = threadIdx.x + q * blockDim.x;
                        if (o < P) acc[q] = fmaf(wrow[o], v, acc[q]);
                    }
                }
            }
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int o = threadIdx.x + q * blockDim.x;
            if (o < P) x[E + o] = fmaxf(acc[q], 0.f);
        }
    }
}

// Backward of LSTMCell + Hidden2Normal for one active row per CTA (128 threads = units): the only
// kernel on the sequential chain of the BPTT.
//   in : gates_pre [R,512] of this step (with bias), c_prev (state before the step, null = zeros),
//        incoming dh = dg_next[r] . Whh_next (recurrent part of the LATER step's gate gradient,
//        W_hh in torch layout [4H, H]) + pass_prev[r] (what by-passed the cell there); both null
//        at the last step.  dc [R,128] in place; upstream dnormal [M,5] (row-indexed by track)
//   out: dgates [R,512], dc (gradient wrt c_prev), hs [R,128] (h of this step), dn_raw [R,8],
//        pass_cur [R,128] (masked rows: dh goes straight through, lstm.py:158-166)
__global__ void __launch_bounds__(4 * kBH) bwd_cell_head_kernel(
    const int* __restrict__ rows, const int* __restrict__ masked, const float* __restrict__ gates_pre,
    const float* __restrict__ c_prev, const float* __restrict__ dg_next, const float* __restrict__ Whh_next,
    const float* __restrict__ dh_rec, const float* __restrict__ pass_prev, float* __restrict__ pass_cur,
    float* __restrict__ dc,
    const float* __restrict__ dnormal, const float* __restrict__ Wn, const float* __restrict__ bn,
    float* __restrict__ dgates, float* __restrict__ hs, float* __restrict__ dn_raw, int R) {
    __shared__ float red[5][kBH];
    __shared__ float dn_s[5];
    __shared__ __align__(16) float dgn_s[4 * kBH];
    __shared__ float part_s[4][kBH];
    const int r = blockIdx.x, u = threadIdx.x & (kBH - 1), quarter = threadIdx.x >> 7;
    const int m = rows[r];
    float* dg = dgates + (size_t)r * 4 * kBH;
    float dh_in = 0.f;
    if (dh_rec) {       // many rows: dg_next . W_hh was done as one GEMM
        dh_in = dh_rec[(size_t)r * kBH + u] + pass_prev[(size_t)r * kBH + u];
    } else if (dg_next) {      // 4 x 128 threads: each quarter of the CTA reduces one gate block of the mat-vec
        dgn_s[threadIdx.x] = dg_next[(size_t)r * 4 * kBH + threadIdx.x];
        __syncthreads();
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
        const float* wq = Whh_next + (size_t)quarter * kBH * kBH + u;
        const float* dq = dgn_s + quarter * kBH;
#pragma unroll 4
        for (int g = 0; g < kBH; g += 4) {
            a0 = fmaf(dq[g + 0], wq[(size_t)(g + 0) * kBH], a0);
            a1 = fmaf(dq[g + 1], wq[(size_t)(g + 1) * kBH], a1);
            a2 = fmaf(dq[g + 2], wq[(size_t)(g + 2) * kBH], a2);
            a3 = fmaf(dq[g + 3], wq[(size_t)(g + 3) * kBH], a3);
        }
        part_s[quarter][u] = (a0 + a1) + (a2 + a3);
        __syncthreads();
        dh_in = (part_s[0][u] + part_s[1][u]) + (part_s[2][u] + part_s[3][u]) + pass_prev[(size_t)r * kBH + u];
    }
    if (quarter != 0) return;       // the cell / head math below is one thread per unit
    if (masked[r]) {   // absent track: state passes through, no parameter gradient
#pragma unroll
        for (int g = 0; g < 4; ++g) dg[g * kBH + u] = 0.f;
        hs[(size_t)r * kBH + u] = 0.f;
        if (u < 8) dn_raw[r * 8 + u] = 0.f;
        pass_cur[(size_t)r * kBH + u] = dh_in;
        return;        // dc stays as it is
    }
    pass_cur[(size_t)r * kBH + u] = 0.f;
    const float* gp = gates_pre + (size_t)r * 4 * kBH;
    const float ig = sigm(gp[u]), fg = sigm(gp[kBH + u]), gg = tanhf(gp[2 * kBH + u]), og = sigm(gp[3 * kBH + u]);
    const float cp = c_prev ? c_prev[(size_t)m * kBH + u] : 0.f;
    const float cn = fg * cp + ig * gg;
    const float tc = tanhf(cn);
    const float hn = og * tc;
    hs[(size_t)r * kBH + u] = hn;
    // head: n_raw = Wn h + bn (modules.py:57); recomputed for the sigmoid derivatives
#pragma unroll
    for (int o = 0; o < 5; ++o) red[o][u] = Wn[o * kBH + u] * hn;
    asm volatile("bar.sync 1, 128;" ::: "memory");
    for (int s = kBH / 2; s > 0; s >>= 1) {
        if (u < s) {
#pragma unroll
            for (int o = 0; o < 5; ++o) red[o][u] += red[o][u + s];
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");
    }
    if (u < 8) {
        float d = 0.f;
        if (u < 5) {
            const float raw = red[u][0] + bn[u];
            d = dnormal[(size_t)m * 5 + u];
            if (isnan(d)) d = 0.f;
            if (u >= 2) {
                const float sg = sigm(raw);
                d *= (u == 4 ? 0.7f : 0.2f) * sg * (1.f - sg);     // modules.py:60-62
            }
            dn_s[u] = d;
        }
        dn_raw[r * 8 + u] = d;
    }
    asm volatile("bar.sync 1, 128;" ::: "memory");
    float dht = dh_in;
#pragma unroll
    for (int o = 0; o < 5; ++o) dht = fmaf(Wn[o * kBH + u], dn_s[o], dht);
    float dct = dc[(size_t)r * kBH + u] + dht * og * (1.f - tc * tc);
    const float dog = dht * tc;
    const float dig = dct * gg, dgg = dct * ig, dfg = dct * cp;
    dg[u] = dig * ig * (1.f - ig);
    dg[kBH + u] = dfg * fg * (1.f - fg);
    dg[2 * kBH + u] = dgg * (1.f - gg * gg);
    dg[3 * kBH + u] = dog * og * (1.f - og);
    dc[(size_t)r * kBH + u] = dct * fg;
}

// ------------------------------------------------------------------------------------------
// Tiled fp32 GEMMs of the backward (64 x 64 tiles, 32-deep slices, register prefetch of the next
// slice so one global-load latency is paid per slice instead of per 16 products).
//   gemm_kernel<BT>:  C[M,N] = A[M,K] . op(B) (+ bias[n]);  op(B) = B[K,N] or (BT) B[N,K]^T
//   gemm_tn_kernel :  C[n][k] (+)= sum_r A[r][n] * B[r][k]   (weight gradients; one CTA owns a
//                     tile of C and walks all rows: deterministic)
// ------------------------------------------------------------------------------------------
constexpr int kGT = 64, kGK = 32;

__device__ __forceinline__ float4 ld4(const float* base, size_t row, int ld, int col, int rows, int cols,
                                      bool vec) {
    // 4 consecutive elements of a row-major matrix, zero outside [rows, cols)
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if ((int)row >= rows) return v;
    const float* p = base + row * (size_t)ld + col;
    if (vec && col + 3 < cols) return *reinterpret_cast<const float4*>(p);
    if (col < cols) v.x = p[0];
    if (col + 1 < cols) v.y = p[1];
    if (col + 2 < cols) v.z = p[2];
    if (col + 3 < cols) v.w = p[3];
    return v;
}

template <bool BT, int TM>
__global__ void __launch_bounds__(TM * 4) gemm_kernel(const float* __restrict__ A, int lda,
                                                      const float* __restrict__ B, int ldb,
                                                      float* __restrict__ Cm, int ldc, int M, int N, int K,
                                                      const float* __restrict__ bias, int vec) {
    constexpr int NT = TM * 4;                 // threads; each owns a 4 x 4 micro-tile of TM x 64
    constexpr int LA = TM * 8 / NT;            // float4 loads per thread for the A slice (TM x 32) = 2
    constexpr int LB = 64 * 8 / NT;            // ... for the B slice (64 x 32): 2 (TM = 64) or 4 (TM = 32)
    __shared__ __align__(16) float As[kGK][TM + 4];
    __shared__ __align__(16) float Bs[kGK][kGT + 4];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int m0 = blockIdx.y * TM, n0 = blockIdx.x * kGT;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    float4 ra[LA], rb[LB];
    auto load = [&](int k0) {
#pragma unroll
        for (int i = 0; i < LA; ++i) {
            const int f = tid + i * NT, row = f >> 3, kq = (f & 7) * 4;      // TM rows x 32 k
            ra[i] = ld4(A, (size_t)(m0 + row), lda, k0 + kq, M, K, vec);
        }
#pragma unroll
        for (int i = 0; i < LB; ++i) {
            const int f = tid + i * NT;
            if (BT) {
                const int row = f >> 3, kq = (f & 7) * 4;                    // 64 n x 32 k
                rb[i] = ld4(B, (size_t)(n0 + row), ldb, k0 + kq, N, K, vec);
            } else {
                const int kk = f >> 4, nq = (f & 15) * 4;                    // 32 k x 64 n
                rb[i] = ld4(B, (size_t)(k0 + kk), ldb, n0 + nq, K, N, vec);
            }
        }
    };
    auto store = [&]() {
#pragma unroll
        for (int i = 0; i < LA; ++i) {
            const int f = tid + i * NT, row = f >> 3, kq = (f & 7) * 4;
            As[kq + 0][row] = ra[i].x; As[kq + 1][row] = ra[i].y; As[kq + 2][row] = ra[i].z; As[kq + 3][row] = ra[i].w;
        }
#pragma unroll
        for (int i = 0; i < LB; ++i) {
            const int f = tid + i * NT;
            if (BT) {
                const int row = f >> 3, kq = (f & 7) * 4;
                Bs[kq + 0][row] = rb[i].x; Bs[kq + 1][row] = rb[i].y; Bs[kq + 2][row] = rb[i].z; Bs[kq + 3][row] = rb[i].w;
            } else {
                const int kk = f >> 4, nq = (f & 15) * 4;
                *reinterpret_cast<float4*>(&Bs[kk][nq]) = rb[i];
            }
        }
    };
    load(0);
    store();
    __syncthreads();
    for (int k0 = 0; k0 < K; k0 += kGK) {
        const bool more = k0 + kGK < K;
        if (more) load(k0 + kGK);
#pragma unroll
        for (int kk = 0; kk < kGK; ++kk) {
            const float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
            const float4 b = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
        if (more) {
            store();
            __syncthreads();
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int m = m0 + ty * 4 + i;
        if (m >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n = n0 + tx * 4 + j;
            if (n < N) Cm[(size_t)m * ldc + n] = acc[i][j] + (bias ? bias[n] : 0.f);
        }
    }
}

template <int TN>
__global__ void __launch_bounds__(TN * 4) gemm_tn_kernel(const float* __restrict__ A, int lda,
                                                         const float* __restrict__ B, int ldb,
                                                         float* __restrict__ Cm, int ldc, int R, int N, int Kc,
                                                         int vec) {
    constexpr int NT = TN * 4;
    constexpr int LA = TN * 8 / NT;            // A slice: 32 rows x TN cols
    constexpr int LB = 64 * 8 / NT;            // B slice: 32 rows x 64 cols
    __shared__ __align__(16) float As[kGK][TN + 4];
    __shared__ __align__(16) float Bs[kGK][kGT + 4];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int n0 = blockIdx.y * TN, k0c = blockIdx.x * kGT;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    float4 ra[LA], rb[LB];
    auto load = [&](int r0) {
#pragma unroll
        for (int i = 0; i < LA; ++i) {
            const int f = tid + i * NT, rr = f / (TN / 4), cq = (f % (TN / 4)) * 4;
            ra[i] = ld4(A, (size_t)(r0 + rr), lda, n0 + cq, R, N, vec);
        }
#pragma unroll
        for (int i = 0; i < LB; ++i) {
            const int f = tid + i * NT, rr = f >> 4, cq = (f & 15) * 4;
            rb[i] = ld4(B, (size_t)(r0 + rr), ldb, k0c + cq, R, Kc, vec);
        }
    };
    auto store = [&]() {
#pragma unroll
        for (int i = 0; i < LA; ++i) {
            const int f = tid + i * NT, rr = f / (TN / 4), cq = (f % (TN / 4)) * 4;
            *reinterpret_cast<float4*>(&As[rr][cq]) = ra[i];
        }
#pragma unroll
        for (int i = 0; i < LB; ++i) {
            const int f = tid + i * NT, rr = f >> 4, cq = (f & 15) * 4;
            *reinterpret_cast<float4*>(&Bs[rr][cq]) = rb[i];
        }
    };
    load(0);
    store();
    __syncthreads();
    for (int r0 = 0; r0 < R; r0 += kGK) {
        const bool more = r0 + kGK < R;
        if (more) load(r0 + kGK);
#pragma unroll
        for (int rr = 0; rr < kGK; ++rr) {
            const float4 a = *reinterpret_cast<const float4*>(&As[rr][ty * 4]);
            const float4 b = *reinterpret_cast<const float4*>(&Bs[rr][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
        if (more) {
            store();
            __syncthreads();
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int n = n0 + ty * 4 + i;
        if (n >= N) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int k = k0c + tx * 4 + j;
            if (k < Kc) Cm[(size_t)n * ldc + k] += acc[i][j];
        }
    }
}

// same product, rows split over gridDim.z: slice z writes its partial tile sums to part[z][n][k]
// (dense N x Kc); reduce_partials_kernel adds the slices in a fixed order.
template <int TN>
__global__ void __launch_bounds__(TN * 4) gemm_tn_split_kernel(const float* __restrict__ A, int lda,
                                                               const float* __restrict__ B, int ldb,
                                                               float* __restrict__ part, int R, int N, int Kc,
                                                               int rows_per_slice, int vec) {
    constexpr int NT = TN * 4;
    constexpr int LA = TN * 8 / NT;
    constexpr int LB = 64 * 8 / NT;
    __shared__ __align__(16) float As[kGK][TN + 4];
    __shared__ __align__(16) float Bs[kGK][kGT + 4];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int n0 = blockIdx.y * TN, k0c = blockIdx.x * kGT;
    const int rbeg = blockIdx.z * rows_per_slice, rend = min(R, rbeg + rows_per_slice);
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    float4 ra[LA], rb[LB];
    auto load = [&](int r0) {
#pragma unroll
        for (int i = 0; i < LA; ++i) {
            const int f = tid + i * NT, rr = f / (TN / 4), cq = (f % (TN / 4)) * 4;
            ra[i] = ld4(A, (size_t)(r0 + rr), lda, n0 + cq, rend, N, vec);
        }
#pragma unroll
        for (int i = 0; i < LB; ++i) {
            const int f = tid + i * NT, rr = f >> 4, cq = (f & 15) * 4;
            rb[i] = ld4(B, (size_t)(r0 + rr), ldb, k0c + cq, rend, Kc, vec);
        }
    };
    auto store = [&]() {
#pragma unroll
        for (int i = 0; i < LA; ++i) {
            const int f = tid + i * NT, rr = f / (TN / 4), cq = (f % (TN / 4)) * 4;
            *reinterpret_cast<float4*>(&As[rr][cq]) = ra[i];
        }
#pragma unroll
        for (int i = 0; i < LB; ++i) {
            const int f = tid + i * NT, rr = f >> 4, cq = (f & 15) * 4;
            *reinterpret_cast<float4*>(&Bs[rr][cq]) = rb[i];
        }
    };
    if (rbeg < rend) {
        load(rbeg);
        store();
    }
    __syncthreads();
    for (int r0 = rbeg; r0 < rend; r0 += kGK) {
        const bool more = r0 + kGK < rend;
        if (more) load(r0 + kGK);
#pragma unroll
        for (int rr = 0; rr < kGK; ++rr) {
            const float4 a = *reinterpret_cast<const float4*>(&As[rr][ty * 4]);
            const float4 b = *reinterpret_cast<const float4*>(&Bs[rr][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
        if (more) {
            store();
            __syncthreads();
        }
    }
    float* out = part + (size_t)blockIdx.z * N * Kc;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int n = n0 + ty * 4 + i;
        if (n >= N) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int k = k0c + tx * 4 + j;
            if (k < Kc) out[(size_t)n * Kc + k] = acc[i][j];
        }
    }
}

// C[n][k] (ldc) += sum_z part[z][n][k];  also used for column sums (N = 1)
__global__ void reduce_partials_kernel(const float* __restrict__ part, int Z, int N, int Kc, float* __restrict__ C,
                                       int ldc, float* __restrict__ C2) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)N * Kc) return;
    float s = 0.f;
    for (int z = 0; z < Z; ++z) s += part[(size_t)z * N * Kc + idx];
    const size_t n = idx / Kc, k = idx - n * Kc;
    C[n * ldc + k] += s;
    if (C2) C2[n * ldc + k] += s;
}

// part[z][n] = sum over the rows of slice z of A[r][n]
__global__ void __launch_bounds__(256) colsum_partial_kernel(const float* __restrict__ A, int lda, int R, int N,
                                                             int rows_per_slice, float* __restrict__ part) {
    __shared__ float sm[8][33];
    const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
    const int n = blockIdx.x * 32 + cx;
    const int rbeg = blockIdx.y * rows_per_slice, rend = min(R, rbeg + rows_per_slice);
    float s = 0.f;
    if (n < N)
        for (int r = rbeg + ry; r < rend; r += 8) s += A[(size_t)r * lda + n];
    sm[ry][cx] = s;
    __syncthreads();
    if (ry == 0 && n < N) {
        float t = 0.f;
#pragma unroll
        for (int q = 0; q < 8; ++q) t += sm[q][cx];
        part[(size_t)blockIdx.y * N + n] = t;
    }
}

// dst[r][o] = ref[r][o] > 0 ? src[r][o] : 0   (row strides given; dst may alias src)
__global__ void masked_copy_kernel(const float* __restrict__ ref, int ld_ref, const float* src, int ld_src,
                                   float* dst, int ld_dst, int rows, int cols) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)rows * cols) return;
    const size_t r = idx / cols;
    const int o = (int)(idx - r * cols);
    dst[r * ld_dst + o] = ref[r * ld_ref + o] > 0.f ? src[r * ld_src + o] : 0.f;
}

// dz = dX_pooled * (pooled > 0) in place (one_layer: pooled = relu(W1 grid + b1))
__global__ void relu_mask_kernel(const float* __restrict__ X, int ldx, float* __restrict__ dX, int ldd, int rows,
                                 int E, int P) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)rows * P) return;
    const size_t r = idx / P;
    const int o = (int)(idx - r * P);
    if (!(X[r * ldx + E + o] > 0.f)) dX[r * ldd + E + o] = 0.f;
}

// InputEmbedding backward (modules.py:24-30) over all saved (step, row) pairs: one CTA per
// embedding unit k, d pre[k] = dX[k] * (emb[k] > 0), fixed-order tree reduction.
__global__ void __launch_bounds__(256) bwd_embed_kernel(const float* __restrict__ X, int ldx,
                                                        const float* __restrict__ dXe, int ldd,
                                                        const float* __restrict__ vel, int rows_total,
                                                        float* __restrict__ dWe, float* __restrict__ dbe) {
    __shared__ float red[3][256];
    const int k = blockIdx.x, t = threadIdx.x;
    float gx = 0.f, gy = 0.f, gb = 0.f;
    for (int r = t; r < rows_total; r += 256) {
        if (X[(size_t)r * ldx + k] > 0.f) {
            const float d = dXe[(size_t)r * ldd + k];
            gx = fmaf(d, vel[2 * r], gx);
            gy = fmaf(d, vel[2 * r + 1], gy);
            gb += d;
        }
    }
    red[0][t] = gx; red[1][t] = gy; red[2][t] = gb;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (t < s) {
            red[0][t] += red[0][t + s]; red[1][t] += red[1][t + s]; red[2][t] += red[2][t + s];
        }
        __syncthreads();
    }
    if (t == 0) {
        dWe[2 * k] += red[0][0];
        dWe[2 * k + 1] += red[1][0];
        dbe[k] += red[2][0];
    }
}


// ------------------------------------------------------------------------------------------
// Social pooling backward (gridbased_pooling.py:145-170 through autograd).  The grid of observer i
// holds lat_j = W_enc h_j + b_enc of the winning neighbour of each occupied cell.
//   * d W1 sees the grid as it was written: winners only.
//   * d lat follows what autograd's index_put_ backward does for `occ[rows, oi] = other_values`
//     (gridbased_pooling.py:290-293): grad_values = grad_occ[oi] for EVERY written pair, so each
//     IN-RANGE pair (i, j) receives d grid_i[cell(i, j), :] = W1[:, cell-slab]^T dz1_i -- also the
//     pairs a later writer of the same cell overwrote; out-of-range pairs were replaced by the
//     constant before the write (:281-282) and receive nothing.
// In-range pairs are bucketed by cell with a stable counting sort (scene by scene, slots
// ascending), so every reduction below runs in a fixed order: results are run-to-run identical,
// no float atomics.  A slot is row * nm1 + jj (neighbour slot jj <-> j = jj + (jj >= i)).
// ------------------------------------------------------------------------------------------
__global__ void pair_count_kernel(const int* __restrict__ scene_off, const int* __restrict__ masked,
                                  const int* __restrict__ pair_cell, const uint8_t* __restrict__ pair_flag,
                                  int nm1, int cells, int* __restrict__ counts) {
    extern __shared__ int hist_s[];
    const int b = blockIdx.x, row0 = scene_off[b], n_s = scene_off[b + 1] - row0;
    for (int c = threadIdx.x; c < cells; c += blockDim.x) hist_s[c] = 0;
    __syncthreads();
    for (int idx = threadIdx.x; idx < n_s * nm1; idx += blockDim.x) {
        const int r = idx / nm1;
        const size_t slot = (size_t)row0 * nm1 + idx;
        if (pair_flag[slot] && !masked[row0 + r]) atomicAdd(&hist_s[pair_cell[slot]], 1);
    }
    __syncthreads();
    for (int c = threadIdx.x; c < cells; c += blockDim.x) counts[(size_t)b * cells + c] = hist_s[c];
}

// base[b][c] = pairs of cell c in scenes before b;  start[c] = pairs in cells before c
__global__ void pair_offsets_kernel(const int* __restrict__ counts, int B, int cells, int* __restrict__ base,
                                    int* __restrict__ start) {
    extern __shared__ int total_s[];
    for (int c = threadIdx.x; c < cells; c += blockDim.x) {
        int run = 0;
        for (int b = 0; b < B; ++b) {
            base[(size_t)b * cells + c] = run;
            run += counts[(size_t)b * cells + c];
        }
        total_s[c] = run;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int run = 0;
        for (int c = 0; c < cells; ++c) {
            start[c] = run;
            run += total_s[c];
        }
        start[cells] = run;
    }
}

// sorted[start[c] + base[b][c] + rank] = slot id, bit 31 set when the pair is NOT the winner of its
// cell (it then takes part in d lat but not in d W1); rank = earlier slots of the scene in cell c.
// Bit 30 ("dead"): an in-range pair of cell 0 whose observer's LAST writer of cell 0 is an out-of-range
// neighbour (or a padding slot).  The cell then holds the constant 0, and the reference's
// lp_pool2d(occ, 1, pool_size = 1) = sign(x) relu(|x|) has derivative sign(0)^2 = 0 at exactly 0
// (gridbased_pooling.py:304): no gradient reaches any writer of that cell.  (Found by the drop-in test
// against the unmodified Trainer.train_batch; a cell overwritten by a later IN-RANGE writer holds a non-zero
// latent vector and all its writers do receive gradient.)
__global__ void pair_place_kernel(const int* __restrict__ scene_off, const int* __restrict__ masked,
                                  const int* __restrict__ pair_cell, const uint8_t* __restrict__ pair_flag,
                                  const int* __restrict__ win_count, const uint32_t* __restrict__ win_ent, int nm1,
                                  int cells, const int* __restrict__ base, const int* __restrict__ start,
                                  int pad_to_max, unsigned* __restrict__ sorted) {
    extern __shared__ short cell_s[];         // [n_s * nm1] cell of the in-range pairs, -1 otherwise
    const int b = blockIdx.x, row0 = scene_off[b], n_s = scene_off[b + 1] - row0;
    for (int idx = threadIdx.x; idx < n_s * nm1; idx += blockDim.x) {
        const size_t slot = (size_t)row0 * nm1 + idx;
        cell_s[idx] = (short)((pair_flag[slot] && !masked[row0 + idx / nm1]) ? pair_cell[slot] : -1);
    }
    __syncthreads();
    const int n_slots = pad_to_max ? nm1 : n_s - 1;      // neighbour slots that write at all
    for (int idx = threadIdx.x; idx < n_s * nm1; idx += blockDim.x) {
        const int cell = cell_s[idx];
        if (cell < 0) continue;
        int rank = 0;
        for (int q = 0; q < idx; ++q) rank += cell_s[q] == cell;
        const int r = idx / nm1, jj = idx - r * nm1, j = jj + (jj >= r);
        const uint32_t want = ((uint32_t)cell << 16) | (uint32_t)j;
        bool winner = false;
        const int cnt = win_count[row0 + r];
        for (int e = 0; e < cnt; ++e) winner |= win_ent[(size_t)(row0 + r) * nm1 + e] == want;
        bool dead = false;
        if (cell == 0) {
            // last writer of cell 0 for this observer: in-range pairs of cell 0 and every out-of-range slot write it
            for (int q = n_slots - 1; q >= 0; --q) {
                const int cq = cell_s[r * nm1 + q];
                if (cq == 0) break;                                   // an in-range pair wrote last: the cell is alive
                if (cq < 0) { dead = true; break; }                   // out of range (or padding): constant
            }
        }
        sorted[start[cell] + base[(size_t)b * cells + cell] + rank] =
            (unsigned)((size_t)row0 * nm1 + idx) | (winner ? 0u : 0x80000000u) | (dead ? 0x40000000u : 0u);
    }
}

// dgrid[slot][ch] = sum_o dz1[row(slot)][o] * Wt1[cell][ch][o]  for the pairs of one cell
// (64 pairs x C channels per CTA, 64-deep slices of o through shared memory)
constexpr int kDgPairs = 64, kDgK = 64;

template <int C>
__global__ void __launch_bounds__(256) social_dgrid_kernel(const unsigned* __restrict__ sorted,
                                                           const int* __restrict__ start,
                                                           const float* __restrict__ dz1, int d1,
                                                           const float* __restrict__ Wt1, int nm1,
                                                           float* __restrict__ dgrid) {
    constexpr int CQ = C / 4;                       // channels per thread
    __shared__ __align__(16) float As[kDgPairs][kDgK + 4];
    __shared__ __align__(16) float Bs[C][kDgK + 4];
    __shared__ int slot_s[kDgPairs];
    const int cell = blockIdx.x;
    const int tid = threadIdx.x;
    const int pr = tid >> 2, cq = tid & 3;
    // a cell can hold more pairs than gridDim.y * 64 (several neighbours of one observer in the same cell, all
    // scenes of the batch): every CTA walks its chunks with stride gridDim.y
    for (int p0 = start[cell] + blockIdx.y * kDgPairs; p0 < start[cell + 1]; p0 += gridDim.y * kDgPairs) {
    const int p1 = min(start[cell + 1], p0 + kDgPairs);
    const int np = p1 - p0;
    __syncthreads();
    if (tid < kDgPairs) slot_s[tid] = tid < np ? (int)(sorted[p0 + tid] & 0x7fffffffu) : -1;       // bit 30 (dead) kept
    __syncthreads();
    float acc[CQ];
#pragma unroll
    for (int q = 0; q < CQ; ++q) acc[q] = 0.f;
    const float* Wc = Wt1 + (size_t)cell * C * d1;
    for (int k0 = 0; k0 < d1; k0 += kDgK) {
        for (int idx = tid; idx < kDgPairs * (kDgK / 4); idx += 256) {
            const int r = idx / (kDgK / 4), c4 = (idx % (kDgK / 4)) * 4;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            const int slot = slot_s[r] < 0 ? -1 : (slot_s[r] & 0x3fffffff);
            if (slot >= 0) {
                const float* src = dz1 + (size_t)(slot / nm1) * d1 + k0 + c4;
                if (k0 + c4 + 3 < d1) v = *reinterpret_cast<const float4*>(src);
                else {
                    if (k0 + c4 < d1) v.x = src[0];
                    if (k0 + c4 + 1 < d1) v.y = src[1];
                    if (k0 + c4 + 2 < d1) v.z = src[2];
                }
            }
            *reinterpret_cast<float4*>(&As[r][c4]) = v;
        }
        for (int idx = tid; idx < C * (kDgK / 4); idx += 256) {
            const int r = idx / (kDgK / 4), c4 = (idx % (kDgK / 4)) * 4;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            const float* src = Wc + (size_t)r * d1 + k0 + c4;
            if (k0 + c4 + 3 < d1) v = *reinterpret_cast<const float4*>(src);
            else {
                if (k0 + c4 < d1) v.x = src[0];
                if (k0 + c4 + 1 < d1) v.y = src[1];
                if (k0 + c4 + 2 < d1) v.z = src[2];
            }
            *reinterpret_cast<float4*>(&Bs[r][c4]) = v;
        }
        __syncthreads();
#pragma unroll 4
        for (int o = 0; o < kDgK; o += 4) {
            const float4 a = *reinterpret_cast<const float4*>(&As[pr][o]);
#pragma unroll
            for (int q = 0; q < CQ; ++q) {
                const float4 w = *reinterpret_cast<const float4*>(&Bs[cq * CQ + q][o]);
                acc[q] = fmaf(a.x, w.x, fmaf(a.y, w.y, fmaf(a.z, w.z, fmaf(a.w, w.w, acc[q]))));
            }
        }
        __syncthreads();
    }
    if (pr < np) {
        const bool dead = (slot_s[pr] & 0x40000000) != 0;             // its cell holds the constant: zero gradient
        float* out = dgrid + (size_t)(slot_s[pr] & 0x3fffffff) * C + cq * CQ;
#pragma unroll
        for (int q = 0; q < CQ; ++q) out[q] = dead ? 0.f : acc[q];
    }
    }
}


// ------------------------------------------------------------------------------------------
// social_dgrid on the tensor cores (warp-level mma.sync, 3-pass bf16 split, fp32 accumulation): per grid cell the
// pairs of the cell form a GEMM  dgrid[pairs, 16] = dz1[rows of the pairs, d1] . Wt1[cell]^T[d1, 16]  whose A rows are
// gathered.  One CTA = one cell (its weight slab as bf16 hi | lo in shared memory, loaded once), 64 pairs per chunk:
// warp = (16-pair tile, half of the d1 range); the A fragments come straight from global memory (a quad reads 32
// contiguous bytes of a dz1 row per load) and are split into (hi, lo) in registers.  The FFMA version above needed
// five shared-memory loads per 16 FMAs and ran at 8.6 TFLOP/s.
// ------------------------------------------------------------------------------------------
__global__ void split_bf16_flat_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ hi,
                                  __nv_bfloat16* __restrict__ lo, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const float v = src[i];
        const __nv_bfloat16 h = __float2bfloat16_rn(v);
        hi[i] = h;
        lo[i] = __float2bfloat16_rn(v - __bfloat162float(h));
    }
}

__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void split2(const float2 v, uint32_t& hi, uint32_t& lo) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(v.x, v.y);
    const __nv_bfloat162 l = __floats2bfloat162_rn(v.x - __low2float(h), v.y - __high2float(h));
    hi = *reinterpret_cast<const uint32_t*>(&h);
    lo = *reinterpret_cast<const uint32_t*>(&l);
}

constexpr int kDmPairs = 64, kDmYs = 8;
static size_t dgrid_mma_smem(int d1) { return (size_t)2 * 16 * (d1 + 8) * sizeof(__nv_bfloat16) + 4 * 16 * 16 * sizeof(float) + kDmPairs * sizeof(int); }

__global__ void __launch_bounds__(256) social_dgrid_mma_kernel(const unsigned* __restrict__ sorted, const int* __restrict__ start,
                                                               const float* __restrict__ dz1, int d1,
                                                               const __nv_bfloat16* __restrict__ w_hi,
                                                               const __nv_bfloat16* __restrict__ w_lo, int nm1,
                                                               float* __restrict__ dgrid) {
    extern __shared__ __align__(16) unsigned char smem_dm[];
    const int ldw = d1 + 8;                                       // bf16 elements per weight row (+8: conflict-free fragments)
    __nv_bfloat16* Bh = reinterpret_cast<__nv_bfloat16*>(smem_dm);
    __nv_bfloat16* Bl = Bh + 16 * ldw;
    float* red = reinterpret_cast<float*>(Bl + 16 * ldw);         // [4 pair tiles][16 rows][16 channels]
    int* slot_s = reinterpret_cast<int*>(red + 4 * 16 * 16);
    const int cell = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int p_begin = start[cell] + blockIdx.y * kDmPairs, p_end = start[cell + 1];
    if (p_begin >= p_end) return;
    for (int idx = tid; idx < 16 * (d1 / 8); idx += 256) {
        const int r = idx / (d1 / 8), c8 = (idx - r * (d1 / 8)) * 8;
        *reinterpret_cast<uint4*>(Bh + r * ldw + c8) = *reinterpret_cast<const uint4*>(w_hi + ((size_t)cell * 16 + r) * d1 + c8);
        *reinterpret_cast<uint4*>(Bl + r * ldw + c8) = *reinterpret_cast<const uint4*>(w_lo + ((size_t)cell * 16 + r) * d1 + c8);
    }
    const int pt = warp & 3, kh = warp >> 2, g = lane >> 2, t = lane & 3;
    const int khalf = d1 / 2;
    for (int p0 = p_begin; p0 < p_end; p0 += gridDim.y * kDmPairs) {
        const int np = min(kDmPairs, p_end - p0);
        __syncthreads();
        if (tid < kDmPairs) slot_s[tid] = tid < np ? (int)(sorted[p0 + tid] & 0x7fffffffu) : -1;
        __syncthreads();
        const int s0 = slot_s[pt * 16 + g], s1 = slot_s[pt * 16 + g + 8];
        const float* a0p = s0 < 0 ? nullptr : dz1 + (size_t)((s0 & 0x3fffffff) / nm1) * d1 + kh * khalf + 2 * t;
        const float* a1p = s1 < 0 ? nullptr : dz1 + (size_t)((s1 & 0x3fffffff) / nm1) * d1 + kh * khalf + 2 * t;
        float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
        const float2 z2 = make_float2(0.f, 0.f);
        const uint32_t* bh0 = reinterpret_cast<const uint32_t*>(Bh + g * ldw + kh * khalf + 2 * t);
        const uint32_t* bl0 = reinterpret_cast<const uint32_t*>(Bl + g * ldw + kh * khalf + 2 * t);
        const int ldw2 = 8 * ldw / 2;                              // 32-bit words between channel g and g + 8
#pragma unroll 4
        for (int k0 = 0; k0 < khalf; k0 += 16) {
            const float2 v00 = a0p ? *reinterpret_cast<const float2*>(a0p + k0) : z2;
            const float2 v10 = a1p ? *reinterpret_cast<const float2*>(a1p + k0) : z2;
            const float2 v01 = a0p ? *reinterpret_cast<const float2*>(a0p + k0 + 8) : z2;
            const float2 v11 = a1p ? *reinterpret_cast<const float2*>(a1p + k0 + 8) : z2;
            uint32_t ah[4], al[4];
            split2(v00, ah[0], al[0]); split2(v10, ah[1], al[1]); split2(v01, ah[2], al[2]); split2(v11, ah[3], al[3]);
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
                const uint32_t h0 = bh0[nt * ldw2 + k0 / 2], h1 = bh0[nt * ldw2 + k0 / 2 + 4];
                const uint32_t l0 = bl0[nt * ldw2 + k0 / 2], l1 = bl0[nt * ldw2 + k0 / 2 + 4];
                mma_bf16_16816(acc[nt], ah, h0, h1);
                mma_bf16_16816(acc[nt], al, h0, h1);
                mma_bf16_16816(acc[nt], ah, l0, l1);
            }
        }
        // the two halves of the d1 range: warps 4..7 hand their sums to warps 0..3
        float* rp = red + pt * 256;
        if (kh == 1) {
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
                rp[g * 16 + nt * 8 + 2 * t] = acc[nt][0]; rp[g * 16 + nt * 8 + 2 * t + 1] = acc[nt][1];
                rp[(g + 8) * 16 + nt * 8 + 2 * t] = acc[nt][2]; rp[(g + 8) * 16 + nt * 8 + 2 * t + 1] = acc[nt][3];
            }
        }
        __syncthreads();
        if (kh == 0) {
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int sl = half ? s1 : s0;
                if (sl < 0) continue;
                const bool dead = (sl & 0x40000000) != 0;          // its cell holds the constant: zero gradient
                float* out = dgrid + (size_t)(sl & 0x3fffffff) * 16;
                const int r = g + 8 * half;
#pragma unroll
                for (int nt = 0; nt < 2; ++nt) {
                    const float x = acc[nt][2 * half] + rp[r * 16 + nt * 8 + 2 * t];
                    const float y = acc[nt][2 * half + 1] + rp[r * 16 + nt * 8 + 2 * t + 1];
                    *reinterpret_cast<float2*>(out + nt * 8 + 2 * t) = dead ? make_float2(0.f, 0.f) : make_float2(x, y);
                }
            }
        }
    }
}

// per scene: dlat[j] = sum over the observers i (rows ascending) whose pair (i, j) is in range of
// that pair's dgrid slot; then the social part of d h_prev[j] = W_enc^T dlat[j] is added to the
// by-pass buffer that the next (earlier) step's cell kernel reads.
__global__ void __launch_bounds__(256) social_scene_reduce_kernel(
    const int* __restrict__ scene_off, const int* __restrict__ masked, const uint8_t* __restrict__ pair_flag,
    int nm1, int C, const float* __restrict__ dgrid, const float* __restrict__ Wenc, float* __restrict__ dlat,
    float* __restrict__ dh_add) {
    extern __shared__ float dl_s[];       // [n_s][C]
    const int b = blockIdx.x, row0 = scene_off[b], n_s = scene_off[b + 1] - row0;
    for (int idx = threadIdx.x; idx < n_s * C; idx += blockDim.x) {
        const int j = idx / C, ch = idx - j * C;
        float sum = 0.f;
        for (int r = 0; r < n_s; ++r) {
            if (r == j || masked[row0 + r]) continue;
            const size_t slot = (size_t)(row0 + r) * nm1 + (j - (j > r));
            if (pair_flag[slot]) sum += dgrid[slot * C + ch];
        }
        dl_s[idx] = sum;
        dlat[(size_t)(row0 + j) * C + ch] = sum;
    }
    __syncthreads();
    if (dh_add) {
        for (int idx = threadIdx.x; idx < n_s * kBH; idx += blockDim.x) {
            const int j = idx / kBH, u = idx - j * kBH;
            float a = 0.f;
            for (int ch = 0; ch < C; ++ch) a = fmaf(dl_s[j * C + ch], Wenc[ch * kBH + u], a);
            dh_add[(size_t)(row0 + j) * kBH + u] += a;
        }
    }
}


// dWt1 on the tensor cores (warp-level mma.sync, 3-pass bf16 split): per cell
//   dWt1[cell][16 ch][d1] += lat^T [16 ch x pairs] . dz1[rows of the pairs][d1]
// M = the 16 latent channels, K = the pairs of the cell (16 per k-step), N = 32 output columns per warp (4 n-tiles).
// The A fragments (latent vectors of the winning pairs, zero for overwritten ones) come from shared memory, the B
// fragments straight from the gathered dz1 rows (lane (g, t) reads column o0 + g of the rows of pairs 2t, 2t+1, 2t+8,
// 2t+9); one CTA = (cell, 256 columns).  The FFMA kernel below it is kept for C != 16.
__global__ void __launch_bounds__(256) social_dw1_mma_kernel(const unsigned* __restrict__ sorted, const int* __restrict__ start,
                                                             int nm1, const int* __restrict__ row_scene,
                                                             const int* __restrict__ scene_off, const float* __restrict__ lat,
                                                             const float* __restrict__ dz1, int d1, float* __restrict__ dWt1) {
    __shared__ float lat_s[32][17];          // [pair][channel], +1: conflict-free column reads
    __shared__ int row_s[32];
    const int cell = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const int p0 = start[cell], p1 = start[cell + 1];
    if (p0 >= p1) return;
    const int obase = blockIdx.y * 256 + warp * 32;
    const bool active = obase < d1;          // d1 % 32 == 0: a warp is entirely inside or outside
    float acc[4][4];
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
        for (int k = 0; k < 4; ++k) acc[nt][k] = 0.f;
    for (int pb = p0; pb < p1; pb += 32) {
        const int nb = min(32, p1 - pb);
        __syncthreads();
        for (int idx = tid; idx < 32 * 16; idx += 256) {
            const int tt = idx >> 4, ch = idx & 15;
            float v = 0.f;
            int rowi = 0;
            if (tt < nb) {
                const unsigned sv = sorted[pb + tt];
                const int slot = (int)(sv & 0x3fffffffu);
                const int i = slot / nm1, jj = slot - i * nm1;
                const int s0 = scene_off[row_scene[i]];
                const int j = jj + (jj >= i - s0);
                // overwritten pairs are not in the grid: they contribute to d lat only
                v = (sv & 0x80000000u) ? 0.f : lat[(size_t)(s0 + j) * 16 + ch];
                rowi = i;
            }
            lat_s[tt][ch] = v;
            if (ch == 0) row_s[tt] = rowi;       // padded pairs read row 0 with a zero latent vector
        }
        __syncthreads();
        if (!active) continue;
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
            if (ks * 16 >= nb) break;
            const int kb = ks * 16;
            uint32_t ah[4], al[4];
            split2(make_float2(lat_s[kb + 2 * t][g], lat_s[kb + 2 * t + 1][g]), ah[0], al[0]);
            split2(make_float2(lat_s[kb + 2 * t][g + 8], lat_s[kb + 2 * t + 1][g + 8]), ah[1], al[1]);
            split2(make_float2(lat_s[kb + 2 * t + 8][g], lat_s[kb + 2 * t + 9][g]), ah[2], al[2]);
            split2(make_float2(lat_s[kb + 2 * t + 8][g + 8], lat_s[kb + 2 * t + 9][g + 8]), ah[3], al[3]);
            const float* r0 = dz1 + (size_t)row_s[kb + 2 * t] * d1 + obase + g;
            const float* r1 = dz1 + (size_t)row_s[kb + 2 * t + 1] * d1 + obase + g;
            const float* r2 = dz1 + (size_t)row_s[kb + 2 * t + 8] * d1 + obase + g;
            const float* r3 = dz1 + (size_t)row_s[kb + 2 * t + 9] * d1 + obase + g;
#pragma unroll
            for (int nt = 0; nt < 4; ++nt) {
                uint32_t bh0, bl0, bh1, bl1;
                split2(make_float2(__ldg(r0 + nt * 8), __ldg(r1 + nt * 8)), bh0, bl0);
                split2(make_float2(__ldg(r2 + nt * 8), __ldg(r3 + nt * 8)), bh1, bl1);
                mma_bf16_16816(acc[nt], ah, bh0, bh1);
                mma_bf16_16816(acc[nt], al, bh0, bh1);
                mma_bf16_16816(acc[nt], ah, bl0, bl1);
            }
        }
    }
    if (active) {
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
            float* d0 = dWt1 + ((size_t)cell * 16 + g) * d1 + obase + nt * 8 + 2 * t;
            float* d8 = dWt1 + ((size_t)cell * 16 + g + 8) * d1 + obase + nt * 8 + 2 * t;
            float2 v0 = *reinterpret_cast<float2*>(d0), v8 = *reinterpret_cast<float2*>(d8);
            v0.x += acc[nt][0]; v0.y += acc[nt][1]; v8.x += acc[nt][2]; v8.y += acc[nt][3];
            *reinterpret_cast<float2*>(d0) = v0;
            *reinterpret_cast<float2*>(d8) = v8;
        }
    }
}

// dWt1[cell][ch][o] += sum over the cell's pairs (sorted order) of dz1[i][o] * lat_j[ch]
template <int C>
__global__ void __launch_bounds__(256) social_dw1_kernel(const unsigned* __restrict__ sorted,
                                                         const int* __restrict__ start, int nm1,
                                                         const int* __restrict__ row_scene,
                                                         const int* __restrict__ scene_off,
                                                         const float* __restrict__ lat,
                                                         const float* __restrict__ dz1, int d1,
                                                         float* __restrict__ dWt1) {
    __shared__ float lat_s[32][C];
    __shared__ int row_s[32];
    const int cell = blockIdx.x, o = blockIdx.y * 256 + threadIdx.x;
    const int p0 = start[cell], p1 = start[cell + 1];
    if (p0 >= p1) return;
    float acc[C];
#pragma unroll
    for (int c = 0; c < C; ++c) acc[c] = 0.f;
    for (int pb = p0; pb < p1; pb += 32) {
        const int nb = min(32, p1 - pb);
        __syncthreads();
        for (int idx = threadIdx.x; idx < nb * C; idx += 256) {
            const int t = idx / C, ch = idx - t * C;
            const unsigned sv = sorted[pb + t];
            const int slot = (int)(sv & 0x3fffffffu);
            const int i = slot / nm1, jj = slot - i * nm1;
            const int s0 = scene_off[row_scene[i]];
            const int j = jj + (jj >= i - s0);
            // overwritten pairs are not in the grid: they contribute to d lat only
            lat_s[t][ch] = (sv & 0x80000000u) ? 0.f : lat[(size_t)(s0 + j) * C + ch];
            if (ch == 0) row_s[t] = i;
        }
        __syncthreads();
        if (o < d1) {
#pragma unroll 4
            for (int t = 0; t < nb; ++t) {
                const float dz = dz1[(size_t)row_s[t] * d1 + o];
#pragma unroll
                for (int c = 0; c < C; ++c) acc[c] = fmaf(dz, lat_s[t][c], acc[c]);
            }
        }
    }
    if (o < d1) {
#pragma unroll
        for (int c = 0; c < C; ++c) dWt1[((size_t)cell * C + c) * d1 + o] += acc[c];
    }
}

// dW1[o][ch * cells + cell] += dWt1[cell][ch][o]   (back to the reference's parameter layout)
__global__ void untranspose_add_kernel(const float* __restrict__ dWt1, float* __restrict__ dW1, int cells, int C,
                                       int d1) {
    const size_t total = (size_t)cells * C * d1;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (size_t)gridDim.x * blockDim.x) {
        const int o = (int)(idx % d1);
        const size_t cc = idx / d1;
        const int ch = (int)(cc % C), cell = (int)(cc / C);
        dW1[(size_t)o * C * cells + (size_t)ch * cells + cell] += dWt1[idx];
    }
}

// hidden1 of a step as fp32: from the bf16 (hi, lo) pair the tensor-core layer consumed, or a copy
__global__ void merge_split_kernel(const __nv_bfloat16* __restrict__ hi, const __nv_bfloat16* __restrict__ lo,
                                   const float* __restrict__ src, float* __restrict__ dst, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        dst[i] = hi ? __bfloat162float(hi[i]) + __bfloat162float(lo[i]) : src[i];
}

__global__ void iota_kernel(int* __restrict__ p, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = i;
}

}  // namespace tb2

using namespace tb2;

namespace tb2 {
int resolve_step_inputs(const tb2_layout* l, const float* observed, int obs_length, const float* truth,
                        const float* positions, int s, Workspace* ws, const float** o1, const float** o2,
                        int* phase, cudaStream_t st);

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }


// ------------------------------------------------------------------------------------------
// Large plain GEMMs of the all-row (social) backward: cuBLAS with FP32 emulation on the bf16 tensor cores
// (CUBLAS_COMPUTE_32F_EMULATED_16BFX9: every fp32 operand is split into three bf16 values, nine products,
// fp32-accurate) -- library code for plain library GEMMs; everything with a gather, a mask or a fused epilogue
// stays in the kernels of this file.  Where a cuBLAS build rejects the emulated mode, plain fp32 cuBLAS is used.
// ------------------------------------------------------------------------------------------
// cuBLAS is bound at run time (dlopen): inside a torch process the already loaded libcublas.so.12 is used, whatever
// its minor version; entry points a build does not have (cublasSetEmulationStrategy) are simply skipped, and without
// the library the FFMA kernels below do the work.
struct CublasApi {
    cublasStatus_t (*create)(cublasHandle_t*) = nullptr;
    cublasStatus_t (*set_stream)(cublasHandle_t, cudaStream_t) = nullptr;
    cublasStatus_t (*gemm_ex)(cublasHandle_t, cublasOperation_t, cublasOperation_t, int, int, int, const void*, const void*,
                              cudaDataType, int, const void*, cudaDataType, int, const void*, void*, cudaDataType, int,
                              cublasComputeType_t, cublasGemmAlgo_t) = nullptr;
    cublasStatus_t (*set_emulation)(cublasHandle_t, cublasEmulationStrategy_t) = nullptr;
    bool ok = false;
};
static const CublasApi& cublas_api() {
    static CublasApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        void* lib = dlopen("libcublas.so.12", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) lib = dlopen("libcublas.so", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) return;
        api.create = reinterpret_cast<decltype(api.create)>(dlsym(lib, "cublasCreate_v2"));
        api.set_stream = reinterpret_cast<decltype(api.set_stream)>(dlsym(lib, "cublasSetStream_v2"));
        api.gemm_ex = reinterpret_cast<decltype(api.gemm_ex)>(dlsym(lib, "cublasGemmEx"));
        api.set_emulation = reinterpret_cast<decltype(api.set_emulation)>(dlsym(lib, "cublasSetEmulationStrategy"));
        api.ok = api.create && api.set_stream && api.gemm_ex;
    });
    return api;
}

static cublasHandle_t cublas_for_device() {
    if (!cublas_api().ok) return nullptr;
    static std::mutex mu;
    static cublasHandle_t handles[64] = {nullptr};
    std::lock_guard<std::mutex> lock(mu);
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
    cublasHandle_t& h = handles[dev & 63];
    if (!h) {
        if (cublas_api().create(&h) != CUBLAS_STATUS_SUCCESS) { h = nullptr; return nullptr; }
        if (cublas_api().set_emulation) cublas_api().set_emulation(h, CUBLAS_EMULATION_STRATEGY_EAGER);
    }
    return h;
}

// column-major view: C(m x n) = alpha * op(A)(m x k) . op(B)(k x n) + beta * C; false = not taken (caller falls back)
static bool cublas_gemm(cublasOperation_t ta, cublasOperation_t tb, int m, int n, int k, const float* A, int lda,
                        const float* B, int ldb, float beta, float* C, int ldc, const char* name, cudaStream_t st) {
    if ((double)m * n * k < 3.2e7) return false;            // small problems: the FFMA kernels (deterministic split order)
    cublasHandle_t h = cublas_for_device();
    if (!h) return false;
    const CublasApi& api = cublas_api();
    static bool emulation_ok = true;
    const float alpha = 1.f;
    KernelTimer kt(name, st);
    if (api.set_stream(h, st) != CUBLAS_STATUS_SUCCESS) return false;
    cublasStatus_t rc = CUBLAS_STATUS_NOT_SUPPORTED;
    if (emulation_ok) {
        rc = api.gemm_ex(h, ta, tb, m, n, k, &alpha, A, CUDA_R_32F, lda, B, CUDA_R_32F, ldb, &beta, C, CUDA_R_32F, ldc,
                         CUBLAS_COMPUTE_32F_EMULATED_16BFX9, CUBLAS_GEMM_DEFAULT);
        if (rc != CUBLAS_STATUS_SUCCESS) emulation_ok = false;
    }
    if (rc != CUBLAS_STATUS_SUCCESS)
        rc = api.gemm_ex(h, ta, tb, m, n, k, &alpha, A, CUDA_R_32F, lda, B, CUDA_R_32F, ldb, &beta, C, CUDA_R_32F, ldc,
                         CUBLAS_COMPUTE_32F, CUBLAS_GEMM_DEFAULT);
    return rc == CUBLAS_STATUS_SUCCESS;
}

__global__ void fill_bias_rows_kernel(float* __restrict__ C, int ldc, int M, int N, const float* __restrict__ bias) {
    const size_t total = (size_t)M * (N / 4);
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const size_t r = idx / (N / 4);
        const int c4 = (int)(idx - r * (N / 4)) * 4;
        *reinterpret_cast<float4*>(C + r * ldc + c4) = *reinterpret_cast<const float4*>(bias + c4);
    }
}

// C = A . B (+bias), B [K, N] row-major
static int gemm_nn(const float* A, int lda, const float* B, int ldb, float* C, int ldc, int M, int N, int K,
                   const float* bias, cudaStream_t st) {
    {   // row-major C = A . B  <=>  column-major C^T (N x M) = B^T-view (N x K) . A^T-view (K x M)
        const bool bias_ok = !bias || (N % 4 == 0 && ldc % 4 == 0 && aligned16(C) && aligned16(bias));
        if (bias_ok && (double)M * N * K >= 3.2e7) {
            if (bias) {
                fill_bias_rows_kernel<<<1184, 256, 0, st>>>(C, ldc, M, N, bias);
                TB2_LAUNCH_CHECK();
            }
            if (cublas_gemm(CUBLAS_OP_N, CUBLAS_OP_N, N, M, K, B, ldb, A, lda, bias ? 1.f : 0.f, C, ldc, "bwd_gemm_cublas", st))
                return TB2_OK;
        }
    }
    const int vec = (lda % 4 == 0 && ldb % 4 == 0 && aligned16(A) && aligned16(B)) ? 1 : 0;
    const bool small = (size_t)((M + 63) / 64) * ((N + kGT - 1) / kGT) < 148;     // few tiles: halve them
    {
        KernelTimer kt("bwd_gemm", st);
        if (small)
            gemm_kernel<false, 32><<<dim3((N + kGT - 1) / kGT, (M + 31) / 32), 128, 0, st>>>(A, lda, B, ldb, C, ldc, M,
                                                                                         N, K, bias, vec);
        else
            gemm_kernel<false, 64><<<dim3((N + kGT - 1) / kGT, (M + 63) / 64), 256, 0, st>>>(A, lda, B, ldb, C, ldc, M,
                                                                                         N, K, bias, vec);
    }
    TB2_LAUNCH_CHECK();
    return TB2_OK;
}

// C = A . B^T, B [N, K] row-major
static int gemm_nt(const float* A, int lda, const float* B, int ldb, float* C, int ldc, int M, int N, int K,
                   cudaStream_t st) {
    // row-major C = A . B^T, B [N, K]  <=>  column-major C^T (N x M) = (B-view (K x N))^T . A-view (K x M)
    if (cublas_gemm(CUBLAS_OP_T, CUBLAS_OP_N, N, M, K, B, ldb, A, lda, 0.f, C, ldc, "bwd_gemm_cublas", st)) return TB2_OK;
    const int vec = (lda % 4 == 0 && ldb % 4 == 0 && aligned16(A) && aligned16(B)) ? 1 : 0;
    const bool small = (size_t)((M + 63) / 64) * ((N + kGT - 1) / kGT) < 148;
    {
        KernelTimer kt("bwd_gemm", st);
        if (small)
            gemm_kernel<true, 32><<<dim3((N + kGT - 1) / kGT, (M + 31) / 32), 128, 0, st>>>(A, lda, B, ldb, C, ldc, M,
                                                                                        N, K, nullptr, vec);
        else
            gemm_kernel<true, 64><<<dim3((N + kGT - 1) / kGT, (M + 63) / 64), 256, 0, st>>>(A, lda, B, ldb, C, ldc, M,
                                                                                        N, K, nullptr, vec);
    }
    TB2_LAUNCH_CHECK();
    return TB2_OK;
}

// C[n][k] += sum_r A[r][n] B[r][k]; rows are split over CTAs when the output has few tiles
// (partials in `scratch`, summed in a fixed order: run-to-run deterministic)
static int gemm_tn(const float* A, int lda, const float* B, int ldb, float* C, int ldc, int R, int N, int Kc,
                   float* scratch, size_t scratch_floats, cudaStream_t st) {
    if (R <= 0) return TB2_OK;
    // row-major C (N x Kc) += A^T . B  <=>  column-major C^T (Kc x N) += B-view (Kc x R) . (A-view (N x R))^T
    if (cublas_gemm(CUBLAS_OP_N, CUBLAS_OP_T, Kc, N, R, B, ldb, A, lda, 1.f, C, ldc, "bwd_gemm_tn_cublas", st)) return TB2_OK;
    const int vec = (lda % 4 == 0 && ldb % 4 == 0 && aligned16(A) && aligned16(B)) ? 1 : 0;
    const int tiles32 = ((N + 31) / 32) * ((Kc + kGT - 1) / kGT);
    int Z = (2 * 148 + tiles32 - 1) / tiles32;
    if (Z > (R + 127) / 128) Z = (R + 127) / 128;
    while (Z > 1 && (size_t)Z * N * Kc > scratch_floats) --Z;
    if (Z <= 1) {
        KernelTimer kt("bwd_gemm_tn", st);
        gemm_tn_kernel<32><<<dim3((Kc + kGT - 1) / kGT, (N + 31) / 32), 128, 0, st>>>(A, lda, B, ldb, C, ldc, R, N, Kc,
                                                                                  vec);
    } else {
        int rps = (R + Z - 1) / Z;
        rps = (rps + kGK - 1) / kGK * kGK;
        Z = (R + rps - 1) / rps;
        KernelTimer kt("bwd_gemm_tn", st);
        gemm_tn_split_kernel<32><<<dim3((Kc + kGT - 1) / kGT, (N + 31) / 32, Z), 128, 0, st>>>(A, lda, B, ldb, scratch,
                                                                                           R, N, Kc, rps, vec);
        reduce_partials_kernel<<<(unsigned)(((size_t)N * Kc + 255) / 256), 256, 0, st>>>(scratch, Z, N, Kc, C, ldc,
                                                                                      nullptr);
    }
    TB2_LAUNCH_CHECK();
    return TB2_OK;
}

static int colsum(const float* A, int lda, int R, int N, float* out, float* out2, float* scratch,
                  size_t scratch_floats, cudaStream_t st) {
    if (R <= 0) return TB2_OK;
    int Z = (R + 63) / 64;
    if (Z > 64) Z = 64;
    while (Z > 1 && (size_t)Z * N > scratch_floats) --Z;
    const int rps = (R + Z - 1) / Z;
    Z = (R + rps - 1) / rps;
    colsum_partial_kernel<<<dim3((N + 31) / 32, Z), 256, 0, st>>>(A, lda, R, N, rps, scratch);
    reduce_partials_kernel<<<(N + 255) / 256, 256, 0, st>>>(scratch, Z, 1, N, out, N, out2);
    TB2_LAUNCH_CHECK();
    return TB2_OK;
}

// Carving of the backward workspace (floats).  Per (step, row) records are kept so that every
// weight gradient is one reduction over all S * R rows after the time loop.
struct BwdBuffers {
    float *X, *GP, *DG, *HS, *DN, *VEL, *DXIN, *G;     // [S][R][K | 512 | 512 | 128 | 8 | 2 | E+P | C n n]
    float *pass[2], *dc;                               // [R][128] chain state
    float* scratch;                                    // partial sums of the row-split reductions
    size_t scratch_floats;
    int* masked;                                       // [S][R]
};

static size_t carve_bwd(const tb2_lstm* m, size_t R, size_t S, void* base, BwdBuffers* b) {
    const size_t K = (size_t)m->K_gate, E = (size_t)m->E, P = (size_t)(m->P > 0 ? m->P : 0);
    size_t off = 0;
    auto take = [&](size_t n) {
        float* p = base ? reinterpret_cast<float*>(base) + off : nullptr;
        off += (n + 3) & ~(size_t)3;       // keep every array 16-byte aligned
        return p;
    };
    BwdBuffers tmp;
    BwdBuffers* o = b ? b : &tmp;
    const size_t CG = (size_t)m->C * (size_t)m->cells;
    o->X = take(S * R * K);
    o->GP = take(S * R * 512);
    o->DG = take(S * R * 512);
    o->HS = take(S * R * 128);
    o->DN = take(S * R * 8);
    o->VEL = take(S * R * 2);
    o->DXIN = take(S * R * (E + P));
    o->G = take(P ? S * R * CG : 4);
    o->pass[0] = take(R * 128);
    o->pass[1] = take(R * 128);
    o->dc = take(R * 128);
    size_t big = 512 * K;
    if (P * CG > big) big = P * CG;
    o->scratch_floats = 8 * big;
    o->scratch = take(o->scratch_floats);
    o->masked = reinterpret_cast<int*>(take(S * R));
    return off * sizeof(float) + 256;
}
}  // namespace tb2

namespace tb2 {


// fp32 window [rows x cols] (leading dimension ld_src) -> bf16 (hi, lo) at column col_off of a [rows x ld_dst] matrix
__global__ void split2d_kernel(const float* __restrict__ src, int ld_src, int rows, int cols, __nv_bfloat16* __restrict__ hi,
                               __nv_bfloat16* __restrict__ lo, int ld_dst, int col_off) {
    const size_t total = (size_t)rows * cols;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const size_t r = idx / cols;
        const int c = (int)(idx - r * cols);
        const float v = src[r * ld_src + c];
        const __nv_bfloat16 h = __float2bfloat16_rn(v);
        hi[r * ld_dst + col_off + c] = h;
        lo[r * ld_dst + col_off + c] = __float2bfloat16_rn(v - __bfloat162float(h));
    }
}
// src [R x Cc] row-major -> bf16 (hi, lo) of its transpose [Cc x R] (weights: a few hundred KB, once per backward)
__global__ void transpose_split_kernel(const float* __restrict__ src, int R, int Cc, __nv_bfloat16* __restrict__ hi,
                                       __nv_bfloat16* __restrict__ lo) {
    const size_t total = (size_t)R * Cc;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const size_t c = idx / R;
        const int r = (int)(idx - c * R);
        const float v = src[(size_t)r * Cc + c];
        const __nv_bfloat16 h = __float2bfloat16_rn(v);
        hi[idx] = h;
        lo[idx] = __float2bfloat16_rn(v - __bfloat162float(h));
    }
}
static int split2d(const float* src, int ld_src, size_t rows, int cols, __nv_bfloat16* hi, __nv_bfloat16* lo, int ld_dst,
                   int col_off, cudaStream_t st) {
    KernelTimer kt("bwd_split", st);
    const size_t total = rows * (size_t)cols;
    const unsigned blocks = (unsigned)std::min<size_t>((total + 255) / 256, 148 * 16);
    split2d_kernel<<<blocks, 256, 0, st>>>(src, ld_src, (int)rows, cols, hi, lo, ld_dst, col_off);
    TB2_LAUNCH_CHECK();
    return TB2_OK;
}

struct SocBuffers {
    float *X, *GP, *DG, *HS, *DN, *VEL, *DXIN, *H1, *DH1, *LAT, *DLAT, *DGRID, *dWt1;
    float *pass[2], *dc, *zero_h, *scratch;
    size_t scratch_floats;
    int *masked, *rows, *winc, *counts, *base, *start, *pcell;
    unsigned* sorted;
    uint8_t* pflag;
    uint32_t* wine;
    __nv_bfloat16 *Wt1_hi, *Wt1_lo;                       // bf16 split of the cell-major first-layer weights (dgrid on mma.sync)
    // 3-pass tcgen05 versions of the row GEMMs (dense_layer_tc_kernel): bf16 (hi, lo) operands
    __nv_bfloat16 *X_hi, *X_lo;                           // [S][M][K]
    __nv_bfloat16 *DG_hi[2], *DG_lo[2];                   // [M][512], steps s and s + 1
    __nv_bfloat16 *DZ2_hi, *DZ2_lo;                       // [M][P]
    __nv_bfloat16 *Wcat_hi[2], *Wcat_lo[2];               // [512][K] = [W_ih | W_hh] per phase
    __nv_bfloat16 *WhhT_hi[2], *WhhT_lo[2];               // [128][512]
    __nv_bfloat16 *WihT_hi[2], *WihT_lo[2];               // [E + P][512]
    __nv_bfloat16 *W2T_hi, *W2T_lo;                       // [d1][P]
    float* zero_bias;                                     // [max(d1, 512)]
};

static size_t carve_social(const tb2_lstm* m, const tb2_layout* l, size_t S, void* basep, SocBuffers* b) {
    const size_t M = (size_t)l->M, K = (size_t)m->K_gate, E = (size_t)m->E, P = (size_t)m->P;
    const size_t d1 = (size_t)m->mlp_dims[1], C = (size_t)m->C, cells = (size_t)m->cells;
    const size_t nm1 = (size_t)(l->n_max > 1 ? l->n_max - 1 : 1);
    size_t off = 0;
    auto take = [&](size_t n) {
        float* p = basep ? reinterpret_cast<float*>(basep) + off : nullptr;
        off += (n + 3) & ~(size_t)3;
        return p;
    };
    SocBuffers tmp;
    SocBuffers* o = b ? b : &tmp;
    o->X = take(S * M * K);
    o->GP = take(S * M * 512);
    o->DG = take(S * M * 512);
    o->HS = take(S * M * 128);
    o->DN = take(S * M * 8);
    o->VEL = take(S * M * 2);
    o->DXIN = take(S * M * (E + P));
    o->H1 = take(m->n_mlp == 2 ? S * M * d1 : 4);
    o->DH1 = take(M * (d1 > 128 ? d1 : 128));     // also holds the [M,128] recurrent d h of a step
    o->LAT = take(S * M * C);
    o->DLAT = take(S * M * C);
    o->DGRID = take(M * nm1 * C);
    o->dWt1 = take(cells * C * d1);
    o->pass[0] = take(M * 128);
    o->pass[1] = take(M * 128);
    o->dc = take(M * 128);
    o->zero_h = take(M * 128);
    size_t big = 512 * K;
    if (P * d1 > big) big = P * d1;
    o->scratch_floats = 8 * big;
    o->scratch = take(o->scratch_floats);
    o->masked = reinterpret_cast<int*>(take(S * M));
    o->rows = reinterpret_cast<int*>(take(M));
    o->winc = reinterpret_cast<int*>(take(S * M));
    o->wine = reinterpret_cast<uint32_t*>(take(S * M * nm1));
    o->sorted = reinterpret_cast<unsigned*>(take(M * nm1));
    o->pcell = reinterpret_cast<int*>(take(S * M * nm1));
    o->pflag = reinterpret_cast<uint8_t*>(take((S * M * nm1 + 3) / 4));
    o->counts = reinterpret_cast<int*>(take((size_t)l->B * cells));
    o->base = reinterpret_cast<int*>(take((size_t)l->B * cells));
    o->start = reinterpret_cast<int*>(take(cells + 1));
    o->Wt1_hi = reinterpret_cast<__nv_bfloat16*>(take((cells * C * d1 + 1) / 2));
    o->Wt1_lo = reinterpret_cast<__nv_bfloat16*>(take((cells * C * d1 + 1) / 2));
    auto take_bf16 = [&](size_t n) { return reinterpret_cast<__nv_bfloat16*>(take((n + 1) / 2)); };
    o->X_hi = take_bf16(S * M * K);
    o->X_lo = take_bf16(S * M * K);
    for (int i = 0; i < 2; ++i) {
        o->DG_hi[i] = take_bf16(M * 512);
        o->DG_lo[i] = take_bf16(M * 512);
        o->Wcat_hi[i] = take_bf16(512 * K);
        o->Wcat_lo[i] = take_bf16(512 * K);
        o->WhhT_hi[i] = take_bf16(128 * 512);
        o->WhhT_lo[i] = take_bf16(128 * 512);
        o->WihT_hi[i] = take_bf16((E + P) * 512);
        o->WihT_lo[i] = take_bf16((E + P) * 512);
    }
    o->DZ2_hi = take_bf16(M * P);
    o->DZ2_lo = take_bf16(M * P);
    o->W2T_hi = take_bf16(d1 * P);
    o->W2T_lo = take_bf16(d1 * P);
    o->zero_bias = take(d1 > 512 ? d1 : 512);
    return off * sizeof(float) + 256;
}

template <int C>
static int social_pair_kernels(const tb2_lstm* m, const tb2_layout* l, const SocBuffers& b, const float* lat,
                               int nm1, int d1, cudaStream_t st) {
    if (C == 16 && d1 % 32 == 0 && b.Wt1_hi != nullptr && dgrid_mma_smem(d1) <= 200 * 1024) {
        static DynSmemConfig configured;
        TB2_CHECK_CUDA(configured.ensure(social_dgrid_mma_kernel, dgrid_mma_smem(d1), 48 * 1024));
        KernelTimer kt("social_dgrid_mma", st);
        social_dgrid_mma_kernel<<<dim3(m->cells, kDmYs), 256, dgrid_mma_smem(d1), st>>>(
            b.sorted, b.start, b.DH1, d1, b.Wt1_hi, b.Wt1_lo, nm1, b.DGRID);
    } else {
        KernelTimer kt("social_dgrid", st);
        social_dgrid_kernel<C><<<dim3(m->cells, (l->M + kDgPairs - 1) / kDgPairs), 256, 0, st>>>(
            b.sorted, b.start, b.DH1, d1, m->Wt1, nm1, b.DGRID);
    }
    TB2_LAUNCH_CHECK();
    if (C == 16 && d1 % 32 == 0) {
        KernelTimer kt("social_dw1_mma", st);
        social_dw1_mma_kernel<<<dim3(m->cells, (d1 + 255) / 256), 256, 0, st>>>(
            b.sorted, b.start, nm1, l->row_scene, l->scene_off, lat, b.DH1, d1, b.dWt1);
    } else {
        KernelTimer kt("social_dw1", st);
        social_dw1_kernel<C><<<dim3(m->cells, (d1 + 255) / 256), 256, 0, st>>>(
            b.sorted, b.start, nm1, l->row_scene, l->scene_off, lat, b.DH1, d1, b.dWt1);
    }
    TB2_LAUNCH_CHECK();
    return TB2_OK;
}

// BPTT through social pooling: every track of a scene receives gradient, so the backward runs on
// all M rows (see the kernel comments above for the scatter part).
static int social_backward(const tb2_lstm* m, const tb2_layout* l, const tb2_lstm_weights* w,
                           const float* observed, int obs_length, const float* truth, int n_decode,
                           const float* positions, const float* states, const float* d_normals,
                           const tb2_lstm_grads* g, Workspace& ws, void* bwd_workspace, cudaStream_t st,
                           const TrainCache* cache = nullptr) {
    const int S = obs_length - 1 + n_decode, S_enc = obs_length - 1;
    const int Mi = l->M, K = m->K_gate, E = m->E, P = m->P, EP = E + P, C = m->C, cells = m->cells;
    const int d1 = m->mlp_dims[1];
    const bool two = m->n_mlp == 2;
    const size_t M = (size_t)Mi;
    const int nm1 = l->n_max > 1 ? l->n_max - 1 : 1;
    TB2_REQUIRE(g->pool_embedding_weight0 && g->pool_embedding_bias0 && g->pool_encoding_weight &&
                g->pool_encoding_bias && (!two || (g->pool_embedding_weight1 && g->pool_embedding_bias1)),
                "social backward needs gradient buffers for pool.hidden_dim_encoding and pool.embedding");
    SocBuffers b;
    carve_social(m, l, (size_t)S, bwd_workspace, &b);
    if (cache) {      // the forward kept its per-step winners / latent vectors: same [S][M][...] layouts
        b.LAT = cache->lat;
        b.winc = cache->win_count;
        b.wine = cache->win_ent;
        b.pcell = cache->pair_cell;
        b.pflag = cache->pair_flag;
    }
    TB2_CHECK_CUDA(cudaMemsetAsync(b.dc, 0, M * 128 * sizeof(float), st));
    TB2_CHECK_CUDA(cudaMemsetAsync(b.dWt1, 0, (size_t)cells * C * d1 * sizeof(float), st));
    TB2_CHECK_CUDA(cudaMemsetAsync(b.zero_h, 0, M * 128 * sizeof(float), st));      // state before step 0
    iota_kernel<<<(Mi + 255) / 256, 256, 0, st>>>(b.rows, Mi);
    TB2_LAUNCH_CHECK();
    split_bf16_flat_kernel<<<1184, 256, 0, st>>>(m->Wt1, b.Wt1_hi, b.Wt1_lo, (size_t)cells * C * d1);
    TB2_LAUNCH_CHECK();
    int rc;
    const bool tc2 = two && m->W_hi[1] != nullptr;
    // (A) forward quantities of every step: winners + lat, hidden1, X = [emb | pooled | h_prev]
    for (int s = 0; s < S; ++s) {
        const float *o1, *o2;
        int phase;
        if ((rc = resolve_step_inputs(l, observed, obs_length, truth, positions, s, &ws, &o1, &o2, &phase, st))) return rc;
        const float* h_prev = s > 0 ? states + ((size_t)(s - 1) * 2 + 0) * M * kBH : nullptr;
        Workspace w2 = ws;
        w2.lat = b.LAT + (size_t)s * M * C;
        w2.win_count = b.winc + (size_t)s * M;
        w2.win_ent = b.wine + (size_t)s * M * nm1;
        w2.pair_cell = b.pcell + (size_t)s * M * nm1;
        w2.pair_flag = b.pflag + (size_t)s * M * nm1;
        if (cache) {
            // hidden1 and the pooled vector of the forward, as fp32 (hi + lo of the bf16 pair the next kernel consumed)
            if (two) {
                merge_split_kernel<<<1024, 256, 0, st>>>((const __nv_bfloat16*)cache->h1_hi + (size_t)s * M * d1,
                                                         (const __nv_bfloat16*)cache->h1_lo + (size_t)s * M * d1, nullptr,
                                                         b.H1 + (size_t)s * M * d1, M * d1);
                TB2_LAUNCH_CHECK();
            }
            merge_split_kernel<<<512, 256, 0, st>>>((const __nv_bfloat16*)cache->pool_hi + (size_t)s * M * P,
                                                    (const __nv_bfloat16*)cache->pool_lo + (size_t)s * M * P, nullptr, ws.pooled,
                                                    M * P);
            TB2_LAUNCH_CHECK();
        } else {
            if ((rc = launch_pool_prepare(m, l, h_prev ? h_prev : b.zero_h, o1, o2, 1, 1, 0, &w2, st))) return rc;
            if ((rc = launch_pool_mlp(m, l, &w2, ws.pooled, nullptr, nullptr, st))) return rc;
            if (two) {
                merge_split_kernel<<<1024, 256, 0, st>>>(tc2 ? (const __nv_bfloat16*)ws.act[0] : nullptr,
                                                         tc2 ? (const __nv_bfloat16*)ws.act[1] : nullptr, ws.act[0],
                                                         b.H1 + (size_t)s * M * d1, M * d1);
                TB2_LAUNCH_CHECK();
            }
        }
        {
            KernelTimer kt("bwd_gather", st);
            bwd_gather_kernel<<<Mi, 256, 0, st>>>(b.rows, Mi, (const float2*)o1, (const float2*)o2, m->We, m->be,
                                                  h_prev, nullptr, nullptr, nullptr, nullptr, nullptr, nm1, C, cells,
                                                  ws.pooled, b.X + (size_t)s * M * K, nullptr,
                                                  b.VEL + (size_t)s * M * 2, b.masked + (size_t)s * M, E, P, K);
        }
        TB2_LAUNCH_CHECK();
    }
    // The row GEMMs (rows = all tracks) run on the 3-pass tcgen05 kernel of the forward (dense_layer_tc_kernel:
    // Y = A . W^T + bias, bf16 (hi, lo) operands, fp32 accumulation) when the shapes allow it: A and the (transposed)
    // weights are split once, the outputs stay fp32.  Other shapes: cuBLAS / FFMA GEMMs.
    const bool tcg = K == EP + 128 && dense_tc_supported(K, 512) && dense_tc_supported(512, 128) &&
                     dense_tc_supported(512, EP) && (!two || dense_tc_supported(P, d1));
    if (tcg) {
        TB2_CHECK_CUDA(cudaMemsetAsync(b.zero_bias, 0, (size_t)(d1 > 512 ? d1 : 512) * sizeof(float), st));
        for (int phase = 0; phase < 2; ++phase) {
            const float* Wih_p = phase == TB2_PHASE_ENCODER ? w->encoder_weight_ih : w->decoder_weight_ih;
            const float* Whh_p = phase == TB2_PHASE_ENCODER ? w->encoder_weight_hh : w->decoder_weight_hh;
            if ((rc = split2d(Wih_p, EP, 512, EP, b.Wcat_hi[phase], b.Wcat_lo[phase], K, 0, st))) return rc;
            if ((rc = split2d(Whh_p, 128, 512, 128, b.Wcat_hi[phase], b.Wcat_lo[phase], K, EP, st))) return rc;
            transpose_split_kernel<<<256, 256, 0, st>>>(Whh_p, 512, 128, b.WhhT_hi[phase], b.WhhT_lo[phase]);
            TB2_LAUNCH_CHECK();
            transpose_split_kernel<<<512, 256, 0, st>>>(Wih_p, 512, EP, b.WihT_hi[phase], b.WihT_lo[phase]);
            TB2_LAUNCH_CHECK();
        }
        if (two) {
            transpose_split_kernel<<<1024, 256, 0, st>>>(w->pool_embedding_weight[1], P, d1, b.W2T_hi, b.W2T_lo);
            TB2_LAUNCH_CHECK();
        }
        if ((rc = split2d(b.X, K, (size_t)S * M, K, b.X_hi, b.X_lo, K, 0, st))) return rc;
    }
    // (B) gate pre-activations of all steps
    for (int phase = 0; phase < 2; ++phase) {
        const int s0 = phase == TB2_PHASE_ENCODER ? 0 : S_enc;
        const int ns = phase == TB2_PHASE_ENCODER ? S_enc : S - S_enc;
        if (ns <= 0) continue;
        if (tcg) {
            if ((rc = launch_dense_tc(b.X_hi + (size_t)s0 * M * K, b.X_lo + (size_t)s0 * M * K, b.Wcat_hi[phase],
                                      b.Wcat_lo[phase], m->bg[phase], b.GP + (size_t)s0 * M * 512, nullptr, nullptr, ns * Mi,
                                      K, 512, 0, st)))
                return rc;
            continue;
        }
        if ((rc = gemm_nn(b.X + (size_t)s0 * M * K, K, m->WgT[phase], 512, b.GP + (size_t)s0 * M * 512, 512,
                          ns * Mi, 512, K, m->bg[phase], st)))
            return rc;
    }
    // (C) reverse time: cell -> input gradient -> grid MLP -> scatter to the neighbours' hidden states
    const size_t place_smem = (size_t)l->n_max * nm1 * sizeof(short);
    TB2_REQUIRE(place_smem <= 200 * 1024 && cells < 32768, "scene too large for the social backward");
    {
        static DynSmemConfig configured;
        TB2_CHECK_CUDA(configured.ensure(pair_place_kernel, place_smem, 48 * 1024));
    }
    int cur = 0;
    for (int s = S - 1; s >= 0; --s, cur ^= 1) {
        const int phase = s < S_enc ? TB2_PHASE_ENCODER : TB2_PHASE_DECODER;
        const float* c_prev = s > 0 ? states + ((size_t)(s - 1) * 2 + 1) * M * kBH : nullptr;
        const bool last = s == S - 1;
        const int next_phase = (s + 1) < S_enc ? TB2_PHASE_ENCODER : TB2_PHASE_DECODER;
        const float* Whh_next = next_phase == TB2_PHASE_ENCODER ? w->encoder_weight_hh : w->decoder_weight_hh;
        const float* Wih = phase == TB2_PHASE_ENCODER ? w->encoder_weight_ih : w->decoder_weight_ih;
        float* DGs = b.DG + (size_t)s * M * 512;
        float* DXs = b.DXIN + (size_t)s * M * EP;
        const float* Xs = b.X + (size_t)s * M * K;
        // recurrent part of d h: all rows are active, so dgates(s+1) . W_hh is a GEMM (DH1 is free here)
        float* dh_rec = nullptr;
        if (!last) {
            dh_rec = b.DH1;
            if (tcg) {      // dgates(s + 1) was split at the end of the previous iteration
                if ((rc = launch_dense_tc(b.DG_hi[(s + 1) & 1], b.DG_lo[(s + 1) & 1], b.WhhT_hi[next_phase], b.WhhT_lo[next_phase],
                                          b.zero_bias, dh_rec, nullptr, nullptr, Mi, 512, 128, 0, st)))
                    return rc;
            } else if ((rc = gemm_nn(b.DG + (size_t)(s + 1) * M * 512, 512, Whh_next, 128, dh_rec, 128, Mi, 128, 512, nullptr,
                                     st)))
                return rc;
        }
        {
            KernelTimer kt("bwd_cell_head", st);
            bwd_cell_head_kernel<<<Mi, 4 * kBH, 0, st>>>(
                b.rows, b.masked + (size_t)s * M, b.GP + (size_t)s * M * 512, c_prev, nullptr, Whh_next, dh_rec,
                b.pass[cur ^ 1], b.pass[cur], b.dc,
                d_normals + (size_t)s * M * 5, m->Wn, m->bn, DGs, b.HS + (size_t)s * M * 128,
                b.DN + (size_t)s * M * 8, Mi);
        }
        TB2_LAUNCH_CHECK();
        if (tcg) {
            if ((rc = split2d(DGs, 512, M, 512, b.DG_hi[s & 1], b.DG_lo[s & 1], 512, 0, st))) return rc;
            if ((rc = launch_dense_tc(b.DG_hi[s & 1], b.DG_lo[s & 1], b.WihT_hi[phase], b.WihT_lo[phase], b.zero_bias, DXs,
                                      nullptr, nullptr, Mi, 512, EP, 0, st)))
                return rc;
        } else if ((rc = gemm_nn(DGs, 512, Wih, EP, DXs, EP, Mi, EP, 512, nullptr, st))) return rc;
        const unsigned eb = (unsigned)((M * d1 + 255) / 256);
        if (two) {
            const float* H1s = b.H1 + (size_t)s * M * d1;
            relu_mask_kernel<<<(unsigned)((M * P + 255) / 256), 256, 0, st>>>(Xs, K, DXs, EP, Mi, E, P);   // dz2
            TB2_LAUNCH_CHECK();
            // d hidden1 = dz2 . W2 (torch layout [P, d1] is the [K = P, N = d1] operand), then the ReLU mask
            if (tcg) {
                if ((rc = split2d(DXs + E, EP, M, P, b.DZ2_hi, b.DZ2_lo, P, 0, st))) return rc;
                if ((rc = launch_dense_tc(b.DZ2_hi, b.DZ2_lo, b.W2T_hi, b.W2T_lo, b.zero_bias, b.DH1, nullptr, nullptr, Mi, P, d1,
                                          0, st)))
                    return rc;
            } else if ((rc = gemm_nn(DXs + E, EP, w->pool_embedding_weight[1], d1, b.DH1, d1, Mi, d1, P, nullptr, st))) return rc;
            masked_copy_kernel<<<eb, 256, 0, st>>>(H1s, d1, b.DH1, d1, b.DH1, d1, Mi, d1);
            TB2_LAUNCH_CHECK();
            // dW2 / db2: one reduction over the rows of ALL steps after the loop (dz2 stays in DXIN, hidden1 in H1)
        } else {
            masked_copy_kernel<<<eb, 256, 0, st>>>(Xs + E, K, DXs + E, EP, b.DH1, d1, Mi, d1);
            TB2_LAUNCH_CHECK();
        }
        if ((rc = colsum(b.DH1, d1, Mi, d1, g->pool_embedding_bias0, nullptr, b.scratch, b.scratch_floats, st))) return rc;
        const int* winc = b.winc + (size_t)s * M;
        const uint32_t* wine = b.wine + (size_t)s * M * nm1;
        const int* pcell = b.pcell + (size_t)s * M * nm1;
        const uint8_t* pflag = b.pflag + (size_t)s * M * nm1;
        const int* msk = b.masked + (size_t)s * M;
        const float* lat = b.LAT + (size_t)s * M * C;
        {
            KernelTimer kt("social_pair_sort", st);
            pair_count_kernel<<<l->B, 256, cells * sizeof(int), st>>>(l->scene_off, msk, pcell, pflag, nm1, cells,
                                                                       b.counts);
            pair_offsets_kernel<<<1, 1024, cells * sizeof(int), st>>>(b.counts, l->B, cells, b.base, b.start);
            pair_place_kernel<<<l->B, 256, place_smem, st>>>(
                l->scene_off, msk, pcell, pflag, winc, wine, nm1, cells, b.base, b.start, l->pad_to_max, b.sorted);
        }
        TB2_LAUNCH_CHECK();
        switch (C) {
            case 4: rc = social_pair_kernels<4>(m, l, b, lat, nm1, d1, st); break;
            case 8: rc = social_pair_kernels<8>(m, l, b, lat, nm1, d1, st); break;
            case 16: rc = social_pair_kernels<16>(m, l, b, lat, nm1, d1, st); break;
            case 32: rc = social_pair_kernels<32>(m, l, b, lat, nm1, d1, st); break;
            default: set_error("social latent_dim must be 4, 8, 16 or 32"); return TB2_ERR_UNSUPPORTED;
        }
        if (rc) return rc;
        {
            KernelTimer kt("social_scene_reduce", st);
            social_scene_reduce_kernel<<<l->B, 256, (size_t)l->n_max * C * sizeof(float), st>>>(
                l->scene_off, msk, pflag, nm1, C, b.DGRID, w->pool_encoding_weight, b.DLAT + (size_t)s * M * C,
                s > 0 ? b.pass[cur] : nullptr);
        }
        TB2_LAUNCH_CHECK();
    }
    if (two) {
        if ((rc = gemm_tn(b.DXIN + E, EP, b.H1, d1, g->pool_embedding_weight1, d1, S * Mi, P, d1, b.scratch, b.scratch_floats, st)))
            return rc;
        if ((rc = colsum(b.DXIN + E, EP, S * Mi, P, g->pool_embedding_bias1, nullptr, b.scratch, b.scratch_floats, st))) return rc;
    }
    // (D) parameter gradients: one reduction over all (step, row) records per tensor
    for (int phase = 0; phase < 2; ++phase) {
        const int s0 = phase == TB2_PHASE_ENCODER ? 0 : S_enc;
        const int ns = phase == TB2_PHASE_ENCODER ? S_enc : S - S_enc;
        if (ns <= 0) continue;
        const float* DG = b.DG + (size_t)s0 * M * 512;
        const float* X = b.X + (size_t)s0 * M * K;
        const int rows = ns * Mi;
        float* gWih = phase == TB2_PHASE_ENCODER ? g->encoder_weight_ih : g->decoder_weight_ih;
        float* gWhh = phase == TB2_PHASE_ENCODER ? g->encoder_weight_hh : g->decoder_weight_hh;
        float* gbih = phase == TB2_PHASE_ENCODER ? g->encoder_bias_ih : g->decoder_bias_ih;
        float* gbhh = phase == TB2_PHASE_ENCODER ? g->encoder_bias_hh : g->decoder_bias_hh;
        if ((rc = gemm_tn(DG, 512, X, K, gWih, EP, rows, 512, EP, b.scratch, b.scratch_floats, st))) return rc;
        if ((rc = gemm_tn(DG, 512, X + EP, K, gWhh, 128, rows, 512, 128, b.scratch, b.scratch_floats, st))) return rc;
        if ((rc = colsum(DG, 512, rows, 512, gbih, gbhh, b.scratch, b.scratch_floats, st))) return rc;
    }
    if ((rc = gemm_tn(b.DN, 8, b.HS, 128, g->hidden2normal_weight, 128, S * Mi, 5, 128, b.scratch, b.scratch_floats, st)))
        return rc;
    if ((rc = colsum(b.DN, 8, S * Mi, 5, g->hidden2normal_bias, nullptr, b.scratch, b.scratch_floats, st))) return rc;
    bwd_embed_kernel<<<E - 2, 256, 0, st>>>(b.X, K, b.DXIN, EP, b.VEL, S * Mi, g->input_embedding_weight,
                                            g->input_embedding_bias);
    TB2_LAUNCH_CHECK();
    untranspose_add_kernel<<<2048, 256, 0, st>>>(b.dWt1, g->pool_embedding_weight0, cells, C, d1);
    TB2_LAUNCH_CHECK();
    // lat_j = W_enc h_j + b_enc (gridbased_pooling.py:160-167): h of step s-1 is states[s-1]
    for (int s = 1; s < S; ++s) {
        const float* h_prev = states + ((size_t)(s - 1) * 2 + 0) * M * kBH;
        if ((rc = gemm_tn(b.DLAT + (size_t)s * M * C, C, h_prev, 128, g->pool_encoding_weight, 128, Mi, C, 128,
                          b.scratch, b.scratch_floats, st)))
            return rc;
    }
    if ((rc = colsum(b.DLAT, C, S * Mi, C, g->pool_encoding_bias, nullptr, b.scratch, b.scratch_floats, st))) return rc;
    return TB2_OK;
}
}  // namespace tb2

extern "C" {

size_t tb2_lstm_backward_workspace_bytes(const tb2_lstm* m, const tb2_layout* l, int32_t num_active,
                                         int32_t num_steps) {
    if (!m || !l || num_active < 0 || num_steps < 0) return 0;
    if (m->cfg.pool_type == TB2_POOL_SOCIAL)
        return carve_social(m, l, (size_t)(num_steps > 0 ? num_steps : 1), nullptr, nullptr);
    return carve_bwd(m, (size_t)(num_active > 0 ? num_active : 1), (size_t)(num_steps > 0 ? num_steps : 1),
                     nullptr, nullptr);
}

static int sequence_backward_impl(const tb2_lstm* m, const tb2_layout* l, const tb2_lstm_weights* w,
                               const float* observed, int32_t obs_length, const float* truth, int32_t n_decode,
                               const float* positions, const float* states, const float* d_normals,
                               const int32_t* active_rows, int32_t num_active, const tb2_lstm_grads* g,
                               void* workspace, size_t workspace_bytes, void* bwd_workspace,
                               size_t bwd_workspace_bytes, void* stream, const void* cache, size_t cache_bytes);

int tb2_lstm_sequence_backward(const tb2_lstm* m, const tb2_layout* l, const tb2_lstm_weights* w,
                               const float* observed, int32_t obs_length, const float* truth, int32_t n_decode,
                               const float* positions, const float* states, const float* d_normals,
                               const int32_t* active_rows, int32_t num_active, const tb2_lstm_grads* g,
                               void* workspace, size_t workspace_bytes, void* bwd_workspace,
                               size_t bwd_workspace_bytes, void* stream) {
    return sequence_backward_impl(m, l, w, observed, obs_length, truth, n_decode, positions, states, d_normals, active_rows,
                                  num_active, g, workspace, workspace_bytes, bwd_workspace, bwd_workspace_bytes, stream, nullptr, 0);
}

int tb2_lstm_sequence_backward_cached(const tb2_lstm* m, const tb2_layout* l, const tb2_lstm_weights* w,
                                      const float* observed, int32_t obs_length, const float* truth, int32_t n_decode,
                                      const float* positions, const float* states, const float* d_normals,
                                      const int32_t* active_rows, int32_t num_active, const tb2_lstm_grads* g,
                                      void* workspace, size_t workspace_bytes, void* bwd_workspace,
                                      size_t bwd_workspace_bytes, const void* cache, size_t cache_bytes, void* stream) {
    return sequence_backward_impl(m, l, w, observed, obs_length, truth, n_decode, positions, states, d_normals, active_rows,
                                  num_active, g, workspace, workspace_bytes, bwd_workspace, bwd_workspace_bytes, stream, cache,
                                  cache_bytes);
}

static int sequence_backward_impl(const tb2_lstm* m, const tb2_layout* l, const tb2_lstm_weights* w,
                               const float* observed, int32_t obs_length, const float* truth, int32_t n_decode,
                               const float* positions, const float* states, const float* d_normals,
                               const int32_t* active_rows, int32_t num_active, const tb2_lstm_grads* g,
                               void* workspace, size_t workspace_bytes, void* bwd_workspace,
                               size_t bwd_workspace_bytes, void* stream, const void* cache, size_t cache_bytes) {
    TB2_REQUIRE(m && l && w && g, "null handle");
    TB2_REQUIRE(m->weights_set, "tb2_lstm_set_weights has not been called");
    TB2_REQUIRE(observed && positions && states && d_normals && active_rows, "null argument");
    TB2_REQUIRE(obs_length >= 2 && n_decode >= 0, "need obs_length >= 2 and n_decode >= 0");
    TB2_REQUIRE(m->H == kBH, "hidden_dim must be 128");
    const bool social = m->cfg.pool_type == TB2_POOL_SOCIAL;
    if (social && (m->n_mlp < 1 || m->n_mlp > 2 || !m->cfg.pool_to_input || m->cfg.constant != 0.f)) {
        set_error("social training backward supports one_layer / two_layer embeddings with constant = 0");
        return TB2_ERR_UNSUPPORTED;
    }
    if (!social && m->cfg.pool_type != TB2_POOL_NONE &&
        (m->n_mlp != 1 || !m->cfg.pool_to_input || m->cfg.constant != 0.f || m->P > 1024 || m->C > 2)) {
        set_error("training backward supports one_layer grid embeddings with constant = 0 and pool_to_input");
        return TB2_ERR_UNSUPPORTED;
    }
    const int S = obs_length - 1 + n_decode;
    TB2_REQUIRE(workspace && workspace_bytes >= carve_workspace(m, l, nullptr, nullptr), "workspace too small");
    TB2_REQUIRE(bwd_workspace && bwd_workspace_bytes >= tb2_lstm_backward_workspace_bytes(m, l, num_active, S),
                "backward workspace too small");
    if (num_active == 0) return TB2_OK;
    cudaStream_t st = (cudaStream_t)stream;
    Workspace ws;
    carve_workspace(m, l, workspace, &ws);
    if (social) {    // every track of a scene receives gradient: all rows, active_rows is ignored
        TrainCache tc;
        const size_t need = cache ? carve_train_cache(m, l, (size_t)S, const_cast<void*>(cache), &tc) : 0;
        TB2_REQUIRE(!cache || (need > 0 && cache_bytes >= need), "training cache too small (tb2_lstm_train_cache_bytes)");
        return social_backward(m, l, w, observed, obs_length, truth, n_decode, positions, states, d_normals, g, ws,
                               bwd_workspace, st, cache ? &tc : nullptr);
    }
    const int R = num_active, K = m->K_gate, E = m->E, P = m->P, EP = E + P;
    const size_t M = (size_t)l->M;
    BwdBuffers b;
    carve_bwd(m, (size_t)R, (size_t)S, bwd_workspace, &b);
    TB2_CHECK_CUDA(cudaMemsetAsync(b.dc, 0, (size_t)R * 128 * sizeof(float), st));
    const int nm1 = l->n_max > 1 ? l->n_max - 1 : 1;
    const bool pooled = m->cfg.pool_type != TB2_POOL_NONE;
    const size_t CG = (size_t)m->C * (size_t)m->cells;
    const int S_enc = obs_length - 1;
    int rc;
    // (A) inputs of every step for the active rows: winners -> X = [emb | pooled | h_prev], grid rows
    for (int s = 0; s < S; ++s) {
        const float *o1, *o2;
        int phase;
        if ((rc = resolve_step_inputs(l, observed, obs_length, truth, positions, s, &ws, &o1, &o2, &phase, st))) return rc;
        const float* h_prev = s > 0 ? states + ((size_t)(s - 1) * 2 + 0) * M * kBH : nullptr;
        if (pooled && (rc = launch_pool_prepare(m, l, h_prev, o1, o2, 1, 0, 0, &ws, st))) return rc;   // winners
        {
            KernelTimer kt("bwd_gather", st);
            bwd_gather_kernel<<<R, 256, 0, st>>>(active_rows, R, (const float2*)o1, (const float2*)o2, m->We, m->be,
                                                 h_prev, ws.win_count, ws.win_ent, ws.win_val, m->Wt1, m->base1,
                                                 nm1, m->C, m->cells, nullptr, b.X + (size_t)s * R * K,
                                                 pooled ? b.G + (size_t)s * R * CG : nullptr,
                                                 b.VEL + (size_t)s * R * 2, b.masked + (size_t)s * R, E, P, K);
        }
        TB2_LAUNCH_CHECK();
    }
    // (B) gate pre-activations of all steps: one GEMM per cell (encoder / decoder weights)
    for (int phase = 0; phase < 2; ++phase) {
        const int s0 = phase == TB2_PHASE_ENCODER ? 0 : S_enc;
        const int ns = phase == TB2_PHASE_ENCODER ? S_enc : S - S_enc;
        if (ns <= 0) continue;
        if ((rc = gemm_nn(b.X + (size_t)s0 * R * K, K, m->WgT[phase], 512, b.GP + (size_t)s0 * R * 512, 512, ns * R,
                          512, K, m->bg[phase], st)))
            return rc;
    }
    // (C) the sequential chain: one kernel per step
    int cur = 0;
    for (int s = S - 1; s >= 0; --s, cur ^= 1) {
        const float* c_prev = s > 0 ? states + ((size_t)(s - 1) * 2 + 1) * M * kBH : nullptr;
        const bool last = s == S - 1;
        const int next_phase = (s + 1) < S_enc ? TB2_PHASE_ENCODER : TB2_PHASE_DECODER;
        const float* Whh_next = next_phase == TB2_PHASE_ENCODER ? w->encoder_weight_hh : w->decoder_weight_hh;
        {
            KernelTimer kt("bwd_cell_head", st);
            bwd_cell_head_kernel<<<R, 4 * kBH, 0, st>>>(
                active_rows, b.masked + (size_t)s * R, b.GP + (size_t)s * R * 512, c_prev,
                last ? nullptr : b.DG + (size_t)(s + 1) * R * 512, Whh_next, nullptr, b.pass[cur ^ 1], b.pass[cur], b.dc,
                d_normals + (size_t)s * M * 5, m->Wn, m->bn, b.DG + (size_t)s * R * 512,
                b.HS + (size_t)s * R * 128, b.DN + (size_t)s * R * 8, R);
        }
        TB2_LAUNCH_CHECK();
    }
    // (D) + (E) input gradients of all steps and the parameter gradients: one reduction per tensor
    for (int phase = 0; phase < 2; ++phase) {
        const int s0 = phase == TB2_PHASE_ENCODER ? 0 : S_enc;
        const int ns = phase == TB2_PHASE_ENCODER ? S_enc : S - S_enc;
        if (ns <= 0) continue;
        const float* DG = b.DG + (size_t)s0 * R * 512;
        const float* X = b.X + (size_t)s0 * R * K;
        const int rows = ns * R;
        float* gWih = phase == TB2_PHASE_ENCODER ? g->encoder_weight_ih : g->decoder_weight_ih;
        float* gWhh = phase == TB2_PHASE_ENCODER ? g->encoder_weight_hh : g->decoder_weight_hh;
        float* gbih = phase == TB2_PHASE_ENCODER ? g->encoder_bias_ih : g->decoder_bias_ih;
        float* gbhh = phase == TB2_PHASE_ENCODER ? g->encoder_bias_hh : g->decoder_bias_hh;
        const float* Wih = phase == TB2_PHASE_ENCODER ? w->encoder_weight_ih : w->decoder_weight_ih;
        // dX_in = dgates . W_ih   (torch layout [4H, E+P] is the [K = 4H, N = E+P] operand as it stands)
        if ((rc = gemm_nn(DG, 512, Wih, EP, b.DXIN + (size_t)s0 * R * EP, EP, rows, EP, 512, nullptr, st))) return rc;
        if ((rc = gemm_tn(DG, 512, X, K, gWih, EP, rows, 512, EP, b.scratch, b.scratch_floats, st))) return rc;
        if ((rc = gemm_tn(DG, 512, X + EP, K, gWhh, 128, rows, 512, 128, b.scratch, b.scratch_floats, st))) return rc;
        if ((rc = colsum(DG, 512, rows, 512, gbih, gbhh, b.scratch, b.scratch_floats, st))) return rc;
    }
    if ((rc = gemm_tn(b.DN, 8, b.HS, 128, g->hidden2normal_weight, 128, S * R, 5, 128, b.scratch, b.scratch_floats, st)))
        return rc;
    if ((rc = colsum(b.DN, 8, S * R, 5, g->hidden2normal_bias, nullptr, b.scratch, b.scratch_floats, st))) return rc;
    bwd_embed_kernel<<<E - 2, 256, 0, st>>>(b.X, K, b.DXIN, EP, b.VEL, S * R, g->input_embedding_weight,
                                            g->input_embedding_bias);
    TB2_LAUNCH_CHECK();
    if (pooled) {
        relu_mask_kernel<<<(unsigned)(((size_t)S * R * P + 255) / 256), 256, 0, st>>>(b.X, K, b.DXIN, EP, S * R, E, P);
        TB2_LAUNCH_CHECK();
        if ((rc = gemm_tn(b.DXIN + E, EP, b.G, (int)CG, g->pool_embedding_weight0, (int)CG, S * R, P, (int)CG,
                          b.scratch, b.scratch_floats, st)))
            return rc;
        if ((rc = colsum(b.DXIN + E, EP, S * R, P, g->pool_embedding_bias0, nullptr, b.scratch, b.scratch_floats, st)))
            return rc;
    }
    return TB2_OK;
}

}  // extern "C"
