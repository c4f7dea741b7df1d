// Fused recurrence step: input embedding + LSTMCell gates + cell update + Gaussian head +
// position feedback, one launch per timestep.
//
// Replaces (reference: trajnetbaselines/lstm/) LSTM.step lstm.py:118-168 minus the pooling
// call: InputEmbedding.forward modules.py:24-30, torch.nn.LSTMCell (lstm.py:84-85,154),
// Hidden2Normal.forward modules.py:56-64, the masked write-back lstm.py:158-166 and the
// position update lstm.py:232,255.  The reference keeps h/c as Python lists of M tensors and
// stacks/unstacks them every step; here they are flat [M, H] arrays updated in place.
//
// Tiling: CTA = 32 tracks x all 4H gate columns, 256 threads; thread (warp w, lane l) owns
// rows 4w..4w+3 and hidden units 4l..4l+3 of all four gates, so the LSTM pointwise math needs
// no exchange and the 5-wide Gaussian head is a warp-shuffle reduction.  The A operand
// [emb | pooled | h] is assembled on the fly in shared memory (the embedding is recomputed
// from the 2-float velocity, never stored); W^T streams from L2 through a cp.async
// double buffer.
#include <math_constants.h>

#include <cuda_bf16.h>

#include "common.cuh"

namespace tb2 {

constexpr int kGH = 128;            // hidden_dim this kernel is specialised for
constexpr int kGN = 4 * kGH;        // gate columns
constexpr int kGM = 32;             // tracks per CTA
constexpr int kGThreads = 256;

struct GateParams {
    const float2* obs1;
    const float2* obs2;
    const float* pooled;   // [M, P] or null
    const float* h_in;
    const float* c_in;
    float* h_out;
    float* c_out;
    float* normal_out;     // [M, 5]
    float2* pos_out;       // [M] or null
    const float* We;       // [E-2, 2]
    const float* be;
    const float* WgT;      // [K_pad, 4H]
    const float* bg;       // [4H]
    const float* Wn;       // [5, H]
    const float* bn;
    int M, E, P, K, K_pad, add_pooled_to_h;
};

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

__global__ void __launch_bounds__(kGThreads, 2) lstm_gates_kernel(GateParams p) {
    extern __shared__ __align__(16) float smem_gates[];
    float (*Ws)[kGateBK][kGN] = reinterpret_cast<float (*)[kGateBK][kGN]>(smem_gates);               // 64 KB
    float (*As)[kGateBK][kGM] = reinterpret_cast<float (*)[kGateBK][kGM]>(smem_gates + 2 * kGateBK * kGN);  // 4 KB
    __shared__ float2 vel4[kGM];                            // 4 * (obs2 - obs1)
    __shared__ float2 obs2s[kGM];
    __shared__ int maskS[kGM];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int row0 = blockIdx.x * kGM;

    if (tid < kGM) {
        int m = row0 + tid;
        float2 a = make_float2(CUDART_NAN_F, CUDART_NAN_F), b = a;
        if (m < p.M) {
            a = p.obs1[m];
            b = p.obs2[m];
        }
        maskS[tid] = !(isnan(a.x) || isnan(b.x));                           // lstm.py:118
        vel4[tid] = make_float2((b.x - a.x) * 4.0f, (b.y - a.y) * 4.0f);   // modules.py:27 (scale)
        obs2s[tid] = b;
    }
    __syncthreads();

    float acc[4][4][4];   // [row][gate][unit]
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int g = 0; g < 4; ++g)
#pragma unroll
            for (int u = 0; u < 4; ++u) acc[r][g][u] = 0.f;

    const int nchunks = p.K_pad / kGateBK;

    auto load_w = [&](int buf, int chunk) {
        // 16 x 512 floats = 2048 float4, 8 per thread
        const float4* src = reinterpret_cast<const float4*>(p.WgT + (size_t)chunk * kGateBK * kGN);
        float4* dst = reinterpret_cast<float4*>(&Ws[buf][0][0]);
#pragma unroll
        for (int q = 0; q < (kGateBK * kGN / 4) / kGThreads; ++q) {
            int idx = tid + q * kGThreads;
            cp_async16(dst + idx, src + idx);
        }
    };
    auto load_a = [&](int buf, int chunk) {
        // 16 k x 32 rows = 512 values, 2 per thread; thread -> (kk = idx / 32, r = idx % 32)
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            int idx = tid + q * kGThreads;
            int kk = idx >> 5, r = idx & 31;
            int k = chunk * kGateBK + kk;
            int m = row0 + r;
            float v = 0.f;
            if (m < p.M && maskS[r]) {
                if (k < p.E) {
                    if (k < p.E - 2) {
                        float2 vv = vel4[r];
                        float e = fmaf(p.We[2 * k + 1], vv.y, fmaf(p.We[2 * k], vv.x, p.be[k]));
                        v = fmaxf(e, 0.f);
                    }
                } else if (k < p.E + p.P) {
                    v = p.pooled[(size_t)m * p.P + (k - p.E)];
                } else if (k < p.K) {
                    int u = k - p.E - p.P;
                    v = p.h_in[(size_t)m * kGH + u];
                    if (p.add_pooled_to_h) v += p.pooled[(size_t)m * kGH + u];   // lstm.py:151
                }
            }
            As[buf][kk][r] = v;
        }
    };

    load_w(0, 0);
    cp_async_commit();
    load_a(0, 0);
    for (int ch = 0; ch < nchunks; ++ch) {
        const int buf = ch & 1;
        if (ch + 1 < nchunks) {
            load_w(buf ^ 1, ch + 1);
            cp_async_commit();
            load_a(buf ^ 1, ch + 1);
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < kGateBK; ++kk) {
            const float4 a4 = *reinterpret_cast<const float4*>(&As[buf][kk][warp * 4]);
            const float a[4] = {a4.x, a4.y, a4.z, a4.w};
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                const float4 w4 = *reinterpret_cast<const float4*>(&Ws[buf][kk][g * kGH + lane * 4]);
                const float w[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
                for (int r = 0; r < 4; ++r)
#pragma unroll
                    for (int u = 0; u < 4; ++u) acc[r][g][u] = fmaf(a[r], w[u], acc[r][g][u]);
            }
        }
        __syncthreads();
    }

    // epilogue: LSTM pointwise + Gaussian head
    float bgr[4][4];
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        const float4 b4 = *reinterpret_cast<const float4*>(p.bg + g * kGH + lane * 4);
        bgr[g][0] = b4.x; bgr[g][1] = b4.y; bgr[g][2] = b4.z; bgr[g][3] = b4.w;
    }
    float wn[5][4];
#pragma unroll
    for (int o = 0; o < 5; ++o) {
        const float4 w4 = *reinterpret_cast<const float4*>(p.Wn + o * kGH + lane * 4);
        wn[o][0] = w4.x; wn[o][1] = w4.y; wn[o][2] = w4.z; wn[o][3] = w4.w;
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int rl = warp * 4 + r;
        const int m = row0 + rl;
        if (m >= p.M) continue;                       // warp-uniform
        const size_t off = (size_t)m * kGH + lane * 4;
        const float4 c4 = *reinterpret_cast<const float4*>(p.c_in + off);
        if (!maskS[rl]) {                             // warp-uniform: absent track keeps its state
            if (p.h_out != p.h_in) *reinterpret_cast<float4*>(p.h_out + off) = *reinterpret_cast<const float4*>(p.h_in + off);
            if (p.c_out != p.c_in) *reinterpret_cast<float4*>(p.c_out + off) = c4;
            if (lane < 5) p.normal_out[(size_t)m * 5 + lane] = CUDART_NAN_F;
            if (lane == 0 && p.pos_out) p.pos_out[m] = make_float2(CUDART_NAN_F, CUDART_NAN_F);
            continue;
        }
        const float cold[4] = {c4.x, c4.y, c4.z, c4.w};
        float hn[4], cn[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            float ig = sigmoidf_(acc[r][0][u] + bgr[0][u]);
            float fg = sigmoidf_(acc[r][1][u] + bgr[1][u]);
            float gg = tanhf(acc[r][2][u] + bgr[2][u]);
            float og = sigmoidf_(acc[r][3][u] + bgr[3][u]);
            cn[u] = fg * cold[u] + ig * gg;
            hn[u] = og * tanhf(cn[u]);
        }
        *reinterpret_cast<float4*>(p.h_out + off) = make_float4(hn[0], hn[1], hn[2], hn[3]);
        *reinterpret_cast<float4*>(p.c_out + off) = make_float4(cn[0], cn[1], cn[2], cn[3]);
        float part[5];
#pragma unroll
        for (int o = 0; o < 5; ++o) {
            float s = 0.f;
#pragma unroll
            for (int u = 0; u < 4; ++u) s = fmaf(hn[u], wn[o][u], s);
            part[o] = s;
        }
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1)
#pragma unroll
            for (int o = 0; o < 5; ++o) part[o] += __shfl_xor_sync(0xffffffffu, part[o], d);
        if (lane == 0) {
            float n0 = part[0] + p.bn[0], n1 = part[1] + p.bn[1];
            float n2 = 0.01f + 0.2f * sigmoidf_(part[2] + p.bn[2]);       // modules.py:60-62
            float n3 = 0.01f + 0.2f * sigmoidf_(part[3] + p.bn[3]);
            float n4 = 0.7f * sigmoidf_(part[4] + p.bn[4]);
            float* no = p.normal_out + (size_t)m * 5;
            no[0] = n0; no[1] = n1; no[2] = n2; no[3] = n3; no[4] = n4;
            if (p.pos_out) {
                float2 b = obs2s[rl];
                p.pos_out[m] = make_float2(b.x + n0, b.y + n1);          // lstm.py:232,255
            }
        }
    }
}

int launch_gates(const tb2_lstm* m, const tb2_layout* l, int phase, const float* obs1,
                 const float* obs2, const float* pooled, const float* h_in, const float* c_in,
                 float* h_out, float* c_out, float* normal_out, float* pos_out, cudaStream_t st) {
    TB2_REQUIRE(m->H == kGH, "hidden_dim must be 128");
    GateParams p;
    p.obs1 = (const float2*)obs1;
    p.obs2 = (const float2*)obs2;
    p.pooled = pooled;
    p.h_in = h_in;
    p.c_in = c_in;
    p.h_out = h_out;
    p.c_out = c_out;
    p.normal_out = normal_out;
    p.pos_out = (float2*)pos_out;
    p.We = m->We;
    p.be = m->be;
    p.WgT = m->WgT[phase];
    p.bg = m->bg[phase];
    p.Wn = m->Wn;
    p.bn = m->bn;
    p.M = l->M;
    p.E = m->E;
    p.P = m->P;
    p.K = m->K_gate;
    p.K_pad = m->K_gate_pad;
    p.add_pooled_to_h = (m->cfg.pool_type != TB2_POOL_NONE && !m->cfg.pool_to_input) ? 1 : 0;
    const size_t smem = (size_t)2 * kGateBK * (kGN + kGM) * sizeof(float);
    static DynSmemConfig configured;
    TB2_CHECK_CUDA(configured.ensure(lstm_gates_kernel, smem));
    int blocks = (l->M + kGM - 1) / kGM;
    {
        KernelTimer kt("lstm_gates", st);
        lstm_gates_kernel<<<blocks, kGThreads, smem, st>>>(p);
    }
    TB2_LAUNCH_CHECK();
    return TB2_OK;
}

// ------------------------------------------------------------------------------------------
// weight repack (device side, asynchronous): reference state_dict layout -> kernel layouts.
// ------------------------------------------------------------------------------------------
__global__ void repack_gates_kernel(const float* __restrict__ w_ih, const float* __restrict__ w_hh,
                                    const float* __restrict__ b_ih, const float* __restrict__ b_hh,
                                    float* __restrict__ WgT, float* __restrict__ bg, int in_dim, int H,
                                    int K_pad) {
    // WgT[k][n]: k < in_dim -> w_ih[n][k]; k < in_dim + H -> w_hh[n][k - in_dim]; else 0
    const int N = 4 * H;
    size_t total = (size_t)K_pad * N;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (size_t)gridDim.x * blockDim.x) {
        int k = (int)(idx / N), n = (int)(idx - (size_t)k * N);
        float v = 0.f;
        if (k < in_dim) v = w_ih[(size_t)n * in_dim + k];
        else if (k < in_dim + H) v = w_hh[(size_t)n * H + (k - in_dim)];
        WgT[idx] = v;
        if (k == 0) bg[n] = b_ih[n] + b_hh[n];
    }
}

__global__ void add_bias_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ out, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = a[i] + b[i];
}

// outT[c][o] = sum_m Win[o][m] * w[m][c]   (E x E matrices; AttentionMLPPooling: in-projection after wq / wk / wv)
__global__ void combine_proj_kernel(const float* __restrict__ Win, const float* __restrict__ w, float* __restrict__ outT, int E) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= E * E) return;
    const int c = idx / E, o = idx - c * E;
    float acc = 0.f;
    for (int mm = 0; mm < E; ++mm) acc = fmaf(Win[(size_t)o * E + mm], w[(size_t)mm * E + c], acc);
    outT[idx] = acc;
}

__global__ void transpose_kernel(const float* __restrict__ W, float* __restrict__ WT, int N, int K) {
    // W [N, K] -> WT [K, N]
    size_t total = (size_t)N * K;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (size_t)gridDim.x * blockDim.x) {
        int k = (int)(idx / N), n = (int)(idx - (size_t)k * N);
        WT[idx] = W[(size_t)n * K + k];
    }
}

__global__ void repack_layer1_kernel(const float* __restrict__ W1, const float* __restrict__ b1,
                                     float* __restrict__ Wt, float* __restrict__ base, int OUT, int C,
                                     int cells, float constant) {
    // Wt[cell][c][o] = W1[o][c * cells + cell]   (grid flattened channel-major, :107,294-295)
    size_t total = (size_t)cells * C * OUT;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (size_t)gridDim.x * blockDim.x) {
        int o = (int)(idx % OUT);
        int cc = (int)(idx / OUT);
        int c = cc % C, cell = cc / C;
        Wt[idx] = W1[(size_t)o * C * cells + (size_t)c * cells + cell];
    }
    // base[o] = b1[o] + constant * sum_k W1[o][k]
    for (int o = blockIdx.x * blockDim.x + threadIdx.x; o < OUT; o += gridDim.x * blockDim.x) {
        float s = 0.f;
        if (constant != 0.f) {
            const float* row = W1 + (size_t)o * C * cells;
            for (int k = 0; k < C * cells; ++k) s += row[k];
        }
        base[o] = b1[o] + constant * s;
    }
}

__global__ void copy_kernel(const float* __restrict__ src, float* __restrict__ dst, size_t n) {
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < n;
         idx += (size_t)gridDim.x * blockDim.x)
        dst[idx] = src[idx];
}

static int copy_dev(const float* src, float* dst, size_t n, cudaStream_t st) {
    copy_kernel<<<(unsigned)((n + 255) / 256 > 1024 ? 1024 : (n + 255) / 256), 256, 0, st>>>(src, dst, n);
    TB2_LAUNCH_CHECK();
    return TB2_OK;
}

int launch_repack(tb2_lstm* m, const tb2_lstm_weights* w, cudaStream_t st) {
    TB2_REQUIRE(w->input_embedding_weight && w->input_embedding_bias, "input embedding weights missing");
    TB2_REQUIRE(w->encoder_weight_ih && w->encoder_weight_hh && w->encoder_bias_ih && w->encoder_bias_hh,
                "encoder weights missing");
    TB2_REQUIRE(w->decoder_weight_ih && w->decoder_weight_hh && w->decoder_bias_ih && w->decoder_bias_hh,
                "decoder weights missing");
    TB2_REQUIRE(w->hidden2normal_weight && w->hidden2normal_bias, "hidden2normal weights missing");
    int rc;
    if ((rc = copy_dev(w->input_embedding_weight, m->We, (size_t)(m->E - 2) * 2, st))) return rc;
    if ((rc = copy_dev(w->input_embedding_bias, m->be, (size_t)(m->E - 2), st))) return rc;
    if ((rc = copy_dev(w->hidden2normal_weight, m->Wn, (size_t)5 * m->H, st))) return rc;
    if ((rc = copy_dev(w->hidden2normal_bias, m->bn, 5, st))) return rc;
    const float* wih[2] = {w->encoder_weight_ih, w->decoder_weight_ih};
    const float* whh[2] = {w->encoder_weight_hh, w->decoder_weight_hh};
    const float* bih[2] = {w->encoder_bias_ih, w->decoder_bias_ih};
    const float* bhh[2] = {w->encoder_bias_hh, w->decoder_bias_hh};
    for (int ph = 0; ph < 2; ++ph) {
        repack_gates_kernel<<<512, 256, 0, st>>>(wih[ph], whh[ph], bih[ph], bhh[ph], m->WgT[ph], m->bg[ph],
                                                 m->E + m->P, m->H, m->K_gate_pad);
        TB2_LAUNCH_CHECK();
        if (m->Wg_hi[ph] &&
            (rc = launch_repack_gates_tc(wih[ph], whh[ph], m->Wg_hi[ph], m->Wg_lo[ph], m->E + m->P, m->H, st)))
            return rc;
    }
    if (m->cfg.pool_type == TB2_POOL_TRAJECTRON) {
        TB2_REQUIRE(w->pool_spatial_weight && w->pool_spatial_bias, "pool.embedding.0 (Trajectron pooling) missing");
        if ((rc = copy_dev(w->pool_spatial_weight, m->mp_Ws, (size_t)m->cfg.out_dim * 8, st))) return rc;
        if ((rc = copy_dev(w->pool_spatial_bias, m->mp_bs, (size_t)m->cfg.out_dim, st))) return rc;
    }
    if (m->cfg.pool_type == TB2_POOL_NN_LSTM || m->cfg.pool_type == TB2_POOL_TRAJECTRON) {
        const tb2_lstm_config& c = m->cfg;
        const int Hp = c.mlp_dim_hidden;
        TB2_REQUIRE(w->pool_lstm_weight_ih && w->pool_lstm_weight_hh && w->pool_lstm_bias_ih && w->pool_lstm_bias_hh &&
                    w->pool_out_weight && w->pool_out_bias, "pool.pool_lstm / pool.hidden2pool parameters missing");
        transpose_kernel<<<256, 256, 0, st>>>(w->pool_lstm_weight_ih, m->pl_WihT, 4 * Hp, c.out_dim);
        TB2_LAUNCH_CHECK();
        transpose_kernel<<<256, 256, 0, st>>>(w->pool_lstm_weight_hh, m->pl_WhhT, 4 * Hp, Hp);
        TB2_LAUNCH_CHECK();
        add_bias_kernel<<<(4 * Hp + 255) / 256, 256, 0, st>>>(w->pool_lstm_bias_ih, w->pool_lstm_bias_hh, m->pl_b, 4 * Hp);
        TB2_LAUNCH_CHECK();
        transpose_kernel<<<128, 256, 0, st>>>(w->pool_out_weight, m->mp_WoT, c.out_dim, Hp);
        TB2_LAUNCH_CHECK();
        if ((rc = copy_dev(w->pool_out_bias, m->mp_bo, (size_t)c.out_dim, st))) return rc;
    }
    if (m->cfg.pool_type == TB2_POOL_NN_MLP || m->cfg.pool_type == TB2_POOL_NN_LSTM) {
        const tb2_lstm_config& c = m->cfg;
        TB2_REQUIRE(w->pool_spatial_weight && w->pool_spatial_bias, "pool.embedding.0 (nearest-neighbour pooling) missing");
        if ((rc = copy_dev(w->pool_spatial_weight, m->mp_Ws, (size_t)c.mlp_dim_spatial * (c.mlp_dim_vel ? 4 : 2), st))) return rc;
        if ((rc = copy_dev(w->pool_spatial_bias, m->mp_bs, (size_t)c.mlp_dim_spatial, st))) return rc;
    }
    if (m->cfg.pool_type == TB2_POOL_ATTN_MLP) {
        const int Ea = m->cfg.mlp_dim_spatial + m->cfg.mlp_dim_vel + m->cfg.mlp_dim_hidden;
        TB2_REQUIRE(w->pool_attn_wq && w->pool_attn_wk && w->pool_attn_wv && w->pool_attn_in_proj_weight &&
                    w->pool_attn_in_proj_bias && w->pool_attn_out_proj_weight && w->pool_attn_out_proj_bias,
                    "pool.wq / wk / wv / multihead_attn parameters missing");
        // in-projection . w{q,k,v}: A[o][c] = sum_m Win[o][m] w[m][c], stored transposed [c][o]
        const float* wqkv[3] = {w->pool_attn_wq, w->pool_attn_wk, w->pool_attn_wv};
        float* outT[3] = {m->at_AqT, m->at_AkT, m->at_AvT};
        for (int i = 0; i < 3; ++i) {
            combine_proj_kernel<<<(Ea * Ea + 255) / 256, 256, 0, st>>>(w->pool_attn_in_proj_weight + (size_t)i * Ea * Ea, wqkv[i],
                                                                     outT[i], Ea);
            TB2_LAUNCH_CHECK();
        }
        if ((rc = copy_dev(w->pool_attn_in_proj_bias, m->at_bqkv, (size_t)3 * Ea, st))) return rc;
        transpose_kernel<<<64, 256, 0, st>>>(w->pool_attn_out_proj_weight, m->at_WoT, Ea, Ea);
        TB2_LAUNCH_CHECK();
        if ((rc = copy_dev(w->pool_attn_out_proj_bias, m->at_bo, (size_t)Ea, st))) return rc;
    }
    if (m->cfg.pool_type == TB2_POOL_HIDDEN_MLP || m->cfg.pool_type == TB2_POOL_ATTN_MLP) {
        const tb2_lstm_config& c = m->cfg;
        const int D = c.mlp_dim_spatial + c.mlp_dim_vel + c.mlp_dim_hidden;
        TB2_REQUIRE(w->pool_spatial_weight && w->pool_spatial_bias && w->pool_out_weight && w->pool_out_bias,
                    "pool.spatial_embedding / pool.out_projection missing");
        TB2_REQUIRE(c.mlp_dim_vel == 0 || (w->pool_vel_weight && w->pool_vel_bias), "pool.vel_embedding missing");
        TB2_REQUIRE(c.mlp_dim_hidden == 0 || (w->pool_hidden_weight && w->pool_hidden_bias), "pool.hidden_embedding missing");
        if ((rc = copy_dev(w->pool_spatial_weight, m->mp_Ws, (size_t)c.mlp_dim_spatial * 2, st))) return rc;
        if ((rc = copy_dev(w->pool_spatial_bias, m->mp_bs, (size_t)c.mlp_dim_spatial, st))) return rc;
        if (c.mlp_dim_vel) {
            if ((rc = copy_dev(w->pool_vel_weight, m->mp_Wv, (size_t)c.mlp_dim_vel * 2, st))) return rc;
            if ((rc = copy_dev(w->pool_vel_bias, m->mp_bv, (size_t)c.mlp_dim_vel, st))) return rc;
        }
        if (c.mlp_dim_hidden) {
            transpose_kernel<<<64, 256, 0, st>>>(w->pool_hidden_weight, m->mp_WhT, c.mlp_dim_hidden, m->H);
            TB2_LAUNCH_CHECK();
            if ((rc = copy_dev(w->pool_hidden_bias, m->mp_bh, (size_t)c.mlp_dim_hidden, st))) return rc;
        }
        transpose_kernel<<<128, 256, 0, st>>>(w->pool_out_weight, m->mp_WoT, c.out_dim, D);
        TB2_LAUNCH_CHECK();
        if ((rc = copy_dev(w->pool_out_bias, m->mp_bo, (size_t)c.out_dim, st))) return rc;
    }
    if (m->cfg.pool_type == TB2_POOL_SOCIAL) {
        TB2_REQUIRE(w->pool_encoding_weight && w->pool_encoding_bias, "pool.hidden_dim_encoding missing");
        transpose_kernel<<<64, 256, 0, st>>>(w->pool_encoding_weight, m->WencT, m->C, m->H);
        TB2_LAUNCH_CHECK();
        if ((rc = copy_dev(w->pool_encoding_bias, m->benc, (size_t)m->C, st))) return rc;
    }
    if (m->cfg.pool_type != TB2_POOL_NONE && m->cfg.pool_type < TB2_POOL_HIDDEN_MLP && m->n_mlp >= 1) {
        TB2_REQUIRE(w->pool_embedding_weight[0] && w->pool_embedding_bias[0], "pool.embedding.0 missing");
        repack_layer1_kernel<<<1024, 256, 0, st>>>(w->pool_embedding_weight[0], w->pool_embedding_bias[0],
                                                   m->Wt1, m->base1, m->mlp_dims[1], m->C, m->cells,
                                                   m->cfg.constant);
        TB2_LAUNCH_CHECK();
        if (m->Wt1_hi &&
            (rc = launch_repack_layer1_mma(w->pool_embedding_weight[0], m->Wt1_hi, m->Wt1_lo, m->mlp_dims[1], m->cells, st)))
            return rc;
        if (m->Wt1_nat_hi &&
            (rc = launch_repack_layer1_nat(w->pool_embedding_weight[0], m->Wt1_nat_hi, m->Wt1_nat_lo, m->mlp_dims[1], m->cells, st)))
            return rc;
        if (m->Wt1_sw_hi &&
            (rc = launch_repack_layer1_sw(w->pool_embedding_weight[0], m->Wt1_sw_hi, m->Wt1_sw_lo, m->mlp_dims[1], m->cells, st)))
            return rc;
        for (int layer = 1; layer < m->n_mlp; ++layer) {
            TB2_REQUIRE(w->pool_embedding_weight[layer] && w->pool_embedding_bias[layer], "pool.embedding layer missing");
            transpose_kernel<<<512, 256, 0, st>>>(w->pool_embedding_weight[layer], m->WT[layer],
                                                  m->mlp_dims[layer + 1], m->mlp_dims[layer]);
            TB2_LAUNCH_CHECK();
            if ((rc = copy_dev(w->pool_embedding_bias[layer], m->bl[layer], (size_t)m->mlp_dims[layer + 1], st))) return rc;
            if (m->W_hi[layer] &&
                (rc = launch_split_bf16(w->pool_embedding_weight[layer], m->W_hi[layer], m->W_lo[layer],
                                        (size_t)m->mlp_dims[layer] * m->mlp_dims[layer + 1], st)))
                return rc;
        }
    }
    m->weights_set = true;
    return TB2_OK;
}

}  // namespace tb2
