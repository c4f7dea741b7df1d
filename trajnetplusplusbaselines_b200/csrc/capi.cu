// extern "C" boundary of libtrajnet_b200 (see include/trajnet_b200.h).
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

#include "common.cuh"

namespace tb2 {

static thread_local std::string g_error;
std::atomic<uint64_t> g_launch_count{0};

void set_error(const std::string& msg) { g_error = msg; }

// ---- optional per-kernel CUDA-event timing ---------------------------------------------------
struct ProfRec { const char* name; cudaEvent_t a, b; };
static bool g_profiling = false;
static std::vector<ProfRec> g_prof;

KernelTimer::KernelTimer(const char* name, cudaStream_t s) : slot(-1), st(s) {
    if (!g_profiling) return;
    ProfRec r;
    r.name = name;
    if (cudaEventCreate(&r.a) != cudaSuccess || cudaEventCreate(&r.b) != cudaSuccess) return;
    cudaEventRecord(r.a, st);
    g_prof.push_back(r);
    slot = (int)g_prof.size() - 1;
}
KernelTimer::~KernelTimer() {
    if (slot >= 0) cudaEventRecord(g_prof[slot].b, st);
}

static int dev_alloc(std::vector<void*>& owned, void** out, size_t bytes) {
    *out = nullptr;
    if (bytes == 0) bytes = 16;
    TB2_CHECK_CUDA(cudaMalloc(out, bytes));
    owned.push_back(*out);
    return TB2_OK;
}

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

size_t carve_workspace(const tb2_lstm* m, const tb2_layout* l, void* base, Workspace* ws) {
    const size_t M = (size_t)l->M;
    const size_t nm1 = (size_t)(l->n_max > 1 ? l->n_max - 1 : 1);
    size_t off = 0;
    auto take = [&](size_t bytes) {
        size_t o = off;
        off = align_up(off + bytes, 256);
        return base ? (void*)((char*)base + o) : (void*)nullptr;
    };
    Workspace w;
    w.obs1 = (float*)take(M * 2 * sizeof(float));
    w.obs2 = (float*)take(M * 2 * sizeof(float));
    w.lat = (float*)take(M * (size_t)std::max(m->C, 1) * sizeof(float));
    w.win_count = (int*)take(M * sizeof(int));
    w.win_ent = (uint32_t*)take(M * nm1 * sizeof(uint32_t));
    w.win_val = (float*)take(M * nm1 * 2 * sizeof(float));
    w.pair_cell = (int*)take(M * nm1 * sizeof(int));
    w.pair_flag = (uint8_t*)take(M * nm1);
    w.cell_row = nullptr;
    if (m->Wt1_sw_hi != nullptr && m->cells <= 256) w.cell_row = (uint8_t*)take(M * (size_t)m->cells);
    size_t wmax = 1;
    for (int i = 1; i <= m->n_mlp; ++i) wmax = std::max(wmax, (size_t)m->mlp_dims[i]);
    w.act[0] = (float*)take(M * wmax * sizeof(float));
    w.act[1] = (float*)take(M * wmax * sizeof(float));
    w.act2 = (float*)take(m->n_mlp > 2 ? M * wmax * sizeof(float) : 16);
    w.pooled = (float*)take(M * (size_t)std::max(m->pool_out, 1) * sizeof(float));
    w.emb_hi = take(M * 64 * 2);
    w.emb_lo = take(M * 64 * 2);
    w.pool_hi = take(M * (size_t)std::max(m->P, 1) * 2);
    w.pool_lo = take(M * (size_t)std::max(m->P, 1) * 2);
    for (int i = 0; i < 2; ++i) {
        w.hs_hi[i] = take(M * 128 * 2);
        w.hs_lo[i] = take(M * 128 * 2);
    }
    w.pool_feat = w.pool_h = w.pool_c = w.scene_sum = nullptr;
    if (m->cfg.pool_type == TB2_POOL_TRAJECTRON) w.scene_sum = (float*)take((size_t)l->B * 4 * sizeof(float));
    if (m->cfg.pool_type == TB2_POOL_NN_LSTM || m->cfg.pool_type == TB2_POOL_TRAJECTRON) {
        w.pool_feat = (float*)take(M * (size_t)m->cfg.out_dim * sizeof(float));
        w.pool_h = (float*)take(M * (size_t)m->cfg.mlp_dim_hidden * sizeof(float));
        w.pool_c = (float*)take(M * (size_t)m->cfg.mlp_dim_hidden * sizeof(float));
    }
    w.bytes = off;
    w.write_pairs = 0;
    if (ws) *ws = w;
    return off;
}

size_t carve_train_cache(const tb2_lstm* m, const tb2_layout* l, size_t S, void* base, TrainCache* out) {
    const bool two = m->n_mlp == 2;
    if (m->cfg.pool_type != TB2_POOL_SOCIAL || m->Wg_hi[0] == nullptr || m->n_mlp < 1 || m->n_mlp > 2 || !m->cfg.pool_to_input ||
        (two && m->W_hi[1] == nullptr))
        return 0;
    const size_t M = (size_t)l->M, C = (size_t)m->C, nm1 = (size_t)(l->n_max > 1 ? l->n_max - 1 : 1);
    const size_t d1 = (size_t)m->mlp_dims[1], P = (size_t)m->P;
    size_t off = 0;
    auto take = [&](size_t bytes) {
        void* p = base ? (void*)((char*)base + off) : nullptr;
        off += (bytes + 255) & ~(size_t)255;
        return p;
    };
    TrainCache c;
    c.lat = (float*)take(S * M * C * sizeof(float));
    c.win_count = (int*)take(S * M * sizeof(int));
    c.win_ent = (uint32_t*)take(S * M * nm1 * sizeof(uint32_t));
    c.pair_cell = (int*)take(S * M * nm1 * sizeof(int));
    c.pair_flag = (uint8_t*)take(S * M * nm1);
    c.h1_hi = two ? take(S * M * d1 * 2) : nullptr;
    c.h1_lo = two ? take(S * M * d1 * 2) : nullptr;
    c.pool_hi = take(S * M * P * 2);
    c.pool_lo = take(S * M * P * 2);
    if (out) *out = c;
    return off;
}

// Inputs of recurrence step s (encoder: lstm.py:226-232; decoder feedback rule: lstm.py:240-250).
// positions[s'] is the output of step s' (obs2 + mu).  May launch resolve_obs into ws->obs1/obs2.
int resolve_step_inputs(const tb2_layout* l, const float* observed, int obs_length, const float* truth,
                        const float* positions, int s, Workspace* ws, const float** o1, const float** o2,
                        int* phase, cudaStream_t st) {
    const size_t frame = (size_t)l->M * 2;
    int rc;
    if (s < obs_length - 1) {
        *phase = TB2_PHASE_ENCODER;
        *o1 = observed + (size_t)s * frame;
        *o2 = observed + (size_t)(s + 1) * frame;
        return TB2_OK;
    }
    *phase = TB2_PHASE_DECODER;
    const int k = s - (obs_length - 1);
    // positions[-1] = output of step s-1, positions[-2] = output of step s-2
    // (or observed[-1] when obs_length == 2, lstm.py:222-223)
    const float* pos_m1 = positions + (size_t)(s - 1) * frame;
    const float* pos_m2 = (s >= 2) ? positions + (size_t)(s - 2) * frame
                                   : observed + (size_t)(obs_length - 1) * frame;
    // obs1 = seq[k]: seq[0] = observed[-1] (always a tensor -> primary rows only)
    if (k == 0) {
        if ((rc = launch_resolve_obs(l, observed + (size_t)(obs_length - 1) * frame, pos_m2, ws->obs1, st))) return rc;
        *o1 = ws->obs1;
    } else if (truth) {
        if ((rc = launch_resolve_obs(l, truth + (size_t)(k - 1) * frame, pos_m2, ws->obs1, st))) return rc;
        *o1 = ws->obs1;
    } else {
        *o1 = pos_m2;                                                      // :242 all rows predicted
    }
    if (truth) {
        if ((rc = launch_resolve_obs(l, truth + (size_t)k * frame, pos_m1, ws->obs2, st))) return rc;
        *o2 = ws->obs2;
    } else {
        *o2 = pos_m1;                                                      // :247
    }
    return TB2_OK;
}

}  // namespace tb2

using namespace tb2;

extern "C" {

const char* tb2_last_error(void) { return g_error.c_str(); }
int tb2_version(void) { return 100; }
uint64_t tb2_launch_count(void) { return g_launch_count.load(); }

int tb2_profile_begin(void) {
    for (auto& r : g_prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    g_prof.clear();
    g_profiling = true;
    return TB2_OK;
}

int tb2_profile_end(char* json_out, size_t capacity) {
    g_profiling = false;
    TB2_CHECK_CUDA(cudaDeviceSynchronize());
    struct Agg { const char* name; double ms; long n; };
    std::vector<Agg> agg;
    for (auto& r : g_prof) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, r.a, r.b);
        bool found = false;
        for (auto& a : agg) if (std::strcmp(a.name, r.name) == 0) { a.ms += ms; a.n++; found = true; break; }
        if (!found) agg.push_back({r.name, (double)ms, 1});
        cudaEventDestroy(r.a);
        cudaEventDestroy(r.b);
    }
    g_prof.clear();
    std::string s = "{";
    for (size_t i = 0; i < agg.size(); ++i) {
        char buf[256];
        snprintf(buf, sizeof(buf), "%s\"%s\": {\"launches\": %ld, \"total_ms\": %.6f}", i ? ", " : "",
                 agg[i].name, agg[i].n, agg[i].ms);
        s += buf;
    }
    s += "}";
    TB2_REQUIRE(json_out && capacity > s.size(), "profile buffer too small");
    std::memcpy(json_out, s.c_str(), s.size() + 1);
    return TB2_OK;
}

int tb2_lstm_create(const tb2_lstm_config* cfg, tb2_lstm** out) {
    TB2_REQUIRE(cfg && out, "null argument");
    *out = nullptr;
    TB2_REQUIRE(cfg->hidden_dim == 128, "hidden_dim must be 128 (kernel specialisation)");
    TB2_REQUIRE(cfg->embedding_dim >= 4 && cfg->embedding_dim <= 1024, "embedding_dim out of range");
    TB2_REQUIRE(cfg->pool_type >= TB2_POOL_NONE && cfg->pool_type <= TB2_POOL_TRAJECTRON, "bad pool_type");
    tb2_lstm* m = new (std::nothrow) tb2_lstm();
    TB2_REQUIRE(m, "out of host memory");
    m->cfg = *cfg;
    m->H = cfg->hidden_dim;
    m->E = cfg->embedding_dim;
    m->weights_set = false;
    m->C = 0; m->cells = 0; m->n_mlp = 0; m->P = 0; m->pool_out = 0;
    m->We = m->be = m->Wn = m->bn = m->WencT = m->benc = m->Wt1 = m->base1 = nullptr;
    m->Wt1_hi = m->Wt1_lo = m->Wt1_nat_hi = m->Wt1_nat_lo = m->Wt1_sw_hi = m->Wt1_sw_lo = nullptr;
    for (int i = 0; i < 2; ++i) { m->WgT[i] = m->bg[i] = nullptr; m->Wg_hi[i] = m->Wg_lo[i] = nullptr; }
    for (int i = 0; i < kMaxMlpLayers; ++i) { m->WT[i] = m->bl[i] = nullptr; m->W_hi[i] = m->W_lo[i] = nullptr; }
    m->mp_Ws = m->mp_bs = m->mp_Wv = m->mp_bv = m->mp_WhT = m->mp_bh = m->mp_WoT = m->mp_bo = nullptr;
    m->at_AqT = m->at_AkT = m->at_AvT = m->at_bqkv = m->at_WoT = m->at_bo = nullptr;
    m->pl_WihT = m->pl_WhhT = m->pl_b = nullptr;
    auto fail = [&](int rc) { tb2_lstm_destroy(m); return rc; };
    if (cfg->pool_type == TB2_POOL_TRAJECTRON) {
        if (!(cfg->mlp_dim_hidden >= 1 && cfg->mlp_dim_hidden <= 512 && cfg->out_dim >= 1 && cfg->out_dim <= 1024)) {
            set_error("invalid argument: Trajectron pooling needs 1 <= hidden_dim <= 512 and out_dim <= 1024");
            return fail(TB2_ERR_INVALID);
        }
        m->pool_out = cfg->out_dim;
        if (cfg->pool_to_input) m->P = m->pool_out;
        else if (m->pool_out != m->H) { set_error("invalid argument: pool_to_input=0 needs out_dim == hidden_dim"); return fail(TB2_ERR_INVALID); }
    }
    if (cfg->pool_type == TB2_POOL_NN_LSTM &&
        !(cfg->mlp_dim_hidden >= 1 && cfg->mlp_dim_hidden <= 512 && cfg->out_dim <= 1024 && cfg->mlp_dim_vel != 0)) {
        set_error("invalid argument: nearest-neighbour LSTM pooling needs 1 <= hidden_dim <= 512, out_dim <= 1024 and velocities");
        return fail(TB2_ERR_INVALID);
    }
    if (cfg->pool_type == TB2_POOL_TRAJECTRON) {
        // validated above
    } else
    if (cfg->pool_type == TB2_POOL_NN_MLP || cfg->pool_type == TB2_POOL_NN_LSTM) {
        if (!(cfg->n >= 1 && cfg->n <= 32 && cfg->mlp_dim_spatial >= 1 && cfg->out_dim == cfg->n * cfg->mlp_dim_spatial)) {
            set_error("invalid argument: nearest-neighbour pooling needs 1 <= n <= 32 and out_dim == n * mlp_dim_spatial");
            return fail(TB2_ERR_INVALID);
        }
        m->pool_out = cfg->out_dim;
        if (cfg->pool_to_input) m->P = m->pool_out;
        else if (m->pool_out != m->H) { set_error("invalid argument: pool_to_input=0 needs out_dim == hidden_dim"); return fail(TB2_ERR_INVALID); }
    } else
    if (cfg->pool_type == TB2_POOL_ATTN_MLP) {
        const int Ea = cfg->mlp_dim_spatial + cfg->mlp_dim_vel + cfg->mlp_dim_hidden;
        if (!(cfg->mlp_dim_spatial >= 1 && cfg->mlp_dim_vel >= 0 && cfg->mlp_dim_hidden >= 0 && cfg->out_dim >= 1 && Ea <= 128)) {
            set_error("invalid argument: attention pooling needs mlp_dim <= 128 (kernel specialisation)");
            return fail(TB2_ERR_INVALID);
        }
        m->pool_out = cfg->out_dim;
        if (cfg->pool_to_input) m->P = m->pool_out;
        else if (m->pool_out != m->H) { set_error("invalid argument: pool_to_input=0 needs out_dim == hidden_dim"); return fail(TB2_ERR_INVALID); }
    } else
    if (cfg->pool_type == TB2_POOL_HIDDEN_MLP) {
        if (!(cfg->mlp_dim_spatial >= 1 && cfg->mlp_dim_vel >= 0 && cfg->mlp_dim_hidden >= 0 && cfg->out_dim >= 1 &&
              cfg->mlp_dim_spatial + cfg->mlp_dim_vel + cfg->mlp_dim_hidden <= 4096)) {
            set_error("invalid argument: hidden-state MLP pooling widths");
            return fail(TB2_ERR_INVALID);
        }
        m->pool_out = cfg->out_dim;
        if (cfg->pool_to_input) m->P = m->pool_out;
        else if (m->pool_out != m->H) { set_error("invalid argument: pool_to_input=0 needs out_dim == hidden_dim"); return fail(TB2_ERR_INVALID); }
    } else
    if (cfg->pool_type != TB2_POOL_NONE) {
        if (cfg->pool_size != 1 || cfg->blur_size != 1) {
            set_error("pool_size / blur_size != 1 are not built (the reference CLI never sets them)");
            return fail(TB2_ERR_UNSUPPORTED);
        }
        if (!(cfg->n >= 1 && cfg->n <= 64 && cfg->cell_side > 0.f)) { set_error("invalid argument: grid size"); return fail(TB2_ERR_INVALID); }
        if (!(cfg->num_layers >= 0 && cfg->num_layers <= kMaxMlpLayers)) { set_error("invalid argument: num_layers"); return fail(TB2_ERR_INVALID); }
        m->C = cfg->pool_type == TB2_POOL_OCCUPANCY ? 1 : cfg->pool_type == TB2_POOL_DIRECTIONAL ? 2 : cfg->latent_dim;
        if (cfg->pool_type == TB2_POOL_SOCIAL && !(m->C == 4 || m->C == 8 || m->C == 16 || m->C == 32)) {
            set_error("social latent_dim must be 4, 8, 16 or 32");
            return fail(TB2_ERR_UNSUPPORTED);
        }
        m->cells = cfg->n * cfg->n;
        m->n_mlp = cfg->num_layers;
        m->mlp_dims[0] = m->C * m->cells;
        for (int i = 1; i <= m->n_mlp; ++i)
            m->mlp_dims[i] = (i == m->n_mlp) ? cfg->out_dim : cfg->layer_dims[i - 1];
        m->pool_out = m->n_mlp == 0 ? m->mlp_dims[0] : cfg->out_dim;
        for (int i = 1; i <= m->n_mlp; ++i)
            if (m->mlp_dims[i] < 1) { set_error("invalid argument: MLP width"); return fail(TB2_ERR_INVALID); }
        if (cfg->pool_to_input) m->P = m->pool_out;
        else if (m->pool_out != m->H) { set_error("invalid argument: pool_to_input=0 needs out_dim == hidden_dim"); return fail(TB2_ERR_INVALID); }
    }
    m->K_gate = m->E + m->P + m->H;
    m->K_gate_pad = (m->K_gate + kGateBK - 1) / kGateBK * kGateBK;
    int rc;
#define ALLOC(ptr, count) if ((rc = dev_alloc(m->owned, (void**)&(ptr), (size_t)(count) * sizeof(float)))) return fail(rc)
    ALLOC(m->We, (m->E - 2) * 2);
    ALLOC(m->be, m->E - 2);
    ALLOC(m->Wn, 5 * m->H);
    ALLOC(m->bn, 5);
    for (int ph = 0; ph < 2; ++ph) {
        ALLOC(m->WgT[ph], (size_t)m->K_gate_pad * 4 * m->H);
        ALLOC(m->bg[ph], 4 * m->H);
    }
    const bool use_tc = !tc_disabled();
    if (use_tc && gates_tc_supported(m)) {
        const size_t half = ((size_t)4 * m->H * m->K_gate + 1) / 2;
        for (int ph = 0; ph < 2; ++ph) {
            float *hi, *lo;
            ALLOC(hi, half);
            ALLOC(lo, half);
            m->Wg_hi[ph] = hi;
            m->Wg_lo[ph] = lo;
        }
    }
    if (cfg->pool_type == TB2_POOL_SOCIAL) {
        ALLOC(m->WencT, m->H * m->C);
        ALLOC(m->benc, m->C);
    }
    if (cfg->pool_type == TB2_POOL_TRAJECTRON) {
        ALLOC(m->mp_Ws, (size_t)cfg->out_dim * 8);
        ALLOC(m->mp_bs, cfg->out_dim);
    }
    if (cfg->pool_type == TB2_POOL_NN_LSTM || cfg->pool_type == TB2_POOL_TRAJECTRON) {
        const size_t Hp = (size_t)cfg->mlp_dim_hidden;
        ALLOC(m->pl_WihT, (size_t)cfg->out_dim * 4 * Hp);
        ALLOC(m->pl_WhhT, Hp * 4 * Hp);
        ALLOC(m->pl_b, 4 * Hp);
        ALLOC(m->mp_WoT, Hp * (size_t)cfg->out_dim);
        ALLOC(m->mp_bo, cfg->out_dim);
    }
    if (cfg->pool_type == TB2_POOL_NN_MLP || cfg->pool_type == TB2_POOL_NN_LSTM) {
        ALLOC(m->mp_Ws, cfg->mlp_dim_spatial * 4);
        ALLOC(m->mp_bs, cfg->mlp_dim_spatial);
    } else
    if (cfg->pool_type == TB2_POOL_ATTN_MLP) {
        const size_t Ea = (size_t)(cfg->mlp_dim_spatial + cfg->mlp_dim_vel + cfg->mlp_dim_hidden);
        ALLOC(m->at_AqT, Ea * Ea);
        ALLOC(m->at_AkT, Ea * Ea);
        ALLOC(m->at_AvT, Ea * Ea);
        ALLOC(m->at_bqkv, 3 * Ea);
        ALLOC(m->at_WoT, Ea * Ea);
        ALLOC(m->at_bo, Ea);
    }
    if (cfg->pool_type == TB2_POOL_HIDDEN_MLP || cfg->pool_type == TB2_POOL_ATTN_MLP) {
        const int D = cfg->mlp_dim_spatial + cfg->mlp_dim_vel + cfg->mlp_dim_hidden;
        ALLOC(m->mp_Ws, cfg->mlp_dim_spatial * 2);
        ALLOC(m->mp_bs, cfg->mlp_dim_spatial);
        ALLOC(m->mp_Wv, std::max(cfg->mlp_dim_vel, 1) * 2);
        ALLOC(m->mp_bv, std::max(cfg->mlp_dim_vel, 1));
        ALLOC(m->mp_WhT, (size_t)m->H * std::max(cfg->mlp_dim_hidden, 1));
        ALLOC(m->mp_bh, std::max(cfg->mlp_dim_hidden, 1));
        ALLOC(m->mp_WoT, (size_t)D * cfg->out_dim);
        ALLOC(m->mp_bo, cfg->out_dim);
    }
    if (m->n_mlp >= 1) {
        ALLOC(m->Wt1, (size_t)m->cells * m->C * m->mlp_dims[1]);
        ALLOC(m->base1, m->mlp_dims[1]);
        if (cfg->pool_type == TB2_POOL_SOCIAL && m->C == 16 && use_tc) {
            const size_t half = ((size_t)m->cells * 16 * m->mlp_dims[1] + 1) / 2;
            float *hi, *lo;
            ALLOC(hi, 2 * half);      // interleaved (hi | lo) slabs
            ALLOC(lo, 4);
            m->Wt1_hi = hi;
            m->Wt1_lo = lo;
            float *nh, *nl;
            ALLOC(nh, half);
            ALLOC(nl, half);
            m->Wt1_nat_hi = nh;
            m->Wt1_nat_lo = nl;
            float *sh, *sl;
            ALLOC(sh, 2 * half);      // hi and lo interleaved by 8-row group (one bulk copy per slab)
            ALLOC(sl, 4);
            m->Wt1_sw_hi = sh;
            m->Wt1_sw_lo = sl;
        }
        for (int layer = 1; layer < m->n_mlp; ++layer) {
            ALLOC(m->WT[layer], (size_t)m->mlp_dims[layer] * m->mlp_dims[layer + 1]);
            ALLOC(m->bl[layer], m->mlp_dims[layer + 1]);
            if (layer == 1 && use_tc && dense_tc_supported(m->mlp_dims[1], m->mlp_dims[2])) {
                const size_t half = ((size_t)m->mlp_dims[1] * m->mlp_dims[2] + 1) / 2;   // bf16 pairs in float units
                float *hi, *lo;
                ALLOC(hi, half);
                ALLOC(lo, half);
                m->W_hi[1] = hi;
                m->W_lo[1] = lo;
            }
        }
    }
#undef ALLOC
    *out = m;
    return TB2_OK;
}

int tb2_lstm_destroy(tb2_lstm* m) {
    if (!m) return TB2_OK;
    for (cudaEvent_t ev : m->step_events) cudaEventDestroy(ev);
    for (void* p : m->owned) cudaFree(p);
    delete m;
    return TB2_OK;
}

int tb2_lstm_set_weights(tb2_lstm* m, const tb2_lstm_weights* w, void* stream) {
    TB2_REQUIRE(m && w, "null argument");
    return launch_repack(m, w, (cudaStream_t)stream);
}

int tb2_layout_create(const int64_t* off, int32_t B, tb2_layout** out) {
    TB2_REQUIRE(off && out && B >= 1, "null / empty batch_split");
    *out = nullptr;
    TB2_REQUIRE(off[0] == 0, "batch_split must start at 0");
    tb2_layout* l = new (std::nothrow) tb2_layout();
    TB2_REQUIRE(l, "out of host memory");
    l->B = B;
    l->scene_off_host.resize(B + 1);
    int n_max = 0;
    for (int b = 0; b <= B; ++b) {
        if (b > 0 && off[b] <= off[b - 1]) { delete l; set_error("invalid argument: batch_split must be strictly increasing"); return TB2_ERR_INVALID; }
        if (off[b] > 0x7fffffff / 4) { delete l; set_error("invalid argument: too many tracks"); return TB2_ERR_INVALID; }
        l->scene_off_host[b] = (int)off[b];
        if (b > 0) n_max = std::max(n_max, (int)(off[b] - off[b - 1]));
    }
    l->M = (int)off[B];
    l->n_max = n_max;
    l->scene_off = l->row_scene = nullptr;
    l->group_off[0] = l->group_off[1] = nullptr;
    auto fail = [&](int rc) { tb2_layout_destroy(l); return rc; };
    int rc;
    if ((rc = dev_alloc(l->owned, (void**)&l->scene_off, (size_t)(B + 1) * sizeof(int)))) return fail(rc);
    if ((rc = dev_alloc(l->owned, (void**)&l->row_scene, (size_t)l->M * sizeof(int)))) return fail(rc);
    std::vector<int> row_scene(l->M);
    for (int b = 0; b < B; ++b)
        for (int r = l->scene_off_host[b]; r < l->scene_off_host[b + 1]; ++r) row_scene[r] = b;
    if (cudaMemcpy(l->scene_off, l->scene_off_host.data(), (size_t)(B + 1) * sizeof(int), cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMemcpy(l->row_scene, row_scene.data(), (size_t)l->M * sizeof(int), cudaMemcpyHostToDevice) != cudaSuccess) {
        set_error(std::string("cudaMemcpy(layout): ") + cudaGetErrorString(cudaGetLastError()));
        return fail(TB2_ERR_CUDA);
    }
    // scene groups for sparse_layer1_kernel: [0] large (wide layers), [1] small (narrow layers)
    const int caps[2] = {160, 40};
    for (int g = 0; g < 2; ++g) {
        int cap = std::max(caps[g], n_max);
        std::vector<int> go;
        go.push_back(0);
        int rows = 0;
        for (int b = 0; b < B; ++b) {
            int n_b = l->scene_off_host[b + 1] - l->scene_off_host[b];
            if (rows + n_b > cap) { go.push_back(b); rows = 0; }
            rows += n_b;
        }
        go.push_back(B);
        l->group_cap[g] = cap;
        l->num_groups[g] = (int)go.size() - 1;
        if ((rc = dev_alloc(l->owned, (void**)&l->group_off[g], go.size() * sizeof(int)))) return fail(rc);
        if (cudaMemcpy(l->group_off[g], go.data(), go.size() * sizeof(int), cudaMemcpyHostToDevice) != cudaSuccess) {
            set_error(std::string("cudaMemcpy(groups): ") + cudaGetErrorString(cudaGetLastError()));
            return fail(TB2_ERR_CUDA);
        }
    }
    *out = l;
    return TB2_OK;
}

int tb2_layout_destroy(tb2_layout* l) {
    if (!l) return TB2_OK;
    for (void* p : l->owned) cudaFree(p);
    delete l;
    return TB2_OK;
}

int32_t tb2_layout_num_tracks(const tb2_layout* l) { return l ? l->M : -1; }
int32_t tb2_layout_max_scene(const tb2_layout* l) { return l ? l->n_max : -1; }
int tb2_layout_set_padding(tb2_layout* l, int32_t pad_to_batch_max) {
    TB2_REQUIRE(l, "null layout");
    l->pad_to_max = pad_to_batch_max ? 1 : 0;
    return TB2_OK;
}

size_t tb2_lstm_workspace_bytes(const tb2_lstm* m, const tb2_layout* l) {
    if (!m || !l) return 0;
    return carve_workspace(m, l, nullptr, nullptr);
}

static int check_ready(const tb2_lstm* m, const tb2_layout* l, void* ws, size_t ws_bytes) {
    TB2_REQUIRE(m && l, "null handle");
    TB2_REQUIRE(m->weights_set, "tb2_lstm_set_weights has not been called");
    TB2_REQUIRE(ws && ws_bytes >= carve_workspace(m, l, nullptr, nullptr), "workspace too small");
    TB2_REQUIRE(((uintptr_t)ws & 255) == 0, "workspace must be 256-byte aligned");
    return TB2_OK;
}

int tb2_grid_indices(const tb2_lstm* m, const tb2_layout* l, const float* obs, int32_t* cell_out,
                     uint8_t* in_range_out, void* stream) {
    TB2_REQUIRE(m && l && obs && cell_out && in_range_out, "null argument");
    TB2_REQUIRE(m->cfg.pool_type >= TB2_POOL_OCCUPANCY && m->cfg.pool_type <= TB2_POOL_SOCIAL, "model has no grid pooling");
    // The pair tables are produced straight into the caller's buffers: no workspace needed.
    Workspace ws;
    std::memset(&ws, 0, sizeof(ws));
    // pool_prepare writes winners too; give it scratch inside a temporary allocation
    size_t bytes = carve_workspace(m, l, nullptr, nullptr);
    void* tmp = nullptr;
    TB2_CHECK_CUDA(cudaMalloc(&tmp, bytes));
    carve_workspace(m, l, tmp, &ws);
    cudaStream_t st = (cudaStream_t)stream;
    // occupancy-style call: obs1 is irrelevant for the indices, pass obs for both
    tb2_lstm tmp_model = *m;
    tmp_model.owned.clear();
    tmp_model.cfg.pool_type = TB2_POOL_OCCUPANCY;   // indices do not depend on the payload
    int rc = launch_pool_prepare(&tmp_model, l, nullptr, obs, obs, 0, 1, 0, &ws, st);
    if (rc == TB2_OK) rc = launch_grid_indices_copy(l, &ws, cell_out, in_range_out, st);
    cudaError_t e = cudaStreamSynchronize(st);       // debug export: synchronous so tmp can be freed
    cudaFree(tmp);
    if (rc != TB2_OK) return rc;
    TB2_CHECK_CUDA(e);
    return TB2_OK;
}

int tb2_pool_forward(const tb2_lstm* m, const tb2_layout* l, const float* hidden, const float* obs1,
                     const float* obs2, float* pooled_out, void* workspace, size_t workspace_bytes,
                     void* stream) {
    int rc = check_ready(m, l, workspace, workspace_bytes);
    if (rc) return rc;
    TB2_REQUIRE(m->cfg.pool_type != TB2_POOL_NONE, "model has no interaction pooling");
    TB2_REQUIRE(obs1 && obs2 && pooled_out, "null argument");
    TB2_REQUIRE((m->cfg.pool_type != TB2_POOL_SOCIAL && m->cfg.pool_type != TB2_POOL_HIDDEN_MLP &&
                 m->cfg.pool_type != TB2_POOL_ATTN_MLP) || hidden,
                "this pooling needs hidden states");
    Workspace ws;
    carve_workspace(m, l, workspace, &ws);
    cudaStream_t st = (cudaStream_t)stream;
    if (m->cfg.pool_type == TB2_POOL_HIDDEN_MLP) return launch_hidden_mlp_pool(m, l, hidden, obs1, obs2, pooled_out, st);
    if (m->cfg.pool_type == TB2_POOL_NN_MLP) return launch_nn_mlp_pool(m, l, obs1, obs2, pooled_out, st);
    if (m->cfg.pool_type == TB2_POOL_NN_LSTM || m->cfg.pool_type == TB2_POOL_TRAJECTRON) {      // stateful: advances the LSTM state kept in the workspace
        if (m->cfg.pool_type == TB2_POOL_NN_LSTM) rc = launch_nn_mlp_pool(m, l, obs1, obs2, ws.pool_feat, st);
        else rc = launch_trajectron_feat(m, l, obs1, obs2, ws.scene_sum, ws.pool_feat, st);
        if (rc) return rc;
        return launch_pool_lstm_cell(m, l, ws.pool_feat, ws.pool_h, ws.pool_c, pooled_out, st);
    }
    if (m->cfg.pool_type == TB2_POOL_ATTN_MLP) return launch_attn_mlp_pool(m, l, hidden, obs1, obs2, pooled_out, st);
    if ((rc = launch_pool_prepare(m, l, hidden, obs1, obs2, 0, 0, 0, &ws, st))) return rc;
    return launch_pool_mlp(m, l, &ws, pooled_out, nullptr, nullptr, st);
}

// hs_cur: index (0/1) of the ping-pong buffer holding the bf16 split of h_in (tensor-core gates)
static int step_impl(const tb2_lstm* m, const tb2_layout* l, int phase, const float* obs1,
                     const float* obs2, const float* h_in, const float* c_in, float* h_out,
                     float* c_out, float* normal_out, float* pos_out, Workspace* ws, int hs_cur,
                     cudaStream_t st) {
    int rc;
    const bool tc = m->Wg_hi[0] != nullptr;
    const float* pooled = nullptr;
    if (m->cfg.pool_type >= TB2_POOL_HIDDEN_MLP) {
        // non-grid interaction module: one kernel per scene -> pooled fp32, split for the tensor-core gate kernel
        if (m->cfg.pool_type == TB2_POOL_NN_MLP) rc = launch_nn_mlp_pool(m, l, obs1, obs2, ws->pooled, st);
        else if (m->cfg.pool_type == TB2_POOL_NN_LSTM || m->cfg.pool_type == TB2_POOL_TRAJECTRON) {
            if (m->cfg.pool_type == TB2_POOL_NN_LSTM) rc = launch_nn_mlp_pool(m, l, obs1, obs2, ws->pool_feat, st);
            else rc = launch_trajectron_feat(m, l, obs1, obs2, ws->scene_sum, ws->pool_feat, st);
            if (!rc) rc = launch_pool_lstm_cell(m, l, ws->pool_feat, ws->pool_h, ws->pool_c, ws->pooled, st);
        }
        else if (m->cfg.pool_type == TB2_POOL_ATTN_MLP) rc = launch_attn_mlp_pool(m, l, h_in, obs1, obs2, ws->pooled, st);
        else rc = launch_hidden_mlp_pool(m, l, h_in, obs1, obs2, ws->pooled, st);
        if (rc) return rc;
        if (tc && (rc = launch_split_rows(ws->pooled, ws->pool_hi, ws->pool_lo, (size_t)l->M * m->P, st))) return rc;
        pooled = ws->pooled;
    } else
    if (m->cfg.pool_type != TB2_POOL_NONE) {
        if ((rc = launch_pool_prepare(m, l, h_in, obs1, obs2, 1, ws->write_pairs, tc ? 1 : 0, ws, st))) return rc;
        if (tc) rc = launch_pool_mlp(m, l, ws, nullptr, ws->pool_hi, ws->pool_lo, st);
        else rc = launch_pool_mlp(m, l, ws, ws->pooled, nullptr, nullptr, st);
        if (rc) return rc;
        pooled = ws->pooled;
    }
    if (tc) {
        if ((m->cfg.pool_type == TB2_POOL_NONE || m->cfg.pool_type >= TB2_POOL_HIDDEN_MLP) &&     // grid pools: pool_prepare already wrote emb
            (rc = launch_embed_split(m, l->M, obs1, obs2, ws->emb_hi, ws->emb_lo, st)))
            return rc;
        return launch_gates_tc(m, l, phase, obs1, obs2, ws->emb_hi, ws->emb_lo, ws->pool_hi, ws->pool_lo,
                               ws->hs_hi[hs_cur], ws->hs_lo[hs_cur], ws->hs_hi[hs_cur ^ 1], ws->hs_lo[hs_cur ^ 1],
                               h_in, c_in, h_out, c_out, normal_out, pos_out, st);
    }
    return launch_gates(m, l, phase, obs1, obs2, pooled, h_in, c_in, h_out, c_out, normal_out, pos_out, st);
}

int tb2_lstm_step_forward(const tb2_lstm* m, const tb2_layout* l, int32_t phase, const float* obs1,
                          const float* obs2, const float* h_in, const float* c_in, float* h_out,
                          float* c_out, float* normal_out, float* pos_out, void* workspace,
                          size_t workspace_bytes, void* stream) {
    int rc = check_ready(m, l, workspace, workspace_bytes);
    if (rc) return rc;
    TB2_REQUIRE(phase == TB2_PHASE_ENCODER || phase == TB2_PHASE_DECODER, "bad phase");
    TB2_REQUIRE(obs1 && obs2 && h_in && c_in && h_out && c_out && normal_out, "null argument");
    Workspace ws;
    carve_workspace(m, l, workspace, &ws);
    cudaStream_t st = (cudaStream_t)stream;
    if (m->Wg_hi[0] &&
        (rc = launch_split_rows(h_in, ws.hs_hi[0], ws.hs_lo[0], (size_t)l->M * m->H, st)))
        return rc;
    return step_impl(m, l, phase, obs1, obs2, h_in, c_in, h_out, c_out, normal_out, pos_out, &ws, 0, st);
}

// Steps [first_step, last_step) of the time loop.  first_step == 0 starts from the zero state
// (lstm.py:207-210); otherwise h / c hold the state after step first_step - 1 (possibly edited by
// the caller, e.g. the noise injection of the S-GAN generator between encoder and decoder,
// sgan/sgan.py:200-221,373) and positions_out holds the positions of the earlier steps.
struct HostSink {              // optional: per-step device-to-host streaming of the outputs
    float* normals_host;
    float* positions_host;
    cudaStream_t copy_stream;
    std::vector<cudaEvent_t>* events;
};

static int forward_steps_impl(const tb2_lstm* m, const tb2_layout* l, const float* observed,
                              int32_t obs_length, const float* truth, int32_t n_decode, int32_t first_step,
                              int32_t last_step, float* normals_out, float* positions_out, float* h, float* c,
                              float* states_out, void* workspace, size_t workspace_bytes, void* stream,
                              const HostSink* sink, const TrainCache* cache = nullptr) {
    int rc = check_ready(m, l, workspace, workspace_bytes);
    if (rc) return rc;
    TB2_REQUIRE(observed && normals_out && positions_out && h && c, "null argument");
    TB2_REQUIRE(obs_length >= 2 && n_decode >= 0, "need obs_length >= 2 and n_decode >= 0");
    const int S = obs_length - 1 + n_decode;
    TB2_REQUIRE(first_step >= 0 && first_step <= last_step && last_step <= S, "bad step range");
    Workspace ws;
    carve_workspace(m, l, workspace, &ws);
    cudaStream_t st = (cudaStream_t)stream;
    const size_t M = (size_t)l->M, H = (size_t)m->H;
    const size_t frame = M * 2;
    if (first_step == 0 && ws.pool_h) {       // pool.reset(...) lstm.py:213-216
        TB2_CHECK_CUDA(cudaMemsetAsync(ws.pool_h, 0, M * (size_t)m->cfg.mlp_dim_hidden * sizeof(float), st));
        TB2_CHECK_CUDA(cudaMemsetAsync(ws.pool_c, 0, M * (size_t)m->cfg.mlp_dim_hidden * sizeof(float), st));
    }
    if (first_step == 0) {
        TB2_CHECK_CUDA(cudaMemsetAsync(h, 0, M * H * sizeof(float), st));     // lstm.py:207-210
        TB2_CHECK_CUDA(cudaMemsetAsync(c, 0, M * H * sizeof(float), st));
        if (m->Wg_hi[0]) {
            TB2_CHECK_CUDA(cudaMemsetAsync(ws.hs_hi[0], 0, M * H * 2, st));
            TB2_CHECK_CUDA(cudaMemsetAsync(ws.hs_lo[0], 0, M * H * 2, st));
        }
    } else if (m->Wg_hi[0]) {      // bf16 split of the incoming state for the tensor-core gate kernel
        if ((rc = launch_split_rows(h, ws.hs_hi[first_step & 1], ws.hs_lo[first_step & 1], M * H, st))) return rc;
    }
    const float* h_prev = h;
    const float* c_prev = c;
    for (int s = first_step; s < last_step; ++s) {
        const float* o1;
        const float* o2;
        int phase;
        if ((rc = resolve_step_inputs(l, observed, obs_length, truth, positions_out, s, &ws, &o1, &o2, &phase, st)))
            return rc;
        float* h_next = states_out ? states_out + ((size_t)s * 2 + 0) * M * H : h;
        float* c_next = states_out ? states_out + ((size_t)s * 2 + 1) * M * H : c;
        Workspace wstep = ws;
        if (cache) {        // this step's winners, latent vectors, hidden1 and pooled vector stay where the backward reads them
            const size_t nm1 = (size_t)(l->n_max > 1 ? l->n_max - 1 : 1), us = (size_t)s;
            wstep.lat = cache->lat + us * M * m->C;
            wstep.win_count = cache->win_count + us * M;
            wstep.win_ent = cache->win_ent + us * M * nm1;
            wstep.pair_cell = cache->pair_cell + us * M * nm1;
            wstep.pair_flag = cache->pair_flag + us * M * nm1;
            if (cache->h1_hi) {
                wstep.act[0] = (float*)((char*)cache->h1_hi + us * M * (size_t)m->mlp_dims[1] * 2);
                wstep.act[1] = (float*)((char*)cache->h1_lo + us * M * (size_t)m->mlp_dims[1] * 2);
            }
            wstep.pool_hi = (char*)cache->pool_hi + us * M * (size_t)m->P * 2;
            wstep.pool_lo = (char*)cache->pool_lo + us * M * (size_t)m->P * 2;
            wstep.write_pairs = 1;
        }
        if ((rc = step_impl(m, l, phase, o1, o2, h_prev, c_prev, h_next, c_next,
                            normals_out + (size_t)s * M * 5, positions_out + (size_t)s * frame, &wstep, s & 1, st)))
            return rc;
        h_prev = h_next;
        c_prev = c_next;
        if (sink) {     // this step's results -> host, behind the step, beside the following steps
            cudaEvent_t ev = (*sink->events)[(size_t)s];
            TB2_CHECK_CUDA(cudaEventRecord(ev, st));
            TB2_CHECK_CUDA(cudaStreamWaitEvent(sink->copy_stream, ev, 0));
            TB2_CHECK_CUDA(cudaMemcpyAsync(sink->normals_host + (size_t)s * M * 5, normals_out + (size_t)s * M * 5,
                                           M * 5 * sizeof(float), cudaMemcpyDeviceToHost, sink->copy_stream));
            TB2_CHECK_CUDA(cudaMemcpyAsync(sink->positions_host + (size_t)s * frame, positions_out + (size_t)s * frame,
                                           frame * sizeof(float), cudaMemcpyDeviceToHost, sink->copy_stream));
        }
    }
    if (states_out && last_step > first_step) {
        TB2_CHECK_CUDA(cudaMemcpyAsync(h, h_prev, M * H * sizeof(float), cudaMemcpyDeviceToDevice, st));
        TB2_CHECK_CUDA(cudaMemcpyAsync(c, c_prev, M * H * sizeof(float), cudaMemcpyDeviceToDevice, st));
    }
    return TB2_OK;
}

int tb2_lstm_forward_steps(const tb2_lstm* m, const tb2_layout* l, const float* observed,
                           int32_t obs_length, const float* truth, int32_t n_decode, int32_t first_step,
                           int32_t last_step, float* normals_out, float* positions_out, float* h, float* c,
                           float* states_out, void* workspace, size_t workspace_bytes, void* stream) {
    return forward_steps_impl(m, l, observed, obs_length, truth, n_decode, first_step, last_step, normals_out,
                              positions_out, h, c, states_out, workspace, workspace_bytes, stream, nullptr);
}

int tb2_lstm_forward_sequence_host(tb2_lstm* m, const tb2_layout* l, const float* observed, int32_t obs_length,
                                   const float* truth, int32_t n_decode, float* normals_out, float* positions_out,
                                   float* h, float* c, void* workspace, size_t workspace_bytes,
                                   float* normals_host, float* positions_host, void* stream, void* copy_stream) {
    TB2_REQUIRE(m && normals_host && positions_host && copy_stream, "null argument");
    TB2_REQUIRE(obs_length >= 2 && n_decode >= 0, "need obs_length >= 2 and n_decode >= 0");
    const int S = obs_length - 1 + n_decode;
    while ((int)m->step_events.size() < S) {
        cudaEvent_t ev;
        TB2_CHECK_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        m->step_events.push_back(ev);
    }
    HostSink sink{normals_host, positions_host, (cudaStream_t)copy_stream, &m->step_events};
    return forward_steps_impl(m, l, observed, obs_length, truth, n_decode, 0, S, normals_out, positions_out, h, c,
                              nullptr, workspace, workspace_bytes, stream, &sink);
}

int tb2_pool_state_reset(const tb2_lstm* m, const tb2_layout* l, void* workspace, size_t workspace_bytes, void* stream) {
    int rc = check_ready(m, l, workspace, workspace_bytes);
    if (rc) return rc;
    Workspace ws;
    carve_workspace(m, l, workspace, &ws);
    if (ws.pool_h) {
        const size_t n = (size_t)l->M * (size_t)m->cfg.mlp_dim_hidden * sizeof(float);
        TB2_CHECK_CUDA(cudaMemsetAsync(ws.pool_h, 0, n, (cudaStream_t)stream));
        TB2_CHECK_CUDA(cudaMemsetAsync(ws.pool_c, 0, n, (cudaStream_t)stream));
    }
    return TB2_OK;
}

size_t tb2_lstm_train_cache_bytes(const tb2_lstm* m, const tb2_layout* l, int32_t num_steps) {
    if (!m || !l || num_steps < 1) return 0;
    return carve_train_cache(m, l, (size_t)num_steps, nullptr, nullptr);
}

int tb2_lstm_forward_sequence_train(const tb2_lstm* m, const tb2_layout* l, const float* observed, int32_t obs_length,
                                    const float* truth, int32_t n_decode, float* normals_out, float* positions_out,
                                    float* h, float* c, float* states_out, void* cache, size_t cache_bytes,
                                    void* workspace, size_t workspace_bytes, void* stream) {
    TB2_REQUIRE(m && l, "null handle");
    TB2_REQUIRE(obs_length >= 2 && n_decode >= 0, "need obs_length >= 2 and n_decode >= 0");
    TB2_REQUIRE(states_out, "a training forward keeps the per-step states");
    const int S = obs_length - 1 + n_decode;
    TrainCache tc;
    const size_t need = carve_train_cache(m, l, (size_t)S, cache, &tc);
    TB2_REQUIRE(!cache || (need > 0 && cache_bytes >= need), "training cache too small (tb2_lstm_train_cache_bytes)");
    return forward_steps_impl(m, l, observed, obs_length, truth, n_decode, 0, S, normals_out, positions_out, h, c,
                              states_out, workspace, workspace_bytes, stream, nullptr, cache ? &tc : nullptr);
}

int tb2_lstm_forward_sequence(const tb2_lstm* m, const tb2_layout* l, const float* observed,
                              int32_t obs_length, const float* truth, int32_t n_decode,
                              float* normals_out, float* positions_out, float* h, float* c,
                              float* states_out, void* workspace, size_t workspace_bytes, void* stream) {
    TB2_REQUIRE(obs_length >= 2 && n_decode >= 0, "need obs_length >= 2 and n_decode >= 0");
    return tb2_lstm_forward_steps(m, l, observed, obs_length, truth, n_decode, 0, obs_length - 1 + n_decode,
                                  normals_out, positions_out, h, c, states_out, workspace, workspace_bytes, stream);
}

}  // extern "C"
