// Shared host/device declarations of libtrajnet_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include <atomic>
#include <list>
#include <string>
#include <vector>

#include "trajnet_b200.h"

namespace tb2 {

void set_error(const std::string& msg);
extern std::atomic<uint64_t> g_launch_count;

#define TB2_CHECK_CUDA(expr)                                                              \
    do {                                                                                  \
        cudaError_t _e = (expr);                                                          \
        if (_e != cudaSuccess) {                                                          \
            ::tb2::set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));         \
            return TB2_ERR_CUDA;                                                          \
        }                                                                                 \
    } while (0)

#define TB2_REQUIRE(cond, msg)                                                            \
    do {                                                                                  \
        if (!(cond)) {                                                                    \
            ::tb2::set_error(std::string("invalid argument: ") + (msg));                  \
            return TB2_ERR_INVALID;                                                       \
        }                                                                                 \
    } while (0)

#define TB2_LAUNCH_CHECK()                                                                \
    do {                                                                                  \
        ::tb2::g_launch_count.fetch_add(1, std::memory_order_relaxed);                    \
        TB2_CHECK_CUDA(cudaGetLastError());                                               \
    } while (0)

// Programmatic dependent launch: the kernels of a recurrence step are launched with
// cudaLaunchAttributeProgrammaticStreamSerialization, so the next kernel's CTAs become resident
// and run their prologue (barrier init, TMEM allocation, tensor-map prefetch) while the previous
// kernel drains.  Every thread executes grid_dep_wait() before its first access to global memory
// (it returns once the preceding grid has completed and its writes are visible), then
// grid_dep_launch() lets the following kernel start its own prologue.  TB2_PDL=0 switches the
// launch attribute off (the two instructions are then no-ops).
#ifdef __CUDACC__
__device__ __forceinline__ void grid_dep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void grid_dep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

inline bool pdl_enabled() {
    static const bool on = [] { const char* e = getenv("TB2_PDL"); return !(e && e[0] == '0'); }();
    return on;
}

// TB2_DISABLE_TC=1: fp32 FFMA kernels instead of the tensor-core ones, for parity runs of the tcgen05 path.  Read
// when a model is created (its weights are laid out for one path or the other).
inline bool tc_disabled() {
    const char* e = getenv("TB2_DISABLE_TC");
    return e && e[0] == '1';
}

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                              Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
#endif

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) applies to the CURRENT device: the size a launch
// site has configured is remembered per device, so a second model on another GPU of the same
// process configures its own copy of the kernel.
struct DynSmemConfig {
    size_t bytes[64];      // zero-initialised (function-local static)
    template <typename K>
    cudaError_t ensure(K kernel, size_t smem, size_t preset = 0) {
        int dev = 0;
        cudaError_t e = cudaGetDevice(&dev);
        if (e != cudaSuccess) return e;
        size_t& have = bytes[dev & 63];
        if (have < preset) have = preset;          // e.g. the 48 KB every kernel may use without opting in
        if (smem <= have) return cudaSuccess;
        e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) have = smem;
        return e;
    }
};

// Optional per-kernel timing (tb2_profile_begin / tb2_profile_end): CUDA events recorded on the
// launching stream around every kernel of the library.  Off by default (zero overhead).
struct KernelTimer {
    KernelTimer(const char* name, cudaStream_t st);
    ~KernelTimer();
    int slot;
    cudaStream_t st;
};

constexpr int kMaxMlpLayers = 3;
constexpr int kGateBK = 16;        // K-chunk of the gate GEMM; weight rows are padded to it

}  // namespace tb2

// Opaque handle bodies ---------------------------------------------------------------------
struct tb2_lstm {
    tb2_lstm_config cfg;
    int H, E, C, cells, n_mlp;
    int P;                 // pooled width fed to the LSTM input (0 if none / pool_to_input == 0)
    int pool_out;          // width of the pool output (grid width when n_mlp == 0)
    int mlp_dims[tb2::kMaxMlpLayers + 1];  // [grid_dim, d1, ..]
    int K_gate, K_gate_pad;
    bool weights_set;
    // device buffers (owned)
    float* We;             // [E-2, 2]
    float* be;             // [E-2]
    float* WgT[2];         // [K_gate_pad, 4H]  rows: emb | pooled | h
    float* bg[2];          // [4H] = b_ih + b_hh
    float* Wn;             // [5, H]
    float* bn;             // [5]
    float* WencT;          // [H, C]
    float* benc;           // [C]
    float* Wt1;            // [cells, C, d1]  cell-major slabs of pool.embedding.0.weight
    float* base1;          // [d1] = b1 + constant * rowsum(W1)
    void* Wt1_hi;          // social, C == 16: bf16 [cells, d1, 16] (hi, lo) slabs for sparse_layer1_mma
    void* Wt1_lo;
    void* Wt1_nat_hi;      // social, C == 16: bf16 [cells, d1, 16] natural k order (TMA source of sparse_layer1_tc)
    void* Wt1_nat_lo;
    void* Wt1_sw_hi;       // social, C == 16: the same slabs as a SWIZZLE_32B shared-memory image (bulk-copy source of
    void* Wt1_sw_lo;       // sparse_layer1_pair)
    float* WT[tb2::kMaxMlpLayers];   // layers >= 2: [K, N] transposed
    float* bl[tb2::kMaxMlpLayers];   // biases of layers >= 2
    void* W_hi[tb2::kMaxMlpLayers];  // layer 1 (the second Linear): bf16 [N, K] (hi, lo) split for the tcgen05 path (null: FFMA path)
    void* W_lo[tb2::kMaxMlpLayers];
    std::vector<cudaEvent_t> step_events;     // tb2_lstm_forward_sequence_host: one event per recurrence step
    // HiddenStateMLPPooling (TB2_POOL_HIDDEN_MLP)
    float *mp_Ws, *mp_bs, *mp_Wv, *mp_bv, *mp_WhT, *mp_bh, *mp_WoT, *mp_bo;
    // AttentionMLPPooling (TB2_POOL_ATTN_MLP): in-projection . wq / wk / wv combined and transposed [E in][E out], biases,
    // out-projection transposed
    float *at_AqT, *at_AkT, *at_AvT, *at_bqkv, *at_WoT, *at_bo;
    // NearestNeighborLSTM (TB2_POOL_NN_LSTM): interaction-encoder LSTMCell, weights transposed [in][4 Hp], fused bias
    float *pl_WihT, *pl_WhhT, *pl_b;
    void* Wg_hi[2];        // gate weights [4H (rank, gate, unit), K_gate] bf16 split (null: FFMA gates)
    void* Wg_lo[2];
    std::vector<void*> owned;
};

struct tb2_layout {
    int B, M, n_max;
    int pad_to_max = 1;    // 1: scenes padded to the batch maximum like the reference's batched call (padded
                           // slots clobber grid cell 0); 0: every scene as if it were called on its own
    std::vector<int> scene_off_host;
    int* scene_off;        // [B+1] device
    int* row_scene;        // [M]   device
    // scene groups for the sparse grid-MLP kernel: consecutive scenes, <= cap rows each
    int group_cap[2];
    int num_groups[2];
    int* group_off[2];     // [G+1] scene indices, device
    // round tables of sparse_layer1_pair (one per (layer width, unit count)), built on first use
    struct PairPlan { int OUT, units_max, units, rounds_per_unit; void* dev; };
    std::list<PairPlan> pair_plans;           // (list: entries are handed out by pointer)
    std::vector<void*> owned;
};

namespace tb2 {

struct Workspace {
    float* obs1;           // [M,2] resolved step inputs
    float* obs2;           // [M,2]
    float* lat;            // [M,C]
    int* win_count;        // [M]
    uint32_t* win_ent;     // [M, nm1]  cell << 16 | scene-local j
    float* win_val;        // [M, nm1, 2]
    int* pair_cell;        // [M, nm1]
    uint8_t* pair_flag;    // [M, nm1]
    uint8_t* cell_row;     // [M, cells] social, cells <= 256: per-row cell map (scene-local winner index, 0xFF none,
                           // 0xFE NaN-padded slot) read by sparse_layer1_pair; null otherwise
    float* act[2];         // ping-pong MLP activations [M, max width]
    float* act2;           // third scratch (three_layer with a tensor-core second layer)
    float* pooled;         // [M, pool_out]
    void* emb_hi;          // [M, 64] bf16 split operands of the tensor-core gate kernel
    void* emb_lo;
    void* pool_hi;         // [M, P]
    void* pool_lo;
    void* hs_hi[2];        // [M, 128] ping-pong split of the hidden state
    void* hs_lo[2];
    size_t bytes;
    int write_pairs;       // pool_prepare also exports the pair tables (training forward with a cache)
    float* pool_feat;      // [M, out_dim] neighbour features of NearestNeighborLSTM (null otherwise)
    float* pool_h;         // [M, Hp] state of its interaction-encoder LSTM, kept over the steps of a sequence
    float* pool_c;
    float* scene_sum;      // [B, 4] TrajectronPooling: sum of (pos, vel) over the visible tracks of every scene
};

// Per-step forward quantities a training forward keeps for the social backward (tb2_lstm_forward_sequence_train):
// the backward then skips its own pool_prepare / grid-embedding recomputation.  Layouts match the backward's
// own per-step arrays ([S][M][...]).
struct TrainCache {
    float* lat;            // [S][M][C]
    int* win_count;        // [S][M]
    uint32_t* win_ent;     // [S][M][nm1]
    int* pair_cell;        // [S][M][nm1]
    uint8_t* pair_flag;    // [S][M * nm1]
    void* h1_hi;           // [S][M][d1] bf16 (two_layer) or null
    void* h1_lo;
    void* pool_hi;         // [S][M][P] bf16
    void* pool_lo;
};
// 0 when the configuration keeps no cache (anything but social pooling on the tensor-core path)
size_t carve_train_cache(const tb2_lstm* m, const tb2_layout* l, size_t S, void* base, TrainCache* out);
size_t carve_workspace(const tb2_lstm* m, const tb2_layout* l, void* base, Workspace* ws);

// kernels.cu launchers (all asynchronous on `st`)
int launch_resolve_obs(const tb2_layout* l, const float* base, const float* pred, float* out,
                       cudaStream_t st);
int launch_pool_prepare(const tb2_lstm* m, const tb2_layout* l, const float* hidden,
                        const float* obs1, const float* obs2, int skip_masked, int write_pairs,
                        int write_emb, Workspace* ws, cudaStream_t st);
// pooled_out fp32 and/or (pool_hi, pool_lo) bf16 split (either may be null, not both)
int launch_pool_mlp(const tb2_lstm* m, const tb2_layout* l, Workspace* ws, float* pooled_out,
                    void* pool_hi, void* pool_lo, cudaStream_t st);
int launch_gates(const tb2_lstm* m, const tb2_layout* l, int phase, const float* obs1,
                 const float* obs2, const float* pooled, const float* h_in, const float* c_in,
                 float* h_out, float* c_out, float* normal_out, float* pos_out, cudaStream_t st);
int launch_repack(tb2_lstm* m, const tb2_lstm_weights* w, cudaStream_t st);
int launch_repack_layer1_mma(const float* W1, void* hi, void* lo, int OUT, int cells, cudaStream_t st);
int launch_repack_layer1_nat(const float* W1, void* hi, void* lo, int OUT, int cells, cudaStream_t st);
bool sparse_tc_supported(const tb2_lstm* m, const tb2_layout* l, int gsel);
int launch_sparse_tc(const tb2_lstm* m, const tb2_layout* l, int gsel, Workspace* ws, float* out, void* out_hi,
                     void* out_lo, cudaStream_t st);
// round-2 kernel of the same layer (pedestrians on the M side, CTA pair with cta_group::2)
bool sparse_pair_supported(const tb2_lstm* m, const tb2_layout* l);
int launch_sparse_pair(const tb2_lstm* m, const tb2_layout* l, Workspace* ws, float* out, void* out_hi, void* out_lo,
                       cudaStream_t st);
int launch_repack_layer1_sw(const float* W1, void* hi, void* lo, int OUT, int cells, cudaStream_t st);
int launch_hidden_mlp_pool(const tb2_lstm* m, const tb2_layout* l, const float* hidden, const float* obs1,
                           const float* obs2, float* out, cudaStream_t st);
int launch_attn_mlp_pool(const tb2_lstm* m, const tb2_layout* l, const float* hidden, const float* obs1, const float* obs2,
                         float* out, cudaStream_t st);
int launch_trajectron_feat(const tb2_lstm* m, const tb2_layout* l, const float* obs1, const float* obs2, float* scene_sum,
                           float* feat, cudaStream_t st);
int launch_pool_lstm_cell(const tb2_lstm* m, const tb2_layout* l, const float* feat, float* h, float* c, float* out,
                          cudaStream_t st);
int launch_nn_mlp_pool(const tb2_lstm* m, const tb2_layout* l, const float* obs1, const float* obs2, float* out,
                       cudaStream_t st);
bool dense_tc_supported(int K, int N);
int launch_dense_tc(const void* a_hi, const void* a_lo, const void* w_hi, const void* w_lo, const float* bias,
                    float* Y, void* Y_hi, void* Y_lo, int M, int K, int N, int relu, cudaStream_t st);
bool gates_tc_supported(const tb2_lstm* m);
int launch_repack_gates_tc(const float* w_ih, const float* w_hh, void* hi, void* lo, int in_dim, int H, cudaStream_t st);
int launch_embed_split(const tb2_lstm* m, int M, const float* obs1, const float* obs2, void* hi, void* lo, cudaStream_t st);
int launch_split_rows(const float* src, void* hi, void* lo, size_t n, cudaStream_t st);
int launch_gates_tc(const tb2_lstm* m, const tb2_layout* l, int phase, const float* obs1, const float* obs2,
                    const void* emb_hi, const void* emb_lo, const void* pool_hi, const void* pool_lo,
                    const void* hs_in_hi, const void* hs_in_lo, void* hs_out_hi, void* hs_out_lo,
                    const float* h_in, const float* c_in, float* h_out, float* c_out, float* normal_out,
                    float* pos_out, cudaStream_t st);
int launch_split_bf16(const float* src, void* hi, void* lo, size_t n, cudaStream_t st);
int launch_grid_indices_copy(const tb2_layout* l, const Workspace* ws, int32_t* cell_out,
                             uint8_t* flag_out, cudaStream_t st);

}  // namespace tb2
