// Internal (not part of the C-ABI): packed device-side weights and the per-geometry plan.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <string>
#include <unordered_map>
#include <vector>

#include "common.cuh"

namespace cb2 {

// fp32 weights are stored TRANSPOSED ([in][out]) so that a thread owning output column c reads
// consecutive addresses across the warp.  fp16 copies keep nn.Linear's [out][in] layout, which is
// exactly the K-major B operand a tcgen05.mma wants (one 128x128 block per matrix, 128 rows apart).
struct EncLayerW {
    const float *W1a_t, *W1b_t, *W1c_t, *b1, *W2_t, *b2, *W3_t, *b3;
    const float *W11a_t, *W11b_t, *W11c_t, *b11, *W12_t, *b12, *W13_t, *b13;
    const float *Win_t, *bin, *Wout_t, *bout;
    const __half *W1b_h, *W2_h, *W11b_h, *W12_h, *W13_h;
    const __half *W1a_h, *W1c_h, *W11a_h, *W11c_h, *W3_h, *Win_h /* 4 blocks */, *Wout_h /* 4 blocks */;
    const __half *b2_16, *b12_16, *b13_16;      // fp16 copies of the biases the tensor-core epilogues add
};

struct DecLayerW {
    // W1 = [W1a | W1b | W1c | W1d] over inputs [h_V_i | 2 h_E | 2 h_S_j | h_V_j + h_Venc_j]
    const float *W1a_t, *W1b2_t /* 2*W1b^T */, *W1d_t, *b1, *TS /* [30][128] = 2 * W_s @ W1c^T */;
    const float *W2_t, *b2, *W3_t, *b3, *Win_t, *bin, *Wout_t, *bout;
    const __half *W1b2_h, *W2_h;
    const __half *W1a_h, *W1d_h, *W3_h, *Win_h /* 4 blocks */, *Wout_h /* 4 blocks */;
    const __half* b2_16;
};

struct DenoiserModel {
    int k_neighbors = 64;
    int vocab = 30;
    // timestep embedder + every adaLN projection concatenated (enc0..2, dec0..2, final)
    const float *freqs /* [128] sinusoid frequencies */, *te_w0_t, *te_b0, *te_w2_t, *te_b2, *ada_w_t, *ada_b;
    const float *xin_w_t /* [3][128] */, *xin_b;
    // featuriser: PT[65][128] = (W_pos[:,d] + b_pos) @ W_edge[:, :16]^T ; wedge_t rows = 144 rbf + 7 ori + 1 pad
    const float *pos_table, *wedge_t, *ln_w, *ln_b, *we_t, *we_b;
    EncLayerW enc[3];
    DecLayerW dec[3];
    const float *fin_w_t /* [128][6] */, *fin_b;
    float* dev_f32 = nullptr;
    __half* dev_f16 = nullptr;
    __half* dev_vec16 = nullptr;
    int n_f16_blocks = 0;
};

enum Precision { PREC_F32 = 0, PREC_F16 = 1 };
enum UpdateKind { UPDATE_DDPM = 0, UPDATE_DDIM = 1 };

// One plan = one geometry: F frames of padded length L, NB members (member b uses frame
// frame_of[b]), K neighbours.  Owns every intermediate buffer of the denoiser.
struct Plan {
    const DenoiserModel* model = nullptr;
    int F = 0, NB = 0, L = 0, K = 0, precision = PREC_F32;
    int T_rows = 0;                 // rows currently held in `mod`
    // per-frame
    float* X = nullptr;             // [F, L, 3]
    int* lengths = nullptr;         // [F]
    int* cg_z = nullptr;            // [F, L]
    int* frame_of = nullptr;        // [NB]
    int* nbr_idx = nullptr;         // [F, L, K]
    float* nbr_dist = nullptr;      // [F, L, K]
    void* hE0 = nullptr;            // [F, L, K, 128] fp32 | fp16
    float* E_dbg = nullptr;         // optional [F, L, K, 128] (norm_edges output) for parity tests
    // per-member
    void* hE = nullptr;             // [NB, L, K, 128] fp32 | fp16
    float* hV = nullptr;            // [NB*L, 128]
    float* hVenc = nullptr;         // [NB*L, 128]
    float* P = nullptr;             // [2][NB*L, 256] per-node halves of the edge MLPs' first layer: [own | gathered]
    __half* P16[2] = {nullptr, nullptr};    // fp16 tier: [NB*L, 256] = [own half + bias | gathered half] of the two first-layer splits
    __half* mod16 = nullptr;                // fp16 tier: [mod_capacity, 3, 256] edge-stream adaLN: gate (1 + scale) | gate * shift
    int num_sms = 148;
    bool all_full = false;                    // every frame has L residues (no padding, hence no neighbour mask)
    unsigned long long* tc_trace = nullptr;   // debug: stage timestamps of one tensor-core edge pipeline ("tc_trace" buffer)
    float* silu_c = nullptr;        // [mod_capacity, 128] scratch of the timestep embedder
    float* S = nullptr;             // [NB*L, 128]  aggregated messages
    float* out6 = nullptr;          // [NB*L, 6]
    float* mod = nullptr;           // [T_rows, 6016] adaLN table
    int mod_capacity = 0;
    int* mod_row = nullptr;         // [NB] row of `mod` used by each member (forward() path)
    float* tvals = nullptr;         // [mod_capacity] timestep values staging
    // sampling-loop state
    float* coef = nullptr;          // [T, 8] per-step update scalars (fp32): p_sample or DDIM rows, as update_kind says
    int coef_steps = 0;
    int update_kind = 0;            // UPDATE_DDPM | UPDATE_DDIM, uniform over the schedule (the fused update selects on it)
    bool coef_noisy = true;         // the update reads its noise (DDPM always; DDIM when some sigma != 0)
    // latent inpainting (cb2_plan_set_inpaint): plan-owned copies, allocated on first use; their addresses never change
    bool inpaint = false;           // kept rows are overwritten after every update (uniform per launch, like update_kind)
    int inpaint_steps = 0;          // T of the uploaded inpainting table (must equal coef_steps to sample)
    unsigned char* inp_keep = nullptr;   // [NB*L] 1 = keep this row's latent
    float* inp_x0 = nullptr;        // [NB*L, 3] normalised latent to keep
    float* inp_eps = nullptr;       // [NB*L, 3] the fixed draw of the kept rows (saved from the initial noise)
    float* inp_coef = nullptr;      // [mod_capacity + 1, 2] rows s: {sqrt(acp_prev[s]), sqrt(1 - acp_prev[s])}, row T: head
    std::vector<float> inp_coef_host;    // what inp_coef holds (re-uploaded only when it changes)
    cudaGraphExec_t graph = nullptr;
    const void* graph_key[4] = {nullptr, nullptr, nullptr, nullptr};
    int graph_steps = 0;
    bool graph_all_full = false;    // the captured launches chose the masked / unmasked message kernels from all_full
    bool graph_inpaint = false;     // the captured loop applies the inpainting overwrite
    std::vector<void*> allocs;
    void* tmaps = nullptr;          // host-side CUtensorMap storage of the tcgen05 edge kernels
    void* node_tc = nullptr;        // ... and of the tcgen05 node kernels
    long long launches = 0;         // kernels launched through this plan (bench: gpu_launches)
};

// ---- kernel launchers (each returns a cudaError as int) ----
int launch_knn(const float* X, const int* lengths, int F, int L, int K, float* D, int* idx, cudaStream_t s);
int launch_edge_features(const DenoiserModel& m, const float* X, const int* lengths, const int* idx, const float* D,
                         int F, int L, int K, float* E_dbg, void* hE0, int precision, cudaStream_t s);
int launch_edge_raw_features(const float* X, const int* idx, const float* D, int F, int L, int K, float* raw_out, cudaStream_t s);
int launch_timestep_mod(const DenoiserModel& m, const float* tvals, int n, float* scratch_silu_c, float* mod, __half* mod16, cudaStream_t s);
int launch_p_sample(const float* x, const float* out6, const float* noise, const float* coef_rows, const int* step_of_row,
                    int rows_per_b, int n_rows, int C, float* x_next, cudaStream_t s);
int launch_ddim_sample(const float* x, const float* out6, const float* noise, const float* coef_rows, const int* step_of_row,
                       int rows_per_b, int n_rows, int C, float* x_next, cudaStream_t s);
// in place on the loop's initial latent x: eps = x and x = q_head[0] x0 + q_head[1] eps on the kept rows
int launch_inpaint_init(const unsigned char* keep, const float* x0, const float* q_head, int n_rows, float* x, float* eps, cudaStream_t s);
float* plan_P(Plan& p, int which);

// The fused update's kept-row overwrite reads the plan's inpainting buffers with `inpaint_row` = the step's
// {sqrt(acp_prev), sqrt(1 - acp_prev)}; nullptr = no inpainting.
struct NodeArgs;   // node.cu
int launch_node_init(Plan& p, const float* x, const float* mod_base, int mod_stride_b, cudaStream_t s);
int launch_node_update(Plan& p, int phase /*0..2 enc, 3..5 dec*/, const float* mod_base, int mod_stride_b,
                       const float* x_t, const float* noise, float* x_next, const float* coef_row, const float* inpaint_row,
                       cudaStream_t s);
int launch_edge_f32(Plan& p, int mode, int layer, const float* mod_base, int mod_stride_b, cudaStream_t s);
int launch_edge_tc(Plan& p, int mode, int layer, const float* mod_base, int mod_stride_b, cudaStream_t s);
int edge_tc_prepare(Plan& p);
int node_tc_prepare(Plan& p);
void node_tc_release(Plan& p);
int launch_node_init_tc(Plan& p, const float* x, cudaStream_t s);
int launch_node_update_tc(Plan& p, int phase, const float* mod_base, int mod_stride_b, const float* x_t, const float* noise,
                          float* x_next, const float* coef_row, const float* inpaint_row, cudaStream_t s);
void edge_tc_release(Plan& p);
const unsigned int* edge_tc_trap_log();      // debug (CB2_TRAP_DEBUG): record of a timed-out barrier wait, or nullptr

enum EdgeMode { EDGE_ENC_NODE = 0, EDGE_ENC_EDGE = 1, EDGE_DEC = 2 };

}  // namespace cb2
