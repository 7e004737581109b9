// Per-node (per-residue) kernels of the denoiser.
//
//  * timestep_mod:  TimestepEmbedder (reference models/latent_model.py:37-75) + every adaLN
//    projection `Linear(SiLU(c))` of the 3 encoder layers, 3 decoder layers and the final layer
//    (protein_mpnn_utils.py:228-232,288-292; latent_model.py:27-30) -> one [n, 6016] table.  It depends
//    only on t, so the sampler computes its 100 rows once instead of 7 small GEMMs per step.
//  * node_update:  everything EncLayer_diffusion / DecLayer_diffusion do per node after the
//    neighbour aggregation (protein_mpnn_utils.py:247-259 and :307-317): dh = (W3 . sum_k m_k + cnt b3)/30
//    (W3 is linear, so it is applied once per node after the masked sum instead of once per edge),
//    LayerNorm + adaLN modulate/gate, position-wise FFN 128->512->128, second LayerNorm/adaLN, node
//    mask; then the per-node halves of the NEXT edge MLP's first layer
//    (W1 [h_V_i | h_E | h_V_j] = W1a h_V_i + W1b h_E + W1c h_V_j: the a/c products are per node),
//    and for the last decoder layer FinalLayer (latent_model.py:21-35) fused with the DDPM
//    p_sample update (diffusion_and_flow/gaussian_diffusion.py:303-318,345-351,440-446) or, on a
//    DDIM schedule, IDDPM's ddim_sample update (ddim_update, common.cuh).  With latent inpainting on,
//    the kept rows are then overwritten with the forward marginal of their latent (inpaint_level).
//  * inpaint_init:  before the first step, saves the kept rows' initial noise as their fixed draw and
//    puts them at the head level of the schedule; for partial-noise refinement (all_rows) every row
//    starts at the level of its own x0 there.
//
// fp32 SIMT: 16 rows per CTA, 128 threads, thread = output column (see tile_gemm.cuh).
#include "model.h"
#include "tile_gemm.cuh"

namespace cb2 {

namespace {

// ------------------------------------------------------------------ timestep / adaLN table
__global__ void __launch_bounds__(128) timestep_cond_kernel(const float* __restrict__ tvals, const float* __restrict__ freqs,
                                                            const float* __restrict__ w0_t, const float* __restrict__ b0,
                                                            const float* __restrict__ w2_t, const float* __restrict__ b2,
                                                            float* __restrict__ silu_c /* [n][128] */) {
    __shared__ float emb[256];
    __shared__ float hid[128];
    const int n = blockIdx.x, c = threadIdx.x;
    const float t = tvals[n];
    const float arg = t * freqs[c];
    emb[c] = cosf(arg);
    emb[128 + c] = sinf(arg);
    __syncthreads();
    float a = b0[c];
    for (int k = 0; k < 256; ++k) a = fmaf(emb[k], w0_t[k * 128 + c], a);
    hid[c] = silu(a);
    __syncthreads();
    float o = b2[c];
    for (int k = 0; k < 128; ++k) o = fmaf(hid[k], w2_t[k * 128 + c], o);
    silu_c[n * 128 + c] = silu(o);       // every consumer applies SiLU first
}

__global__ void __launch_bounds__(128) adaln_table_kernel(const float* __restrict__ silu_c, const float* __restrict__ ada_w_t,
                                                          const float* __restrict__ ada_b, float* __restrict__ mod) {
    __shared__ float s[128];
    const int n = blockIdx.x, col = blockIdx.y * 128 + threadIdx.x;
    s[threadIdx.x] = silu_c[n * 128 + threadIdx.x];
    __syncthreads();
    float o = ada_b[col];
    for (int k = 0; k < 128; ++k) o = fmaf(s[k], ada_w_t[(size_t)k * CB2_MOD_TOTAL + col], o);
    mod[(size_t)n * CB2_MOD_TOTAL + col] = o;
}

// edge-stream adaLN of the three encoder layers in the form the tensor-core epilogue consumes:
// mod16[n][l] = [gate3 (1 + scale3) | gate3 * shift3] as fp16 (protein_mpnn_utils.py:270)
__global__ void __launch_bounds__(128) mod16_kernel(const float* __restrict__ mod, __half* __restrict__ mod16) {
    const int n = blockIdx.x, l = blockIdx.y, c = threadIdx.x;
    const float* m = mod + (size_t)n * CB2_MOD_TOTAL + CB2_MOD_ENC_OFF(l);
    const float gate = m[1024 + c];
    __half* o = mod16 + ((size_t)n * 3 + l) * 256;
    o[c] = __float2half_rn(gate * (1.0f + m[896 + c]));
    o[128 + c] = __float2half_rn(gate * m[768 + c]);
}

// ------------------------------------------------------------------ node update
struct Proj {                // P[n] = [Wa h + ba | Wc h' (+ table[z])],  h' = h (+ h_enc)
    const float *Wa_t, *ba, *Wc_t, *table;
    float* out;              // [N, 256]
    int add_enc;             // 0: h' = h, 1: h' = h + hVenc[n], 2: h' = 2 h (this kernel is producing hVenc)
};

struct NodeParams {
    int N, L, K;
    int do_update;           // 0: node_init (h = x_in(x)), 1: message update
    int masked_count;        // 1: cnt = sum_k mask_i mask_j (encoder), 0: cnt = K (decoder)
    const float* x;          // [N,3] (node_init)
    const float *xin_w_t, *xin_b;
    const float* S;          // [N,128]
    const float *W3_t, *b3, *Win_t, *bin, *Wout_t, *bout;
    const float* mod;        // table base (already offset to this layer's block); row b at mod + b*mod_stride
    int mod_stride;
    const int *lengths, *frame_of, *nbr_idx, *cg_z;   // per-frame graph (nbr_idx [F,L,K])
    float *hV, *hVenc;       // hVenc written when write_enc
    int write_enc;
    Proj proj[2];
    int n_proj;
    // final layer + p_sample (do_final)
    int do_final;
    const float *fin_mod, *fin_w_t, *fin_b;   // fin_mod row b at fin_mod + b*mod_stride
    float* out6;             // [N,6]
    const float *x_t, *noise, *coef;          // p_sample inputs (nullable -> forward() only); DDIM: noise may be null
    float* x_next;
    int ddim;                // the fused update is DDIM (coef = a DDIM row) instead of p_sample
};

constexpr int NR = 16;

__device__ __forceinline__ void rows_ln(float* sB, float* sStat, int tid) {
    // LayerNorm statistics (eps 1e-6, no affine) of the NR rows in sB[NR][128]; 4 warps.
    const int warp = tid >> 5, lane = tid & 31;
    for (int r = warp; r < NR; r += 4) {
        float4 v4 = *reinterpret_cast<float4*>(sB + r * 128 + lane * 4);
        float v[4] = {v4.x, v4.y, v4.z, v4.w};
        float mean, rstd;
        warp_ln_stats(v, 1e-6f, mean, rstd);
        if (lane == 0) { sStat[r * 2] = mean; sStat[r * 2 + 1] = rstd; }
    }
}

// INPAINT: the final update is followed by the inpainting overwrite of the rows `ir` keeps (the last node launch of a step with
// latent inpainting on); otherwise `ir` is unused.
template <bool INPAINT>
__global__ void __launch_bounds__(128) node_update_kernel(NodeParams p, InpaintRows ir) {
    extern __shared__ __align__(16) float smem[];
    float* sA = smem;                  // [16][128] current h
    float* sMid = sA + NR * 128;       // [16][512] S rows, then FFN hidden
    float* sB = sMid + NR * 512;       // [16][128] scratch
    __shared__ float sStat[NR * 2];
    __shared__ float sCnt[NR];
    __shared__ int sMem[NR];           // member index b per row
    __shared__ float sMask[NR];

    const int tid = threadIdx.x, c = tid;
    const int n0 = blockIdx.x * NR;

    if (tid < NR) {
        const int n = n0 + tid;
        int b = 0;
        float mk = 0.f, cnt = (float)p.K;
        if (n < p.N) {
            b = n / p.L;
            const int i = n - b * p.L;
            const int f = p.frame_of[b];
            const int len = p.lengths[f];
            mk = i < len ? 1.f : 0.f;
            if (p.masked_count && len < p.L) {
                int cn = 0;
                if (i < len) {
                    const int* row = p.nbr_idx + ((size_t)f * p.L + i) * p.K;
                    for (int k = 0; k < p.K; ++k) cn += row[k] < len ? 1 : 0;
                }
                cnt = (float)cn;
            }
        }
        sMem[tid] = b; sMask[tid] = mk; sCnt[tid] = cnt;
    }

    float h[NR];
    if (p.do_update) {
        for (int t = tid; t < NR * 32; t += 128) {     // S rows -> sMid (row stride 128), float4
            const int r = t >> 5, q = t & 31;
            const int n = n0 + r;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (n < p.N) v = *reinterpret_cast<const float4*>(p.S + (size_t)n * 128 + q * 4);
            *reinterpret_cast<float4*>(sMid + r * 128 + q * 4) = v;
        }
        __syncthreads();
        float acc[NR];
        zero_acc(acc);
        tile_gemm<NR, 128, 128>(sMid, p.W3_t + c, 128, acc);
        const float b3 = p.b3[c];
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            const int n = n0 + r;
            const float hv = n < p.N ? p.hV[(size_t)n * 128 + c] : 0.f;
            sB[r * 128 + c] = hv + (acc[r] + sCnt[r] * b3) / 30.0f;
        }
        __syncthreads();
        rows_ln(sB, sStat, tid);
        __syncthreads();
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            const float* m = p.mod + (size_t)sMem[r] * p.mod_stride;
            const float hn = (sB[r * 128 + c] - sStat[r * 2]) * sStat[r * 2 + 1];
            h[r] = m[256 + c] * (hn * (1.0f + m[128 + c]) + m[c]);       // gate1 * modulate(norm1, shift1, scale1)
            sA[r * 128 + c] = h[r];
        }
        __syncthreads();
        // FFN 128 -> 512 (GELU) -> 128
        for (int pass = 0; pass < 4; ++pass) {
            zero_acc(acc);
            tile_gemm<NR, 128, 128>(sA, p.Win_t + pass * 128 + c, 512, acc);
            const float bi = p.bin[pass * 128 + c];
#pragma unroll
            for (int r = 0; r < NR; ++r) sMid[r * 512 + pass * 128 + c] = gelu_erf(acc[r] + bi);
        }
        __syncthreads();
        zero_acc(acc);
        tile_gemm<NR, 512, 512>(sMid, p.Wout_t + c, 128, acc);
        const float bo = p.bout[c];
#pragma unroll
        for (int r = 0; r < NR; ++r) sB[r * 128 + c] = h[r] + (acc[r] + bo);
        __syncthreads();
        rows_ln(sB, sStat, tid);
        __syncthreads();
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            const float* m = p.mod + (size_t)sMem[r] * p.mod_stride;
            const float hn = (sB[r * 128 + c] - sStat[r * 2]) * sStat[r * 2 + 1];
            h[r] = sMask[r] * (m[640 + c] * (hn * (1.0f + m[512 + c]) + m[384 + c]));   // mask * gate2 * modulate(norm2, shift2, scale2)
        }
        __syncthreads();   // everyone is done reading sA / sB
    } else {
        __syncthreads();
        const float w0 = p.xin_w_t[c], w1 = p.xin_w_t[128 + c], w2 = p.xin_w_t[256 + c], bb = p.xin_b[c];
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            const int n = n0 + r;
            float v = 0.f;
            if (n < p.N) {
                const float* xr = p.x + (size_t)n * 3;
                v = fmaf(xr[2], w2, fmaf(xr[1], w1, fmaf(xr[0], w0, bb)));
            }
            h[r] = v;
        }
    }
#pragma unroll
    for (int r = 0; r < NR; ++r) {
        const int n = n0 + r;
        sA[r * 128 + c] = h[r];
        if (n < p.N) {
            p.hV[(size_t)n * 128 + c] = h[r];
            if (p.write_enc) p.hVenc[(size_t)n * 128 + c] = h[r];
        }
    }
    __syncthreads();

    // per-node halves of the next edge MLPs
    for (int j = 0; j < p.n_proj; ++j) {
        const Proj pj = p.proj[j];
        float acc[NR];
        zero_acc(acc);
        tile_gemm<NR, 128, 128>(sA, pj.Wa_t + c, 128, acc);
        const float ba = pj.ba[c];
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            const int n = n0 + r;
            if (n < p.N) pj.out[(size_t)n * 256 + c] = acc[r] + ba;
        }
        const float* src = sA;
        if (pj.add_enc) {
            __syncthreads();
#pragma unroll
            for (int r = 0; r < NR; ++r) {
                const int n = n0 + r;
                float e = h[r];
                if (pj.add_enc == 1) e = n < p.N ? p.hVenc[(size_t)n * 128 + c] : 0.f;
                sB[r * 128 + c] = h[r] + e;
            }
            __syncthreads();
            src = sB;
        }
        zero_acc(acc);
        tile_gemm<NR, 128, 128>(src, pj.Wc_t + c, 128, acc);
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            const int n = n0 + r;
            if (n < p.N) {
                float v = acc[r];
                if (pj.table != nullptr) {
                    const int b = sMem[r];
                    const int z = p.cg_z[(size_t)p.frame_of[b] * p.L + (n - b * p.L)];
                    v += pj.table[z * 128 + c];
                }
                pj.out[(size_t)n * 256 + 128 + c] = v;
            }
        }
    }

    if (p.do_final) {
        __syncthreads();
        const int warp = tid >> 5, lane = tid & 31;
        for (int r = warp; r < NR; r += 4) {
            const int n = n0 + r;
            if (n >= p.N) continue;
            float4 v4 = *reinterpret_cast<float4*>(sA + r * 128 + lane * 4);
            float v[4] = {v4.x, v4.y, v4.z, v4.w};
            float mean, rstd;
            warp_ln_stats(v, 1e-6f, mean, rstd);
            const float* m = p.fin_mod + (size_t)sMem[r] * p.mod_stride;     // [shift | scale]
            float o[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int col = lane * 4 + q;
                const float fm = (v[q] - mean) * rstd * (1.0f + m[128 + col]) + m[col];
#pragma unroll
                for (int u = 0; u < 6; ++u) o[u] = fmaf(fm, p.fin_w_t[col * 6 + u], o[u]);
            }
#pragma unroll
            for (int u = 0; u < 6; ++u) o[u] = warp_sum(o[u]) + p.fin_b[u];
            if (lane < 6) p.out6[(size_t)n * 6 + lane] = o[lane];
            if (p.x_next != nullptr && lane < 3 && p.ddim) {
                const float* nz = p.noise != nullptr ? p.noise + (size_t)n * 3 + lane : nullptr;
                p.x_next[(size_t)n * 3 + lane] = ddim_update(p.x_t[(size_t)n * 3 + lane], o[lane], p.coef, nz);
            } else if (p.x_next != nullptr && lane < 3) {
                // learned-range variance + epsilon parameterisation (gaussian_diffusion.py:303-318,345-351,440-446)
                const float eps = o[lane], vv = o[3 + lane];
                const float min_log = p.coef[0], max_log = p.coef[1];
                const float x = p.x_t[(size_t)n * 3 + lane];
                const float frac = (vv + 1.0f) / 2.0f;
                const float logvar = frac * max_log + (1.0f - frac) * min_log;
                const float x0 = p.coef[2] * x - p.coef[3] * eps;
                const float mean_ = p.coef[4] * x0 + p.coef[5] * x;
                p.x_next[(size_t)n * 3 + lane] = mean_ + p.coef[6] * expf(0.5f * logvar) * p.noise[(size_t)n * 3 + lane];
            }
            if constexpr (INPAINT) {
                if (lane < 3 && ir.keep[n]) {
                    const size_t k = (size_t)n * 3 + lane;
                    p.x_next[k] = inpaint_level(ir.level, ir.x0[k], ir.eps[k]);
                }
            }
        }
    }
}

__global__ void p_sample_kernel(const float* __restrict__ x, const float* __restrict__ out6, const float* __restrict__ noise,
                                const float* __restrict__ coef_rows, const int* __restrict__ step_of_row, int rows_per_b,
                                int n_rows, int C, float* __restrict__ x_next) {
    // Stand-alone DDPM update for callers that run their own denoiser (generic p_sample path).
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_rows * C) return;
    const int row = t / C, d = t - row * C;
    const float* cf = coef_rows + (size_t)step_of_row[row / rows_per_b] * 8;
    const float eps = out6[(size_t)row * 2 * C + d], vv = out6[(size_t)row * 2 * C + C + d];
    const float xv = x[t];
    const float frac = (vv + 1.0f) / 2.0f;
    const float logvar = frac * cf[1] + (1.0f - frac) * cf[0];
    const float x0 = cf[2] * xv - cf[3] * eps;
    const float mean_ = cf[4] * x0 + cf[5] * xv;
    x_next[t] = mean_ + cf[6] * expf(0.5f * logvar) * noise[t];
}

__global__ void ddim_sample_kernel(const float* __restrict__ x, const float* __restrict__ out6, const float* __restrict__ noise,
                                   const float* __restrict__ coef_rows, const int* __restrict__ step_of_row, int rows_per_b,
                                   int n_rows, int C, float* __restrict__ x_next) {
    // Stand-alone DDIM update for callers that run their own denoiser (generic ddim_sample path); noise may be null.
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_rows * C) return;
    const int row = t / C, d = t - row * C;
    const float* cf = coef_rows + (size_t)step_of_row[row / rows_per_b] * 8;
    x_next[t] = ddim_update(x[t], out6[(size_t)row * 2 * C + d], cf, noise != nullptr ? noise + t : nullptr);
}

// all_rows is uniform per launch; eps is saved for kept rows only, as the overwrite reads it for them alone.
__global__ void inpaint_init_kernel(const unsigned char* __restrict__ keep, const float* __restrict__ x0, const float* __restrict__ q_head,
                                    int n_rows, int all_rows, float* __restrict__ x, float* __restrict__ eps) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_rows * 3) return;
    const bool kept = keep[t / 3] != 0;
    if (!kept && !all_rows) return;
    const float e = x[t];
    if (kept) eps[t] = e;
    x[t] = inpaint_level(q_head, x0[t], e);
}

}  // namespace

int launch_timestep_mod(const DenoiserModel& m, const float* tvals, int n, float* scratch_silu_c, float* mod, __half* mod16, cudaStream_t s) {
    timestep_cond_kernel<<<n, 128, 0, s>>>(tvals, m.freqs, m.te_w0_t, m.te_b0, m.te_w2_t, m.te_b2, scratch_silu_c);
    CB2_LAUNCH_CHECK();
    adaln_table_kernel<<<dim3(n, CB2_MOD_TOTAL / 128), 128, 0, s>>>(scratch_silu_c, m.ada_w_t, m.ada_b, mod);
    CB2_LAUNCH_CHECK();
    if (mod16 != nullptr) {
        mod16_kernel<<<dim3(n, 3), 128, 0, s>>>(mod, mod16);
        CB2_LAUNCH_CHECK();
    }
    return 0;
}

int launch_p_sample(const float* x, const float* out6, const float* noise, const float* coef_rows, const int* step_of_row,
                    int rows_per_b, int n_rows, int C, float* x_next, cudaStream_t s) {
    const int total = n_rows * C;
    p_sample_kernel<<<(total + 255) / 256, 256, 0, s>>>(x, out6, noise, coef_rows, step_of_row, rows_per_b, n_rows, C, x_next);
    CB2_LAUNCH_CHECK();
    return 0;
}

int launch_ddim_sample(const float* x, const float* out6, const float* noise, const float* coef_rows, const int* step_of_row,
                       int rows_per_b, int n_rows, int C, float* x_next, cudaStream_t s) {
    const int total = n_rows * C;
    ddim_sample_kernel<<<(total + 255) / 256, 256, 0, s>>>(x, out6, noise, coef_rows, step_of_row, rows_per_b, n_rows, C, x_next);
    CB2_LAUNCH_CHECK();
    return 0;
}

int launch_inpaint_init(const unsigned char* keep, const float* x0, const float* q_head, int n_rows, bool all_rows, float* x, float* eps,
                        cudaStream_t s) {
    const int total = n_rows * 3;
    inpaint_init_kernel<<<(total + 255) / 256, 256, 0, s>>>(keep, x0, q_head, n_rows, all_rows ? 1 : 0, x, eps);
    CB2_LAUNCH_CHECK();
    return 0;
}

static int node_launch(Plan& p, NodeParams& np, cudaStream_t s, const InpaintRows* ir = nullptr) {
    const size_t smem = (size_t)(NR * 128 + NR * 512 + NR * 128) * 4;
    static bool attr = false;
    if (!attr) {
        CB2_CUDA(cudaFuncSetAttribute(node_update_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CB2_CUDA(cudaFuncSetAttribute(node_update_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr = true;
    }
    if (ir != nullptr) node_update_kernel<true><<<(np.N + NR - 1) / NR, 128, smem, s>>>(np, *ir);
    else node_update_kernel<false><<<(np.N + NR - 1) / NR, 128, smem, s>>>(np, InpaintRows{});
    CB2_LAUNCH_CHECK();
    p.launches++;
    return 0;
}

static void base_params(Plan& p, NodeParams& np) {
    np = NodeParams{};
    np.N = p.NB * p.L; np.L = p.L; np.K = p.K;
    np.lengths = p.lengths; np.frame_of = p.frame_of; np.nbr_idx = p.nbr_idx; np.cg_z = p.cg_z;
    np.hV = p.hV; np.hVenc = p.hVenc; np.S = p.S;
}

float* plan_P(Plan& p, int which);   // capi.cu: P buffer 0 (for node-message kernels) / 1 (for enc_edge)

int launch_node_init(Plan& p, const float* x, const float* mod_base, int mod_stride_b, cudaStream_t s) {
    (void)mod_base; (void)mod_stride_b;
    const DenoiserModel& m = *p.model;
    NodeParams np;
    base_params(p, np);
    np.do_update = 0;
    np.x = x; np.xin_w_t = m.xin_w_t; np.xin_b = m.xin_b;
    np.n_proj = 1;
    np.proj[0] = Proj{m.enc[0].W1a_t, m.enc[0].b1, m.enc[0].W1c_t, nullptr, plan_P(p, 0), 0};
    return node_launch(p, np, s);
}

int launch_node_update(Plan& p, int phase, const float* mod_base, int mod_stride_b, const float* x_t, const float* noise,
                       float* x_next, const float* coef_row, const float* inpaint_row, cudaStream_t s) {
    const DenoiserModel& m = *p.model;
    NodeParams np;
    base_params(p, np);
    np.do_update = 1;
    np.mod_stride = mod_stride_b;
    if (phase < 3) {
        const EncLayerW& e = m.enc[phase];
        np.masked_count = 1;
        np.W3_t = e.W3_t; np.b3 = e.b3; np.Win_t = e.Win_t; np.bin = e.bin; np.Wout_t = e.Wout_t; np.bout = e.bout;
        np.mod = mod_base + CB2_MOD_ENC_OFF(phase);
        np.n_proj = 2;
        np.proj[0] = Proj{e.W11a_t, e.b11, e.W11c_t, nullptr, plan_P(p, 1), 0};          // this layer's edge update
        if (phase < 2) {
            const EncLayerW& nx = m.enc[phase + 1];
            np.proj[1] = Proj{nx.W1a_t, nx.b1, nx.W1c_t, nullptr, plan_P(p, 0), 0};        // next layer's node message
        } else {
            const DecLayerW& d = m.dec[0];
            np.write_enc = 1;
            np.proj[1] = Proj{d.W1a_t, d.b1, d.W1d_t, d.TS, plan_P(p, 0), 2};              // h_V + h_Venc = 2 h_V here
        }
    } else {
        const int l = phase - 3;
        const DecLayerW& d = m.dec[l];
        np.masked_count = 0;
        np.W3_t = d.W3_t; np.b3 = d.b3; np.Win_t = d.Win_t; np.bin = d.bin; np.Wout_t = d.Wout_t; np.bout = d.bout;
        np.mod = mod_base + CB2_MOD_DEC_OFF(l);
        if (l < 2) {
            const DecLayerW& nx = m.dec[l + 1];
            np.n_proj = 1;
            np.proj[0] = Proj{nx.W1a_t, nx.b1, nx.W1d_t, nx.TS, plan_P(p, 0), 1};
        } else {
            np.n_proj = 0;
            np.do_final = 1;
            np.fin_mod = mod_base + CB2_MOD_FIN_OFF;
            np.fin_w_t = m.fin_w_t; np.fin_b = m.fin_b;
            np.out6 = p.out6;
            np.x_t = x_t; np.noise = noise; np.x_next = x_next; np.coef = coef_row;
            np.ddim = p.update_kind == UPDATE_DDIM;
            if (inpaint_row != nullptr) {
                const InpaintRows ir{p.inp_keep, p.inp_x0, p.inp_eps, inpaint_row};
                return node_launch(p, np, s, &ir);
            }
        }
    }
    return node_launch(p, np, s);
}

}  // namespace cb2
