// tcgen05 tier of the per-node kernels (same maths as node.cu; reference models/protein_mpnn_utils.py:247-259,
// :307-317, models/latent_model.py:21-35,214, diffusion_and_flow/gaussian_diffusion.py:303-318,345-351,440-446).
//
// The node kernels are latency chains (W3 -> LN -> FFN -> LN -> projections) over few rows (B L nodes), so they are laid
// out TRANSPOSED: every MMA computes D[feature, node] = W[feature, :] . act[node, :] with the weight block as the
// 128-row A operand and a narrow tile of NT = 32 nodes as the B operand (N = 32).  A TMEM lane is then a feature and a
// column a node, the per-warp epilogue work scales with the nodes of the CTA, and the grid is N / 32 CTAs instead of
// N / 128.  Warps 0-15 are the epilogue warps: thread (feature quarter, node group) owns one feature lane and 8 node
// columns; LayerNorm statistics (over features = across lanes) use a shuffle transpose-reduce plus one shared-memory
// exchange between the four feature quarters.  Warp 16 (one lane) issues the MMAs, warp 17 (one lane) streams the fp16
// weight blocks through five 32 KB slots with TMA in consumption order; the first five blocks are requested before the
// dependency wait, so they land while the previous kernel drains.
//
//   P1  acc = W3 . S^T                          EA  h1 = gate1 * mod(LN(h_V + (acc + cnt b3)/30))
//   P2  4 x acc_c = Win[c] . h1^T               EG  mid_c = 2 GELU(acc_c + b_in)
//   P3  acc = sum_c (Wout[:, c]/2) . mid_c^T    EB  h2 = mask * gate2 * mod(LN(h1 + acc + b_out))   (+ FinalLayer, p_sample / DDIM,
//                                                                                                       inpainting overwrite)
//   P4  own / gathered halves of the next edge MLPs' first layer        EP  -> P16 (fp16 [own + bias | gathered (+ table)])
//
// State h_V stays fp32 in HBM; only MMA operands are fp16 (fp32 accumulation in TMEM).
#include "node_tc_body.cuh"

namespace cb2 {

using namespace tc;

namespace {

template <bool INPAINT>
__device__ __forceinline__ void node_tc_run(const CUtensorMap& wmap, const NodeTcParams& p, const InpaintRows& ir) {
    extern __shared__ __align__(1024) unsigned char smem[];
    __shared__ uint32_t s_tmem;
    const int tid = threadIdx.x, warp = tid >> 5;
    if (tid == 0) trace_window(p.trace, p.trace_slot, false);
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    pdl_launch_dependents();               // the next kernel of the step may start its prologue on the SMs this grid leaves idle
    if (warp == 16) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(&s_tmem)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = s_tmem;
    node_block<INPAINT>(smem, tmem_base, &wmap, p, blockIdx.x * NT, p.N, true, ir);
    if (tid == 0) trace_window(p.trace, p.trace_slot, true);
    if (warp == 16) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
}

__global__ void __launch_bounds__(NODE_CTA_THREADS, 1) node_tc_kernel(const __grid_constant__ CUtensorMap wmap, const NodeTcParams p) {
    node_tc_run<false>(wmap, p, InpaintRows{});
}

// the last node launch of a step with latent inpainting on
__global__ void __launch_bounds__(NODE_CTA_THREADS, 1) node_tc_inpaint_kernel(const __grid_constant__ CUtensorMap wmap, const NodeTcParams p,
                                                                             const __grid_constant__ InpaintRows ir) {
    node_tc_run<true>(wmap, p, ir);
}


struct NodeTcState { CUtensorMap wmap; };

int node_tc_launch(Plan& p, NodeTcParams& np, cudaStream_t s, const InpaintRows* ir = nullptr) {
    const NodeTcState& st = *reinterpret_cast<const NodeTcState*>(p.node_tc);
    const dim3 grid((np.N + NT - 1) / NT), block(NODE_CTA_THREADS);
    if (ir != nullptr) CB2_CUDA(launch_pdl(node_tc_inpaint_kernel, grid, block, NODE_TC_SMEM, s, st.wmap, np, *ir));
    else CB2_CUDA(launch_pdl(node_tc_kernel, grid, block, NODE_TC_SMEM, s, st.wmap, np));
    CB2_LAUNCH_CHECK();
    p.launches++;
    return 0;
}

void base_params(Plan& p, NodeTcParams& np) {
    np = NodeTcParams{};
    np.N = p.NB * p.L; np.L = p.L; np.K = p.K;
    np.lengths = p.lengths; np.frame_of = p.frame_of; np.nbr_idx = p.nbr_idx; np.cg_z = p.cg_z;
    np.hV = p.hV; np.hVenc = p.hVenc; np.S = p.S;
    np.trace = p.tc_trace; np.trace_slot = p.launches & 2047;
}

}  // namespace

int node_tc_prepare(Plan& p) {
    EncodeTiledFn fn = nullptr;
    if (get_encode_fn(&fn)) return 1;
    NodeTcState* st = new NodeTcState();
    p.node_tc = st;
    if (encode_rows_map(fn, &st->wmap, p.model->dev_f16, (size_t)p.model->n_f16_blocks * 128, 128)) return 1;
    CB2_CUDA(cudaFuncSetAttribute(node_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)NODE_TC_SMEM));
    CB2_CUDA(cudaFuncSetAttribute(node_tc_inpaint_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)NODE_TC_SMEM));
    return 0;
}

void node_tc_release(Plan& p) {
    delete reinterpret_cast<NodeTcState*>(p.node_tc);
    p.node_tc = nullptr;
}

int launch_node_init_tc(Plan& p, const float* x, cudaStream_t s) {
    const DenoiserModel& m = *p.model;
    auto row_of = [&](const __half* w) { return (int)((w - m.dev_f16) / 128); };
    NodeTcParams np;
    base_params(p, np);
    np.do_update = 0;
    np.x = x; np.xin_w_t = m.xin_w_t; np.xin_b = m.xin_b;
    np.n_proj = 1;
    np.proj[0] = ProjTc{row_of(m.enc[0].W1a_h), row_of(m.enc[0].W1c_h), m.enc[0].b1, nullptr, p.P16[0], 0};
    return node_tc_launch(p, np, s);
}

void node_tc_update_params(Plan& p, int phase, const float* mod_base, int mod_stride_b, const float* x_t, const float* noise,
                           float* x_next, const float* coef_row, tc::NodeTcParams& np) {
    const DenoiserModel& m = *p.model;
    auto row_of = [&](const __half* w) { return (int)((w - m.dev_f16) / 128); };
    base_params(p, np);
    np.do_update = 1;
    np.mod_stride = mod_stride_b;
    if (phase < 3) {
        const EncLayerW& e = m.enc[phase];
        np.masked_count = 1;
        np.w3_row = row_of(e.W3_h); np.win_row = row_of(e.Win_h); np.wout_row = row_of(e.Wout_h);
        np.b3 = e.b3; np.bin = e.bin; np.bout = e.bout;
        np.mod = mod_base + CB2_MOD_ENC_OFF(phase);
        np.n_proj = 2;
        np.proj[0] = ProjTc{row_of(e.W11a_h), row_of(e.W11c_h), e.b11, nullptr, p.P16[1], 0};
        if (phase < 2) {
            const EncLayerW& nx = m.enc[phase + 1];
            np.proj[1] = ProjTc{row_of(nx.W1a_h), row_of(nx.W1c_h), nx.b1, nullptr, p.P16[0], 0};
        } else {
            const DecLayerW& d = m.dec[0];
            np.write_enc = 1;
            np.proj[1] = ProjTc{row_of(d.W1a_h), row_of(d.W1d_h), d.b1, d.TS, p.P16[0], 2};
        }
    } else {
        const int l = phase - 3;
        const DecLayerW& d = m.dec[l];
        np.masked_count = 0;
        np.w3_row = row_of(d.W3_h); np.win_row = row_of(d.Win_h); np.wout_row = row_of(d.Wout_h);
        np.b3 = d.b3; np.bin = d.bin; np.bout = d.bout;
        np.mod = mod_base + CB2_MOD_DEC_OFF(l);
        if (l < 2) {
            const DecLayerW& nx = m.dec[l + 1];
            np.n_proj = 1;
            np.proj[0] = ProjTc{row_of(nx.W1a_h), row_of(nx.W1d_h), nx.b1, nx.TS, p.P16[0], 1};
        } else {
            np.n_proj = 0;
            np.do_final = 1;
            np.fin_mod = mod_base + CB2_MOD_FIN_OFF;
            np.fin_w_t = m.fin_w_t; np.fin_b = m.fin_b;
            np.out6 = p.out6;
            np.x_t = x_t; np.noise = noise; np.x_next = x_next; np.coef = coef_row;
            np.ddim = p.update_kind == UPDATE_DDIM;
        }
    }
}

int launch_node_update_tc(Plan& p, int phase, const float* mod_base, int mod_stride_b, const float* x_t, const float* noise,
                          float* x_next, const float* coef_row, const float* inpaint_row, cudaStream_t s) {
    NodeTcParams np;
    node_tc_update_params(p, phase, mod_base, mod_stride_b, x_t, noise, x_next, coef_row, np);
    if (inpaint_row != nullptr && np.do_final) {
        const InpaintRows ir{p.inp_keep, p.inp_x0, p.inp_eps, inpaint_row};
        return node_tc_launch(p, np, s, &ir);
    }
    return node_tc_launch(p, np, s);
}

}  // namespace cb2
