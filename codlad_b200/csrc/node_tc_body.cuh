// Device-side body of the tcgen05 node update (see node_tc.cu for the design notes), kept apart from the kernel wrapper so that
// it can be run on an arbitrary node range of an arbitrary CTA (a fused message + node launch was measured: no gain at
// configs[1], the node phase loses its weight prefetch under the dependency wait -- DESIGN.md section 4).
#pragma once
#include "model.h"
#include "tc_common.cuh"

namespace cb2 {
namespace tc {

struct ProjTc {
    int wa_row, wc_row;          // weight blocks (rows of the packed fp16 weight tensor)
    const float *ba, *table;     // own-half bias; optional per-residue-type table added to the gathered half
    __half* out16;               // [N, 256] fp16: [own half + bias | gathered half (+ table)]
    int add_enc;                 // 0: h' = h, 1: h' = h + hVenc, 2: h' = 2 h
};

struct NodeTcParams {
    int N, L, K;
    int do_update, masked_count;
    const float *x, *xin_w_t, *xin_b;
    const float* S;
    int w3_row, win_row, wout_row;           // win/wout: 4 consecutive 128-row blocks each
    const float *b3, *bin, *bout;
    const float* mod;
    int mod_stride;
    const int *lengths, *frame_of, *nbr_idx, *cg_z;
    float *hV, *hVenc;
    int write_enc;
    ProjTc proj[2];
    int n_proj;
    int do_final;
    const float *fin_mod, *fin_w_t, *fin_b;
    float* out6;
    const float *x_t, *noise, *coef;
    float* x_next;
    int ddim;                    // the fused update is DDIM (coef = a DDIM row; noise may be null) instead of p_sample
    unsigned long long* trace;   // debug timeline of CTA 0 (nullptr = off)
    int trace_slot;              // debug: launch window slot (trace_window)
};

constexpr int NODE_EPI_THREADS = 512;
constexpr int NODE_CTA_THREADS = NODE_EPI_THREADS + 64;     // + MMA warp + TMA warp (one lane each)
constexpr int NT = 32;                       // nodes per CTA = the N extent of every MMA
constexpr int NPTH = NT / 4;                 // nodes per epilogue thread
constexpr int ACT_HALF = NT * 128;           // bytes of one K half (64 features) of an activation tile
constexpr int ACT_BYTES = 2 * ACT_HALF;      // [NT nodes][128 features] fp16, K-major SW128
constexpr int N_SLOT = 5;                    // 32 KB weight slots
constexpr int N_ACT = 6;                     // activation tiles: 0 = S / h2, 1 = h1 / h', 2..5 = FFN hidden chunks
constexpr int MAX_WT = 13;                   // weight tiles of one launch: W3, 4 Win, 4 Wout, 2 x (own, gathered)
constexpr int R1 = 0, R2 = NT, R3 = 5 * NT;  // TMEM column regions: W3 output | 4 FFN-in chunks (reused by the projections) | FFN-out
static_assert(NT == 32, "the LayerNorm transpose-reduce below is written for 8 nodes per thread");

__device__ __forceinline__ void node_epi_sync() { asm volatile("bar.sync 1, 512;" ::: "memory"); }
// the four warps (feature quarters) that share a node group: named barrier 2 + group, 128 threads
__device__ __forceinline__ void node_group_sync(int cq) { asm volatile("bar.sync %0, 128;" ::"r"(cq + 2) : "memory"); }

// byte offset of (node r, feature f) inside an activation tile
__device__ __forceinline__ uint32_t act_off(int r, int f) {
    return (uint32_t)((f >> 6) * ACT_HALF + r * 128 + ((((f >> 3) & 7) ^ (r & 7)) << 4) + (f & 7) * 2);
}
__device__ __forceinline__ void sts_h(unsigned char* p, __half h) { *reinterpret_cast<__half*>(p) = h; }

__device__ __forceinline__ int weight_rows(const NodeTcParams& p, int* rows) {
    int n = 0;
    if (p.do_update) {
        rows[n++] = p.w3_row;
        for (int c = 0; c < 4; ++c) rows[n++] = p.win_row + 128 * c;
        for (int c = 0; c < 4; ++c) rows[n++] = p.wout_row + 128 * c;
    }
    for (int j = 0; j < p.n_proj; ++j) { rows[n++] = p.proj[j].wa_row; rows[n++] = p.proj[j].wc_row; }
    return n;
}

constexpr int N_BAR = 20;                    // mbarriers of one node block (see node_block)
constexpr size_t NODE_TC_SMEM = (size_t)N_SLOT * TILE_BYTES + (size_t)N_ACT * ACT_BYTES + 2 * 4 * 4 * 16 * 4 + 4 * NT * 4 + N_BAR * 8 + 16;

// One block of NT nodes [node0, min(node0 + NT, n_end)) through the whole node update.  Called by every thread of a 576-thread CTA
// (16 epilogue warps, MMA warp 16, TMA warp 17) with `smem` = the CTA's dynamic shared memory (NODE_TC_SMEM bytes, 1024-aligned,
// free of live mbarriers) and an allocated 512-column TMEM region.  `dep_wait`: the epilogue warps execute griddepcontrol.wait
// before their first read of activations (stand-alone kernel); the fused caller has already waited.  INPAINT: the final update
// is followed by the inpainting overwrite of the rows `ir` keeps.
template <bool INPAINT>
__device__ __forceinline__ void node_block(unsigned char* smem, const uint32_t tmem_base, const CUtensorMap* wmap_p, const NodeTcParams& p,
                                           const int node0, const int n_end, const bool dep_wait, const InpaintRows& ir) {
    unsigned char* sW = smem;                                          // N_SLOT weight slots (A operands)
    unsigned char* sAct = sW + N_SLOT * TILE_BYTES;                    // N_ACT activation tiles (B operands)
    float* sRed = reinterpret_cast<float*>(sAct + N_ACT * ACT_BYTES);  // [2 uses][4 node groups][4 feature quarters][16] LayerNorm partials
    int* sB = reinterpret_cast<int*>(sRed + 2 * 4 * 4 * 16);           // per node: member
    float* sMk = reinterpret_cast<float*>(sB + NT);                    //           node mask
    float* sCnt = sMk + NT;                                            //           masked-neighbour count
    int* sZ = reinterpret_cast<int*>(sCnt + NT);                       //           residue type
    uint64_t* sBar = reinterpret_cast<uint64_t*>(sZ + NT);             // [0..4] slot full, [5..9] slot free, [10] MMAs done, [11] operands ready,
                                                                       // [12..15] FFN-in chunk c accumulated, [16..19] FFN hidden chunk c written

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    auto bar_full = [&](int s) { return smem_u32(&sBar[s]); };
    auto bar_free = [&](int s) { return smem_u32(&sBar[N_SLOT + s]); };
    const uint32_t bar_mma = smem_u32(&sBar[10]), bar_act = smem_u32(&sBar[11]);
    auto bar_chunk = [&](int c) { return smem_u32(&sBar[12 + c]); };
    auto bar_mid = [&](int c) { return smem_u32(&sBar[16 + c]); };
    if (tid == 0) {
        for (int s = 0; s < N_SLOT; ++s) { mbar_init(bar_full(s), 1); mbar_init(bar_free(s), 1); }
        mbar_init(bar_mma, 1); mbar_init(bar_act, NODE_EPI_THREADS / 32);
        for (int c = 0; c < 4; ++c) { mbar_init(bar_chunk(c), 1); mbar_init(bar_mid(c), NODE_EPI_THREADS / 32); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (tid < NT) {
        // per-node metadata (member, node mask, residue type, masked-neighbour count): static plan data, read before the
        // dependency wait
        const int n = min(node0 + tid, n_end - 1);
        const int b = n / p.L, i = n - b * p.L;
        const int f = __ldg(p.frame_of + b);
        const int len = __ldg(p.lengths + f);
        float cnt = (float)p.K;
        if (p.masked_count && len < p.L) {
            int cn = 0;
            if (i < len) {
                const int* row = p.nbr_idx + ((size_t)f * p.L + i) * p.K;
                for (int k = 0; k < p.K; ++k) cn += __ldg(row + k) < len ? 1 : 0;
            }
            cnt = (float)cn;
        }
        sB[tid] = b; sMk[tid] = i < len ? 1.f : 0.f; sCnt[tid] = cnt; sZ[tid] = __ldg(p.cg_z + (size_t)f * p.L + i);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    constexpr uint32_t IDESC = umma_idesc(128, NT, 0, 0);
    auto act_tile = [&](int t) { return sAct + t * ACT_BYTES; };

    if (warp >= 16) {
        if (warp == 17) {
            // ------------------------------------------------------------------ TMA warp (issues through an elected lane): streams the weight tiles, in the order the
            // MMAs consume them, through the slots (tile i -> slot i % N_SLOT; a slot is reloaded once its MMAs have completed)
            int rows[MAX_WT];
            const int nt = weight_rows(p, rows);
            for (int i = 0; i < nt; ++i) {
                const int slot = i % N_SLOT, use = i / N_SLOT;
                if (use > 0) mbar_wait(bar_free(slot), (uint32_t)((use - 1) & 1));
                if (elect_one()) {
                    mbar_expect_tx(bar_full(slot), (uint32_t)TILE_BYTES);
                    for (int h = 0; h < 2; ++h)
                        tma_load_2d(smem_u32(sW + slot * TILE_BYTES + h * HALF_BYTES), wmap_p, h * 64, rows[i], bar_full(slot));
                }
                __syncwarp();
            }
        } else if (warp == 16) {
            // ------------------------------------------------------------------ MMA lane: D[feature, node] = W[feature, :] . act[node, :]
            // (the whole warp runs the control flow; the instructions are issued by an elected lane)
#ifdef CB2_TRACE_CTRL                                                   // debug builds only (tools/dev/build_variant.sh -DCB2_TRACE_CTRL)
            unsigned long long* ctrace = (p.trace != nullptr && blockIdx.x == 0 && lane == 0) ? p.trace + 512 : nullptr;
            int n_ct = 0;
            auto cmark = [&](int ev) {
                if (ctrace != nullptr && n_ct < 400) {
                    unsigned long long t;
                    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
                    ctrace[1 + n_ct] = (t << 8) | (unsigned long long)ev;
                    ctrace[0] = (unsigned long long)(++n_ct);
                }
            };
#else
            auto cmark = [](int) {};
#endif
            cmark(0);
            uint32_t ph_act = 0;
            int ti = 0;
            auto gemm = [&](int act, int d_col, bool accumulate) {            // next weight tile x activation tile `act`
                const int slot = ti % N_SLOT;
                mbar_wait(bar_full(slot), (uint32_t)((ti / N_SLOT) & 1));
                tc_fence_after();
                cmark(6);
                // descriptors of k-step 0; a k-step advances only the (16-byte granular) start-address field
                const uint64_t a0 = umma_desc(smem_u32(sW + slot * TILE_BYTES), 16, 1024), b0 = umma_desc(smem_u32(act_tile(act)), 16, 1024);
                if (elect_one()) {
#pragma unroll
                    for (int k = 0; k < 8; ++k)
                        umma_f16(tmem_base + (uint32_t)d_col, a0 + (uint64_t)(((k >> 2) * HALF_BYTES + (k & 3) * 32) >> 4),
                                 b0 + (uint64_t)(((k >> 2) * ACT_HALF + (k & 3) * 32) >> 4), IDESC, (accumulate || k > 0) ? 1u : 0u);
                    umma_commit(bar_free(slot));
                }
                __syncwarp();
                cmark(7);
                ++ti;
            };
            auto commit_phase = [&]() { if (elect_one()) umma_commit(bar_mma); __syncwarp(); cmark(4); };
            auto wait_act = [&]() { mbar_wait(bar_act, ph_act); ph_act ^= 1; tc_fence_after(); cmark(2); };
            if (p.do_update) {
                wait_act(); gemm(0, R1, false); commit_phase();
                // FFN: the four 128-feature chunks flow through chunk by chunk -- chunk c's GELU epilogue starts when its own GEMM has
                // completed, and its share of the output GEMM when its hidden tile is written (no phase-wide hand-offs)
                wait_act();
                for (int c = 0; c < 4; ++c) { gemm(1, R2 + c * NT, false); if (elect_one()) umma_commit(bar_chunk(c)); __syncwarp(); }
                for (int c = 0; c < 4; ++c) { mbar_wait(bar_mid(c), 0); tc_fence_after(); cmark(8); gemm(2 + c, R3, c > 0); }
                commit_phase();
            }
            if (p.n_proj > 0) {
                wait_act();
                for (int j = 0; j < p.n_proj; ++j) {
                    gemm(0, R2 + (2 * j) * NT, false);
                    gemm(p.proj[j].add_enc ? 1 : 0, R2 + (2 * j + 1) * NT, false);
                }
                commit_phase();
            }
        }
    } else {
        // ------------------------------------------------------------------ epilogue warps: thread = (feature, 8 nodes)
        const int quarter = warp & 3, cq = warp >> 2;
        const int fl = quarter * 32 + lane;                 // feature (within a 128-feature chunk) = TMEM lane
        const int nl0 = cq * NPTH;                          // first of this thread's nodes (CTA-local)
        const uint32_t tmem_lane = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)nl0;
        uint32_t ph_mma = 0;
        int red_use = 0;
        float v[NPTH];                                      // fp32 node state: feature fl of nodes nl0 .. nl0+7
        auto publish = [&]() { fence_async_smem(); tc_fence_before(); __syncwarp(); if (lane == 0) mbar_arrive(bar_act); };    // one arrival per warp
        auto wait_mma = [&]() { mbar_wait(bar_mma, ph_mma); ph_mma ^= 1; tc_fence_after(); };
        auto live = [&](int i) { return node0 + nl0 + i < n_end; };
        auto gnode = [&](int i) { return (size_t)(node0 + nl0 + i); };
        // fp16 store of this thread's 8 values into an activation tile (row = node, column = feature fl)
        auto store_act = [&](unsigned char* tile, const float* x) {
#pragma unroll
            for (int i = 0; i < NPTH; ++i) sts_h(tile + act_off(nl0 + i, fl), __float2half_rn(x[i]));
        };
        // LayerNorm statistics over the 128 features of each of this thread's nodes (no affine, eps 1e-6).  Within a warp the
        // 16 partial sums (8 nodes x {sum, sum of squares}) are transpose-reduced with shuffles (each step halves the values a
        // lane carries); the four feature quarters then meet in shared memory.  Fixed order -> deterministic.
        auto node_stats = [&](float* mean, float* rstd) {
            float q[16];
#pragma unroll
            for (int i = 0; i < 8; ++i) { q[i] = v[i]; q[8 + i] = v[i] * v[i]; }
#pragma unroll
            for (int cnt = 8, off = 16; cnt >= 1; cnt >>= 1, off >>= 1) {
                const bool upper = (lane & off) != 0;
#pragma unroll
                for (int j = 0; j < cnt; ++j) {
                    const float send = upper ? q[j] : q[j + cnt];
                    const float keep = upper ? q[j + cnt] : q[j];
                    q[j] = keep + __shfl_xor_sync(0xffffffffu, send, off);
                }
            }
            q[0] += __shfl_xor_sync(0xffffffffu, q[0], 1);
            // lane holds value index (bit 4 -> 8, bit 3 -> 4, bit 2 -> 2, bit 1 -> 1)
            const int idx = ((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1);
            float* red = sRed + ((red_use & 1) * 16 + cq * 4) * 16;
            if ((lane & 1) == 0) red[quarter * 16 + idx] = q[0];
            node_group_sync(cq);
            float tot[16];
#pragma unroll
            for (int k4 = 0; k4 < 4; ++k4) {
                const float4 a = *reinterpret_cast<const float4*>(red + 0 * 16 + k4 * 4), b = *reinterpret_cast<const float4*>(red + 1 * 16 + k4 * 4);
                const float4 c = *reinterpret_cast<const float4*>(red + 2 * 16 + k4 * 4), d = *reinterpret_cast<const float4*>(red + 3 * 16 + k4 * 4);
                tot[k4 * 4] = (a.x + b.x) + (c.x + d.x); tot[k4 * 4 + 1] = (a.y + b.y) + (c.y + d.y);
                tot[k4 * 4 + 2] = (a.z + b.z) + (c.z + d.z); tot[k4 * 4 + 3] = (a.w + b.w) + (c.w + d.w);
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                mean[i] = tot[i] * (1.0f / 128.0f);
                rstd[i] = rsqrtf(fmaxf(tot[8 + i] * (1.0f / 128.0f) - mean[i] * mean[i], 0.f) + 1e-6f);
            }
            ++red_use;
        };
        // v <- gate * (LN(v) (1 + scale) + shift) [* node mask], modulation rows of each node's member
        const int b_first = sB[nl0], b_last = sB[nl0 + NPTH - 1];
        struct ModRow { float sh, sc, gt; };
        // (the common case -- all 8 nodes in one member -- fetches its modulation row ahead of the accumulator wait)
        auto fetch_mod = [&](const float* mod_sh) {
            const float* m = mod_sh + (size_t)b_first * p.mod_stride + fl;
            return ModRow{__ldg(m), __ldg(m + 128), __ldg(m + 256)};
        };
        auto modulate = [&](const float* mod_sh, const ModRow& mr, bool masked) {
            float mean[8], rstd[8];
            node_stats(mean, rstd);
            float A = mr.gt * (1.0f + mr.sc), Bv = mr.gt * mr.sh;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                if (b_first != b_last) {
                    const float* m = mod_sh + (size_t)sB[nl0 + i] * p.mod_stride + fl;
                    const float sh = __ldg(m), sc = __ldg(m + 128), gt = __ldg(m + 256);
                    A = gt * (1.0f + sc); Bv = gt * sh;
                }
                const float t = fmaf((v[i] - mean[i]) * rstd[i], A, Bv);
                v[i] = masked ? sMk[nl0 + i] * t : t;
            }
        };

        const int enc_mode = p.n_proj > 0 ? p.proj[p.n_proj - 1].add_enc : 0;     // only the decoder-facing projection uses h'
        // operands of the projection epilogue that do not depend on this launch's arithmetic: fetched early
        float pj_ba[2] = {0.f, 0.f}, pj_tab[NPTH], h_enc[NPTH];
        int tab_j = -1;
#pragma unroll
        for (int i = 0; i < NPTH; ++i) { pj_tab[i] = 0.f; h_enc[i] = 0.f; }
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            if (j < p.n_proj) {
                pj_ba[j] = __ldg(p.proj[j].ba + fl);
                if (p.proj[j].table != nullptr) {
                    tab_j = j;
#pragma unroll
                    for (int i = 0; i < NPTH; ++i) pj_tab[i] = __ldg(p.proj[j].table + sZ[nl0 + i] * 128 + fl);
                }
            }
        }
        if (dep_wait) pdl_wait();                       // S / h_V / x are produced by the previous kernels of the step
        if (enc_mode == 1) {
#pragma unroll
            for (int i = 0; i < NPTH; ++i) h_enc[i] = live(i) ? p.hVenc[gnode(i) * 128 + fl] : 0.f;
        }
        if (p.do_update) {
            // ---- E0: S -> fp16 operand tile (cooperative: one 8-feature chunk per thread); h_V -> v ----
            {
                const int node = tid >> 4, c16 = tid & 15;
                uint32_t o[4] = {0u, 0u, 0u, 0u};
                if (node0 + node < n_end) {
                    uint32_t r8[8];
                    ldg256_coherent(p.S + (size_t)(node0 + node) * 128 + c16 * 8, r8);
#pragma unroll
                    for (int e = 0; e < 4; ++e) o[e] = f2_to_h2(__uint_as_float(r8[2 * e]), __uint_as_float(r8[2 * e + 1]));
                }
                *reinterpret_cast<uint4*>(act_tile(0) + (c16 >> 3) * ACT_HALF + node * 128 + (((c16 & 7) ^ (node & 7)) << 4)) = make_uint4(o[0], o[1], o[2], o[3]);
            }
#pragma unroll
            for (int i = 0; i < NPTH; ++i) v[i] = live(i) ? p.hV[gnode(i) * 128 + fl] : 0.f;
            publish();
            // ---- EA: h1 = gate1 * (LN(h_V + (acc + cnt b3)/30) (1 + scale1) + shift1) ----
            {
                const float b3 = __ldg(p.b3 + fl);
                const ModRow mr = fetch_mod(p.mod);
                wait_mma();
                float acc[8];
                tmem_ld8(tmem_lane + R1, acc);
#pragma unroll
                for (int i = 0; i < NPTH; ++i) v[i] += (acc[i] + sCnt[nl0 + i] * b3) * (1.0f / 30.0f);
                modulate(p.mod, mr, false);
                store_act(act_tile(1), v);
            }
            publish();
            // ---- EG: FFN hidden = 2 GELU(Win h1 + b_in) (the 1/2 lives in the packed W_out), four 128-feature chunks ----
            {
                float bi[4];
#pragma unroll
                for (int c = 0; c < 4; ++c) bi[c] = __ldg(p.bin + c * 128 + fl);
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    mbar_wait(bar_chunk(c), 0);
                    tc_fence_after();
                    float acc[8];
                    tmem_ld8(tmem_lane + (uint32_t)(R2 + c * NT), acc);
                    unsigned char* dst = act_tile(2 + c);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const __half2 g = gelu2_h2(as_h2(pack_sat(acc[2 * j] + bi[c], acc[2 * j + 1] + bi[c])));
                        sts_h(dst + act_off(nl0 + 2 * j, fl), __low2half(g));
                        sts_h(dst + act_off(nl0 + 2 * j + 1, fl), __high2half(g));
                    }
                    fence_async_smem(); tc_fence_before(); __syncwarp();
                    if (lane == 0) mbar_arrive(bar_mid(c));
                }
            }
            // ---- EB: h2 = mask * gate2 * (LN(h1 + acc + b_out) (1 + scale2) + shift2) ----
            {
                const float bo = __ldg(p.bout + fl);
                const ModRow mr = fetch_mod(p.mod + 384);
                wait_mma();
                float acc[8];
                tmem_ld8(tmem_lane + R3, acc);
#pragma unroll
                for (int i = 0; i < NPTH; ++i) v[i] += acc[i] + bo;
                modulate(p.mod + 384, mr, true);
            }
        } else {
            // ---- node init: h = x_in(x) ----
            const float w0 = __ldg(p.xin_w_t + fl), w1 = __ldg(p.xin_w_t + 128 + fl), w2 = __ldg(p.xin_w_t + 256 + fl), bb = __ldg(p.xin_b + fl);
#pragma unroll
            for (int i = 0; i < NPTH; ++i) {
                v[i] = 0.f;
                if (live(i)) {
                    const float* x = p.x + gnode(i) * 3;
                    v[i] = fmaf(x[2], w2, fmaf(x[1], w1, fmaf(x[0], w0, bb)));
                }
            }
        }
        // ---- stage the projection operands, then write h_V (and the decoder's frozen encoder state): the global stores come after the
        //      hand-off so that the projection GEMMs do not wait for them (the hand-off's fence drains the thread's memory operations) ----
        auto write_state = [&]() {
#pragma unroll
            for (int i = 0; i < NPTH; ++i) {
                if (live(i)) {
                    p.hV[gnode(i) * 128 + fl] = v[i];
                    if (p.write_enc) p.hVenc[gnode(i) * 128 + fl] = v[i];
                }
            }
        };
        if (p.n_proj == 0) write_state();
        if (p.n_proj > 0) {
            store_act(act_tile(0), v);
            if (enc_mode) {
                float hp[NPTH];
#pragma unroll
                for (int i = 0; i < NPTH; ++i)
                    hp[i] = enc_mode == 1 ? (live(i) ? v[i] + h_enc[i] : 0.f) : 2.0f * v[i];
                store_act(act_tile(1), hp);
            }
            publish();
            write_state();
            // ---- EP: own halves (+ bias) and gathered halves (+ residue-type table) -> P16 (fp16) ----
            wait_mma();
            for (int j = 0; j < p.n_proj; ++j) {
                const ProjTc pj = p.proj[j];
#pragma unroll
                for (int which = 0; which < 2; ++which) {
                    float acc[8];
                    tmem_ld8(tmem_lane + (uint32_t)(R2 + (2 * j + which) * NT), acc);
#pragma unroll
                    for (int i = 0; i < NPTH; ++i) {
                        if (live(i)) {
                            const float add = which == 0 ? (j == 0 ? pj_ba[0] : pj_ba[1]) : (j == tab_j ? pj_tab[i] : 0.f);
                            pj.out16[gnode(i) * 256 + which * 128 + fl] = __float2half_rn(acc[i] + add);
                        }
                    }
                }
            }
        }
        if (p.do_final) {
            // ---- FinalLayer (adaLN modulate + Linear 128 -> 6) fused with the DDPM p_sample (or DDIM) update and the inpainting
            //      overwrite of kept rows.  The fp32 rows are parked in shared memory (the FFN hidden tiles are dead); each warp
            //      then owns two nodes, lanes across features ----
            float* sH = reinterpret_cast<float*>(act_tile(2));
#pragma unroll
            for (int i = 0; i < NPTH; ++i) sH[(nl0 + i) * 128 + fl] = v[i];
            node_epi_sync();
#pragma unroll 1
            for (int t = 0; t < 2; ++t) {
                const int nl = warp * 2 + t, n = node0 + nl;
                if (n >= n_end) break;
                float h[4], sum = 0.f, sq = 0.f;
#pragma unroll
                for (int k = 0; k < 4; ++k) { h[k] = sH[nl * 128 + lane + 32 * k]; sum += h[k]; sq = fmaf(h[k], h[k], sq); }
#pragma unroll
                for (int off = 16; off >= 1; off >>= 1) { sum += __shfl_xor_sync(0xffffffffu, sum, off); sq += __shfl_xor_sync(0xffffffffu, sq, off); }
                const float mean = sum * (1.0f / 128.0f);
                const float rstd = rsqrtf(fmaxf(sq * (1.0f / 128.0f) - mean * mean, 0.f) + 1e-6f);
                const float* fm = p.fin_mod + (size_t)sB[nl] * p.mod_stride;      // [shift | scale]
                float o[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int c = lane + 32 * k;
                    const float tt = fmaf((h[k] - mean) * rstd, 1.0f + __ldg(fm + 128 + c), __ldg(fm + c));
                    const float2* w = reinterpret_cast<const float2*>(p.fin_w_t + c * 6);
                    const float2 w0 = __ldg(w), w1 = __ldg(w + 1), w2 = __ldg(w + 2);
                    o[0] = fmaf(tt, w0.x, o[0]); o[1] = fmaf(tt, w0.y, o[1]); o[2] = fmaf(tt, w1.x, o[2]);
                    o[3] = fmaf(tt, w1.y, o[3]); o[4] = fmaf(tt, w2.x, o[4]); o[5] = fmaf(tt, w2.y, o[5]);
                }
#pragma unroll
                for (int u = 0; u < 6; ++u) {
#pragma unroll
                    for (int off = 16; off >= 1; off >>= 1) o[u] += __shfl_xor_sync(0xffffffffu, o[u], off);
                    o[u] += __ldg(p.fin_b + u);
                }
                if (lane < 6) {
                    float mine = o[0];
#pragma unroll
                    for (int u = 1; u < 6; ++u) mine = lane == u ? o[u] : mine;
                    p.out6[(size_t)n * 6 + lane] = mine;
                }
                if (p.x_next != nullptr && lane < 3 && p.ddim) {
                    const float eps = lane == 0 ? o[0] : (lane == 1 ? o[1] : o[2]);
                    const float* nz = p.noise != nullptr ? p.noise + (size_t)n * 3 + lane : nullptr;
                    p.x_next[(size_t)n * 3 + lane] = ddim_update(p.x_t[(size_t)n * 3 + lane], eps, p.coef, nz);
                } else if (p.x_next != nullptr && lane < 3) {
                    const float eps = lane == 0 ? o[0] : (lane == 1 ? o[1] : o[2]);
                    const float vv = lane == 0 ? o[3] : (lane == 1 ? o[4] : o[5]);
                    const float x = p.x_t[(size_t)n * 3 + lane];
                    const float frac = (vv + 1.0f) / 2.0f;
                    const float logvar = frac * p.coef[1] + (1.0f - frac) * p.coef[0];
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
    tc_fence_before();
    __syncthreads();
    if (tid == 0)                                     // the shared memory (and these barrier words) may be re-used by the caller
        for (int i = 0; i < N_BAR; ++i) asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_u32(&sBar[i])) : "memory");
    __syncthreads();
}


}  // namespace tc

// host side (node_tc.cu): parameters of the node update `phase` (0..2 encoder layers, 3..5 decoder layers) for a fused launch
void node_tc_update_params(Plan& p, int phase, const float* mod_base, int mod_stride_b, const float* x_t, const float* noise,
                           float* x_next, const float* coef_row, tc::NodeTcParams& np);

}  // namespace cb2
