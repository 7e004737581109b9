// C ABI (include/codlad_b200.h): model packing, plan management and the step-loop driver.
#include <math.h>
#include <stdarg.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <string>
#include <vector>

#include "../../include/codlad_b200.h"
#include "decode.h"
#include "model.h"
#include "repair.h"

namespace cb2 {

static thread_local char g_err[1024] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

float* plan_P(Plan& p, int which) { return p.P + (size_t)which * p.NB * p.L * 256; }

namespace {

struct TensorTable {
    std::map<std::string, const cb2_tensor*> by_name;
    TensorTable(const cb2_tensor* t, int n) {
        for (int i = 0; i < n; ++i) by_name[t[i].name] = &t[i];
    }
    const float* get(const std::string& name, long long numel) const {
        auto it = by_name.find(name);
        if (it == by_name.end()) { set_error("missing tensor '%s'", name.c_str()); return nullptr; }
        if (it->second->numel != numel) {
            set_error("tensor '%s': numel %lld, expected %lld", name.c_str(), it->second->numel, numel);
            return nullptr;
        }
        return it->second->data;
    }
};

// Host-side staging of packed weights; offsets are turned into device pointers after one upload.
struct Packer {
    std::vector<float> buf;
    size_t reserve(size_t n) {
        size_t off = (buf.size() + 63) & ~(size_t)63;     // 256-byte alignment for float4 / TMA
        buf.resize(off + n, 0.0f);
        return off;
    }
    // dst[k][o] = scale * W[o][col0 + k]   for W [out][in_total]
    size_t transposed(const float* W, int out, int in_total, int col0, int ncols, float scale = 1.0f) {
        size_t off = reserve((size_t)ncols * out);
        for (int k = 0; k < ncols; ++k)
            for (int o = 0; o < out; ++o) buf[off + (size_t)k * out + o] = scale * W[(size_t)o * in_total + col0 + k];
        return off;
    }
    size_t copy(const float* v, size_t n) {
        size_t off = reserve(n);
        memcpy(&buf[off], v, n * sizeof(float));
        return off;
    }
};

struct HalfPacker {
    std::vector<__half> buf;
    // dst[o][k] = fp16(scale * W[o][col0 + k]), one 128 x 128 block (consecutive blocks are 128 rows apart)
    size_t block(const float* W, int in_total, int col0, float scale = 1.0f) {
        size_t off = buf.size();
        buf.resize(off + 128 * 128);
        for (int o = 0; o < 128; ++o)
            for (int k = 0; k < 128; ++k) buf[off + (size_t)o * 128 + k] = __float2half_rn(scale * W[(size_t)o * in_total + col0 + k]);
        return off;
    }
};

#define GET(var, name, numel)                               \
    const float* var = tt.get(name, (long long)(numel));    \
    if (!var) return 1;

template <typename T>
int dev_alloc(std::vector<void*>& owned, T** ptr, size_t count) {
    void* q = nullptr;
    CB2_CUDA(cudaMalloc(&q, count * sizeof(T) > 0 ? count * sizeof(T) : 16));
    owned.push_back(q);
    *ptr = reinterpret_cast<T*>(q);
    return 0;
}

}  // namespace
}  // namespace cb2

using namespace cb2;

struct cb2_denoiser { DenoiserModel m; };
struct cb2_vae { VaeModel v; };
struct cb2_plan {
    Plan p;
    // decode-side buffers
    float* ca_full = nullptr;
    int *csr_row = nullptr, *csr_col = nullptr;
    int E = 0;              // edges of the current radius graph
    int E_cap = 0;          // edges csr_col / edge_w hold; both are owned here (not in p.allocs) and replaced when they grow
    signed char* orders = nullptr;
    int* slot_atom = nullptr;
    long long* out_off = nullptr;
    float *edge_w = nullptr, *S40 = nullptr, *phi = nullptr, *ic = nullptr, *zq = nullptr;
    int* vq_idx = nullptr;
    float *xa = nullptr, *xb = nullptr;     // ping-pong latents of the sampling loop
    float4* clash_bounds = nullptr;         // [NB*L] residue centre + radius of cb2_plan_residue_clashes (and cb2_plan_relax)
    RelaxBufs relax{};                      // cb2_plan_relax; sized by the plan's geometry, so allocated once, on first use
    int keep_debug = 0;
    bool frames_ready = false, topo_ready = false;
};

extern "C" {

int cb2_abi_version(void) { return CB2_ABI_VERSION; }
const char* cb2_last_error(void) { return cb2::g_err; }

// ------------------------------------------------------------------------------------------- denoiser
int cb2_denoiser_create(const cb2_tensor* tensors, int n_tensors, const float* freqs128, int k_neighbors, cb2_denoiser** out) {
    if (!tensors || !freqs128 || !out) { set_error("denoiser_create: null argument"); return 1; }
    TensorTable tt(tensors, n_tensors);
    Packer pk;
    HalfPacker bp;
    const int H = CB2_H;
    std::map<std::string, size_t> off;
    std::map<std::string, size_t> boff;

    off["freqs"] = pk.copy(freqs128, 128);
    GET(te0w, "t_embedder.mlp.0.weight", H * 256) GET(te0b, "t_embedder.mlp.0.bias", H)
    GET(te2w, "t_embedder.mlp.2.weight", H * H) GET(te2b, "t_embedder.mlp.2.bias", H)
    off["te_w0_t"] = pk.transposed(te0w, H, 256, 0, 256); off["te_b0"] = pk.copy(te0b, H);
    off["te_w2_t"] = pk.transposed(te2w, H, H, 0, H); off["te_b2"] = pk.copy(te2b, H);

    // adaLN projections concatenated along the output axis, transposed to [128][6016]
    {
        size_t wo = pk.reserve((size_t)H * CB2_MOD_TOTAL), bo = pk.reserve(CB2_MOD_TOTAL);
        off["ada_w_t"] = wo; off["ada_b"] = bo;
        int col = 0;
        auto put = [&](const std::string& pre, int width) -> int {
            const float* w = tt.get(pre + ".adaLN_modulation.1.weight", (long long)width * H);
            const float* b = tt.get(pre + ".adaLN_modulation.1.bias", width);
            if (!w || !b) return 1;
            for (int o = 0; o < width; ++o) {
                pk.buf[bo + col + o] = b[o];
                for (int k = 0; k < H; ++k) pk.buf[wo + (size_t)k * CB2_MOD_TOTAL + col + o] = w[(size_t)o * H + k];
            }
            col += width;
            return 0;
        };
        for (int l = 0; l < 3; ++l) if (put("encoder_layers." + std::to_string(l), CB2_MOD_ENC)) return 1;
        for (int l = 0; l < 3; ++l) if (put("decoder_layers." + std::to_string(l), CB2_MOD_DEC)) return 1;
        if (put("W_out", CB2_MOD_FIN)) return 1;
    }
    GET(xinw, "x_in.weight", H * 3) GET(xinb, "x_in.bias", H)
    off["xin_w_t"] = pk.transposed(xinw, H, 3, 0, 3); off["xin_b"] = pk.copy(xinb, H);

    // featuriser
    GET(posw, "features.embeddings.linear.weight", 16 * 66) GET(posb, "features.embeddings.linear.bias", 16)
    GET(edgew, "features.edge_embedding.weight", H * 167)
    GET(lnw, "features.norm_edges.weight", H) GET(lnb, "features.norm_edges.bias", H)
    GET(wew, "W_e.weight", H * H) GET(web, "W_e.bias", H)
    {
        size_t o = pk.reserve(65 * H);
        for (int d = 0; d < 65; ++d)
            for (int c = 0; c < H; ++c) {
                double a = 0.0;
                for (int q = 0; q < 16; ++q) a += (double)(posw[q * 66 + d] + posb[q]) * (double)edgew[(size_t)c * 167 + q];
                pk.buf[o + (size_t)d * H + c] = (float)a;
            }
        off["pos_table"] = o;
        size_t w = pk.reserve(152 * H);
        for (int r = 0; r < 151; ++r)
            for (int c = 0; c < H; ++c) pk.buf[w + (size_t)r * H + c] = edgew[(size_t)c * 167 + 16 + r];
        off["wedge_t"] = w;
    }
    off["ln_w"] = pk.copy(lnw, H); off["ln_b"] = pk.copy(lnb, H);
    off["we_t"] = pk.transposed(wew, H, H, 0, H); off["we_b"] = pk.copy(web, H);

    GET(ws, "W_s.weight", 30 * H)
    for (int l = 0; l < 3; ++l) {
        const std::string p = "encoder_layers." + std::to_string(l), k = "e" + std::to_string(l) + ".";
        GET(w1, p + ".W1.weight", H * 3 * H) GET(b1, p + ".W1.bias", H) GET(w2, p + ".W2.weight", H * H) GET(b2, p + ".W2.bias", H)
        GET(w3, p + ".W3.weight", H * H) GET(b3, p + ".W3.bias", H)
        GET(w11, p + ".W11.weight", H * 3 * H) GET(b11, p + ".W11.bias", H) GET(w12, p + ".W12.weight", H * H) GET(b12, p + ".W12.bias", H)
        GET(w13, p + ".W13.weight", H * H) GET(b13, p + ".W13.bias", H)
        GET(win, p + ".dense.W_in.weight", 4 * H * H) GET(bin, p + ".dense.W_in.bias", 4 * H)
        GET(wout, p + ".dense.W_out.weight", H * 4 * H) GET(bout, p + ".dense.W_out.bias", H)
        off[k + "W1a_t"] = pk.transposed(w1, H, 3 * H, 0, H); off[k + "W1b_t"] = pk.transposed(w1, H, 3 * H, H, H);
        off[k + "W1c_t"] = pk.transposed(w1, H, 3 * H, 2 * H, H); off[k + "b1"] = pk.copy(b1, H);
        off[k + "W2_t"] = pk.transposed(w2, H, H, 0, H); off[k + "b2"] = pk.copy(b2, H);
        off[k + "W3_t"] = pk.transposed(w3, H, H, 0, H); off[k + "b3"] = pk.copy(b3, H);
        off[k + "W11a_t"] = pk.transposed(w11, H, 3 * H, 0, H); off[k + "W11b_t"] = pk.transposed(w11, H, 3 * H, H, H);
        off[k + "W11c_t"] = pk.transposed(w11, H, 3 * H, 2 * H, H); off[k + "b11"] = pk.copy(b11, H);
        off[k + "W12_t"] = pk.transposed(w12, H, H, 0, H); off[k + "b12"] = pk.copy(b12, H);
        off[k + "W13_t"] = pk.transposed(w13, H, H, 0, H); off[k + "b13"] = pk.copy(b13, H);
        off[k + "Win_t"] = pk.transposed(win, 4 * H, H, 0, H); off[k + "bin"] = pk.copy(bin, 4 * H);
        off[k + "Wout_t"] = pk.transposed(wout, H, 4 * H, 0, 4 * H); off[k + "bout"] = pk.copy(bout, H);
        // fp16 blocks that consume a GELU activation are packed x 0.5: the tensor-core epilogues emit 2 GELU (tc_common.cuh)
        boff[k + "W1b"] = bp.block(w1, 3 * H, H); boff[k + "W2"] = bp.block(w2, H, 0, 0.5f);
        boff[k + "W11b"] = bp.block(w11, 3 * H, H); boff[k + "W12"] = bp.block(w12, H, 0, 0.5f); boff[k + "W13"] = bp.block(w13, H, 0, 0.5f);
        boff[k + "W1a"] = bp.block(w1, 3 * H, 0); boff[k + "W1c"] = bp.block(w1, 3 * H, 2 * H);
        boff[k + "W11a"] = bp.block(w11, 3 * H, 0); boff[k + "W11c"] = bp.block(w11, 3 * H, 2 * H);
        boff[k + "W3"] = bp.block(w3, H, 0);
        for (int q = 0; q < 4; ++q) { size_t o = bp.block(win + (size_t)q * H * H, H, 0); if (q == 0) boff[k + "Win"] = o; }
        for (int q = 0; q < 4; ++q) { size_t o = bp.block(wout, 4 * H, q * H, 0.5f); if (q == 0) boff[k + "Wout"] = o; }
    }
    for (int l = 0; l < 3; ++l) {
        const std::string p = "decoder_layers." + std::to_string(l), k = "d" + std::to_string(l) + ".";
        GET(w1, p + ".W1.weight", H * 4 * H) GET(b1, p + ".W1.bias", H) GET(w2, p + ".W2.weight", H * H) GET(b2, p + ".W2.bias", H)
        GET(w3, p + ".W3.weight", H * H) GET(b3, p + ".W3.bias", H)
        GET(win, p + ".dense.W_in.weight", 4 * H * H) GET(bin, p + ".dense.W_in.bias", 4 * H)
        GET(wout, p + ".dense.W_out.weight", H * 4 * H) GET(bout, p + ".dense.W_out.bias", H)
        off[k + "W1a_t"] = pk.transposed(w1, H, 4 * H, 0, H); off[k + "W1b2_t"] = pk.transposed(w1, H, 4 * H, H, H, 2.0f);
        off[k + "W1d_t"] = pk.transposed(w1, H, 4 * H, 3 * H, H); off[k + "b1"] = pk.copy(b1, H);
        {
            size_t o = pk.reserve(30 * H);      // TS[z][c] = 2 * sum_k W_s[z][k] W1[c][256 + k]
            for (int z = 0; z < 30; ++z)
                for (int c = 0; c < H; ++c) {
                    double a = 0.0;
                    for (int q = 0; q < H; ++q) a += (double)ws[z * H + q] * (double)w1[(size_t)c * 4 * H + 2 * H + q];
                    pk.buf[o + (size_t)z * H + c] = (float)(2.0 * a);
                }
            off[k + "TS"] = o;
        }
        off[k + "W2_t"] = pk.transposed(w2, H, H, 0, H); off[k + "b2"] = pk.copy(b2, H);
        off[k + "W3_t"] = pk.transposed(w3, H, H, 0, H); off[k + "b3"] = pk.copy(b3, H);
        off[k + "Win_t"] = pk.transposed(win, 4 * H, H, 0, H); off[k + "bin"] = pk.copy(bin, 4 * H);
        off[k + "Wout_t"] = pk.transposed(wout, H, 4 * H, 0, 4 * H); off[k + "bout"] = pk.copy(bout, H);
        boff[k + "W1b2"] = bp.block(w1, 4 * H, H, 2.0f); boff[k + "W2"] = bp.block(w2, H, 0, 0.5f);
        boff[k + "W1a"] = bp.block(w1, 4 * H, 0); boff[k + "W1d"] = bp.block(w1, 4 * H, 3 * H);
        boff[k + "W3"] = bp.block(w3, H, 0);
        for (int q = 0; q < 4; ++q) { size_t o = bp.block(win + (size_t)q * H * H, H, 0); if (q == 0) boff[k + "Win"] = o; }
        for (int q = 0; q < 4; ++q) { size_t o = bp.block(wout, 4 * H, q * H, 0.5f); if (q == 0) boff[k + "Wout"] = o; }
    }
    GET(finw, "W_out.linear.weight", 6 * H) GET(finb, "W_out.linear.bias", 6)
    off["fin_w_t"] = pk.transposed(finw, 6, H, 0, H); off["fin_b"] = pk.copy(finb, 6);

    cb2_denoiser* d = new cb2_denoiser();
    DenoiserModel& m = d->m;
    m.k_neighbors = k_neighbors;
    CB2_CUDA(cudaMalloc(&m.dev_f32, pk.buf.size() * sizeof(float)));
    CB2_CUDA(cudaMemcpy(m.dev_f32, pk.buf.data(), pk.buf.size() * sizeof(float), cudaMemcpyHostToDevice));
    {
        std::vector<__half> v16;
        std::map<std::string, size_t> voff;
        auto putv = [&](const std::string& key, const float* src) {
            voff[key] = v16.size();
            for (int q = 0; q < H; ++q) v16.push_back(__float2half_rn(src[q]));
        };
        for (int l = 0; l < 3; ++l) {
            const std::string pe = "encoder_layers." + std::to_string(l), pd = "decoder_layers." + std::to_string(l);
            putv("e" + std::to_string(l) + ".b2", tt.get(pe + ".W2.bias", H));
            putv("e" + std::to_string(l) + ".b12", tt.get(pe + ".W12.bias", H));
            putv("e" + std::to_string(l) + ".b13", tt.get(pe + ".W13.bias", H));
            putv("d" + std::to_string(l) + ".b2", tt.get(pd + ".W2.bias", H));
        }
        CB2_CUDA(cudaMalloc(&m.dev_vec16, v16.size() * sizeof(__half)));
        CB2_CUDA(cudaMemcpy(m.dev_vec16, v16.data(), v16.size() * sizeof(__half), cudaMemcpyHostToDevice));
        for (int l = 0; l < 3; ++l) {
            m.enc[l].b2_16 = m.dev_vec16 + voff.at("e" + std::to_string(l) + ".b2");
            m.enc[l].b12_16 = m.dev_vec16 + voff.at("e" + std::to_string(l) + ".b12");
            m.enc[l].b13_16 = m.dev_vec16 + voff.at("e" + std::to_string(l) + ".b13");
            m.dec[l].b2_16 = m.dev_vec16 + voff.at("d" + std::to_string(l) + ".b2");
        }
    }
    CB2_CUDA(cudaMalloc(&m.dev_f16, bp.buf.size() * sizeof(__half)));
    CB2_CUDA(cudaMemcpy(m.dev_f16, bp.buf.data(), bp.buf.size() * sizeof(__half), cudaMemcpyHostToDevice));
    m.n_f16_blocks = (int)(bp.buf.size() / (128 * 128));
    auto F = [&](const std::string& key) { return (const float*)(m.dev_f32 + off.at(key)); };
    auto B = [&](const std::string& key) { return (const __half*)(m.dev_f16 + boff.at(key)); };
    m.freqs = F("freqs"); m.te_w0_t = F("te_w0_t"); m.te_b0 = F("te_b0"); m.te_w2_t = F("te_w2_t"); m.te_b2 = F("te_b2");
    m.ada_w_t = F("ada_w_t"); m.ada_b = F("ada_b"); m.xin_w_t = F("xin_w_t"); m.xin_b = F("xin_b");
    m.pos_table = F("pos_table"); m.wedge_t = F("wedge_t"); m.ln_w = F("ln_w"); m.ln_b = F("ln_b"); m.we_t = F("we_t"); m.we_b = F("we_b");
    for (int l = 0; l < 3; ++l) {
        const std::string k = "e" + std::to_string(l) + ".";
        EncLayerW& e = m.enc[l];
        e.W1a_t = F(k + "W1a_t"); e.W1b_t = F(k + "W1b_t"); e.W1c_t = F(k + "W1c_t"); e.b1 = F(k + "b1");
        e.W2_t = F(k + "W2_t"); e.b2 = F(k + "b2"); e.W3_t = F(k + "W3_t"); e.b3 = F(k + "b3");
        e.W11a_t = F(k + "W11a_t"); e.W11b_t = F(k + "W11b_t"); e.W11c_t = F(k + "W11c_t"); e.b11 = F(k + "b11");
        e.W12_t = F(k + "W12_t"); e.b12 = F(k + "b12"); e.W13_t = F(k + "W13_t"); e.b13 = F(k + "b13");
        e.Win_t = F(k + "Win_t"); e.bin = F(k + "bin"); e.Wout_t = F(k + "Wout_t"); e.bout = F(k + "bout");
        e.W1b_h = B(k + "W1b"); e.W2_h = B(k + "W2"); e.W11b_h = B(k + "W11b"); e.W12_h = B(k + "W12"); e.W13_h = B(k + "W13");
        e.W1a_h = B(k + "W1a"); e.W1c_h = B(k + "W1c"); e.W11a_h = B(k + "W11a"); e.W11c_h = B(k + "W11c");
        e.W3_h = B(k + "W3"); e.Win_h = B(k + "Win"); e.Wout_h = B(k + "Wout");
    }
    for (int l = 0; l < 3; ++l) {
        const std::string k = "d" + std::to_string(l) + ".";
        DecLayerW& e = m.dec[l];
        e.W1a_t = F(k + "W1a_t"); e.W1b2_t = F(k + "W1b2_t"); e.W1d_t = F(k + "W1d_t"); e.b1 = F(k + "b1"); e.TS = F(k + "TS");
        e.W2_t = F(k + "W2_t"); e.b2 = F(k + "b2"); e.W3_t = F(k + "W3_t"); e.b3 = F(k + "b3");
        e.Win_t = F(k + "Win_t"); e.bin = F(k + "bin"); e.Wout_t = F(k + "Wout_t"); e.bout = F(k + "bout");
        e.W1b2_h = B(k + "W1b2"); e.W2_h = B(k + "W2");
        e.W1a_h = B(k + "W1a"); e.W1d_h = B(k + "W1d"); e.W3_h = B(k + "W3"); e.Win_h = B(k + "Win"); e.Wout_h = B(k + "Wout");
    }
    m.fin_w_t = F("fin_w_t"); m.fin_b = F("fin_b");
    *out = d;
    return 0;
}

void cb2_denoiser_destroy(cb2_denoiser* d) {
    if (!d) return;
    cudaFree(d->m.dev_f32);
    cudaFree(d->m.dev_f16);
    cudaFree(d->m.dev_vec16);
    delete d;
}

// ------------------------------------------------------------------------------------------- VAE decode side
int cb2_vae_create(const cb2_tensor* tensors, int n_tensors, const float* mean3, const float* std3, int angle_variant, cb2_vae** out) {
    if (!tensors || !mean3 || !std3 || !out) { set_error("vae_create: null argument"); return 1; }
    TensorTable tt(tensors, n_tensors);
    Packer pk;
    std::map<std::string, size_t> off;
    const std::string P = "equivaraintconv.";
    auto itcb = tt.by_name.find("quantize._codebook.embed");
    if (itcb == tt.by_name.end() || itcb->second->numel % 3 != 0) { set_error("missing/invalid quantize._codebook.embed"); return 1; }
    const int M = (int)(itcb->second->numel / 3);
    off["codebook"] = pk.copy(itcb->second->data, (size_t)M * 3);
    off["mean"] = pk.copy(mean3, 3); off["std"] = pk.copy(std3, 3);
    GET(mow, "map_out.weight", 36 * 3) GET(mob, "map_out.bias", 36)
    off["mapw_t"] = pk.transposed(mow, 36, 3, 0, 3); off["mapb"] = pk.copy(mob, 36);
    GET(remb, P + "res_embed.weight", 25 * 4) off["res_embed"] = pk.copy(remb, 100);
    const int D = 40, T = angle_variant ? 50 : 40;
    auto linear = [&](const std::string& key, const std::string& name, int o, int i) -> int {
        const float* w = tt.get(P + name + ".weight", (long long)o * i);
        const float* b = tt.get(P + name + ".bias", o);
        if (!w || !b) return 1;
        off[key + "_t"] = pk.transposed(w, o, i, 0, i);
        off[key + "_b"] = pk.copy(b, o);
        return 0;
    };
    size_t wd = pk.reserve(4 * 15 * D), bd = pk.reserve(4 * D);
    off["Wd_t"] = wd; off["bd"] = bd;
    for (int b = 0; b < 4; ++b) {
        const std::string s = std::to_string(b);
        if (linear("inv0." + s, "message_blocks." + s + ".inv_dense.0", D, D)) return 1;
        if (linear("inv1." + s, "message_blocks." + s + ".inv_dense.1", D, D)) return 1;
        GET(dw, P + "message_blocks." + s + ".dist_embed.block.1.weight", D * 15)
        GET(db, P + "message_blocks." + s + ".dist_embed.block.1.bias", D)
        for (int q = 0; q < 15; ++q)
            for (int c = 0; c < D; ++c) pk.buf[wd + ((size_t)b * 15 + q) * D + c] = dw[c * 15 + q];
        for (int c = 0; c < D; ++c) pk.buf[bd + b * D + c] = db[c];
        if (linear("db1." + s, "dense_blocks." + s + ".1", D, D)) return 1;
        if (linear("db3." + s, "dense_blocks." + s + ".3", D, D)) return 1;
        if (linear("tb1." + s, "sidechain_torsion_blocks." + s + ".1", T, T)) return 1;
        if (linear("tb3." + s, "sidechain_torsion_blocks." + s + ".3", T, T)) return 1;
    }
    GET(bbd, P + "backbone_dist.weight", 75) GET(scd, P + "sidechain_dist.weight", 250)
    off["bb_dist"] = pk.copy(bbd, 75); off["sc_dist"] = pk.copy(scd, 250);
    if (linear("ba1", "backbone_angle.1", 3, D) || linear("ba3", "backbone_angle.3", 3, 3)) return 1;
    if (linear("bt1", "backbone_torsion.1", 3, D + 3) || linear("bt3", "backbone_torsion.3", 3, 3)) return 1;
    if (angle_variant) {
        if (linear("sa1", "sidechain_angle.1", 10, D) || linear("sa3", "sidechain_angle.3", 10, 10)) return 1;
    } else {
        GET(sae, P + "sidechain_angle.weight", 250) off["sa_embed"] = pk.copy(sae, 250);
    }
    if (linear("ft1", "final_torsion.1", 10, T) || linear("ft3", "final_torsion.3", 10, 10)) return 1;

    cb2_vae* h = new cb2_vae();
    VaeModel& v = h->v;
    v.M = M; v.angle_variant = angle_variant;
    CB2_CUDA(cudaMalloc(&v.dev, pk.buf.size() * sizeof(float)));
    CB2_CUDA(cudaMemcpy(v.dev, pk.buf.data(), pk.buf.size() * sizeof(float), cudaMemcpyHostToDevice));
    auto F = [&](const std::string& key) -> const float* {
        auto it = off.find(key);
        return it == off.end() ? nullptr : (const float*)(v.dev + it->second);
    };
    v.codebook = F("codebook"); v.mean = F("mean"); v.stdv = F("std"); v.mapw_t = F("mapw_t"); v.mapb = F("mapb");
    v.res_embed = F("res_embed"); v.Wd_t = F("Wd_t"); v.bd = F("bd");
    for (int b = 0; b < 4; ++b) {
        const std::string s = std::to_string(b);
        v.inv0_t[b] = F("inv0." + s + "_t"); v.inv0_b[b] = F("inv0." + s + "_b");
        v.inv1_t[b] = F("inv1." + s + "_t"); v.inv1_b[b] = F("inv1." + s + "_b");
        v.db1_t[b] = F("db1." + s + "_t"); v.db1_b[b] = F("db1." + s + "_b");
        v.db3_t[b] = F("db3." + s + "_t"); v.db3_b[b] = F("db3." + s + "_b");
        v.tb1_t[b] = F("tb1." + s + "_t"); v.tb1_b[b] = F("tb1." + s + "_b");
        v.tb3_t[b] = F("tb3." + s + "_t"); v.tb3_b[b] = F("tb3." + s + "_b");
    }
    v.bb_dist = F("bb_dist"); v.sc_dist = F("sc_dist"); v.sa_embed = F("sa_embed");
    v.ba1_t = F("ba1_t"); v.ba1_b = F("ba1_b"); v.ba3_t = F("ba3_t"); v.ba3_b = F("ba3_b");
    v.bt1_t = F("bt1_t"); v.bt1_b = F("bt1_b"); v.bt3_t = F("bt3_t"); v.bt3_b = F("bt3_b");
    v.sa1_t = F("sa1_t"); v.sa1_b = F("sa1_b"); v.sa3_t = F("sa3_t"); v.sa3_b = F("sa3_b");
    v.ft1_t = F("ft1_t"); v.ft1_b = F("ft1_b"); v.ft3_t = F("ft3_t"); v.ft3_b = F("ft3_b");
    CB2_CUDA(cudaMalloc(&v.e2, (size_t)M * sizeof(float)));
    if (int e = launch_codebook_norms(v.codebook, M, v.e2, 0)) return e;
    CB2_CUDA(cudaStreamSynchronize(0));
    *out = h;
    return 0;
}

void cb2_vae_destroy(cb2_vae* h) {
    if (!h) return;
    cudaFree(h->v.dev);
    cudaFree(h->v.e2);
    delete h;
}

// ------------------------------------------------------------------------------------------- plan
int cb2_plan_create(const cb2_denoiser* d, int F, int NB, int L, int precision, int keep_debug, cb2_plan** out) {
    if (!out || F <= 0 || NB <= 0 || L <= 0) { set_error("plan_create: bad argument"); return 1; }
    if (precision != PREC_F32 && precision != PREC_F16) { set_error("plan_create: unknown precision %d", precision); return 1; }
    cb2_plan* h = new cb2_plan();
    Plan& p = h->p;
    p.model = d ? &d->m : nullptr; p.F = F; p.NB = NB; p.L = L; p.precision = precision;
    h->keep_debug = keep_debug;
    if (!d) {
        // decode-only plan (no denoiser): just the frame geometry the VQ / IC decoder / ic_to_xyz side needs
        int e = 0;
        e |= dev_alloc(p.allocs, &p.X, (size_t)F * L * 3);
        e |= dev_alloc(p.allocs, &p.lengths, F);
        e |= dev_alloc(p.allocs, &p.cg_z, (size_t)F * L);
        e |= dev_alloc(p.allocs, &p.frame_of, NB);
        if (e) { cb2_plan_destroy(h); return e; }
        *out = h;
        return 0;
    }
    p.K = d->m.k_neighbors < L ? d->m.k_neighbors : L;
    const size_t N = (size_t)NB * L, FE = (size_t)F * L * p.K, NE = N * p.K;
    const size_t esz = precision == PREC_F16 ? 2 : 4;
    int e = 0;
    e |= dev_alloc(p.allocs, &p.X, (size_t)F * L * 3);
    e |= dev_alloc(p.allocs, &p.lengths, F);
    e |= dev_alloc(p.allocs, &p.cg_z, (size_t)F * L);
    e |= dev_alloc(p.allocs, &p.frame_of, NB);
    e |= dev_alloc(p.allocs, &p.nbr_idx, FE);
    e |= dev_alloc(p.allocs, &p.nbr_dist, FE);
    e |= dev_alloc(p.allocs, reinterpret_cast<unsigned char**>(&p.hE0), FE * 128 * esz);
    e |= dev_alloc(p.allocs, reinterpret_cast<unsigned char**>(&p.hE), NE * 128 * esz);
    if (keep_debug) e |= dev_alloc(p.allocs, &p.E_dbg, FE * 128);
    e |= dev_alloc(p.allocs, &p.hV, N * 128);
    e |= dev_alloc(p.allocs, &p.hVenc, N * 128);
    e |= dev_alloc(p.allocs, &p.P, 2 * N * 256);
    if (precision == PREC_F16) {
        e |= dev_alloc(p.allocs, &p.P16[0], N * 256);
        e |= dev_alloc(p.allocs, &p.P16[1], N * 256);
    }
    e |= dev_alloc(p.allocs, &p.S, N * 128);
    e |= dev_alloc(p.allocs, &p.out6, N * 6);
    e |= dev_alloc(p.allocs, &h->xa, N * 3);
    e |= dev_alloc(p.allocs, &h->xb, N * 3);
    p.mod_capacity = NB > 1024 ? NB : 1024;
    e |= dev_alloc(p.allocs, &p.mod, (size_t)p.mod_capacity * CB2_MOD_TOTAL);
    if (precision == PREC_F16) e |= dev_alloc(p.allocs, &p.mod16, (size_t)p.mod_capacity * 768);
    e |= dev_alloc(p.allocs, &p.silu_c, (size_t)p.mod_capacity * 128);
    e |= dev_alloc(p.allocs, &p.tvals, p.mod_capacity);
    e |= dev_alloc(p.allocs, &p.coef, (size_t)p.mod_capacity * 8);
    if (e) { cb2_plan_destroy(h); return e; }
    if (precision == PREC_F16) {
        if (int r = edge_tc_prepare(p)) { cb2_plan_destroy(h); return r; }
        if (int r = node_tc_prepare(p)) { cb2_plan_destroy(h); return r; }
    }
    *out = h;
    return 0;
}

void cb2_plan_destroy(cb2_plan* h) {
    if (!h) return;
    if (h->p.graph) cudaGraphExecDestroy(h->p.graph);
    edge_tc_release(h->p);
    node_tc_release(h->p);
    for (void* q : h->p.allocs) cudaFree(q);
    cudaFree(h->csr_col);
    cudaFree(h->edge_w);
    delete h;
}

int cb2_plan_K(const cb2_plan* h) { return h ? h->p.K : 0; }
long long cb2_plan_launches(const cb2_plan* h) { return h ? h->p.launches : 0; }

int cb2_plan_set_frames(cb2_plan* h, const float* X, const int* lengths, const int* cg_z, const int* frame_of, void* stream) {
    if (!h || !X || !lengths || !cg_z || !frame_of) { set_error("set_frames: null argument"); return 1; }
    Plan& p = h->p;
    cudaStream_t s = (cudaStream_t)stream;
    CB2_CUDA(cudaMemcpyAsync(p.X, X, (size_t)p.F * p.L * 3 * sizeof(float), cudaMemcpyDeviceToDevice, s));
    CB2_CUDA(cudaMemcpyAsync(p.lengths, lengths, p.F * sizeof(int), cudaMemcpyDeviceToDevice, s));
    CB2_CUDA(cudaMemcpyAsync(p.cg_z, cg_z, (size_t)p.F * p.L * sizeof(int), cudaMemcpyDeviceToDevice, s));
    CB2_CUDA(cudaMemcpyAsync(p.frame_of, frame_of, p.NB * sizeof(int), cudaMemcpyDeviceToDevice, s));
    if (p.model == nullptr) { h->frames_ready = true; return 0; }      // decode-only plan
    {   // host-side knowledge of the geometry: are there padded residues at all?  (lets the tensor-core message kernels skip
        // the neighbour mask when every frame is full length; once per frame set, not on the step path)
        std::vector<int> len((size_t)p.F);
        CB2_CUDA(cudaMemcpyAsync(len.data(), p.lengths, (size_t)p.F * sizeof(int), cudaMemcpyDeviceToHost, s));
        CB2_CUDA(cudaStreamSynchronize(s));
        p.all_full = true;
        for (int f = 0; f < p.F; ++f) p.all_full = p.all_full && len[f] >= p.L;
    }
    if (int e = launch_knn(p.X, p.lengths, p.F, p.L, p.K, p.nbr_dist, p.nbr_idx, s)) return e;
    if (int e = launch_edge_features(*p.model, p.X, p.lengths, p.nbr_idx, p.nbr_dist, p.F, p.L, p.K, p.E_dbg, p.hE0, p.precision, s)) return e;
    p.launches += 2;
    h->frames_ready = true;
    return 0;
}

}  // extern "C"

namespace {

int edge_dispatch(Plan& p, int mode, int layer, const float* mod_base, int mod_stride, cudaStream_t s) {
    return p.precision == PREC_F16 ? launch_edge_tc(p, mode, layer, mod_base, mod_stride, s)
                                    : launch_edge_f32(p, mode, layer, mod_base, mod_stride, s);
}

// One denoiser forward; when x_next != nullptr the last kernel also applies the p_sample (or DDIM) update, then, when
// inpaint_row != nullptr, the inpainting overwrite of the kept rows.
int run_forward(Plan& p, const float* x, const float* mod_base, int mod_stride, const float* noise, float* x_next,
                const float* coef_row, const float* inpaint_row, cudaStream_t s, int stop_after = -1) {
    int n = 0;
    auto done = [&]() { return stop_after >= 0 && ++n >= stop_after; };     // debug: stop after `stop_after` kernels
    const bool tc = p.precision == PREC_F16 && p.node_tc != nullptr;
    auto node_update = [&](int phase, const float* xt, const float* nz, float* xn, const float* cf, const float* iq) {
        return tc ? launch_node_update_tc(p, phase, mod_base, mod_stride, xt, nz, xn, cf, iq, s)
                  : launch_node_update(p, phase, mod_base, mod_stride, xt, nz, xn, cf, iq, s);
    };
    if (int e = tc ? launch_node_init_tc(p, x, s) : launch_node_init(p, x, mod_base, mod_stride, s)) return e;
    if (done()) return 0;
    for (int l = 0; l < 3; ++l) {
        if (int e = edge_dispatch(p, EDGE_ENC_NODE, l, mod_base, mod_stride, s)) return e;
        if (done()) return 0;
        if (int e = node_update(l, nullptr, nullptr, nullptr, nullptr, nullptr)) return e;
        if (done()) return 0;
        if (int e = edge_dispatch(p, EDGE_ENC_EDGE, l, mod_base, mod_stride, s)) return e;
        if (done()) return 0;
    }
    for (int l = 0; l < 3; ++l) {
        if (int e = edge_dispatch(p, EDGE_DEC, l, mod_base, mod_stride, s)) return e;
        if (done()) return 0;
        const bool last = l == 2;
        if (int e = node_update(3 + l, last ? x : nullptr, last ? noise : nullptr, last ? x_next : nullptr, last ? coef_row : nullptr,
                                last ? inpaint_row : nullptr)) return e;
        if (done()) return 0;
    }
    return 0;
}

}  // namespace

extern "C" {

int cb2_plan_forward_partial(cb2_plan* h, const float* x, const float* t, int stop_after, void* stream) {
    if (!h || !x || !t) { set_error("forward_partial: null argument"); return 1; }
    if (!h->frames_ready || !h->p.model) { set_error("forward_partial: no denoiser frames on this plan"); return 1; }
    Plan& p = h->p;
    cudaStream_t s = (cudaStream_t)stream;
    if (int e = launch_timestep_mod(*p.model, t, p.NB, p.silu_c, p.mod, p.mod16, s)) return e;
    p.coef_steps = 0;
    return run_forward(p, x, p.mod, CB2_MOD_TOTAL, nullptr, nullptr, nullptr, nullptr, s, stop_after);
}

int cb2_plan_forward(cb2_plan* h, const float* x, const float* t, float* out, void* stream) {
    if (!h || !x || !t || !out) { set_error("forward: null argument"); return 1; }
    if (!h->frames_ready || !h->p.model) { set_error("forward: cb2_plan_set_frames has not been called (or decode-only plan)"); return 1; }
    Plan& p = h->p;
    cudaStream_t s = (cudaStream_t)stream;
    if (p.NB > p.mod_capacity) { set_error("forward: NB exceeds table capacity"); return 1; }
    if (int e = launch_timestep_mod(*p.model, t, p.NB, p.silu_c, p.mod, p.mod16, s)) return e;
    p.launches += 2;
    p.coef_steps = 0;   // the table no longer holds a sampling schedule
    if (int e = run_forward(p, x, p.mod, CB2_MOD_TOTAL, nullptr, nullptr, nullptr, nullptr, s)) return e;
    CB2_CUDA(cudaMemcpyAsync(out, p.out6, (size_t)p.NB * p.L * 6 * sizeof(float), cudaMemcpyDeviceToDevice, s));
    return 0;
}

static int set_schedule(cb2_plan* h, const float* t_of_step, const float* coef, int T, int kind, cudaStream_t s) {
    if (!h || !t_of_step || !coef || T <= 0 || !h->p.model) { set_error("set_schedule: bad argument"); return 1; }
    Plan& p = h->p;
    if (T > p.mod_capacity) { set_error("set_schedule: T=%d exceeds capacity %d", T, p.mod_capacity); return 1; }
    CB2_CUDA(cudaMemcpyAsync(p.tvals, t_of_step, T * sizeof(float), cudaMemcpyHostToDevice, s));
    CB2_CUDA(cudaMemcpyAsync(p.coef, coef, (size_t)T * 8 * sizeof(float), cudaMemcpyHostToDevice, s));
    if (int e = launch_timestep_mod(*p.model, p.tvals, T, p.silu_c, p.mod, p.mod16, s)) return e;
    CB2_CUDA(cudaStreamSynchronize(s));     // host staging buffers may be freed by the caller on return
    p.launches += 2;
    p.coef_steps = T;
    p.update_kind = kind;
    p.coef_noisy = kind == UPDATE_DDPM;
    for (int i = 0; i < T && !p.coef_noisy; ++i) p.coef_noisy = coef[(size_t)i * 8 + 4] != 0.0f;      // some DDIM sigma != 0
    if (p.graph) { cudaGraphExecDestroy(p.graph); p.graph = nullptr; }
    return 0;
}

int cb2_plan_set_schedule(cb2_plan* h, const float* t_of_step, const float* coef, int T, void* stream) {
    return set_schedule(h, t_of_step, coef, T, UPDATE_DDPM, (cudaStream_t)stream);
}

int cb2_plan_set_ddim_schedule(cb2_plan* h, const float* t_of_step, const float* ddim_coef, int T, void* stream) {
    return set_schedule(h, t_of_step, ddim_coef, T, UPDATE_DDIM, (cudaStream_t)stream);
}

int cb2_plan_set_inpaint(cb2_plan* h, const unsigned char* keep, const float* x0, const float* q_coef, int T, void* stream) {
    if (!h || !h->p.model) { set_error("set_inpaint: bad argument"); return 1; }
    Plan& p = h->p;
    if (!keep) { p.inpaint = false; return 0; }
    if (!x0 || !q_coef || T <= 0) { set_error("set_inpaint: x0, q_coef and T > 0 are required with a keep mask"); return 1; }
    if (T > p.mod_capacity) { set_error("set_inpaint: T=%d exceeds capacity %d", T, p.mod_capacity); return 1; }
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)p.NB * p.L;
    if (!p.inp_keep) {     // allocated once: the captured loop reads these addresses, so new contents need no recapture
        unsigned char* keep_buf = nullptr;
        float *x0_buf = nullptr, *eps_buf = nullptr, *coef_buf = nullptr;
        int e = 0;
        e |= dev_alloc(p.allocs, &keep_buf, N);
        e |= dev_alloc(p.allocs, &x0_buf, N * 3);
        e |= dev_alloc(p.allocs, &eps_buf, N * 3);
        e |= dev_alloc(p.allocs, &coef_buf, (size_t)(p.mod_capacity + 1) * 2);
        if (e) return e;    // the plan keeps none of them (those that were allocated are freed with it)
        p.inp_keep = keep_buf; p.inp_x0 = x0_buf; p.inp_eps = eps_buf; p.inp_coef = coef_buf;
    }
    CB2_CUDA(cudaMemcpyAsync(p.inp_keep, keep, N, cudaMemcpyDeviceToDevice, s));
    CB2_CUDA(cudaMemcpyAsync(p.inp_x0, x0, N * 3 * sizeof(float), cudaMemcpyDeviceToDevice, s));
    const size_t nq = (size_t)(T + 1) * 2;
    if (p.inp_coef_host.size() != nq || memcmp(p.inp_coef_host.data(), q_coef, nq * sizeof(float)) != 0) {
        p.inp_coef_host.assign(q_coef, q_coef + nq);
        CB2_CUDA(cudaMemcpyAsync(p.inp_coef, q_coef, nq * sizeof(float), cudaMemcpyHostToDevice, s));
        CB2_CUDA(cudaStreamSynchronize(s));     // the caller may free q_coef on return
    }
    p.inpaint_steps = T;
    p.inpaint = true;
    return 0;
}

int cb2_plan_set_start(cb2_plan* h, int steps, void* stream) {
    (void)stream;       // host-side state only
    if (!h || !h->p.model) { set_error("set_start: bad argument"); return 1; }
    if (steps < 0) { set_error("set_start: steps must be >= 0, got %d", steps); return 1; }
    h->p.start_steps = steps;
    return 0;
}

static int enqueue_loop(cb2_plan* h, float* x, const float* noise, cudaStream_t s) {
    Plan& p = h->p;
    const size_t n3 = (size_t)p.NB * p.L * 3;
    CB2_CUDA(cudaMemcpyAsync(h->xa, x, n3 * sizeof(float), cudaMemcpyDeviceToDevice, s));
    const bool refine = p.start_steps > 0;
    const int steps = refine ? p.start_steps : p.coef_steps;
    if (p.inpaint) {
        if (int e = launch_inpaint_init(p.inp_keep, p.inp_x0, p.inp_coef + (size_t)steps * 2, p.NB * p.L, refine, h->xa, p.inp_eps, s)) return e;
        p.launches++;
    }
    float *cur = h->xa, *nxt = h->xb;
    for (int step = steps - 1; step >= 0; --step) {
        const float* mod_row = p.mod + (size_t)step * CB2_MOD_TOTAL;     // every member shares the step -> stride 0
        const float* step_noise = noise != nullptr ? noise + (size_t)step * n3 : nullptr;
        const float* inpaint_row = p.inpaint ? p.inp_coef + (size_t)step * 2 : nullptr;
        if (int e = run_forward(p, cur, mod_row, 0, step_noise, nxt, p.coef + (size_t)step * 8, inpaint_row, s)) {
            char prev[1024];
            snprintf(prev, sizeof(prev), "%s", g_err);
            const unsigned int* tl = edge_tc_trap_log();
            if (tl != nullptr) {
                char w[600]; int n = 0;
                for (int i = 0; i < 18 && n < 560; ++i)
                    if (tl[4 + 2 * i]) n += snprintf(w + n, sizeof(w) - n, " w%d:bar+0x%x/p%u", i, tl[4 + 2 * i] & 0xfffu, tl[5 + 2 * i] >> 16);
                set_error("%s [sampling step %d; block %u timed-out waits:%s]", prev, step, tl[0] - 1u, w);
            }
            else set_error("%s [sampling step %d]", prev, step);
            return e;
        }
        float* t = cur; cur = nxt; nxt = t;
    }
    CB2_CUDA(cudaMemcpyAsync(x, cur, n3 * sizeof(float), cudaMemcpyDeviceToDevice, s));
    return 0;
}

int cb2_plan_sample(cb2_plan* h, float* x, const float* noise, int use_graph, void* stream) {
    if (!h || !x) { set_error("sample: null argument"); return 1; }
    Plan& p = h->p;
    if (!h->frames_ready || p.coef_steps <= 0) { set_error("sample: set_frames / set_schedule must be called first"); return 1; }
    if (!noise && p.coef_noisy) { set_error("sample: noise may be NULL only on a DDIM schedule whose sigma are all zero (eta = 0)"); return 1; }
    if (p.inpaint && p.inpaint_steps != p.coef_steps) {
        set_error("sample: the inpainting table has T=%d, the schedule T=%d", p.inpaint_steps, p.coef_steps);
        return 1;
    }
    if (p.start_steps > p.coef_steps) {
        set_error("sample: the start (%d steps) exceeds the schedule's T=%d", p.start_steps, p.coef_steps);
        return 1;
    }
    if (p.start_steps > 0 && !p.inpaint) {
        set_error("sample: a start of %d steps refines the inpainting latent x0: cb2_plan_set_inpaint must be called first", p.start_steps);
        return 1;
    }
    cudaStream_t s = (cudaStream_t)stream;
    if (!use_graph) return enqueue_loop(h, x, noise, s);
    // (kernel variants are chosen at capture time from the geometry: a frame set with / without padded residues needs its own graph)
    if (!p.graph || p.graph_key[0] != x || p.graph_key[1] != noise || p.graph_steps != p.coef_steps || p.graph_all_full != p.all_full ||
        p.graph_inpaint != p.inpaint || p.graph_start != p.start_steps) {
        if (p.graph) { cudaGraphExecDestroy(p.graph); p.graph = nullptr; }
        cudaStream_t cs;
        CB2_CUDA(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
        const long long before = p.launches;
        CB2_CUDA(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
        int e = enqueue_loop(h, x, noise, cs);
        cudaGraph_t g = nullptr;
        cudaError_t ce = cudaStreamEndCapture(cs, &g);
        p.launches = before;
        if (e || ce != cudaSuccess) {
            if (g) cudaGraphDestroy(g);
            cudaStreamDestroy(cs);
            if (!e) set_error("graph capture failed: %s", cudaGetErrorString(ce));
            return e ? e : (int)ce;
        }
        ce = cudaGraphInstantiate(&p.graph, g, 0);
        cudaGraphDestroy(g);
        cudaStreamDestroy(cs);
        if (ce != cudaSuccess) { set_error("graph instantiate failed: %s", cudaGetErrorString(ce)); p.graph = nullptr; return (int)ce; }
        p.graph_key[0] = x; p.graph_key[1] = noise; p.graph_steps = p.coef_steps; p.graph_all_full = p.all_full;
        p.graph_inpaint = p.inpaint; p.graph_start = p.start_steps;
    }
    CB2_CUDA(cudaGraphLaunch(p.graph, s));
    p.launches += 16LL * (p.start_steps > 0 ? p.start_steps : p.coef_steps) + (p.inpaint ? 1 : 0);
    return 0;
}

// Room for n_edges in csr_col / edge_w.  They grow geometrically and the replaced buffers are freed, so a long run of updates whose
// edge count fluctuates holds at most about 1.5x its largest graph.  Only the eagerly launched decode and the IC filters read these
// buffers (the captured step loop does not), so replacing them needs no graph recapture; the stream is synchronised first because
// earlier decode launches may still be reading the old ones.
static int reserve_edges(cb2_plan* h, int n_edges, cudaStream_t s) {
    if (h->csr_col && n_edges <= h->E_cap) return 0;
    const long long want = h->csr_col ? std::max<long long>(n_edges, (long long)h->E_cap + h->E_cap / 2) : n_edges;
    const int cap = (int)std::min<long long>(want, 0x7fffffff);
    if (h->csr_col) {
        CB2_CUDA(cudaStreamSynchronize(s));
        cudaFree(h->csr_col); cudaFree(h->edge_w);
        h->csr_col = nullptr; h->edge_w = nullptr; h->E_cap = 0;
    }
    const size_t n = cap > 0 ? (size_t)cap : 1;
    CB2_CUDA(cudaMalloc(&h->csr_col, n * sizeof(int)));
    CB2_CUDA(cudaMalloc(&h->edge_w, n * 4 * 40 * sizeof(float)));
    h->E_cap = cap;
    return 0;
}

int cb2_plan_set_topology(cb2_plan* h, const cb2_vae* v, const float* ca_full, const int* csr_row_ptr, const int* csr_col,
                          int n_edges, const signed char* atom_orders, const int* slot_atom, const long long* out_offset,
                          void* stream) {
    if (!h || !v || !ca_full || !csr_row_ptr || !atom_orders || !slot_atom || !out_offset) { set_error("set_topology: null argument"); return 1; }
    Plan& p = h->p;
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)p.NB * p.L, FL = (size_t)p.F * p.L;
    if (!h->ca_full) {
        int e = 0;
        e |= dev_alloc(p.allocs, &h->ca_full, (size_t)p.F * (p.L + 2) * 3);
        e |= dev_alloc(p.allocs, &h->csr_row, FL + 1);
        e |= dev_alloc(p.allocs, &h->orders, FL * 30);
        e |= dev_alloc(p.allocs, &h->slot_atom, FL * 14);
        e |= dev_alloc(p.allocs, &h->out_off, p.NB);
        e |= dev_alloc(p.allocs, &h->S40, N * 40);
        e |= dev_alloc(p.allocs, &h->phi, N * 40);
        e |= dev_alloc(p.allocs, &h->ic, N * 39);
        e |= dev_alloc(p.allocs, &h->zq, N * 3);
        e |= dev_alloc(p.allocs, &h->vq_idx, N);
        if (e) return e;
    }
    if (int e = reserve_edges(h, n_edges, s)) { h->topo_ready = false; return e; }     // no graph buffers: decode refuses
    h->E = n_edges;
    CB2_CUDA(cudaMemcpyAsync(h->ca_full, ca_full, (size_t)p.F * (p.L + 2) * 3 * sizeof(float), cudaMemcpyDeviceToDevice, s));
    CB2_CUDA(cudaMemcpyAsync(h->csr_row, csr_row_ptr, (FL + 1) * sizeof(int), cudaMemcpyDefault, s));
    if (n_edges) CB2_CUDA(cudaMemcpyAsync(h->csr_col, csr_col, (size_t)n_edges * sizeof(int), cudaMemcpyDefault, s));
    CB2_CUDA(cudaMemcpyAsync(h->orders, atom_orders, FL * 30, cudaMemcpyDefault, s));
    CB2_CUDA(cudaMemcpyAsync(h->slot_atom, slot_atom, FL * 14 * sizeof(int), cudaMemcpyDefault, s));
    CB2_CUDA(cudaMemcpyAsync(h->out_off, out_offset, p.NB * sizeof(long long), cudaMemcpyDefault, s));
    if (!h->frames_ready) { set_error("set_topology: call cb2_plan_set_frames first (needs X)"); return 1; }
    if (int e = launch_ic_edge_filters(v->v, p.X, p.F, p.L, h->csr_row, h->csr_col, n_edges, h->edge_w, s)) return e;
    p.launches += 1;
    CB2_CUDA(cudaStreamSynchronize(s));
    h->topo_ready = true;
    return 0;
}

int cb2_plan_set_coords(cb2_plan* h, const cb2_vae* v, const float* ca_full, void* stream) {
    if (!h || !v || !ca_full) { set_error("set_coords: null argument"); return 1; }
    if (!h->topo_ready) { set_error("set_coords: cb2_plan_set_topology has not been called (set_coords keeps its lengths, types and topology)"); return 1; }
    Plan& p = h->p;
    cudaStream_t s = (cudaStream_t)stream;
    const int FL = p.F * p.L;
    CB2_CUDA(cudaMemcpyAsync(h->ca_full, ca_full, (size_t)p.F * (p.L + 2) * 3 * sizeof(float), cudaMemcpyDeviceToDevice, s));
    if (int e = launch_trim_coords(h->ca_full, p.lengths, p.F, p.L, p.X, s)) return e;
    p.launches += 1;
    if (p.model) {
        if (int e = launch_knn(p.X, p.lengths, p.F, p.L, p.K, p.nbr_dist, p.nbr_idx, s)) return e;
        if (int e = launch_edge_features(*p.model, p.X, p.lengths, p.nbr_idx, p.nbr_dist, p.F, p.L, p.K, p.E_dbg, p.hE0, p.precision, s)) return e;
        p.launches += 2;
    }
    if (int e = launch_radius_rows(p.X, p.lengths, p.F, p.L, v->v.cutoff, h->csr_row, s)) return e;
    p.launches += 2;
    int n_edges = 0;
    CB2_CUDA(cudaMemcpyAsync(&n_edges, h->csr_row + FL, sizeof(int), cudaMemcpyDeviceToHost, s));
    CB2_CUDA(cudaStreamSynchronize(s));     // the edge count sizes csr_col / edge_w and the filter launch
    if (int e = reserve_edges(h, n_edges, s)) { h->topo_ready = false; return e; }     // no graph buffers: decode refuses
    h->E = n_edges;
    if (int e = launch_radius_fill(p.X, p.lengths, p.F, p.L, v->v.cutoff, h->csr_row, h->csr_col, s)) return e;
    if (int e = launch_ic_edge_filters(v->v, p.X, p.F, p.L, h->csr_row, h->csr_col, n_edges, h->edge_w, s)) return e;
    p.launches += 2;
    return 0;
}

int cb2_plan_decode(cb2_plan* h, const cb2_vae* v, const float* latent, int denorm, int* idx, float* zq, float* ic_recon,
                    float* xyz, void* stream) {
    if (!h || !v || !latent) { set_error("decode: null argument"); return 1; }
    if (!h->topo_ready) { set_error("decode: cb2_plan_set_topology has not been called"); return 1; }
    Plan& p = h->p;
    cudaStream_t s = (cudaStream_t)stream;
    const int N = p.NB * p.L;
    if (int e = launch_vq_lookup(v->v, latent, N, p.L, p.lengths, p.frame_of, denorm, h->vq_idx, h->zq, h->S40, s)) return e;
    if (int e = launch_ic_decoder(v->v, h->S40, h->phi, N, p.L, p.frame_of, p.lengths, p.cg_z, h->csr_row, h->csr_col, h->E,
                                  h->edge_w, h->ic, s, &p.launches)) return e;
    p.launches += 1;
    if (idx) CB2_CUDA(cudaMemcpyAsync(idx, h->vq_idx, (size_t)N * sizeof(int), cudaMemcpyDeviceToDevice, s));
    if (zq) CB2_CUDA(cudaMemcpyAsync(zq, h->zq, (size_t)N * 3 * sizeof(float), cudaMemcpyDeviceToDevice, s));
    if (ic_recon) CB2_CUDA(cudaMemcpyAsync(ic_recon, h->ic, (size_t)N * 39 * sizeof(float), cudaMemcpyDeviceToDevice, s));
    if (xyz) {
        if (int e = launch_ic_to_xyz(h->ca_full, h->ic, N, p.L, p.frame_of, p.lengths, h->orders, h->slot_atom, h->out_off, xyz,
                                     nullptr, s)) return e;
        p.launches += 1;
    }
    return 0;
}

int cb2_plan_residue_clashes(cb2_plan* h, const float* xyz, float threshold, int grow, int* counts, unsigned char* keep, void* stream) {
    if (!h || !xyz || !counts) { set_error("residue_clashes: null argument"); return 1; }
    if (!h->topo_ready) { set_error("residue_clashes: cb2_plan_set_topology has not been called"); return 1; }
    Plan& p = h->p;
    if (!(threshold > 0.0f) || !isfinite(threshold)) { set_error("residue_clashes: threshold must be finite and positive"); return 1; }
    if (grow < 0 || (grow > 0 && grow >= p.K)) { set_error("residue_clashes: grow=%d outside [0, K=%d)", grow, p.K); return 1; }
    if (!h->clash_bounds)
        if (int e = dev_alloc(p.allocs, &h->clash_bounds, (size_t)p.NB * p.L)) return e;
    if (int e = launch_residue_clashes(xyz, h->slot_atom, h->out_off, p.lengths, p.frame_of, p.nbr_idx, p.NB, p.L, p.K, threshold, grow,
                                       h->clash_bounds, counts, keep, (cudaStream_t)stream)) return e;
    p.launches += keep ? 3 : 2;
    return 0;
}

int cb2_plan_relax(cb2_plan* h, const float* xyz_in, float* xyz_out, float threshold, int iterations, float* max_shift,
                   float* max_restraint_dev, void* stream) {
    if (!h || !xyz_in || !xyz_out) { set_error("relax: null argument"); return 1; }
    if (!h->topo_ready) { set_error("relax: cb2_plan_set_topology has not been called"); return 1; }
    Plan& p = h->p;
    if (!(threshold > 0.0f && threshold <= 2.0f)) { set_error("relax: threshold must lie in (0, 2] A"); return 1; }
    if (iterations < 0 || iterations > 100000) { set_error("relax: iterations=%d outside [0, 100000]", iterations); return 1; }
    const size_t S = (size_t)p.NB * p.L * 14;
    if (S * 16 >= (size_t)1 << 31) { set_error("relax: NB*L=%lld is too large for the restraint lists", (long long)p.NB * p.L); return 1; }
    RelaxBufs& rb = h->relax;
    if (!rb.x0) {
        RelaxBufs nb{};
        int e = 0;
        e |= dev_alloc(p.allocs, &nb.x0, S * 3);
        e |= dev_alloc(p.allocs, &nb.xa, S * 3);
        e |= dev_alloc(p.allocs, &nb.xb, S * 3);
        e |= dev_alloc(p.allocs, &nb.partner, S * 16);
        e |= dev_alloc(p.allocs, &nb.d0, S * 16);
        e |= dev_alloc(p.allocs, &nb.cand, (size_t)p.NB * p.L * ((p.L + 31) / 32));
        e |= dev_alloc(p.allocs, &nb.grid_slot, (size_t)p.F * p.L * 14);
        e |= dev_alloc(p.allocs, &nb.grid_off, p.NB);
        e |= dev_alloc(p.allocs, &nb.nrep, S);
        if (!h->clash_bounds) e |= dev_alloc(p.allocs, &h->clash_bounds, (size_t)p.NB * p.L);
        if (e) return e;    // the plan keeps none of them (those that were allocated are freed with it)
        nb.bounds = h->clash_bounds;
        rb = nb;
    }
    return launch_relax(xyz_in, xyz_out, h->slot_atom, h->out_off, p.lengths, p.frame_of, p.F, p.NB, p.L, threshold, iterations,
                        max_shift, max_restraint_dev, rb, (cudaStream_t)stream, &p.launches);
}

int cb2_plan_buffer(cb2_plan* h, const char* name, void* dst, long long dst_bytes, void* stream) {
    if (!h || !name || !dst) { set_error("plan_buffer: null argument"); return 1; }
    void* src = nullptr;
    long long size = 0;
    void** ptr = &src;
    long long* bytes = &size;
    Plan& p = h->p;
    const size_t N = (size_t)p.NB * p.L, FE = (size_t)p.F * p.L * p.K, esz = p.precision == PREC_F16 ? 2 : 4;
    const std::string n = name;
    if (n == "nbr_idx") { *ptr = p.nbr_idx; *bytes = FE * 4; }
    else if (n == "nbr_dist") { *ptr = p.nbr_dist; *bytes = FE * 4; }
    else if (n == "E") { *ptr = p.E_dbg; *bytes = p.E_dbg ? FE * 128 * 4 : 0; }
    else if (n == "hE0") { *ptr = p.hE0; *bytes = FE * 128 * esz; }
    else if (n == "hE") { *ptr = p.hE; *bytes = N * p.K * 128 * esz; }
    else if (n == "hV") { *ptr = p.hV; *bytes = N * 128 * 4; }
    else if (n == "S") { *ptr = p.S; *bytes = N * 128 * 4; }
    else if (n == "out6") { *ptr = p.out6; *bytes = N * 6 * 4; }
    else if (n == "tc_trace") {
        if (!p.tc_trace) { unsigned long long* t = nullptr; if (dev_alloc(p.allocs, &t, 6144)) return 1; cudaMemsetAsync(t, 0, 49152, (cudaStream_t)stream); p.tc_trace = t; }
        *ptr = p.tc_trace; *bytes = 49152;
    }
    else if (n == "relax_partner") { *ptr = h->relax.partner; *bytes = N * 14 * 16 * 4; }
    else if (n == "relax_d0") { *ptr = h->relax.d0; *bytes = N * 14 * 16 * 4; }
    else if (n == "relax_nrep") { *ptr = h->relax.nrep; *bytes = N * 14 * 4; }
    else if (n == "mod") { *ptr = p.mod; *bytes = (size_t)p.mod_capacity * CB2_MOD_TOTAL * 4; }
    else { set_error("plan_buffer: unknown buffer '%s'", name); return 1; }
    if (!src || dst_bytes > size) { set_error("plan_buffer: '%s' holds %lld bytes, %lld requested", name, size, dst_bytes); return 1; }
    CB2_CUDA(cudaMemcpyAsync(dst, src, (size_t)dst_bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return 0;
}

int cb2_plan_run_edge_kernel(cb2_plan* h, int mode, int layer, void* stream) {
    if (!h || mode < 0 || mode > 2 || layer < 0 || layer > 2) { set_error("run_edge_kernel: bad argument"); return 1; }
    if (!h->frames_ready || h->p.coef_steps <= 0) { set_error("run_edge_kernel: set_frames / set_schedule first"); return 1; }
    return edge_dispatch(h->p, mode, layer, h->p.mod, 0, (cudaStream_t)stream);
}

int cb2_plan_run_stage(cb2_plan* h, const cb2_vae* v, int stage, int layer, float* xyz_scratch, void* stream) {
    if (!h || stage < 0 || stage > 9) { set_error("run_stage: bad argument"); return 1; }
    Plan& p = h->p;
    cudaStream_t s = (cudaStream_t)stream;
    if (!h->frames_ready) { set_error("run_stage: set_frames first"); return 1; }
    if (stage <= 3 && (p.coef_steps <= 0 || !p.model)) { set_error("run_stage: set_schedule first"); return 1; }
    if (stage >= 6 && (!h->topo_ready || !v)) { set_error("run_stage: set_topology first (and pass the vae)"); return 1; }
    const int N = p.NB * p.L;
    switch (stage) {
        case 0: case 1: case 2:
            if (layer < 0 || layer > 2) { set_error("run_stage: layer"); return 1; }
            return edge_dispatch(p, stage, layer, p.mod, 0, s);
        case 3: {
            if (layer < 0 || layer > 5) { set_error("run_stage: phase"); return 1; }
            const bool last = layer == 5, tc = p.precision == PREC_F16 && p.node_tc != nullptr;
            const float *xt = last ? h->xa : nullptr, *nz = last ? h->xa : nullptr, *cf = last ? p.coef : nullptr;
            float* xn = last ? h->xb : nullptr;
            return tc ? launch_node_update_tc(p, layer, p.mod, 0, xt, nz, xn, cf, nullptr, s)
                      : launch_node_update(p, layer, p.mod, 0, xt, nz, xn, cf, nullptr, s);
        }
        case 4: return launch_knn(p.X, p.lengths, p.F, p.L, p.K, p.nbr_dist, p.nbr_idx, s);
        case 5: return launch_edge_features(*p.model, p.X, p.lengths, p.nbr_idx, p.nbr_dist, p.F, p.L, p.K, p.E_dbg, p.hE0, p.precision, s);
        case 6: return launch_vq_lookup(v->v, h->xa, N, p.L, p.lengths, p.frame_of, 1, h->vq_idx, h->zq, h->S40, s);
        case 7: return launch_ic_decoder(v->v, h->S40, h->phi, N, p.L, p.frame_of, p.lengths, p.cg_z, h->csr_row, h->csr_col, h->E, h->edge_w, h->ic, s, &p.launches);
        case 8:
            if (!xyz_scratch) { set_error("run_stage: ic_to_xyz needs xyz_scratch"); return 1; }
            return launch_ic_to_xyz(h->ca_full, h->ic, N, p.L, p.frame_of, p.lengths, h->orders, h->slot_atom, h->out_off, xyz_scratch, nullptr, s);
        default: return launch_ic_edge_filters(v->v, p.X, p.F, p.L, h->csr_row, h->csr_col, h->E, h->edge_w, s);
    }
}

// ------------------------------------------------------------------------------------------- stand-alone kernels
int cb2_knn_topk(const float* X, const int* lengths, int F, int L, int K, float* D, int* idx, void* stream) {
    if (!X || !D || !idx) { set_error("knn_topk: null argument"); return 1; }
    return launch_knn(X, lengths, F, L, K, D, idx, (cudaStream_t)stream);
}

int cb2_radius_graph_rows(const float* X, const int* lengths, int F, int L, float cutoff, int* row_ptr, void* stream) {
    if (!X || !lengths || !row_ptr) { set_error("radius_graph_rows: null argument"); return 1; }
    return launch_radius_rows(X, lengths, F, L, cutoff, row_ptr, (cudaStream_t)stream);
}

int cb2_radius_graph_fill(const float* X, const int* lengths, int F, int L, float cutoff, const int* row_ptr, int* col, void* stream) {
    if (!X || !lengths || !row_ptr || !col) { set_error("radius_graph_fill: null argument"); return 1; }
    return launch_radius_fill(X, lengths, F, L, cutoff, row_ptr, col, (cudaStream_t)stream);
}

int cb2_keyed_normal(uint64_t seed, const int64_t* keys, int NB, int L, uint32_t draw, int first_slice, int n_slices, float* out,
                     void* stream) {
    if (!keys || !out) { set_error("keyed_normal: null argument"); return 1; }
    if (NB < 1 || L < 1 || L >= (1 << 21)) { set_error("keyed_normal: NB=%d must be >= 1 and L=%d in [1, 2^21)", NB, L); return 1; }
    if (first_slice < 0 || n_slices < 1 || first_slice + (long long)n_slices > 2048) {
        set_error("keyed_normal: slices [%d, %lld) must lie in [0, 2048) and hold at least one", first_slice, first_slice + (long long)n_slices);
        return 1;
    }
    return launch_keyed_normal(seed, (const long long*)keys, NB, L, draw, first_slice, n_slices, out, (cudaStream_t)stream);
}

int cb2_vq_lookup(const cb2_vae* v, const float* x, int NB, int L, const int* lengths, const int* frame_of, int denorm,
                  int* idx, float* zq, void* stream) {
    if (!v || !x || !lengths || !frame_of || !idx || !zq) { set_error("vq_lookup: null argument"); return 1; }
    return launch_vq_lookup(v->v, x, NB * L, L, lengths, frame_of, denorm, idx, zq, nullptr, (cudaStream_t)stream);
}

int cb2_p_sample(const float* x, const float* model_out, const float* noise, const float* coef, const int* step_of_member,
                 int rows_per_member, int rows, int C, float* x_next, void* stream) {
    if (!x || !model_out || !noise || !coef || !step_of_member || !x_next) { set_error("p_sample: null argument"); return 1; }
    return launch_p_sample(x, model_out, noise, coef, step_of_member, rows_per_member, rows, C, x_next, (cudaStream_t)stream);
}

int cb2_ddim_sample(const float* x, const float* model_out, const float* noise, const float* coef, const int* step_of_member,
                    int rows_per_member, int rows, int C, float* x_next, void* stream) {
    if (!x || !model_out || !coef || !step_of_member || !x_next) { set_error("ddim_sample: null argument"); return 1; }
    return launch_ddim_sample(x, model_out, noise, coef, step_of_member, rows_per_member, rows, C, x_next, (cudaStream_t)stream);
}

int cb2_ic_to_xyz(const float* ca_full, const float* ic_recon, int NB, int L, const int* frame_of, const int* lengths,
                  const signed char* atom_orders, const int* slot_atom, const long long* out_offset, float* xyz, void* stream) {
    if (!ca_full || !ic_recon || !frame_of || !lengths || !atom_orders || !slot_atom || !out_offset || !xyz) {
        set_error("ic_to_xyz: null argument");
        return 1;
    }
    return launch_ic_to_xyz(ca_full, ic_recon, NB * L, L, frame_of, lengths, atom_orders, slot_atom, out_offset, xyz, nullptr,
                            (cudaStream_t)stream);
}

}  // extern "C"
