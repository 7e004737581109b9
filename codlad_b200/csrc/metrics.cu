// Sample-quality metrics of the evaluation step that follows the sampling path (SURVEY.md section 8f-4; reference
// utils/protein_module.py:245-364, test.py:168-188): bond-graph validity of a generated all-atom structure against its
// reference structure, and RMSD.  The reference builds two dense [Na, Na] distance matrices per structure on the CPU; here one
// kernel walks the pairs once, never materialises a matrix and returns six integer counts per structure.
//
// bond(i, j) = i != j and ||x_i - x_j|| < (r[z_i] + r[z_j]) * scale          (fp32, same operation order as the reference)
// counts per structure: {differing entries, reference bonds, generated bonds} over all atoms and over heavy atoms only
// (z != 1; dropping hydrogens from both structures = restricting the pairs to heavy-heavy ones).  Entries are counted over the
// full symmetric matrix, like `(bonds != ref_bonds).sum()` does.
#include "../../include/codlad_b200.h"
#include "common.cuh"
#include "pair_dist.cuh"

namespace cb2 {

namespace {

constexpr int MT_ROWS = 128;        // rows (atoms i) per CTA = threads per CTA
constexpr int MT_COLS = 256;        // atoms j staged per shared-memory tile

__global__ void __launch_bounds__(MT_ROWS) bond_graph_kernel(const float* __restrict__ xyz_ref, const float* __restrict__ xyz_gen,
                                                             const int* __restrict__ z, const long long* __restrict__ offsets,
                                                             const float* __restrict__ radius, int max_z, float scale,
                                                             unsigned long long* __restrict__ counts) {
    __shared__ float sR[MT_COLS][3], sG[MT_COLS][3], sRad[MT_COLS];
    __shared__ int sHeavy[MT_COLS];
    const int s = blockIdx.y;                                  // grid = (blocks of MT_ROWS atoms of the largest structure, structures)
    const long long base = offsets[s];
    const int na = (int)(offsets[s + 1] - base);
    if ((int)blockIdx.x * MT_ROWS >= na) return;               // smaller structure: nothing in this row block
    const int i = blockIdx.x * MT_ROWS + threadIdx.x;
    const bool live = i < na;
    float ri[3] = {0.f, 0.f, 0.f}, gi[3] = {0.f, 0.f, 0.f}, rad_i = 0.f;
    bool heavy_i = false;
    if (live) {
        for (int d = 0; d < 3; ++d) { ri[d] = xyz_ref[(base + i) * 3 + d]; gi[d] = xyz_gen[(base + i) * 3 + d]; }
        const int zi = z[base + i];
        rad_i = radius[min(max(zi, 0), max_z)];
        heavy_i = zi != 1;
    }
    unsigned int c[6] = {0u, 0u, 0u, 0u, 0u, 0u};        // diff, ref, gen (all atoms) | diff, ref, gen (heavy only)
    for (int j0 = 0; j0 < na; j0 += MT_COLS) {
        __syncthreads();
        for (int t = threadIdx.x; t < MT_COLS; t += MT_ROWS) {
            const int j = j0 + t;
            if (j < na) {
                for (int d = 0; d < 3; ++d) { sR[t][d] = xyz_ref[(base + j) * 3 + d]; sG[t][d] = xyz_gen[(base + j) * 3 + d]; }
                const int zj = z[base + j];
                sRad[t] = radius[min(max(zj, 0), max_z)];
                sHeavy[t] = zj != 1;
            }
        }
        __syncthreads();
        if (!live) continue;
        const int nj = min(MT_COLS, na - j0);
        for (int t = 0; t < nj; ++t) {
            if (j0 + t == i) continue;
            // (x_i - x_j).pow(2).sum(-1).sqrt() < (r_i + r_j) * scale, no fused multiply-add (the reference rounds every operation)
            const float cut = __fmul_rn(__fadd_rn(rad_i, sRad[t]), scale);
            float dr[3], dg[3];
            for (int d = 0; d < 3; ++d) { dr[d] = __fsub_rn(ri[d], sR[t][d]); dg[d] = __fsub_rn(gi[d], sG[t][d]); }
            const float d2r = __fadd_rn(__fadd_rn(__fmul_rn(dr[0], dr[0]), __fmul_rn(dr[1], dr[1])), __fmul_rn(dr[2], dr[2]));
            const float d2g = __fadd_rn(__fadd_rn(__fmul_rn(dg[0], dg[0]), __fmul_rn(dg[1], dg[1])), __fmul_rn(dg[2], dg[2]));
            const bool br = __fsqrt_rn(d2r) < cut, bg = __fsqrt_rn(d2g) < cut;
            const unsigned int hv = (heavy_i && sHeavy[t]) ? 1u : 0u;
            c[0] += br != bg; c[1] += br; c[2] += bg;
            c[3] += hv & (unsigned int)(br != bg); c[4] += hv & (unsigned int)br; c[5] += hv & (unsigned int)bg;
        }
    }
    // CTA reduction: warp shuffles, then one atomic per warp and counter (integer adds: order does not matter)
    for (int k = 0; k < 6; ++k) {
        unsigned int v = c[k];
        for (int off = 16; off >= 1; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
        if ((threadIdx.x & 31) == 0 && v) atomicAdd(counts + (size_t)s * 6 + k, (unsigned long long)v);
    }
}

// per structure: sum over atoms of ||x_gen - x_ref||^2 (all atoms, heavy atoms) in double, and the atom counts
__global__ void __launch_bounds__(256) rmsd_sums_kernel(const float* __restrict__ xyz_ref, const float* __restrict__ xyz_gen, const int* __restrict__ z,
                                                        const long long* __restrict__ offsets, double* __restrict__ out) {
    const int s = blockIdx.x;
    const long long base = offsets[s];
    const int na = (int)(offsets[s + 1] - base);
    double sa = 0.0, sh = 0.0, nh = 0.0;
    for (int i = threadIdx.x; i < na; i += blockDim.x) {
        double d2 = 0.0;
        for (int d = 0; d < 3; ++d) { const double t = (double)xyz_gen[(base + i) * 3 + d] - (double)xyz_ref[(base + i) * 3 + d]; d2 += t * t; }
        sa += d2;
        if (z[base + i] != 1) { sh += d2; nh += 1.0; }
    }
    __shared__ double red[3][8];
    double v[3] = {sa, sh, nh};
    for (int k = 0; k < 3; ++k) {
        for (int off = 16; off >= 1; off >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], off);
        if ((threadIdx.x & 31) == 0) red[k][threadIdx.x >> 5] = v[k];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double t[3] = {0.0, 0.0, 0.0};
        for (int k = 0; k < 3; ++k) for (int w = 0; w < 8; ++w) t[k] += red[k][w];      // fixed order
        out[s * 4 + 0] = t[0]; out[s * 4 + 1] = (double)na; out[s * 4 + 2] = t[1]; out[s * 4 + 3] = t[2];
    }
}

// Minimum RMSD under rigid superposition (what md.rmsd computes for the diversity score, test.py:37-96), per structure pair: the
// 17 sums (centroids, inner products G_a / G_b, 3x3 cross-covariance) are accumulated in double over the atoms, then one thread takes
// the largest eigenvalue of Horn's 4x4 key matrix with cyclic Jacobi rotations: rmsd^2 = (G_a + G_b - 2 lambda_max) / N.
__global__ void __launch_bounds__(256) superposed_rmsd_kernel(const float* __restrict__ A, const float* __restrict__ B, const long long* __restrict__ offsets,
                                                              double* __restrict__ out) {
    const int s = blockIdx.x;
    const long long base = offsets[s];
    const int na = (int)(offsets[s + 1] - base);
    double acc[17];
    for (int k = 0; k < 17; ++k) acc[k] = 0.0;
    for (int i = threadIdx.x; i < na; i += blockDim.x) {
        double a[3], b[3];
        for (int d = 0; d < 3; ++d) { a[d] = (double)A[(base + i) * 3 + d]; b[d] = (double)B[(base + i) * 3 + d]; }
        for (int d = 0; d < 3; ++d) { acc[d] += a[d]; acc[3 + d] += b[d]; acc[6] += a[d] * a[d]; acc[7] += b[d] * b[d]; }
        for (int p = 0; p < 3; ++p) for (int q = 0; q < 3; ++q) acc[8 + 3 * p + q] += a[p] * b[q];
    }
    __shared__ double red[17][8];
    for (int k = 0; k < 17; ++k) {
        double v = acc[k];
        for (int off = 16; off >= 1; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
        if ((threadIdx.x & 31) == 0) red[k][threadIdx.x >> 5] = v;
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    double t[17];
    for (int k = 0; k < 17; ++k) { t[k] = 0.0; for (int w = 0; w < 8; ++w) t[k] += red[k][w]; }       // fixed order
    if (na == 0) { out[s] = 0.0; return; }
    const double n = (double)na;
    double S[3][3];
    for (int p = 0; p < 3; ++p) for (int q = 0; q < 3; ++q) S[p][q] = t[8 + 3 * p + q] - t[p] * t[3 + q] / n;
    const double Ga = t[6] - (t[0] * t[0] + t[1] * t[1] + t[2] * t[2]) / n, Gb = t[7] - (t[3] * t[3] + t[4] * t[4] + t[5] * t[5]) / n;
    double K[4][4] = {
        {S[0][0] + S[1][1] + S[2][2], S[1][2] - S[2][1], S[2][0] - S[0][2], S[0][1] - S[1][0]},
        {S[1][2] - S[2][1], S[0][0] - S[1][1] - S[2][2], S[0][1] + S[1][0], S[2][0] + S[0][2]},
        {S[2][0] - S[0][2], S[0][1] + S[1][0], -S[0][0] + S[1][1] - S[2][2], S[1][2] + S[2][1]},
        {S[0][1] - S[1][0], S[2][0] + S[0][2], S[1][2] + S[2][1], -S[0][0] - S[1][1] + S[2][2]}};
    for (int sweep = 0; sweep < 30; ++sweep) {
        double off = 0.0;
        for (int p = 0; p < 4; ++p) for (int q = p + 1; q < 4; ++q) off += K[p][q] * K[p][q];
        if (off < 1e-30 * (Ga + Gb + 1e-300) * (Ga + Gb + 1e-300)) break;
        for (int p = 0; p < 4; ++p)
            for (int q = p + 1; q < 4; ++q) {
                if (K[p][q] == 0.0) continue;
                const double theta = (K[q][q] - K[p][p]) / (2.0 * K[p][q]);
                const double tt = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                const double c = 1.0 / sqrt(tt * tt + 1.0), sn = tt * c;
                for (int k = 0; k < 4; ++k) { const double kp = K[k][p], kq = K[k][q]; K[k][p] = c * kp - sn * kq; K[k][q] = sn * kp + c * kq; }
                for (int k = 0; k < 4; ++k) { const double pk = K[p][k], qk = K[q][k]; K[p][k] = c * pk - sn * qk; K[q][k] = sn * pk + c * qk; }
            }
    }
    const double lam = fmax(fmax(K[0][0], K[1][1]), fmax(K[2][2], K[3][3]));
    out[s] = sqrt(fmax(0.0, (Ga + Gb - 2.0 * lam) / n));
}


// Pair-list losses of the evaluation step (test.py:97-146: inter_result, clash_result, ged_result).  One row of `idx` is either a pair
// (a, b): d = sqrt(|x_a - x_b|^2 + EPS), or a quad (a, b, c, e): d = distance of the ring centres (x_a + x_b)/2 and (x_c + x_e)/2
// (pi-pi stacking).  Per row: [d < thr_count], max(d - thr_hinge, 0), (d - d_data)^2 with d_data the same distance in `xyz_data`.
// fp32 distances in the reference's operation order; the three sums are accumulated in double, per CTA and then over CTAs in a
// fixed order (deterministic).
constexpr int PL_THREADS = 256, PL_MAX_BLOCKS = 592;

__device__ __forceinline__ float pair_dist(const float* __restrict__ x, const long long* __restrict__ row, int width) {
    if (width == 2) return atom_pair_dist(x + row[0] * 3, x + row[1] * 3);      // pair_dist.cuh, shared with the clash counts
    float d2 = 0.f;
    const float *a = x + row[0] * 3, *b = x + row[1] * 3, *c = x + row[2] * 3, *e = x + row[3] * 3;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float d = __fsub_rn(__fdiv_rn(__fadd_rn(a[k], b[k]), 2.f), __fdiv_rn(__fadd_rn(c[k], e[k]), 2.f));
        d2 = __fadd_rn(d2, __fmul_rn(d, d));
    }
    return __fsqrt_rn(__fadd_rn(d2, PAIR_EPS));
}

__global__ void __launch_bounds__(PL_THREADS) pair_losses_kernel(const float* __restrict__ xyz, const float* __restrict__ xyz_data,
                                                                 const long long* __restrict__ idx, int width, long long P, float thr_count,
                                                                 float thr_hinge, double* __restrict__ part) {
    double acc[3] = {0.0, 0.0, 0.0};
    for (long long r = (long long)blockIdx.x * PL_THREADS + threadIdx.x; r < P; r += (long long)gridDim.x * PL_THREADS) {
        const long long* row = idx + r * width;
        const float d = pair_dist(xyz, row, width);
        acc[0] += d < thr_count ? 1.0 : 0.0;
        acc[1] += (double)fmaxf(__fsub_rn(d, thr_hinge), 0.f);
        if (xyz_data != nullptr) { const float e = __fsub_rn(d, pair_dist(xyz_data, row, width)); acc[2] += (double)__fmul_rn(e, e); }
    }
    __shared__ double red[3][PL_THREADS / 32];
    for (int k = 0; k < 3; ++k) {
        double v = acc[k];
        for (int off = 16; off >= 1; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
        if ((threadIdx.x & 31) == 0) red[k][threadIdx.x >> 5] = v;
    }
    __syncthreads();
    if (threadIdx.x < 3) {
        double t = 0.0;
        for (int w = 0; w < PL_THREADS / 32; ++w) t += red[threadIdx.x][w];
        part[blockIdx.x * 3 + threadIdx.x] = t;
    }
}

__global__ void pair_losses_reduce_kernel(const double* __restrict__ part, int blocks, long long P, double* __restrict__ out) {
    if (threadIdx.x < 3) {
        double t = 0.0;
        for (int b = 0; b < blocks; ++b) t += part[b * 3 + threadIdx.x];
        out[threadIdx.x] = t;
    }
    if (threadIdx.x == 3) out[3] = (double)P;
}

// rows of a SORTED key list that occur exactly once (the `uniques[counts == 1]` of clash_result, test.py:121-123)
__global__ void keys_once_kernel(const long long* __restrict__ keys, long long n, unsigned char* __restrict__ once) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long k = keys[i];
    once[i] = ((i == 0 || keys[i - 1] != k) && (i + 1 == n || keys[i + 1] != k)) ? 1 : 0;
}

double* g_pl_part = nullptr;

}  // namespace

}  // namespace cb2

extern "C" int cb2_superposed_rmsd(const float* A, const float* B, const long long* offsets, int n_struct, double* out, void* stream) {
    using namespace cb2;
    if (!A || !B || !offsets || !out || n_struct < 0) { set_error("superposed_rmsd: bad argument"); return 1; }
    if (n_struct == 0) return 0;
    superposed_rmsd_kernel<<<n_struct, 256, 0, (cudaStream_t)stream>>>(A, B, offsets, out);
    CB2_LAUNCH_CHECK();
    return 0;
}

extern "C" int cb2_eval_bond_graphs(const float* xyz_ref, const float* xyz_gen, const int* atomic_num, const long long* offsets, int n_struct,
                                    int max_atoms, const float* cov_radius, int max_z, float scale, long long* counts, double* sums, void* stream) {
    using namespace cb2;
    if (!xyz_ref || !xyz_gen || !atomic_num || !offsets || !cov_radius || !counts || !sums || n_struct < 0 || max_atoms < 0 || max_z < 1) {
        set_error("eval_bond_graphs: bad argument");
        return 1;
    }
    cudaStream_t s = (cudaStream_t)stream;
    if (n_struct > 65535) { set_error("eval_bond_graphs: at most 65535 structures per call"); return 1; }
    CB2_CUDA(cudaMemsetAsync(counts, 0, (size_t)n_struct * 6 * sizeof(long long), s));
    if (n_struct == 0) return 0;
    if (max_atoms > 0) {
        bond_graph_kernel<<<dim3((max_atoms + MT_ROWS - 1) / MT_ROWS, n_struct), MT_ROWS, 0, s>>>(xyz_ref, xyz_gen, atomic_num, offsets, cov_radius, max_z, scale,
                                                                                                   reinterpret_cast<unsigned long long*>(counts));
        CB2_LAUNCH_CHECK();
    }
    rmsd_sums_kernel<<<n_struct, 256, 0, s>>>(xyz_ref, xyz_gen, atomic_num, offsets, sums);
    CB2_LAUNCH_CHECK();
    return 0;
}

extern "C" int cb2_pair_losses(const float* xyz, const float* xyz_data, const long long* idx, int width, long long n_rows, float thr_count,
                               float thr_hinge, double* out4, void* stream) {
    using namespace cb2;
    if (!xyz || !out4 || (n_rows > 0 && !idx) || (width != 2 && width != 4) || n_rows < 0) { set_error("pair_losses: bad argument"); return 1; }
    cudaStream_t s = (cudaStream_t)stream;
    if (!g_pl_part) CB2_CUDA(cudaMalloc(&g_pl_part, (size_t)PL_MAX_BLOCKS * 3 * sizeof(double)));
    int blocks = (int)((n_rows + PL_THREADS - 1) / PL_THREADS);
    blocks = blocks < 1 ? 1 : (blocks > PL_MAX_BLOCKS ? PL_MAX_BLOCKS : blocks);
    pair_losses_kernel<<<blocks, PL_THREADS, 0, s>>>(xyz, xyz_data, idx, width, n_rows, thr_count, thr_hinge, g_pl_part);
    CB2_LAUNCH_CHECK();
    pair_losses_reduce_kernel<<<1, 32, 0, s>>>(g_pl_part, blocks, n_rows, out4);
    CB2_LAUNCH_CHECK();
    return 0;
}

extern "C" int cb2_keys_once(const long long* sorted_keys, long long n, unsigned char* once, void* stream) {
    using namespace cb2;
    if (n < 0 || (n > 0 && (!sorted_keys || !once))) { set_error("keys_once: bad argument"); return 1; }
    if (n == 0) return 0;
    keys_once_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(sorted_keys, n, once);
    CB2_LAUNCH_CHECK();
    return 0;
}
