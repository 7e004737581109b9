// Restrained clash relaxation of a decoded sample (cb2_plan_relax; Backmapper.relax drives it).  Not in the reference: the short
// restrained minimisation that backmapping pipelines finish with, on the heavy atoms the decoder places, per member.
//
// Objective, for member b with input coordinates x0 (present atoms of real residues only):
//   restraints R_b, built once per call and held at their input distance d0:
//     every intra-residue pair with d0 <= R_RESTRAIN (3 A: the 1-2 and 1-3 pairs, S-C-C included, and ring closures; torsions
//     whose 1-4 distance is longer stay free, so side chains can rotate away from a clash), and the peptide pairs C(i)-N(i+1),
//     CA(i)-N(i+1), O(i)-N(i+1), C(i)-CA(i+1) at any distance;
//   repulsion: every pair (p in residue i, q in residue j != i) that is not a peptide pair and has d < c = threshold + RELAX_MARGIN,
//     i.e. the pair set of cb2_plan_residue_clashes minus the restrained peptide pairs, evaluated at every iteration;
//   E = sum_R K_S (d - d0)^2 + sum_rep K_R (c - d)^2, d = atom_pair_dist (the clash criterion's fp32 distance).
// Update: Jacobi steepest descent with a cap.  Every atom but the C-alphas (slot 3, the coarse-grained trace, never moved) and
// non-finite atoms takes dx = ALPHA F(x_t), scaled to MAX_STEP where longer; forces are read from x_t and x_{t+1} is written to
// the other buffer.  An atom sums its own terms, restraints in list order, then repulsion in (residue, slot) order: no atomics.
// Pairs with a non-finite atom are skipped.  A fixed number of iterations, with no early exit and no host synchronisation.
// A member with no pair closer than c has zero force everywhere (each restraint sits at its d0, computed by the same fp32 code),
// so it comes back bit for bit; a member's result depends on its own atoms alone, whatever the batch or padded length.
//
// Positions live in a slot grid: member b's slot t of residue i is row (b*L + i)*14 + t, absent slots hold NaN (so a pair with
// one never counts).  residue_bounds_kernel (repair.cu) reads the grid through grid_slot / grid_off, tables that map every
// present slot to its own row.
//
// Launches: relax_load_kernel (grid tables, input gather), relax_restraint_kernel (the per-atom restraint lists: at most 13
// intra-residue partners and 3 peptide partners, for N, whose peptide partners are O, C and CA of the residue before; C-alpha and
// C have 1 + 13 + 1 and 13 + 2, O 13 + 1, so RCAP = 16 holds every list), then per iteration relax_step_kernel, preceded every
// REBUILD iterations by the residue bounds and relax_candidates_kernel; finally relax_finish_kernel.
//
// Candidate residues (a Verlet list over residues, one bit per residue pair, written without atomics or a scan): j is a candidate
// of i when |c_i - c_j| <= (r_i + r_j + c + SKIN) * BOUND_SLACK for the bounds at the rebuild.  A step moves an atom by at most
// MAX_STEP (1 + 2^-22) plus the rounding of x + dx, below MAX_STEP + STEP_PAD for coordinates under 10^4 A, so in the REBUILD
// iterations until the next rebuild two atoms approach by at most SKIN = 2 REBUILD (MAX_STEP + STEP_PAD); every pair closer than c
// in that time is therefore in the list, and the pairs evaluated equal a brute-force pass.  The step kernel also skips a candidate
// residue whose sphere at the rebuild, grown by c + SKIN / 2, does not hold the atom: its atoms have moved by at most SKIN / 2.
// A bitmask needs no size read back, so the whole call can be captured in a graph; it takes NB * L * ceil(L/32) words, less than
// one edge-state row of the plan.
#include "../../include/codlad_b200.h"
#include "common.cuh"
#include "pair_dist.cuh"
#include "repair.h"

namespace cb2 {

namespace {

constexpr int SLOTS = 14, SLOT_O = 0, SLOT_N = 1, SLOT_C = 2, SLOT_CA = 3, RCAP = 16;
constexpr float R_RESTRAIN = 3.0f;          // A: intra-residue pairs restrained
constexpr float RELAX_MARGIN = 0.2f;        // A: c = threshold + RELAX_MARGIN
constexpr float K_S = 1.0f, K_R = 10.0f;    // A^-2: restraint and repulsion weights
constexpr float ALPHA = 0.05f;              // A^2: step per unit force
constexpr float MAX_STEP = 0.1f;            // A: cap on one step of one atom
constexpr int REBUILD = 5;                  // iterations between candidate rebuilds
constexpr float STEP_PAD = 0.005f;
constexpr float SKIN = 2.0f * REBUILD * (MAX_STEP + STEP_PAD);
constexpr float BOUND_SLACK = 1.0f + 1e-5f;

// (slot a of residue i, slot b of residue i + 1) is one of the four restrained peptide pairs
__device__ __forceinline__ bool peptide(int a, int b) {
    return (b == SLOT_N && (a == SLOT_C || a == SLOT_CA || a == SLOT_O)) || (a == SLOT_C && b == SLOT_CA);
}

// (r + c + SKIN / 2)^2 with the slack, the squared reach of the atom-sphere test of relax_step_kernel
__device__ __forceinline__ float reach2(float r, float c) { const float q = (r + c + 0.5f * SKIN) * BOUND_SLACK; return q * q; }

__device__ __forceinline__ bool finite3(const float* p) { return isfinite(p[0]) && isfinite(p[1]) && isfinite(p[2]); }

__global__ void __launch_bounds__(128) relax_load_kernel(const float* __restrict__ xyz, const int* __restrict__ slot_atom,
                                                         const long long* __restrict__ out_off, const int* __restrict__ lengths,
                                                         const int* __restrict__ frame_of, int F, int NB, int L,
                                                         int* __restrict__ grid_slot, long long* __restrict__ grid_off,
                                                         float* __restrict__ x0, float* __restrict__ xa) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    const int LS = L * SLOTS;
    if (n < F * LS) {
        const int f = n / LS, r = n - f * LS;
        grid_slot[n] = (r / SLOTS < lengths[f] && slot_atom[n] >= 0) ? r : -1;
    }
    if (n < NB) grid_off[n] = (long long)n * LS;
    if (n < NB * LS) {
        const int b = n / LS, r = n - b * LS, f = frame_of[b];
        const int at = r / SLOTS < lengths[f] ? slot_atom[(size_t)f * LS + r] : -1;
        for (int k = 0; k < 3; ++k) {
            const float v = at >= 0 ? xyz[(out_off[b] + at) * 3 + k] : __int_as_float(0x7fc00000);
            x0[(size_t)n * 3 + k] = v;
            xa[(size_t)n * 3 + k] = v;
        }
    }
}

__global__ void __launch_bounds__(128) relax_restraint_kernel(const float* __restrict__ x0, const int* __restrict__ grid_slot,
                                                              const int* __restrict__ lengths, const int* __restrict__ frame_of,
                                                              int NB, int L, int* __restrict__ partner, float* __restrict__ d0) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    const int LS = L * SLOTS;
    if (n >= NB * LS) return;
    const int b = n / LS, r = n - b * LS, i = r / SLOTS, t = r - i * SLOTS, f = frame_of[b], len = lengths[f];
    const int* gs = grid_slot + (size_t)f * LS;
    const float* x = x0 + (size_t)b * LS * 3;
    int* pn = partner + (size_t)n * RCAP;
    float* dn = d0 + (size_t)n * RCAP;
    int k = 0;
    if (gs[r] >= 0) {
        const float* p = x + (size_t)r * 3;
        auto add = [&](int q, bool pep) {
            if (gs[q] < 0) return;
            const float d = atom_pair_dist(p, x + (size_t)q * 3);
            if (!isfinite(d) || !(pep || d <= R_RESTRAIN)) return;
            pn[k] = q; dn[k] = d; ++k;
        };
        if (i > 0)
            for (int u = 0; u < SLOTS; ++u) if (peptide(u, t)) add(r - SLOTS - t + u, true);
        for (int u = 0; u < SLOTS; ++u) if (u != t) add(r - t + u, false);
        if (i + 1 < len)
            for (int u = 0; u < SLOTS; ++u) if (peptide(t, u)) add(r + SLOTS - t + u, true);
    }
    for (; k < RCAP; ++k) { pn[k] = -1; dn[k] = 0.f; }
}

__global__ void __launch_bounds__(128) relax_candidates_kernel(const float4* __restrict__ bounds, const int* __restrict__ lengths,
                                                               const int* __restrict__ frame_of, int NB, int L, int W, float reach,
                                                               unsigned int* __restrict__ cand) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= NB * L * W) return;
    const int row = n / W, w = n - row * W, b = row / L, i = row - b * L, len = lengths[frame_of[b]];
    const float4 bi = bounds[row];
    unsigned int mask = 0u;
    if (i < len && bi.w >= 0.f) {
        const float ci[3] = {bi.x, bi.y, bi.z};
        for (int jj = 0; jj < 32; ++jj) {
            const int j = w * 32 + jj;
            if (j >= len) break;
            const float4 bj = bounds[(size_t)b * L + j];
            if (j == i || !(bj.w >= 0.f)) continue;
            const float cj[3] = {bj.x, bj.y, bj.z};
            // atom_pair_dist exceeds the centre distance by at most 1.6e-4 A, well inside SKIN's pad
            if (!(atom_pair_dist(ci, cj) > (bi.w + bj.w + reach) * BOUND_SLACK)) mask |= 1u << jj;
        }
    }
    cand[n] = mask;
}

// launched with 128 threads; ptxas keeps it at 40 registers with a spill under __launch_bounds__(128), 47 and none under this cap
__global__ void __maxnreg__(64) relax_step_kernel(const float* __restrict__ cur, const int* __restrict__ partner,
                                                         const float* __restrict__ d0, const unsigned int* __restrict__ cand,
                                                         const float4* __restrict__ bounds, const int* __restrict__ lengths, const int* __restrict__ frame_of, int NB,
                                                         int L, int W, float c, float* __restrict__ nxt, int* __restrict__ nrep) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    const int LS = L * SLOTS;
    if (n >= NB * LS) return;
    const int b = n / LS, r = n - b * LS, i = r / SLOTS, t = r - i * SLOTS;
    const float p[3] = {cur[(size_t)n * 3], cur[(size_t)n * 3 + 1], cur[(size_t)n * 3 + 2]};
    float* out = nxt + (size_t)n * 3;
    // absent slots and padded residues (NaN), the fixed C-alphas and non-finite atoms keep their position
    if (i >= lengths[frame_of[b]] || t == SLOT_CA || !finite3(p)) {
        out[0] = p[0]; out[1] = p[1]; out[2] = p[2];
        nrep[n] = 0;
        return;
    }
    const float* x = cur + (size_t)b * LS * 3;
    float f[3] = {0.f, 0.f, 0.f};
    const int* pn = partner + (size_t)n * RCAP;
    const float* dn = d0 + (size_t)n * RCAP;
    for (int k = 0; k < RCAP; ++k) {
        const int q = pn[k];
        if (q < 0) break;
        const float* xq = x + (size_t)q * 3;
        if (!finite3(xq)) continue;
        const float d = atom_pair_dist(p, xq);
        const float g = -2.f * K_S * (d - dn[k]) / d;
#pragma unroll
        for (int a = 0; a < 3; ++a) f[a] += g * (p[a] - xq[a]);
    }
    int cnt = 0;
    const unsigned int* cw = cand + ((size_t)b * L + i) * W;
    const float4* bb = bounds + (size_t)b * L;
    for (int w = 0; w < W; ++w) {
        for (unsigned int m = cw[w]; m != 0u; m &= m - 1u) {
            const int j = w * 32 + __ffs(m) - 1;
            // an atom of j within c of p is within r_j + SKIN / 2 of j's centre at the rebuild, so p is within r_j + c + SKIN / 2
            const float4 bj = bb[j];
            const float ex = p[0] - bj.x, ey = p[1] - bj.y, ez = p[2] - bj.z;
            if (ex * ex + ey * ey + ez * ez > reach2(bj.w, c)) continue;
#pragma unroll 1
            for (int u = 0; u < SLOTS; ++u) {
                if ((j == i + 1 && peptide(t, u)) || (j == i - 1 && peptide(u, t))) continue;
                const float* xq = x + ((size_t)j * SLOTS + u) * 3;
                const float d = atom_pair_dist(p, xq);      // NaN for absent slots and non-finite atoms: not < c
                if (d < c) {
                    ++cnt;
                    const float g = 2.f * K_R * (c - d) / d;
            #pragma unroll
        for (int a = 0; a < 3; ++a) f[a] += g * (p[a] - xq[a]);
                }
            }
        }
    }
    nrep[n] = cnt;
    if (f[0] == 0.f && f[1] == 0.f && f[2] == 0.f) {            // at rest: the position bit for bit
        out[0] = p[0]; out[1] = p[1]; out[2] = p[2];
        return;
    }
    float dx[3] = {ALPHA * f[0], ALPHA * f[1], ALPHA * f[2]};
    const float len = sqrtf(dx[0] * dx[0] + dx[1] * dx[1] + dx[2] * dx[2]);
    if (len > MAX_STEP) {
        const float s = MAX_STEP / len;
        for (int a = 0; a < 3; ++a) dx[a] *= s;
    }
    for (int a = 0; a < 3; ++a) out[a] = p[a] + dx[a];
}

// One block per member: the output rows, and the member's largest shift and restraint deviation (max is exact, so the
// block's reduction order does not matter).
constexpr int FIN_THREADS = 256;

__global__ void __launch_bounds__(FIN_THREADS) relax_finish_kernel(const float* __restrict__ cur, const float* __restrict__ x0,
                                                                   const int* __restrict__ partner, const float* __restrict__ d0,
                                                                   const int* __restrict__ slot_atom, const long long* __restrict__ out_off,
                                                                   const int* __restrict__ lengths, const int* __restrict__ frame_of,
                                                                   int L, float* __restrict__ xyz_out, float* __restrict__ max_shift,
                                                                   float* __restrict__ max_dev) {
    __shared__ float red[2][FIN_THREADS / 32];
    const int b = blockIdx.x, f = frame_of[b], LS = L * SLOTS, len = lengths[f];
    const float* x = cur + (size_t)b * LS * 3;
    float shift = 0.f, dev = 0.f;
    for (int r = threadIdx.x; r < len * SLOTS; r += FIN_THREADS) {
        const int at = slot_atom[(size_t)f * LS + r];
        if (at < 0) continue;
        const float* p = x + (size_t)r * 3;
        const float* p0 = x0 + ((size_t)b * LS + r) * 3;
        float* o = xyz_out + (out_off[b] + at) * 3;
        o[0] = p[0]; o[1] = p[1]; o[2] = p[2];
        const float sx = p[0] - p0[0], sy = p[1] - p0[1], sz = p[2] - p0[2];
        shift = fmaxf(shift, sqrtf(sx * sx + sy * sy + sz * sz));     // fmaxf drops the NaN of a non-finite atom
        const int* pn = partner + ((size_t)b * LS + r) * RCAP;
        const float* dn = d0 + ((size_t)b * LS + r) * RCAP;
        for (int k = 0; k < RCAP && pn[k] >= 0; ++k) dev = fmaxf(dev, fabsf(atom_pair_dist(p, x + (size_t)pn[k] * 3) - dn[k]));
    }
    for (int o = 16; o > 0; o >>= 1) {
        shift = fmaxf(shift, __shfl_xor_sync(0xffffffffu, shift, o));
        dev = fmaxf(dev, __shfl_xor_sync(0xffffffffu, dev, o));
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { red[0][warp] = shift; red[1][warp] = dev; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < FIN_THREADS / 32; ++w) { shift = fmaxf(shift, red[0][w]); dev = fmaxf(dev, red[1][w]); }
        if (max_shift) max_shift[b] = shift;
        if (max_dev) max_dev[b] = dev;
    }
}

}  // namespace

int launch_relax(const float* xyz_in, float* xyz_out, const int* slot_atom, const long long* out_off, const int* lengths,
                 const int* frame_of, int F, int NB, int L, float threshold, int iterations, float* max_shift, float* max_dev,
                 const RelaxBufs& rb, cudaStream_t s, long long* launches) {
    const int S = NB * L * SLOTS, W = (L + 31) / 32;
    const float c = threshold + RELAX_MARGIN;
    const int n_load = (F > NB ? F : NB) * L * SLOTS;
    relax_load_kernel<<<(n_load + 127) / 128, 128, 0, s>>>(xyz_in, slot_atom, out_off, lengths, frame_of, F, NB, L, rb.grid_slot,
                                                           rb.grid_off, rb.x0, rb.xa);
    CB2_LAUNCH_CHECK();
    relax_restraint_kernel<<<(S + 127) / 128, 128, 0, s>>>(rb.x0, rb.grid_slot, lengths, frame_of, NB, L, rb.partner, rb.d0);
    CB2_LAUNCH_CHECK();
    *launches += 2;
    float *cur = rb.xa, *nxt = rb.xb;
    for (int it = 0; it < iterations; ++it) {
        if (it % REBUILD == 0) {
            if (int e = launch_residue_bounds(cur, rb.grid_slot, rb.grid_off, lengths, frame_of, NB, L, rb.bounds, s)) return e;
            const int nc = NB * L * W;
            relax_candidates_kernel<<<(nc + 127) / 128, 128, 0, s>>>(rb.bounds, lengths, frame_of, NB, L, W, c + SKIN, rb.cand);
            CB2_LAUNCH_CHECK();
            *launches += 2;
        }
        relax_step_kernel<<<(S + 127) / 128, 128, 0, s>>>(cur, rb.partner, rb.d0, rb.cand, rb.bounds, lengths, frame_of, NB, L, W, c, nxt, rb.nrep);
        CB2_LAUNCH_CHECK();
        *launches += 1;
        float* tmp = cur; cur = nxt; nxt = tmp;
    }
    relax_finish_kernel<<<NB, FIN_THREADS, 0, s>>>(cur, rb.x0, rb.partner, rb.d0, slot_atom, out_off, lengths, frame_of, L, xyz_out,
                                                   max_shift, max_dev);
    CB2_LAUNCH_CHECK();
    *launches += 1;
    return 0;
}

}  // namespace cb2
