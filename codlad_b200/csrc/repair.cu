// Clash-driven repair, device side: which residues of a decoded sample clash, and the keep mask of the inpainting pass that
// resamples them (cb2_plan_residue_clashes; Backmapper.repair drives the loop).  Not in the reference: a per-residue form of the
// clash criterion of clash_result (test.py:118-139), which needs no reference structure and no dataset pair lists.
//
// clash_result counts non-bonded atom pairs closer than 1.2 A.  Our structures hold heavy atoms only, 14 slots per residue
// (O, N, C, CA, side chain).  Between two residues the only covalent bond is the peptide bond C(i)-N(i+1), about 1.33 A
// (disulfides are about 2.05 A), so every inter-residue pair closer than the threshold is a clash except the peptide pair.
// counts[b, i] = #{(a in residue i, c in residue j) : j != i in member b, not the peptide pair, d(a, c) < threshold}, with d computed
// as cb2_pair_losses computes it (atom_pair_dist), so a pair is counted once for each of its two residues.
//
// Three launches:
//   1. residue_bounds_kernel: per residue a centre (the CA, slot 3, else the first present atom) and a radius enclosing its present
//      atoms, rounded up by BOUND_SLACK.  A residue without atoms, and every padded residue, gets radius -1.
//   2. residue_clash_kernel: one warp per (member, residue i).  The lanes walk every residue j of the member and test the spheres,
//      |c_i - c_j| <= (r_i + r_j + threshold) * BOUND_SLACK; for a candidate j, each atom of j is tested against the sphere of i
//      grown by the threshold, and only an atom inside it is paired with the atoms of i.  Both tests are conservative, so the
//      counts equal a brute-force pass over all pairs.  (The k-NN graph is not used: K C-alpha neighbours need not include every
//      clash partner.)  The lanes' integer counts are summed by the warp and written once: no atomics, deterministic.
//   3. clash_keep_kernel: keep[b, i] = 0 where residue i or one of its `grow` nearest other residues (the plan's k-NN rows, in
//      distance order, skipping the residue itself) has a clash; 1 elsewhere and on padded rows.
//
// Why the slack is enough: every fp32 operation is correctly rounded (or an FMA, which rounds once), so each computed distance is
// within a few units of 2^-24 of the exact one, relative to itself.  A pair counted as d < threshold is therefore closer than
// threshold * (1 + 4e-7) exactly; the triangle inequality bounds the centre distances exactly, and a relative slack of 1e-5 on the
// bounds covers the rounding of both sides.  Non-finite coordinates never count (d < threshold is false) and make a residue a
// candidate everywhere (its radius becomes +inf; a NaN centre distance passes the `!(d > bound)` tests).
#include "../../include/codlad_b200.h"
#include "common.cuh"
#include "pair_dist.cuh"
#include "repair.h"

namespace cb2 {

namespace {

constexpr int SLOTS = 14, SLOT_N = 1, SLOT_C = 2, SLOT_CA = 3;
constexpr float BOUND_SLACK = 1.0f + 1e-5f;
constexpr int CL_WARPS = 4;

__device__ __forceinline__ float plain_dist(float ax, float ay, float az, float bx, float by, float bz) {
    const float dx = ax - bx, dy = ay - by, dz = az - bz;
    return sqrtf(dx * dx + dy * dy + dz * dz);
}

__global__ void __launch_bounds__(128) residue_bounds_kernel(const float* __restrict__ xyz, const int* __restrict__ slot_atom,
                                                             const long long* __restrict__ out_off, const int* __restrict__ lengths,
                                                             const int* __restrict__ frame_of, int NB, int L, float4* __restrict__ bounds) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= NB * L) return;
    const int b = n / L, i = n - b * L, f = frame_of[b];
    float4 out = make_float4(0.f, 0.f, 0.f, -1.f);
    if (i < lengths[f]) {
        const int* sa = slot_atom + ((size_t)f * L + i) * SLOTS;
        const float* x = xyz + out_off[b] * 3;
        int c = sa[SLOT_CA];
        for (int t = 0; t < SLOTS && c < 0; ++t) c = sa[t];
        if (c >= 0) {
            const float cx = x[(size_t)c * 3], cy = x[(size_t)c * 3 + 1], cz = x[(size_t)c * 3 + 2];
            float r = 0.f;
            for (int t = 0; t < SLOTS; ++t) {
                const int at = sa[t];
                if (at >= 0) r = fmaxf(r, plain_dist(x[(size_t)at * 3], x[(size_t)at * 3 + 1], x[(size_t)at * 3 + 2], cx, cy, cz));
            }
            r *= BOUND_SLACK;
            if (!isfinite(cx) || !isfinite(cy) || !isfinite(cz) || !isfinite(r)) r = INFINITY;
            out = make_float4(cx, cy, cz, r);
        }
    }
    bounds[n] = out;
}

__global__ void __launch_bounds__(CL_WARPS * 32) residue_clash_kernel(const float* __restrict__ xyz, const int* __restrict__ slot_atom,
                                                                      const long long* __restrict__ out_off,
                                                                      const int* __restrict__ lengths, const int* __restrict__ frame_of,
                                                                      const float4* __restrict__ bounds, int NB, int L, float thr,
                                                                      int* __restrict__ counts) {
    __shared__ float sA[CL_WARPS][SLOTS][3];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n = blockIdx.x * CL_WARPS + warp;
    if (n >= NB * L) return;                                   // warp-uniform
    const int b = n / L, i = n - b * L, f = frame_of[b], len = lengths[f];
    const float4 bi = bounds[n];
    unsigned int cnt = 0;
    if (i < len && bi.w >= 0.f) {                              // warp-uniform
        const int* sa = slot_atom + (size_t)f * L * SLOTS;
        const float* x = xyz + out_off[b] * 3;
        const int ai = lane < SLOTS ? sa[(size_t)i * SLOTS + lane] : -1;
        if (ai >= 0)
            for (int k = 0; k < 3; ++k) sA[warp][lane][k] = x[(size_t)ai * 3 + k];
        const unsigned int present = __ballot_sync(0xffffffffu, ai >= 0);     // residue i's present slots
        __syncwarp();
        const float reach = bi.w + thr;                        // sphere of residue i grown by the threshold
        for (int j = lane; j < len; j += 32) {
            if (j == i) continue;
            const float4 bj = bounds[(size_t)b * L + j];
            if (!(bj.w >= 0.f)) continue;
            if (plain_dist(bi.x, bi.y, bi.z, bj.x, bj.y, bj.z) > (reach + bj.w) * BOUND_SLACK) continue;
            for (int tj = 0; tj < SLOTS; ++tj) {
                const int at = sa[(size_t)j * SLOTS + tj];
                if (at < 0) continue;
                const float c[3] = {x[(size_t)at * 3], x[(size_t)at * 3 + 1], x[(size_t)at * 3 + 2]};
                if (plain_dist(c[0], c[1], c[2], bi.x, bi.y, bi.z) > reach * BOUND_SLACK) continue;
                for (unsigned int m = present; m != 0u; m &= m - 1u) {
                    const int ti = __ffs(m) - 1;
                    // the peptide bond C(i)-N(i+1), seen from either residue
                    if ((j == i + 1 && ti == SLOT_C && tj == SLOT_N) || (j == i - 1 && ti == SLOT_N && tj == SLOT_C)) continue;
                    cnt += atom_pair_dist(sA[warp][ti], c) < thr ? 1u : 0u;
                }
            }
        }
    }
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if (lane == 0) counts[n] = (int)cnt;
}

__global__ void __launch_bounds__(128) clash_keep_kernel(const int* __restrict__ counts, const int* __restrict__ nbr_idx,
                                                         const int* __restrict__ lengths, const int* __restrict__ frame_of, int NB, int L,
                                                         int K, int grow, unsigned char* __restrict__ keep) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= NB * L) return;
    const int b = n / L, i = n - b * L, f = frame_of[b];
    bool clash = false;
    if (i < lengths[f]) {
        const int* row = counts + (size_t)b * L;
        clash = row[i] > 0;
        const int* nb = nbr_idx + ((size_t)f * L + i) * K;
        for (int k = 0, taken = 0; k < K && taken < grow && !clash; ++k) {
            const int j = nb[k];
            if (j == i) continue;
            ++taken;
            clash = row[j] > 0;
        }
    }
    keep[n] = clash ? 0 : 1;
}

}  // namespace

int launch_residue_clashes(const float* xyz, const int* slot_atom, const long long* out_off, const int* lengths, const int* frame_of,
                           const int* nbr_idx, int NB, int L, int K, float threshold, int grow, float4* bounds, int* counts,
                           unsigned char* keep, cudaStream_t s) {
    const int N = NB * L;
    if (N <= 0) return 0;
    residue_bounds_kernel<<<(N + 127) / 128, 128, 0, s>>>(xyz, slot_atom, out_off, lengths, frame_of, NB, L, bounds);
    CB2_LAUNCH_CHECK();
    residue_clash_kernel<<<(N + CL_WARPS - 1) / CL_WARPS, CL_WARPS * 32, 0, s>>>(xyz, slot_atom, out_off, lengths, frame_of, bounds, NB, L,
                                                                               threshold, counts);
    CB2_LAUNCH_CHECK();
    if (keep != nullptr) {
        clash_keep_kernel<<<(N + 127) / 128, 128, 0, s>>>(counts, nbr_idx, lengths, frame_of, NB, L, K, grow, keep);
        CB2_LAUNCH_CHECK();
    }
    return 0;
}

}  // namespace cb2
