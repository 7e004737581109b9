// Keyed Gaussian noise for the sampling passes: every value is a pure function of (seed, member key, draw, slice, residue row,
// channel), so a member's start draw and step noise do not depend on the plan it is sampled in -- how many members share it, their
// order, the padded length L -- nor on any draw made before.  The kernel runs before the step loop and fills the buffers the loop
// reads; the loop and its captured graph are untouched.
//
// Generator: Philox4x32-10 (Salmon, Moraes, Dror, Shaw, "Parallel random numbers: as easy as 1, 2, 3", SC'11) with key = seed
// (lo, hi) and counter = (key_b lo, key_b hi, draw, (slice << 21) | i).  One block of four words gives the three channels of one
// row by Box-Muller twice: u = ((w >> 8) + 0.5) 2^-24 in fp32, u in (0, 1] (never 0, so log is finite; above 2^23 the + 0.5 rounds
// to even, so the largest word gives u = 1 exactly, a radius of 0 with probability 2^-24),
// (n0, n1) = sqrt(-2 ln u0) (cospi(2 u1), sinpi(2 u1)), n2 = sqrt(-2 ln u2) cospi(2 u3).
#include "model.h"

namespace cb2 {

constexpr int kNoiseThreads = 256;

struct Philox4 { unsigned int x, y, z, w; };

static __device__ __forceinline__ Philox4 philox4x32_10(Philox4 c, unsigned int k0, unsigned int k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        if (r) { k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
        const unsigned int lo0 = 0xD2511F53u * c.x, hi0 = __umulhi(0xD2511F53u, c.x);
        const unsigned int lo1 = 0xCD9E8D57u * c.z, hi1 = __umulhi(0xCD9E8D57u, c.z);
        c = {hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0};
    }
    return c;
}

// u = ((w >> 8) + 0.5) 2^-24, one correctly rounded addition and an exact scaling: in (0, 1], never 0
static __device__ __forceinline__ float uniform01(unsigned int w) {
    return __fmul_rn(__fadd_rn((float)(w >> 8), 0.5f), 0x1p-24f);
}

// out[s][b][i][0..2], s < n_slices, for slice first_slice + s of member b; one thread per (slice, member, row), padded rows included
__global__ void __launch_bounds__(kNoiseThreads) keyed_normal_kernel(unsigned long long seed, const long long* __restrict__ keys, int NB,
                                                                     int L, unsigned int draw, int first_slice, long long n,
                                                                     float* __restrict__ out) {
    const long long t = (long long)blockIdx.x * kNoiseThreads + threadIdx.x;
    if (t >= n) return;
    const long long r = t / L;
    const int i = (int)(t - r * L);
    const long long s = r / NB;
    const int b = (int)(r - s * NB);
    const unsigned long long key = (unsigned long long)keys[b];
    const Philox4 w = philox4x32_10({(unsigned int)key, (unsigned int)(key >> 32), draw, ((unsigned int)(first_slice + s) << 21) | (unsigned int)i},
                                    (unsigned int)seed, (unsigned int)(seed >> 32));
    const float r01 = sqrtf(-2.0f * logf(uniform01(w.x))), r23 = sqrtf(-2.0f * logf(uniform01(w.z)));
    float s1, c1, s3, c3;
    sincospif(2.0f * uniform01(w.y), &s1, &c1);
    sincospif(2.0f * uniform01(w.w), &s3, &c3);
    float* o = out + t * 3;
    o[0] = r01 * c1;
    o[1] = r01 * s1;
    o[2] = r23 * c3;
}

int launch_keyed_normal(unsigned long long seed, const long long* keys, int NB, int L, unsigned int draw, int first_slice, int n_slices,
                        float* out, cudaStream_t s) {
    const long long n = (long long)n_slices * NB * L;
    const long long blocks = (n + kNoiseThreads - 1) / kNoiseThreads;
    if (blocks > 0x7fffffffLL) { set_error("keyed_normal: %lld rows exceed one launch", n); return 1; }
    keyed_normal_kernel<<<(unsigned)blocks, kNoiseThreads, 0, s>>>(seed, keys, NB, L, draw, first_slice, n, out);
    CB2_LAUNCH_CHECK();
    return 0;
}

}  // namespace cb2
