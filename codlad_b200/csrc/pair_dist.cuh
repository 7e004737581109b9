// Atom-pair distance of the evaluation losses (test.py:27,97-146), shared by cb2_pair_losses (metrics.cu) and the per-residue
// clash counts (repair.cu), so that both apply the same criterion to the same bits.
#pragma once
#include <cuda_runtime.h>

namespace cb2 {

constexpr float PAIR_EPS = 1e-7f;                        // test.py:27

// d = sqrt(|a - b|^2 + EPS) in fp32 with the reference's operation order: rounded differences, squares summed in x, y, z order
// from 0, then EPS, then a correctly rounded sqrt; no fused multiply-add.
__device__ __forceinline__ float atom_pair_dist(const float a[3], const float b[3]) {
    float d2 = 0.f;
#pragma unroll
    for (int k = 0; k < 3; ++k) { const float d = __fsub_rn(a[k], b[k]); d2 = __fadd_rn(d2, __fmul_rn(d, d)); }
    return __fsqrt_rn(__fadd_rn(d2, PAIR_EPS));
}

}  // namespace cb2
