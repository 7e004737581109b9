// Internal: per-residue clash detection on a decoded sample (repair.cu), behind cb2_plan_residue_clashes.
#pragma once
#include <cuda_runtime.h>

namespace cb2 {

// Three launches on a plan's buffers: residue bounds into `bounds` [NB*L] (centre, radius), clash counts [NB*L], and, when
// keep != nullptr, the keep mask [NB*L] grown by `grow` k-NN neighbours (nbr_idx [F, L, K]; may be nullptr when grow == 0).
int launch_residue_clashes(const float* xyz, const int* slot_atom, const long long* out_off, const int* lengths, const int* frame_of,
                           const int* nbr_idx, int NB, int L, int K, float threshold, int grow, float4* bounds, int* counts,
                           unsigned char* keep, cudaStream_t s);

}  // namespace cb2
