// Internal: per-residue clash detection on a decoded sample (repair.cu), behind cb2_plan_residue_clashes, and the restrained
// clash relaxation (relax.cu), behind cb2_plan_relax, which prunes its pair search with the same residue bounds.
#pragma once
#include <cuda_runtime.h>

namespace cb2 {

// Three launches on a plan's buffers: residue bounds into `bounds` [NB*L] (centre, radius), clash counts [NB*L], and, when
// keep != nullptr, the keep mask [NB*L] grown by `grow` k-NN neighbours (nbr_idx [F, L, K]; may be nullptr when grow == 0).
int launch_residue_clashes(const float* xyz, const int* slot_atom, const long long* out_off, const int* lengths, const int* frame_of,
                           const int* nbr_idx, int NB, int L, int K, float threshold, int grow, float4* bounds, int* counts,
                           unsigned char* keep, cudaStream_t s);

// residue_bounds_kernel alone: bounds [NB*L] = (centre, radius) of every residue of the atoms of xyz that slot_atom [F, L*14] and
// out_off [NB] address; radius -1 for padded residues and residues without atoms, +inf where an atom is not finite.  One launch.
int launch_residue_bounds(const float* xyz, const int* slot_atom, const long long* out_off, const int* lengths, const int* frame_of,
                          int NB, int L, float4* bounds, cudaStream_t s);

// Plan-owned buffers of cb2_plan_relax (sizes in relax.cu: relax_buffer_sizes).
struct RelaxBufs {
    float *x0, *xa, *xb;        // [NB*L*14*3] slot-grid positions: the input and the two iterates
    int* partner;               // [NB*L*14*16] restraint partners (member-local slot index), -1 past the end
    float* d0;                  // [NB*L*14*16] their input distances
    unsigned int* cand;         // [NB*L*ceil(L/32)] candidate residues of every residue, one bit each
    int* grid_slot;             // [F*L*14] slot-grid row of each present slot, -1 elsewhere
    long long* grid_off;        // [NB] first slot-grid row of each member
    int* nrep;                  // [NB*L*14] repulsive pairs each atom evaluated in the last iteration
    float4* bounds;             // [NB*L] residue bounds
};

// cb2_plan_relax after its argument checks; adds its launches to *launches.
int launch_relax(const float* xyz_in, float* xyz_out, const int* slot_atom, const long long* out_off, const int* lengths,
                 const int* frame_of, int F, int NB, int L, float threshold, int iterations, float* max_shift, float* max_dev,
                 const RelaxBufs& rb, cudaStream_t s, long long* launches);

}  // namespace cb2
