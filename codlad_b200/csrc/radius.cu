// Directed radius graph of every frame, built on the device from the C-alpha coordinates alone, and the trimmed X of a frame set
// written from its untrimmed trace.  Together with the k-NN / featuriser / IC filter launches this lets a plan move to new
// coordinates without any host work (cb2_plan_set_coords).
//
// The graph has the content and layout of batching.batch_csr(synthetic.radius_graph(...)): a CSR over the F*L padded rows with
// frame-local columns in ascending order, and an edge i -> j when i != j, both are below the frame's length and d <= cutoff, where
// d = sqrt((dx*dx + dy*dy) + dz*dz), dx = x_j - x_i, every operation correctly rounded and no FMA -- what the host forms, and
// exactly symmetric in i and j.  Two passes, deterministic, no atomics: one warp per row counts its edges with ballots, one CTA
// scans the counts into row_ptr, and the fill pass recomputes the row's ballots and writes its columns in order.
#include "model.h"

namespace cb2 {

constexpr int kRadiusWarps = 8;
constexpr int kScanThreads = 1024;

static __device__ __forceinline__ bool within(const float* __restrict__ Xf, int j, float xi, float yi, float zi, float cutoff) {
    const float dx = __fsub_rn(Xf[j * 3 + 0], xi), dy = __fsub_rn(Xf[j * 3 + 1], yi), dz = __fsub_rn(Xf[j * 3 + 2], zi);
    const float s = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
    return __fsqrt_rn(s) <= cutoff;
}

// counts[row] = edges of row (0 on padded rows); one warp per row of the F*L padded rows
__global__ void __launch_bounds__(kRadiusWarps * 32) radius_count_kernel(const float* __restrict__ X, const int* __restrict__ lengths,
                                                                         int F, int L, float cutoff, int* __restrict__ counts) {
    const int lane = threadIdx.x & 31;
    const long long row = (long long)blockIdx.x * kRadiusWarps + (threadIdx.x >> 5);
    if (row >= (long long)F * L) return;
    const int f = (int)(row / L), i = (int)(row - (long long)f * L);
    const int n = min(lengths[f], L);
    int count = 0;
    if (i < n) {
        const float* Xf = X + (size_t)f * L * 3;
        const float xi = Xf[i * 3 + 0], yi = Xf[i * 3 + 1], zi = Xf[i * 3 + 2];
        for (int base = 0; base < n; base += 32) {
            const int j = base + lane;
            const bool e = j < n && j != i && within(Xf, j, xi, yi, zi, cutoff);
            count += __popc(__ballot_sync(0xffffffffu, e));
        }
    }
    if (lane == 0) counts[row] = count;
}

// In place: row_ptr[0..n) holds the counts on entry; on return row_ptr[r] = sum of counts[0..r) for r <= n.  One CTA; each thread
// scans a contiguous run of rows, so the result does not depend on scheduling.
__global__ void __launch_bounds__(kScanThreads) radius_scan_kernel(int* __restrict__ row_ptr, int n) {
    __shared__ int part[kScanThreads];
    const int t = threadIdx.x;
    const int per = (n + kScanThreads - 1) / kScanThreads;
    const int lo = min(t * per, n), hi = min(lo + per, n);
    int s = 0;
    for (int r = lo; r < hi; ++r) s += row_ptr[r];
    part[t] = s;
    __syncthreads();
    for (int o = 1; o < kScanThreads; o <<= 1) {         // Hillis-Steele inclusive scan of the per-thread sums
        const int v = t >= o ? part[t - o] : 0;
        __syncthreads();
        part[t] += v;
        __syncthreads();
    }
    int run = part[t] - s;                                 // exclusive prefix of this thread's run
    for (int r = lo; r < hi; ++r) {
        const int c = row_ptr[r];
        row_ptr[r] = run;
        run += c;
    }
    if (t == kScanThreads - 1) row_ptr[n] = part[t];
}

// col[row_ptr[row] ..] = the row's neighbours in ascending order
__global__ void __launch_bounds__(kRadiusWarps * 32) radius_fill_kernel(const float* __restrict__ X, const int* __restrict__ lengths,
                                                                        int F, int L, float cutoff, const int* __restrict__ row_ptr,
                                                                        int* __restrict__ col) {
    const int lane = threadIdx.x & 31;
    const long long row = (long long)blockIdx.x * kRadiusWarps + (threadIdx.x >> 5);
    if (row >= (long long)F * L) return;
    const int f = (int)(row / L), i = (int)(row - (long long)f * L);
    const int n = min(lengths[f], L);
    if (i >= n) return;
    const float* Xf = X + (size_t)f * L * 3;
    const float xi = Xf[i * 3 + 0], yi = Xf[i * 3 + 1], zi = Xf[i * 3 + 2];
    int* out = col + row_ptr[row];
    int running = 0;
    for (int base = 0; base < n; base += 32) {
        const int j = base + lane;
        const bool e = j < n && j != i && within(Xf, j, xi, yi, zi, cutoff);
        const unsigned m = __ballot_sync(0xffffffffu, e);
        if (e) out[running + __popc(m & ((1u << lane) - 1u))] = j;
        running += __popc(m);
    }
}

// X[f, i] = ca_full[f, 1 + i] for i < lengths[f], 0 on padded rows (batching.pad_frames of the trimmed trace)
__global__ void trim_coords_kernel(const float* __restrict__ ca_full, const int* __restrict__ lengths, int F, int L, float* __restrict__ X) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)F * L * 3) return;
    const long long row = t / 3;
    const int c = (int)(t - row * 3), f = (int)(row / L), i = (int)(row - (long long)f * L);
    X[t] = i < lengths[f] ? ca_full[((size_t)f * (L + 2) + 1 + i) * 3 + c] : 0.0f;
}

int launch_radius_rows(const float* X, const int* lengths, int F, int L, float cutoff, int* row_ptr, cudaStream_t s) {
    if (F <= 0 || L <= 0 || !(cutoff >= 0.0f)) { set_error("radius_graph: bad geometry F=%d L=%d cutoff=%g", F, L, cutoff); return 1; }
    const long long rows = (long long)F * L;
    radius_count_kernel<<<(unsigned)((rows + kRadiusWarps - 1) / kRadiusWarps), kRadiusWarps * 32, 0, s>>>(X, lengths, F, L, cutoff, row_ptr);
    CB2_LAUNCH_CHECK();
    radius_scan_kernel<<<1, kScanThreads, 0, s>>>(row_ptr, (int)rows);
    CB2_LAUNCH_CHECK();
    return 0;
}

int launch_radius_fill(const float* X, const int* lengths, int F, int L, float cutoff, const int* row_ptr, int* col, cudaStream_t s) {
    if (F <= 0 || L <= 0 || !(cutoff >= 0.0f)) { set_error("radius_graph: bad geometry F=%d L=%d cutoff=%g", F, L, cutoff); return 1; }
    const long long rows = (long long)F * L;
    radius_fill_kernel<<<(unsigned)((rows + kRadiusWarps - 1) / kRadiusWarps), kRadiusWarps * 32, 0, s>>>(X, lengths, F, L, cutoff, row_ptr,
                                                                                                           col);
    CB2_LAUNCH_CHECK();
    return 0;
}

int launch_trim_coords(const float* ca_full, const int* lengths, int F, int L, float* X, cudaStream_t s) {
    const long long n = (long long)F * L * 3;
    trim_coords_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(ca_full, lengths, F, L, X);
    CB2_LAUNCH_CHECK();
    return 0;
}

}  // namespace cb2
