// Pieces of the segmented radix selection over non-negative float32 bit patterns shared by visualise.cu (percentiles of
// the magnitudes) and fit_matrix.cu (LMedS medians of the residuals): 3 passes of 12 / 10 / 10 bits, per-block
// shared-memory histograms flushed to one global histogram per segment.
#pragma once
#include "ofk_common.cuh"

namespace ofk {

// Digits of the 32-bit pattern: bits 31..20 (pass 0), 19..10 (pass 1), 9..0 (pass 2). Non-negative floats order like
// their bit patterns.
constexpr int kBins0 = 4096, kBins12 = 1024;
__host__ __device__ constexpr int pass_shift(int pass) { return pass == 0 ? 20 : (pass == 1 ? 10 : 0); }
__host__ __device__ constexpr int pass_bins(int pass) { return pass == 0 ? kBins0 : kBins12; }

// Adds one to sh[bin] for the lanes with `active`. When all active lanes of the warp share one bin (thresholded flows
// put most pixels of a frame into bin 0) that is one atomic for the warp instead of 32 colliding ones. Called by all
// 32 lanes.
__device__ __forceinline__ void hist_add(unsigned int* sh, unsigned int bin, bool active) {
    const unsigned int act = __ballot_sync(0xffffffffu, active);
    if (act == 0) return;
    const int leader = __ffs(act) - 1;
    const unsigned int lead_bin = __shfl_sync(0xffffffffu, bin, leader);
    if (__all_sync(0xffffffffu, !active || bin == lead_bin)) {
        if ((int)(threadIdx.x & 31) == leader) atomicAdd(sh + lead_bin, (unsigned int)__popc(act));
    } else if (active) {
        atomicAdd(sh + bin, 1u);
    }
}

__device__ __forceinline__ void flush_hist(const unsigned int* sh, unsigned int* g, int bins) {
    for (int k = threadIdx.x; k < bins; k += blockDim.x)
        if (sh[k]) atomicAdd(g + k, sh[k]);
}

}  // namespace ofk
