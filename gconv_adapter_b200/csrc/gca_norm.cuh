// Pieces shared by the two normalization tails (gca_layernorm.cu, gca_batchnorm.cu): both backward passes write per-CTA
// partial column sums in the layout [parts][2][d] (sum s * gY * xh, sum s * gY) plus [parts] (the scalar's gradient), and
// one small kernel combines them in a fixed order - no atomics.
#pragma once

#include "gca_common.cuh"

namespace gca {
namespace {

constexpr int kLnThreads = 256;          // 8 warps
constexpr int kLnWarps = kLnThreads / 32;
constexpr int kLnMaxParts = 296;         // per-CTA partials of the backward (2 CTAs per SM)

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}

// one warp per output: lanes stride over the partials, fixed tree
__global__ void __launch_bounds__(kLnThreads)
k_ln_bwd_finalize(const float* __restrict__ partG, const float* __restrict__ partS, int nparts, int d, float* ggamma,
                  float* gbeta, float* gscalar) {
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int w = blockIdx.x * kLnWarps + (threadIdx.x >> 5);
    if (w < 2 * d) {
        const int which = w / d, c = w - which * d;
        float t = 0.f;
        for (int p = lane; p < nparts; p += 32) t += partG[((size_t)p * 2 + which) * d + c];
        t = warp_sum(t);
        float* out = which == 0 ? ggamma : gbeta;
        if (lane == 0 && out) out[c] = t;
    } else if (w == 2 * d && gscalar) {
        float t = 0.f;
        for (int p = lane; p < nparts; p += 32) t += partS[p];
        t = warp_sum(t);
        if (lane == 0) *gscalar = t;
    }
}

}  // namespace
}  // namespace gca
