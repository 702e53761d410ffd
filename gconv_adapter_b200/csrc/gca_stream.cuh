// Device helpers shared by the TMA-fed streaming kernels (gca_stream.cu, gca_stream_bwd.cu): swizzled-box addressing and the
// scaled 2xFP16 split on the legacy tensor path.
#pragma once

#include <cuda_fp16.h>

#include "gca_common.cuh"
#include "gca_device.cuh"

namespace gca {
namespace {

// byte offset of the 16-byte chunk `chunk` of row `row` inside a box of 128-byte rows with the 128-byte swizzle
__device__ __forceinline__ uint32_t box_off(int row, int chunk) { return (uint32_t)(row * 128 + ((chunk ^ (row & 7)) << 4)); }
__device__ __forceinline__ float4 lds4(const uint8_t* p) { return *reinterpret_cast<const float4*>(p); }

// ---- scaled 2xFP16 split ---------------------------------------------------------------------------------------
// The legacy tensor path issues an f16 m16n8k16 at the rate of a tf32 m16n8k8 (8.6 clk per sub-core, measured:
// experiments/mma_rate.cu), i.e. twice the k's per instruction.  fp16 and tf32 carry the same 11 significant bits, so
//     x * 2^e = h0 + h1,  h0 = fp16_rn(x * 2^e),  h1 = fp16_rn(x * 2^e - h0)         A B ~= A0 B0 + A1 B0 + A0 B1
// has the accuracy of the 3xTF32 split (~2^-22 per product) at HALF the tensor-core instructions.  What fp16 lacks is
// range, so every operand block is scaled by an exact power of two that puts its largest magnitude in [2^13, 2^14):
// per 32 x 32 box of the streamed tile (one warp owns a box: a warp-shuffle max, no cross-warp traffic), per H tile, per
// warp for its W fragments.  An element 2^-20 below its block maximum still keeps all 11 bits of h0; below that only
// the absolute error 2^-25 * 2^-e of fp16 subnormals remains, i.e. < 2^-38 of the block maximum.  Accumulators hold
// scaled values and are unscaled (two exact power-of-two multiplies) when they leave the tensor core: per tile.
__device__ __forceinline__ void mma_f16(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ float warp_max(float m) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
    return m;
}
__device__ __forceinline__ float absmax4(float m, const float4& v) {
    return fmaxf(fmaxf(m, fabsf(v.x)), fmaxf(fabsf(v.y), fmaxf(fabsf(v.z), fabsf(v.w))));
}
// scale = 2^(13 - e), inv = 2^(e - 13) for amax = m * 2^e, 1 <= m < 2 (blocks of zeros / denormals: the largest normal scale)
__device__ __forceinline__ void pow2_scale(float amax, float& scale, float& inv) {
    int e = (int)((__float_as_uint(amax) >> 23) & 0xffu);
    e = e < 14 ? 14 : e;
    scale = __uint_as_float((uint32_t)(267 - e) << 23);
    inv = __uint_as_float((uint32_t)(e - 13) << 23);
}
// 8 x 8 b16 transpose across the warp: a projection A-fragment register (lane (g, t) holds row g, k = 2t, 2t+1) becomes
// the weight-gradient B-fragment register of the same block (lane (g, t) holds k = rows 2t, 2t+1 ; n = column g)
__device__ __forceinline__ uint32_t movmatrix_trans(uint32_t a) {
    uint32_t d;
    asm volatile("movmatrix.sync.aligned.m8n8.trans.b16 %0, %1;" : "=r"(d) : "r"(a));
    return d;
}
// (x0, x1) * scale -> packed halves {low = element 0}: hi = rn(.), lo = rn(. - hi)
__device__ __forceinline__ void split_h2(float x0, float x1, float scale, uint32_t& hi, uint32_t& lo) {
    const float a0 = x0 * scale, a1 = x1 * scale;
    const __half2 h = __floats2half2_rn(a0, a1);
    const float2 hf = __half22float2(h);
    const __half2 l = __floats2half2_rn(a0 - hf.x, a1 - hf.y);
    hi = *reinterpret_cast<const uint32_t*>(&h);
    lo = *reinterpret_cast<const uint32_t*>(&l);
}

}  // namespace
}  // namespace gca
