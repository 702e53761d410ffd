// Device-side building blocks shared by the kernel translation units of libgca (sm_100a only):
// 3xTF32 mma.sync helpers, mbarrier / bulk-copy (TMA) / named-barrier wrappers, TMEM loads, and the
// sparse row gather every hop kernel uses.
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "gca_common.cuh"

namespace gca {

constexpr int kLongRow = 96;      // rows longer than this are swept by the whole warp

// ------------------------------------------------------------------------------------------
// Register-level tensor-core helpers (mma.sync m16n8k8, tf32 inputs, fp32 accumulate; 279 TFLOP/s
// measured on B200, 4x the fp32 FMA pipe).  fp32 parity needs the 3xTF32 split: x = hi + lo and
//   A B ~= A_hi B_hi + A_lo B_hi + A_hi B_lo.
// Fragment layout (g = lane >> 2, t = lane & 3):
//   A 16x8: a0 (g, t)  a1 (g+8, t)  a2 (g, t+4)  a3 (g+8, t+4)      B 8x8: b0 (k=t, n=g)  b1 (k=t+4, n=g)
//   C 16x8: c0 (g, 2t) c1 (g, 2t+1) c2 (g+8, 2t) c3 (g+8, 2t+1)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void mma_tf32(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// hi = x with the 13 low mantissa bits cleared (exact tf32), lo = tf32_rn(x - hi)
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
    hi = __float_as_uint(x) & 0xffffe000u;
    lo = (__float_as_uint(x - __uint_as_float(hi)) + 0x1000u) & 0xffffe000u;
}

// ---- named barriers ----
__device__ __forceinline__ void named_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void named_arrive(int id, int count) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory"); }

// ---- mbarrier + bulk copies ----
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t"
        "}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ uint64_t policy_evict_first() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
// 2D tiled bulk copies through a tensor map: rows beyond the tensor are zero-filled on load and clipped on store.
__device__ __forceinline__ void tma_load_box(uint32_t dst, const CUtensorMap* tm, int col, int row, uint32_t bar, uint64_t policy) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3}], [%4], %5;"
                 ::"r"(dst), "l"(tm), "r"(col), "r"(row), "r"(bar), "l"(policy) : "memory");
}
__device__ __forceinline__ void tma_load_box_nohint(uint32_t dst, const CUtensorMap* tm, int col, int row, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(dst), "l"(tm), "r"(col), "r"(row), "r"(bar) : "memory");
}
__device__ __forceinline__ void tma_store_box(const CUtensorMap* tm, int col, int row, uint32_t src, uint64_t policy) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group.L2::cache_hint [%0, {%1, %2}], [%3], %4;"
                 ::"l"(tm), "r"(col), "r"(row), "r"(src), "l"(policy) : "memory");
}
// 1D bulk copy global -> shared (16-byte aligned addresses, size a multiple of 16), completion on an mbarrier
__device__ __forceinline__ void bulk_load_1d(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// L2 prefetch of `bytes` (multiple of 16) bytes at a 16-byte aligned global address, no destination in the SM
__device__ __forceinline__ void prefetch_l2_bulk(const void* p, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ---- TMEM ----
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {       // 32 lanes x 32 consecutive columns, no wait
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
        "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ------------------------------------------------------------------------------------------
// sparse row gather
// ------------------------------------------------------------------------------------------
// CG: the operand was written earlier in the SAME kernel (fused small-graph kernels): coherent L2 loads instead of the
// read-only path.
template <int R, bool CG = false>
__device__ __forceinline__ float4 gather_rows(const float* __restrict__ F, const int* __restrict__ colidx,
                                              int beg, int end, int stride, int sub) {
    // Batches of 8 neighbours: all 8 index loads are issued together, then all 8 row loads, so a row of
    // degree <= 8 costs two dependent memory round trips instead of four.  Missing slots add +0 (exact).
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int e = beg; e < end; e += 8 * stride) {
        int j[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) j[u] = (e + u * stride < end) ? __ldg(colidx + e + u * stride) : -1;
        float4 v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u)
            v[u] = (j[u] < 0) ? make_float4(0.f, 0.f, 0.f, 0.f)
                   : CG   ? __ldcg(reinterpret_cast<const float4*>(F + (size_t)j[u] * R + sub * 4))
                          : ldg4(F + (size_t)j[u] * R + sub * 4);
#pragma unroll
        for (int u = 0; u < 8; ++u) acc = f4_add(acc, v[u]);
    }
    return acc;
}

// Hub rows: sum of the pre-computed partials of the row's work items, in item order, 8 loads in flight.
template <int R>
__device__ __forceinline__ float4 hub_row_sum(const float* __restrict__ hub_part, int first, int nitems, int sub) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int c0 = 0; c0 < nitems; c0 += 8) {
        float4 v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u)
            v[u] = (c0 + u < nitems) ? ldg4(hub_part + (size_t)(first + c0 + u) * R + sub * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int u = 0; u < 8; ++u) acc = f4_add(acc, v[u]);
    }
    return acc;
}

// One CSR row per lane group (R/4 lanes); every lane of the warp must call this.
// Rows up to kLongRow neighbours: the group walks them alone.  Up to kHubDeg: the whole warp sweeps the row
// (fixed shuffle tree).  Longer ("hub") rows: their partial sums were produced by k_hub_partials, one warp per
// kHubChunk neighbours, and are only added up here.  warp_spmm_range takes the row's [beg, end) from the caller, so a
// kernel that loops over row batches can fetch the next batch's row header while the current one gathers.
// hubitem == nullptr: no pre-reduced hub partials exist, rows of any length are swept by the warp.
template <int R, bool CG = false>
__device__ __forceinline__ float4 warp_spmm_range(const int* __restrict__ colidx, const float* __restrict__ F, int row, int beg,
                                                  int end, int lane, const int* __restrict__ hubitem,
                                                  const float* __restrict__ hub_part) {
    constexpr int LPG = R / 4, GPW = 32 / LPG;
    const int sub = lane % LPG, grp = lane / LPG;
    const int deg = end - beg;                           // 0 for lanes without a row
    const bool is_hub = hubitem != nullptr && deg > kHubDeg;
    const bool is_long = deg > kLongRow && !is_hub;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (is_hub) acc = hub_row_sum<R>(hub_part, __ldg(hubitem + row), (deg + kHubChunk - 1) / kHubChunk, sub);
    else if (!is_long) acc = gather_rows<R, CG>(F, colidx, beg, end, 1, sub);
    unsigned longmask = __ballot_sync(0xffffffffu, is_long);
    while (longmask) {                                   // warp-uniform
        const int src = __ffs(longmask) - 1;
        const int g = src / LPG;
        const unsigned gm = (LPG >= 32) ? 0xffffffffu : (((1u << LPG) - 1u) << (g * LPG));
        longmask &= ~gm;
        const int b = __shfl_sync(0xffffffffu, beg, src), e = __shfl_sync(0xffffffffu, end, src);
        float4 part = gather_rows<R, CG>(F, colidx, b + grp, e, GPW, sub);
#pragma unroll
        for (int off = LPG; off < 32; off <<= 1) part = f4_add(part, f4_shfl_xor(part, off));
        if (grp == g) acc = part;
    }
    return acc;
}
template <int R>
__device__ __forceinline__ float4 warp_spmm_rows(const int* __restrict__ rowptr, const int* __restrict__ colidx,
                                                 const float* __restrict__ F, int row, bool valid, int lane,
                                                 const int* __restrict__ hubitem, const float* __restrict__ hub_part) {
    int beg = 0, end = 0;
    if (valid) { beg = __ldg(rowptr + row); end = __ldg(rowptr + row + 1); }
    return warp_spmm_range<R>(colidx, F, row, beg, end, lane, hubitem, hub_part);
}

__device__ __forceinline__ float act_apply(float h, int act) {
    if (act == GCA_ACT_RELU) return h < 0.f ? 0.f : h;
    if (act == GCA_ACT_SILU) return h / (1.f + expf(-h));
    return h;
}
__device__ __forceinline__ float silu_grad(float h) {
    const float sg = 1.f / (1.f + expf(-h));
    return sg * (1.f + h * (1.f - sg));
}

}  // namespace gca
