// Small graphs (cora / pubmed / molecule-batch sized: the first three BASELINE.json configs): the whole forward is ONE
// cooperative kernel and the whole backward is ONE cooperative kernel.  At these sizes the eight launches of the
// streaming path cost ~12 us each in launch + dependent-latency floors (kernel sum 95 us for 0.2 MB of work); here the
// phases of a direction are separated by grid-wide barriers (cooperative_groups::grid_group::sync) instead of kernel
// boundaries and everything stays in L1 / L2.
//
//   forward   A  P'  = dis * (X Wd^T)                     warp per row, reduce-scatter over the lanes
//             B  Z'  = dis * act(dis * (A' P') + bd)      lane group (r/4 lanes) per row
//             C  H2  = dis * (A' Z') ;  Y = s (H2 Wu^T + bu [+ X]) [+ A]   (A: gca_forward_add's addend)
//   backward  A  gH2' = dis * s * (gY Wu)  ;  per-CTA partials of gY^T H2 and of the column sums of gY
//             B  gH1' = dis * act'(.) * dis * (A'^T gH2') ; per-CTA partials of gbd
//             C  gP  = dis * (A'^T gH1') ;  gX = gP Wd [+ s gY]
//             D  per-CTA partials of gP^T X and of <gY, X>
//             E  ordered sums of all partials -> gWd, gbd, gWu, gbu, per-CTA pieces of gscalar ;  F  gscalar
//
// Plain fp32 FMA arithmetic (no tensor cores: 16 MFLOP per step), every sum in a fixed order -> bitwise reproducible.
// Arrays written in one phase and read in a later one are read with coherent loads (ld.global.cg), never through the
// read-only path.  Reference semantics: /root/reference/src/finetune/gconv_adapter.py:92-106 and its autograd.
#include <cooperative_groups.h>

#include <map>
#include <mutex>
#include <tuple>

#include "gca_common.cuh"
#include "gca_device.cuh"
#include "gca_host.cuh"

namespace cg = cooperative_groups;

namespace gca {
namespace {

constexpr int kSmallThreads = 256;
// Measured (profiles/README.md R2-4): kernel time per fwd+bwd 70 us against 95 us for the eight phase launches at cora
// size, but 1.3x SLOWER than them at pubmed size (19,717 rows: the per-warp row loops and eight grid barriers do not
// scale) - hence the low ceiling.
constexpr int kSmallMaxRows = 4096;
constexpr int64_t kSmallMaxElems = 1 << 19;     // n * d
constexpr int kSmallMaxRD = 8192;               // r * d: both weight matrices live in shared memory (64 KB)

struct SmallFwd {
    const int* rowptr; const int* colidx; const float* dis;
    const float* X; int64_t ldx;
    const float* Wd; const float* bd; const float* Wu; const float* bu; const float* scalar;
    int act, skip;
    float* P; float* Zp; float* H1; float* H2; float* Y; int64_t ldy;
    int n, d;
    const float* A; int64_t lda;      // addend of gca_forward_add (k_small_fwd<R, true> only)
};

struct SmallBwd {
    const int* rowptr_t; const int* colidx_t; const float* dis;
    const float* gY; int64_t ldg; const float* X; int64_t ldx;
    const float* Zp; const float* H1; const float* H2;
    const float* Wd; const float* Wu; const float* bu; const float* scalar;
    int act, skip;
    float* gH2; float* gH1; float* gP; float* gX; int64_t ldgx;
    float* partGu; float* partCol; float* partGd; float* partDot; float* partBd; float* gsp;
    float* gWd; float* gbd; float* gWu; float* gbu; float* gscalar;
    int n, d, rpc;          // rpc: rows per CTA in the weight-gradient phases (one partial per CTA)
};

// Warp-wide sums of acc[0..R) by recursive halving: after log2(32) exchange steps lane l holds the sums of indices
// jb .. jb + max(R / 32, 1) - 1 in acc[0..); for R < 32 the lanes that differ only in the low log2(32 / R) bits hold the
// same values.  R + (R < 32 ? log2(32 / R) : 0) - ... shuffles instead of 5 R.
template <int R, int LEN, int M>
__device__ __forceinline__ void reduce_scatter_steps(float (&acc)[R], int lane, int& jb) {
    if constexpr (M >= 1) {
        if constexpr (LEN > 1) {
            constexpr int half = LEN / 2;
            const bool upper = (lane & M) != 0;
#pragma unroll
            for (int i = 0; i < half; ++i) {
                const float send = upper ? acc[i] : acc[i + half];
                const float keep = upper ? acc[i + half] : acc[i];
                acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, M);
            }
            jb += upper ? half : 0;
            reduce_scatter_steps<R, half, M / 2>(acc, lane, jb);
        } else {
            acc[0] += __shfl_xor_sync(0xffffffffu, acc[0], M);
            reduce_scatter_steps<R, 1, M / 2>(acc, lane, jb);
        }
    }
}

// out[row, 0:R] = rowscale * sum_c A[row, c] * Ws[j * d + c]   for the rows this warp owns (warp per row)
template <int R>
__device__ __forceinline__ void small_project(const float* __restrict__ A, int64_t lda, const float* Ws, const float* __restrict__ dis,
                                              float mul, float* out, int n, int d, int wglobal, int wtotal, int lane) {
    constexpr int VPL = R >= 32 ? R / 32 : 1;            // values per lane after the reduce-scatter
    constexpr int DUP = R >= 32 ? 1 : 32 / R;            // lanes holding the same value
    for (int row = wglobal; row < n; row += wtotal) {
        float acc[R];
#pragma unroll
        for (int j = 0; j < R; ++j) acc[j] = 0.f;
        const float* ar = A + (size_t)row * lda;
        for (int c = lane; c < d; c += 32) {
            const float x = __ldg(ar + c);
#pragma unroll
            for (int j = 0; j < R; ++j) acc[j] = fmaf(x, Ws[j * d + c], acc[j]);
        }
        int jb = 0;
        reduce_scatter_steps<R, R, 16>(acc, lane, jb);
        const float sc = __ldg(dis + row) * mul;
        if ((lane & (DUP - 1)) == 0) {
#pragma unroll
            for (int v = 0; v < VPL; ++v) out[(size_t)row * R + jb + v] = sc * acc[v];
        }
    }
}

// h[0..R) <- the R values of lane group g's float4s (every lane of the warp gets them)
template <int R>
__device__ __forceinline__ void bcast_group_row(const float4& mine, int g, float (&h)[R]) {
    constexpr int LPG = R / 4;
#pragma unroll
    for (int q = 0; q < LPG; ++q) {
        const int src = g * LPG + q;
        h[4 * q + 0] = __shfl_sync(0xffffffffu, mine.x, src);
        h[4 * q + 1] = __shfl_sync(0xffffffffu, mine.y, src);
        h[4 * q + 2] = __shfl_sync(0xffffffffu, mine.z, src);
        h[4 * q + 3] = __shfl_sync(0xffffffffu, mine.w, src);
    }
}

// Per-CTA partial of G[j, c] = sum_rows H[row, j] * A[row, c] (+ column sums of A, + <A, B>) over the CTA's rows
// [r0, r1): column block by column block, the 8 warps split the rows, their sums are added in warp order through shared
// memory.  H_CG: H was written earlier in this kernel.
template <int R, bool H_CG>
__device__ __forceinline__ float small_wgrad_partial(const float* __restrict__ A, int64_t lda, const float* H,
                                                     const float* __restrict__ B, int64_t ldb, int r0, int r1, int d,
                                                     float* s_part /*[8][R][32]*/, float* s_col /*[8][32]*/,
                                                     float* partG /*[R][d] of this CTA*/, float* partCol /*[d] or null*/) {
    constexpr int LPG = R / 4, NW = kSmallThreads / 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int ncb = (d + 31) / 32;
    float dot = 0.f;
    auto hrow = [&](int row, int q) {
        const float4* p = reinterpret_cast<const float4*>(H + (size_t)row * R + q * 4);   // same address in every lane
        return H_CG ? __ldcg(p) : __ldg(p);
    };
    for (int cb = 0; cb < ncb; ++cb) {
        const int c = cb * 32 + lane;
        const bool cok = c < d;
        float acc[R];
#pragma unroll
        for (int j = 0; j < R; ++j) acc[j] = 0.f;
        float colsum = 0.f;
        int row = r0 + warp;
        for (; row + NW < r1; row += 2 * NW) {                   // two rows in flight
            const float a0 = cok ? __ldg(A + (size_t)row * lda + c) : 0.f;
            const float a1 = cok ? __ldg(A + (size_t)(row + NW) * lda + c) : 0.f;
            if (B && cok) {
                dot = fmaf(a0, __ldg(B + (size_t)row * ldb + c), dot);
                dot = fmaf(a1, __ldg(B + (size_t)(row + NW) * ldb + c), dot);
            }
            colsum += a0;
            colsum += a1;
#pragma unroll
            for (int q = 0; q < LPG; ++q) {
                const float4 h0 = hrow(row, q), h1 = hrow(row + NW, q);
                acc[4 * q + 0] = fmaf(a1, h1.x, fmaf(a0, h0.x, acc[4 * q + 0]));
                acc[4 * q + 1] = fmaf(a1, h1.y, fmaf(a0, h0.y, acc[4 * q + 1]));
                acc[4 * q + 2] = fmaf(a1, h1.z, fmaf(a0, h0.z, acc[4 * q + 2]));
                acc[4 * q + 3] = fmaf(a1, h1.w, fmaf(a0, h0.w, acc[4 * q + 3]));
            }
        }
        if (row < r1) {
            const float a0 = cok ? __ldg(A + (size_t)row * lda + c) : 0.f;
            if (B && cok) dot = fmaf(a0, __ldg(B + (size_t)row * ldb + c), dot);
            colsum += a0;
#pragma unroll
            for (int q = 0; q < LPG; ++q) {
                const float4 h0 = hrow(row, q);
                acc[4 * q + 0] = fmaf(a0, h0.x, acc[4 * q + 0]);
                acc[4 * q + 1] = fmaf(a0, h0.y, acc[4 * q + 1]);
                acc[4 * q + 2] = fmaf(a0, h0.z, acc[4 * q + 2]);
                acc[4 * q + 3] = fmaf(a0, h0.w, acc[4 * q + 3]);
            }
        }
        __syncthreads();                                          // the previous column block has been read out
#pragma unroll
        for (int j = 0; j < R; ++j) s_part[(warp * R + j) * 32 + lane] = acc[j];
        s_col[warp * 32 + lane] = colsum;
        __syncthreads();
        for (int idx = threadIdx.x; idx < R * 32; idx += kSmallThreads) {
            const int j = idx >> 5, l = idx & 31;
            float t = 0.f;
#pragma unroll
            for (int w = 0; w < NW; ++w) t += s_part[(w * R + j) * 32 + l];
            if (cb * 32 + l < d) partG[(size_t)j * d + cb * 32 + l] = t;
        }
        if (partCol && threadIdx.x < 32 && cb * 32 + (int)threadIdx.x < d) {
            float t = 0.f;
#pragma unroll
            for (int w = 0; w < NW; ++w) t += s_col[w * 32 + threadIdx.x];
            partCol[cb * 32 + threadIdx.x] = t;
        }
    }
    return dot;                                                   // this thread's share of <A, B>
}

// Warp-wide ordered sum of `count` partials spaced `pitch` floats apart (lanes stride over the partials, fixed tree).
__device__ __forceinline__ float warp_sum_partials(const float* base, int count, size_t pitch, int lane) {
    float t = 0.f;
    for (int p = lane; p < count; p += 32) t += __ldcg(base + (size_t)p * pitch);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) t += __shfl_xor_sync(0xffffffffu, t, off);
    return t;
}

__device__ __forceinline__ float block_sum_ordered(float v, float* s_red) {     // fixed-order tree over the CTA
    __syncthreads();
    s_red[threadIdx.x] = v;
    __syncthreads();
    for (int o = kSmallThreads / 2; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) s_red[threadIdx.x] += s_red[threadIdx.x + o];
        __syncthreads();
    }
    return s_red[0];
}

template <int R, bool ADD>
__global__ void __launch_bounds__(kSmallThreads) k_small_fwd(const SmallFwd a) {
    extern __shared__ float sm[];
    constexpr int LPG = R / 4, GPW = 32 / LPG;
    const int n = a.n, d = a.d;
    float* Wd_s = sm;                 // [R][d]
    float* Wut_s = sm + R * d;        // [R][d] = Wu^T
    cg::grid_group grid = cg::this_grid();
    for (int i = threadIdx.x; i < R * d; i += kSmallThreads) {
        Wd_s[i] = __ldg(a.Wd + i);
        Wut_s[(i % R) * d + i / R] = __ldg(a.Wu + i);
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int sub = lane % LPG, grp = lane / LPG;
    const int wglobal = blockIdx.x * (kSmallThreads / 32) + warp, wtotal = gridDim.x * (kSmallThreads / 32);
    const float s = a.scalar ? __ldg(a.scalar) : 1.f;

    small_project<R>(a.X, a.ldx, Wd_s, a.dis, 1.f, a.P, n, d, wglobal, wtotal, lane);
    grid.sync();

    {   // B: first hop + bias + activation
        const float4 b4 = ldg4(a.bd + sub * 4);
        for (int rowbase = wglobal * GPW; rowbase < n; rowbase += wtotal * GPW) {
            const int row = rowbase + grp;
            const bool valid = row < n;
            int beg = 0, end = 0;
            if (valid) { beg = __ldg(a.rowptr + row); end = __ldg(a.rowptr + row + 1); }
            const float4 acc = warp_spmm_range<R, true>(a.colidx, a.P, row, beg, end, lane, nullptr, nullptr);
            if (!valid) continue;
            const float di = __ldg(a.dis + row);
            const size_t o = (size_t)row * R + sub * 4;
            float4 h = make_float4(fmaf(di, acc.x, b4.x), fmaf(di, acc.y, b4.y), fmaf(di, acc.z, b4.z), fmaf(di, acc.w, b4.w));
            if (a.H1) *reinterpret_cast<float4*>(a.H1 + o) = h;
            h = make_float4(act_apply(h.x, a.act), act_apply(h.y, a.act), act_apply(h.z, a.act), act_apply(h.w, a.act));
            *reinterpret_cast<float4*>(a.Zp + o) = f4_scale(h, di);
        }
    }
    grid.sync();

    // C: second hop, then the expansion of the warp's rows (all lanes work on one row at a time)
    for (int rowbase = wglobal * GPW; rowbase < n; rowbase += wtotal * GPW) {
        const int row = rowbase + grp;
        const bool valid = row < n;
        int beg = 0, end = 0;
        if (valid) { beg = __ldg(a.rowptr + row); end = __ldg(a.rowptr + row + 1); }
        float4 acc = warp_spmm_range<R, true>(a.colidx, a.Zp, row, beg, end, lane, nullptr, nullptr);
        const float di = valid ? __ldg(a.dis + row) : 0.f;
        acc = f4_scale(acc, di);
        if (valid) *reinterpret_cast<float4*>(a.H2 + (size_t)row * R + sub * 4) = acc;
        for (int g = 0; g < GPW && rowbase + g < n; ++g) {
            float h[R];
            bcast_group_row<R>(acc, g, h);
            const int rg = rowbase + g;
            const float* xr = a.X + (size_t)rg * a.ldx;
            float* yr = a.Y + (size_t)rg * a.ldy;
            for (int c = lane; c < d; c += 32) {
                float y = __ldg(a.bu + c);
#pragma unroll
                for (int j = 0; j < R; ++j) y = fmaf(h[j], Wut_s[j * d + c], y);
                if (a.skip) y += __ldg(xr + c);
                if constexpr (ADD) yr[c] = __fadd_rn(s * y, __ldcg(a.A + (size_t)rg * a.lda + c));   // (coherent: Y may be A)
                else yr[c] = s * y;
            }
        }
    }
}

template <int R>
__global__ void __launch_bounds__(kSmallThreads) k_small_bwd(const SmallBwd a) {
    extern __shared__ float sm[];
    __shared__ float s_red[kSmallThreads];
    __shared__ float s_gb[kSmallThreads / 32][R];
    constexpr int LPG = R / 4, GPW = 32 / LPG;
    const int n = a.n, d = a.d;
    float* Wd_s = sm;                 // [R][d]
    float* Wut_s = sm + R * d;        // [R][d] = Wu^T
    float* s_part = sm + 2 * R * d;   // [8][R][32]
    float* s_col = s_part + (kSmallThreads / 32) * R * 32;   // [8][32]
    cg::grid_group grid = cg::this_grid();
    for (int i = threadIdx.x; i < R * d; i += kSmallThreads) {
        Wd_s[i] = __ldg(a.Wd + i);
        Wut_s[(i % R) * d + i / R] = __ldg(a.Wu + i);
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int sub = lane % LPG, grp = lane / LPG;
    const int wglobal = blockIdx.x * (kSmallThreads / 32) + warp, wtotal = gridDim.x * (kSmallThreads / 32);
    const float s = a.scalar ? __ldg(a.scalar) : 1.f;

    // A: gH2' rows, and the weight-gradient partials of conv_up (one warp per row segment, column block by column block)
    small_project<R>(a.gY, a.ldg, Wut_s, a.dis, s, a.gH2, n, d, wglobal, wtotal, lane);
    {
        const int r0 = min(n, (int)blockIdx.x * a.rpc), r1 = min(n, r0 + a.rpc);
        small_wgrad_partial<R, false>(a.gY, a.ldg, a.H2, nullptr, 0, r0, r1, d, s_part, s_col,
                                      a.partGu + (size_t)blockIdx.x * R * d, a.partCol + (size_t)blockIdx.x * d);
    }
    grid.sync();

    {   // B: transpose hop + derivative of the activation; bias-gradient partials per CTA
        float4 gb = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int rowbase = wglobal * GPW; rowbase < n; rowbase += wtotal * GPW) {
            const int row = rowbase + grp;
            const bool valid = row < n;
            int beg = 0, end = 0;
            if (valid) { beg = __ldg(a.rowptr_t + row); end = __ldg(a.rowptr_t + row + 1); }
            const float4 acc = warp_spmm_range<R, true>(a.colidx_t, a.gH2, row, beg, end, lane, nullptr, nullptr);
            if (!valid) continue;
            const float di = __ldg(a.dis + row);
            const size_t o = (size_t)row * R + sub * 4;
            float4 g = f4_scale(acc, di);
            if (a.act == GCA_ACT_RELU) {
                const float4 z = ldg4(a.Zp + o);
                g = make_float4(z.x > 0.f ? g.x : 0.f, z.y > 0.f ? g.y : 0.f, z.z > 0.f ? g.z : 0.f, z.w > 0.f ? g.w : 0.f);
            } else if (a.act == GCA_ACT_SILU) {
                const float4 h = ldg4(a.H1 + o);
                g = make_float4(g.x * silu_grad(h.x), g.y * silu_grad(h.y), g.z * silu_grad(h.z), g.w * silu_grad(h.w));
            }
            gb = f4_add(gb, g);
            *reinterpret_cast<float4*>(a.gH1 + o) = f4_scale(g, di);
        }
#pragma unroll
        for (int off = LPG; off < 32; off <<= 1) gb = f4_add(gb, f4_shfl_xor(gb, off));
        if (grp == 0) *reinterpret_cast<float4*>(&s_gb[warp][sub * 4]) = gb;
        __syncthreads();
        if (threadIdx.x < R) {
            float t = 0.f;
#pragma unroll
            for (int w = 0; w < kSmallThreads / 32; ++w) t += s_gb[w][threadIdx.x];
            a.partBd[(size_t)blockIdx.x * R + threadIdx.x] = t;
        }
    }
    grid.sync();

    // C: second transpose hop, gP saved for phase D, expansion into gX
    for (int rowbase = wglobal * GPW; rowbase < n; rowbase += wtotal * GPW) {
        const int row = rowbase + grp;
        const bool valid = row < n;
        int beg = 0, end = 0;
        if (valid) { beg = __ldg(a.rowptr_t + row); end = __ldg(a.rowptr_t + row + 1); }
        float4 acc = warp_spmm_range<R, true>(a.colidx_t, a.gH1, row, beg, end, lane, nullptr, nullptr);
        const float di = valid ? __ldg(a.dis + row) : 0.f;
        acc = f4_scale(acc, di);
        if (valid) *reinterpret_cast<float4*>(a.gP + (size_t)row * R + sub * 4) = acc;
        if (a.gX) {
            for (int g = 0; g < GPW && rowbase + g < n; ++g) {
                float h[R];
                bcast_group_row<R>(acc, g, h);
                const int rg = rowbase + g;
                const float* gyr = a.gY + (size_t)rg * a.ldg;
                float* gxr = a.gX + (size_t)rg * a.ldgx;
                for (int c = lane; c < d; c += 32) {
                    float v = a.skip ? s * __ldg(gyr + c) : 0.f;
#pragma unroll
                    for (int j = 0; j < R; ++j) v = fmaf(h[j], Wd_s[j * d + c], v);
                    gxr[c] = v;
                }
            }
        }
    }
    grid.sync();

    // D: weight-gradient partials of conv_down and <gY, X>
    {
        const int r0 = min(n, (int)blockIdx.x * a.rpc), r1 = min(n, r0 + a.rpc);
        const float dot = small_wgrad_partial<R, true>(a.X, a.ldx, a.gP, a.skip ? a.gY : nullptr, a.ldg, r0, r1, d, s_part, s_col,
                                                       a.partGd + (size_t)blockIdx.x * R * d, nullptr);
        const float t = block_sum_ordered(dot, s_red);
        if (threadIdx.x == 0) a.partDot[blockIdx.x] = t;
    }
    grid.sync();

    // E: ordered sums of the per-CTA partials (one warp per output element, lanes over the partials), pieces of gscalar
    float gs = 0.f;
    const int rd = R * d, np = gridDim.x;
    for (int e = wglobal; e < rd; e += wtotal) {                  // e = j * d + c in both partial arrays
        const float tu = warp_sum_partials(a.partGu + e, np, rd, lane);
        const float td = warp_sum_partials(a.partGd + e, np, rd, lane);
        if (lane == 0) {
            const int j = e / d, c = e - j * d;
            if (a.gWu) a.gWu[(size_t)c * R + j] = s * tu;
            gs = fmaf(tu, __ldg(a.Wu + (size_t)c * R + j), gs);
            if (a.gWd) a.gWd[e] = td;
        }
    }
    for (int c = wglobal; c < d; c += wtotal) {
        const float t = warp_sum_partials(a.partCol + c, np, d, lane);
        if (lane == 0) {
            if (a.gbu) a.gbu[c] = s * t;
            gs = fmaf(t, __ldg(a.bu + c), gs);
        }
    }
    for (int j = wglobal; j < R; j += wtotal) {
        const float t = warp_sum_partials(a.partBd + j, np, R, lane);
        if (lane == 0 && a.gbd) a.gbd[j] = t;
    }
    if (!a.gscalar) return;                                       // (uniform over the grid: no barrier is skipped by a part of it)
    if (a.skip && blockIdx.x == 0 && warp == 0) {
        const float t = warp_sum_partials(a.partDot, np, 1, lane);
        if (lane == 0) gs += t;
    }
    const float mine = block_sum_ordered(gs, s_red);
    if (threadIdx.x == 0) a.gsp[blockIdx.x] = mine;
    grid.sync();
    if (blockIdx.x == 0) {
        const float v = threadIdx.x < gridDim.x ? __ldcg(a.gsp + threadIdx.x) : 0.f;   // gridDim.x <= kSmallThreads
        const float total = block_sum_ordered(v, s_red);
        if (threadIdx.x == 0) *a.gscalar = total;
    }
}

bool small_enabled() {
    static const bool on = [] { const char* e = getenv("GCA_DISABLE_SMALL"); return !(e && e[0] == '1'); }();
    return on;
}

// co-resident CTAs of a kernel with `smem` dynamic bytes, per (device, kernel, smem).  The kernel is part of the key:
// every k_small_fwd<R, ADD> has the same type K, so one cache serves all ranks, and two ranks can ask with the same smem
// (r 64 / d 128 and r 128 / d 64) while their register counts allow different numbers of CTAs per SM.
template <typename K>
int coop_grid_limit(K kernel, size_t smem) {
    static std::mutex mu;
    static std::map<std::tuple<int, const void*, size_t>, int> cache;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 0;
    std::lock_guard<std::mutex> lk(mu);
    const auto key = std::make_tuple(dev, reinterpret_cast<const void*>(kernel), smem);
    auto it = cache.find(key);
    if (it != cache.end()) return it->second;
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kSmallThreads, smem) != cudaSuccess) per_sm = 0;
    const int lim = per_sm * num_sms();
    cache[key] = lim;
    return lim;
}

template <typename K, typename A>
int launch_coop(K kernel, const A& args, int grid, size_t smem, cudaStream_t st, const char* name) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(kSmallThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;
    attr[0].val.cooperative = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    {
        ProfScope ps(name, st, "fused");
        GCA_CUDA(cudaLaunchKernelEx(&cfg, kernel, args));
    }
    GCA_LAUNCH_OK();
    return GCA_OK;
}

inline int small_grid(int n, int limit) {
    int grid = (n + kSmallThreads / 32 - 1) / (kSmallThreads / 32);      // a row per warp in the dense phases
    if (grid > limit) grid = limit;
    if (grid > kSmallThreads) grid = kSmallThreads;                      // gscalar pieces are summed by one CTA
    return grid < 1 ? 1 : grid;
}

template <int R, bool ADD>
int small_forward_t(const SmallFwd& a, cudaStream_t st) {
    const size_t smem = sizeof(float) * 2 * R * a.d;
    GCA_TRY(set_smem(k_small_fwd<R, ADD>, smem));
    const int limit = coop_grid_limit(k_small_fwd<R, ADD>, smem);
    if (limit < 1) return GCA_ERR_UNSUPPORTED;
    return launch_coop(k_small_fwd<R, ADD>, a, small_grid(a.n, limit), smem, st, "small_fwd");
}

template <int R>
int small_backward_t(SmallBwd a, cudaStream_t st) {
    const size_t smem = sizeof(float) * (2 * (size_t)R * a.d + (kSmallThreads / 32) * (R + 1) * 32);
    GCA_TRY(set_smem(k_small_bwd<R>, smem, true));
    const int limit = coop_grid_limit(k_small_bwd<R>, smem);
    if (limit < 1) return GCA_ERR_UNSUPPORTED;
    const int grid = small_grid(a.n, limit);
    a.rpc = (a.n + grid - 1) / grid;
    return launch_coop(k_small_bwd<R>, a, grid, smem, st, "small_bwd");
}

}  // namespace

bool small_path_ok(const gca_graph* g, int d, int r, cudaStream_t st) {
    const int n = g->row_end - g->row_begin;
    if (!(small_enabled() && g->row_begin == 0 && g->row_end == g->N && n > 0 && n <= kSmallMaxRows &&
          (int64_t)n * d <= kSmallMaxElems && r * d <= kSmallMaxRD && shape_ok(d, r)))
        return false;
    // What the fused kernels save is host time (2 launches instead of 8).  Inside a CUDA graph launches cost nothing and the
    // eight phase kernels, overlapped by programmatic dependent launch, replay FASTER (51 vs 56 us per cora-shaped step,
    // profiles/README.md R2-4): a capturing stream takes the phases.
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cap) != cudaSuccess) { (void)cudaGetLastError(); return true; }
    return cap == cudaStreamCaptureStatusNone;
}

int small_forward(const gca_graph* g, const float* X, int64_t ldx, const float* Wd, const float* bd, const float* Wu,
                  const float* bu, const float* scalar, int act, int skip, float* P, float* Zp, float* H1, float* H2, float* Y,
                  int64_t ldy, int d, int r, cudaStream_t st, const float* A, int64_t lda) {
    SmallFwd a{g->rowptr, g->colidx, g->dis, X, ldx, Wd, bd, Wu, bu, scalar, act, skip, P, Zp, H1, H2, Y, ldy, g->N, d, A, lda};
    if (A) { GCA_DISPATCH_R(r, (small_forward_t<R_, true>(a, st))); }
    GCA_DISPATCH_R(r, (small_forward_t<R_, false>(a, st)));
}

int small_backward(const gca_graph* g, const float* gY, int64_t ldg, const float* X, int64_t ldx, const float* Zp,
                   const float* H1, const float* H2, const float* Wd, const float* Wu, const float* bu, const float* scalar,
                   int act, int skip, float* gH2, float* gH1, float* gP, float* gX, int64_t ldgx, const Scratch& S, float* gWd,
                   float* gbd, float* gWu, float* gbu, float* gscalar, int d, int r, cudaStream_t st) {
    const int n = g->N;
    SmallBwd a{g->rowptr_t, g->colidx_t, g->dis, gY, ldg, X, ldx, Zp, H1, H2, Wd, Wu, bu, scalar, act, skip, gH2, gH1, gP, gX, ldgx,
               S.gu, S.col, S.gd, S.dot, S.bd, S.gsp, gWd, gbd, gWu, gbu, gscalar, n, d, 0};
    GCA_DISPATCH_R(r, (small_backward_t<R_>(a, st)));
}

}  // namespace gca
