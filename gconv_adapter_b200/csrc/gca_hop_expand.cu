// K3: hop + expansion.  r-wide gather-SpMM of a row tile fused with the [rows,R] x [R,d] expansion, bias, residual and
// scalar (conv_up + skip + scalar ; gP -> gX), and in the forward optionally + an addend A (ADD: parallel insertion,
// Y = h + adapter(x) in the same pass; gca_fwd_hop2_up_add):
//   k_hop_expand_tc    tcgen05 / TMEM accumulator, tensor-map TMA in and out, 128-row tiles  (r = 16 / 32, d % 64 == 0, d <= 256)
//   k_hop_expand_mma   3xTF32 mma.sync, one kernel per 64-row tile                           (r = 16 / 32, other d)
//   k_hop_expand       FFMA                                                                   (every other shape; r = 128
//                      after a plain hop, by 128-column blocks: PRE)
// Reference semantics: /root/reference/src/finetune/gconv_adapter.py:92-106.
#include "gca_common.cuh"
#include "gca_device.cuh"
#include "gca_host.cuh"
#include "gca_tc.cuh"

namespace gca {
int launch_hub_partials(int r, const Csr& c, const float* F, cudaStream_t st);

namespace {

constexpr int kTileRows = 64;     // rows per CTA tile in k_hop_expand / k_hop_expand_mma

// ------------------------------------------------------------------------------------------
// K3: tile of 64 rows: H[i] = dis[i] * sum_j F[j] staged in shared memory (and saved), then
//     Out[i, :] = alpha * (H[i] W + bias) + beta * Resid[i, :]
// W is kept transposed in shared memory as WT[c][k] so a warp reads 512 contiguous bytes per c.
// Warp w owns rows 8w..8w+7 of the tile, lane l the column quads l, l+32, ...
// PRE (r = 128, where all of W next to the H tile would leave one CTA per SM, or not fit from d = 340): H was left in Hout
// by a plain hop (k_hop, plain mode) and is only read back; the CTA expands the kPreCols output columns of block
// blockIdx.y, so W^T is held kPreCols columns at a time at every d.
// ------------------------------------------------------------------------------------------
constexpr int kPreCols = 128;

template <int R, bool W_IS_DR, bool ADD, bool PRE = false>
__global__ void __launch_bounds__(256, 2)
k_hop_expand(const int* __restrict__ rowptr, const int* __restrict__ colidx, const float* __restrict__ dis,
             const float* __restrict__ F, const float* __restrict__ W, const float* __restrict__ bias,
             const float* __restrict__ resid, int64_t ldr, const float* __restrict__ scalar,
             int alpha_is_scalar, int use_resid, float* __restrict__ Hout, float* __restrict__ Out, int64_t ldo,
             int n, int d,
    const int* __restrict__ hubitem, const float* __restrict__ hub_part, const float* addend, int64_t lda) {
    constexpr int LPG = R / 4, GPW = 32 / LPG;
    extern __shared__ __align__(16) float smem[];
    float* WT = smem;                 // [R][d]   (PRE: [R][dw], columns col0 .. col0 + dw - 1)
    float* Hs;                        // [kTileRows][R]
    int dw = d;
    if constexpr (PRE) {
        const int col0 = blockIdx.y * kPreCols;
        dw = min(kPreCols, d - col0);
        Hs = smem + (size_t)R * kPreCols;
        for (int idx = threadIdx.x; idx < dw * R; idx += blockDim.x) {
            const int c = idx / dw, k = idx - c * dw;
            WT[idx] = W_IS_DR ? W[(size_t)(col0 + k) * R + c] : W[(size_t)c * d + col0 + k];
        }
        bias = bias ? bias + col0 : nullptr;
        resid = resid ? resid + col0 : nullptr;
        Out += col0;
        if constexpr (ADD) addend += col0;
    } else {
        Hs = smem + (size_t)R * d;
        if (Out) {
            for (int idx = threadIdx.x; idx < d * R; idx += blockDim.x) {
                if (W_IS_DR) { const int k = idx / R, c = idx - k * R; WT[c * d + k] = W[idx]; }
                else WT[idx] = W[idx];
            }
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int sub = lane % LPG, grp = lane / LPG;
    const float s = scalar ? __ldg(scalar) : 1.f;
    const float alpha = alpha_is_scalar ? s : 1.f;
    const float beta = use_resid ? s : 0.f;
    const int nq = dw >> 2;
    const int ntiles = (n + kTileRows - 1) / kTileRows;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int trow = tile * kTileRows;
        __syncthreads();              // WT ready / previous tile's readers of Hs are done
        if constexpr (PRE) {
            for (int idx = threadIdx.x; idx < kTileRows * (R / 4); idx += blockDim.x) {
                const int rr = idx / (R / 4);
                reinterpret_cast<float4*>(Hs)[idx] =
                    trow + rr < n ? ldg4(Hout + (size_t)trow * R + (size_t)idx * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        } else
        for (int rr = warp * GPW; rr < kTileRows; rr += 8 * GPW) {
            const int row = trow + rr + grp;
            const bool valid = row < n;
            const float4 acc = warp_spmm_rows<R>(rowptr, colidx, F, row, valid, lane, hubitem, hub_part);
            float4 h = make_float4(0.f, 0.f, 0.f, 0.f);
            if (valid) {
                h = f4_scale(acc, __ldg(dis + row));
                *reinterpret_cast<float4*>(Hout + (size_t)row * R + sub * 4) = h;
            }
            *reinterpret_cast<float4*>(Hs + (rr + grp) * R + sub * 4) = h;
        }
        __syncthreads();
        if (!Out) continue;
        const int r0 = trow + warp * 8;
        const float* hs = Hs + warp * 8 * R;
        for (int q = lane; q < nq; q += 32) {
            float4 xr[8];
            if (use_resid) {
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    xr[i] = (r0 + i < n) ? ldg4_stream(resid + (size_t)(r0 + i) * ldr + q * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            float4 acc[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int c4 = 0; c4 < R / 4; ++c4) {
                const float4 w0 = *reinterpret_cast<const float4*>(WT + (c4 * 4 + 0) * dw + q * 4);
                const float4 w1 = *reinterpret_cast<const float4*>(WT + (c4 * 4 + 1) * dw + q * 4);
                const float4 w2 = *reinterpret_cast<const float4*>(WT + (c4 * 4 + 2) * dw + q * 4);
                const float4 w3 = *reinterpret_cast<const float4*>(WT + (c4 * 4 + 3) * dw + q * 4);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float4 h = *reinterpret_cast<const float4*>(hs + i * R + c4 * 4);
                    acc[i].x = fmaf(h.x, w0.x, acc[i].x); acc[i].y = fmaf(h.x, w0.y, acc[i].y);
                    acc[i].z = fmaf(h.x, w0.z, acc[i].z); acc[i].w = fmaf(h.x, w0.w, acc[i].w);
                    acc[i].x = fmaf(h.y, w1.x, acc[i].x); acc[i].y = fmaf(h.y, w1.y, acc[i].y);
                    acc[i].z = fmaf(h.y, w1.z, acc[i].z); acc[i].w = fmaf(h.y, w1.w, acc[i].w);
                    acc[i].x = fmaf(h.z, w2.x, acc[i].x); acc[i].y = fmaf(h.z, w2.y, acc[i].y);
                    acc[i].z = fmaf(h.z, w2.z, acc[i].z); acc[i].w = fmaf(h.z, w2.w, acc[i].w);
                    acc[i].x = fmaf(h.w, w3.x, acc[i].x); acc[i].y = fmaf(h.w, w3.y, acc[i].y);
                    acc[i].z = fmaf(h.w, w3.z, acc[i].z); acc[i].w = fmaf(h.w, w3.w, acc[i].w);
                }
            }
            float4 xa[ADD ? 8 : 1];
            if constexpr (ADD) {          // (issued after the expansion: the W and H operands are dead by now)
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    xa[i] = (r0 + i < n) ? ld4_addend(addend + (size_t)(r0 + i) * lda + q * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
            if (bias) b4 = ldg4(bias + q * 4);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                if (r0 + i >= n) continue;
                float4 y = make_float4(alpha * (acc[i].x + b4.x), alpha * (acc[i].y + b4.y),
                                       alpha * (acc[i].z + b4.z), alpha * (acc[i].w + b4.w));
                if (use_resid) {
                    y.x = fmaf(beta, xr[i].x, y.x); y.y = fmaf(beta, xr[i].y, y.y);
                    y.z = fmaf(beta, xr[i].z, y.z); y.w = fmaf(beta, xr[i].w, y.w);
                }
                if constexpr (ADD) y = f4_add_rn(y, xa[i]);
                stg4_stream(Out + (size_t)(r0 + i) * ldo + q * 4, y);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// K3-mma: same contract as k_hop_expand, with the [64, R] x [R, d] expansion on the tensor core:
// M = rows (4 m-tiles of 16 per tile), N = output columns, K = R.  The gathered H tile is split into tf32
// hi / lo when it is staged in shared memory; W^T sits in shared memory with an odd row stride so the
// B-fragment loads are conflict-free.  Warp w owns the 32-column blocks w, w+8, ...: lane (g, t) reads the
// residual and writes the output as two float4 (columns cb+8t .. +7) for rows g and g+8 of every m-tile, i.e.
// 8 rows x 128 contiguous bytes per warp instruction.
// ------------------------------------------------------------------------------------------
template <int R, bool W_IS_DR, bool ADD>
__global__ void __launch_bounds__(256, 2)
k_hop_expand_mma(const int* __restrict__ rowptr, const int* __restrict__ colidx, const float* __restrict__ dis,
                 const float* __restrict__ F, const float* __restrict__ W, const float* __restrict__ bias,
                 const float* __restrict__ resid, int64_t ldr, const float* __restrict__ scalar,
                 int alpha_is_scalar, int use_resid, float* __restrict__ Hout, float* __restrict__ Out, int64_t ldo,
                 int n, int d,
    const int* __restrict__ hubitem, const float* __restrict__ hub_part, const float* addend, int64_t lda) {
    constexpr int LPG = R / 4, GPW = 32 / LPG;
    constexpr int RS = R + 4;                       // padded row stride of the H tile
    constexpr int KS = R / 8;                       // k-steps
    extern __shared__ __align__(16) uint32_t smem_u[];
    const int WS = d + 1;                           // odd row stride of W^T
    uint32_t* Wh = smem_u;                          // [R][WS]  tf32 hi
    uint32_t* Wl = Wh + (size_t)R * WS;             // [R][WS]  tf32 lo
    uint32_t* Hh = Wl + (size_t)R * WS;             // [64][RS]
    uint32_t* Hl = Hh + kTileRows * RS;
    if (Out) {
        for (int idx = threadIdx.x; idx < d * R; idx += blockDim.x) {
            int k, c;
            if (W_IS_DR) { k = idx / R; c = idx - k * R; } else { c = idx / d; k = idx - c * d; }
            uint32_t hi, lo;
            split_tf32(W[idx], hi, lo);
            Wh[c * WS + k] = hi;
            Wl[c * WS + k] = lo;
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int sub = lane % LPG, grp = lane / LPG;
    const int g = lane >> 2, t = lane & 3;
    const float s = scalar ? __ldg(scalar) : 1.f;
    const float alpha = alpha_is_scalar ? s : 1.f;
    const float beta = use_resid ? s : 0.f;
    const int nblk = (d + 31) / 32;
    const int ntiles = (n + kTileRows - 1) / kTileRows;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int trow = tile * kTileRows;
        __syncthreads();              // W ready / previous tile's readers of the H tile are done
        for (int rr = warp * GPW; rr < kTileRows; rr += 8 * GPW) {
            const int row = trow + rr + grp;
            const bool valid = row < n;
            const float4 acc = warp_spmm_rows<R>(rowptr, colidx, F, row, valid, lane, hubitem, hub_part);
            float4 h = make_float4(0.f, 0.f, 0.f, 0.f);
            if (valid) {
                h = f4_scale(acc, __ldg(dis + row));
                *reinterpret_cast<float4*>(Hout + (size_t)row * R + sub * 4) = h;
            }
            uint4 hi, lo;
            split_tf32(h.x, hi.x, lo.x); split_tf32(h.y, hi.y, lo.y); split_tf32(h.z, hi.z, lo.z); split_tf32(h.w, hi.w, lo.w);
            *reinterpret_cast<uint4*>(&Hh[(rr + grp) * RS + sub * 4]) = hi;
            *reinterpret_cast<uint4*>(&Hl[(rr + grp) * RS + sub * 4]) = lo;
        }
        __syncthreads();
        if (!Out) continue;
        for (int blk = warp; blk < nblk; blk += 8) {
            const int cb = blk * 32;
            // column permutation inside the 32-column block: n-tile j, n -> col = cb + 4 * perm(n) + j with
            // perm(2t) = t, perm(2t+1) = 4 + t, so the C-fragments of lane (g, t) are the float4s at cb + 4t and
            // cb + 16 + 4t: every load / store instruction covers 64 contiguous bytes (two full sectors) per row.
            const int lc = cb + 4 * ((g >> 1) + 4 * (g & 1));   // B-fragment columns of this lane: lc + j
            const bool lc_ok = lc < d;
            // W fragments of this block: b0 = W[c = 8 ks + t][lc + j], b1 = W[c = 8 ks + t + 4][lc + j]
            uint32_t wh[KS][4][2], wl[KS][4][2];
#pragma unroll
            for (int ks = 0; ks < KS; ++ks)
#pragma unroll
                for (int j = 0; j < 4; ++j)
#pragma unroll
                    for (int h2 = 0; h2 < 2; ++h2) {
                        const int c = ks * 8 + t + 4 * h2;
                        wh[ks][j][h2] = lc_ok ? Wh[c * WS + lc + j] : 0u;
                        wl[ks][j][h2] = lc_ok ? Wl[c * WS + lc + j] : 0u;
                    }
            const int oc = cb + 4 * t, oc1 = cb + 16 + 4 * t;    // output column quads of this lane
            const bool o0 = oc < d, o1 = oc1 < d;
            float4 b4a = make_float4(0.f, 0.f, 0.f, 0.f), b4b = b4a;
            if (bias) { if (o0) b4a = ldg4(bias + oc); if (o1) b4b = ldg4(bias + oc1); }
#pragma unroll(ADD ? 1 : 2)                                 // (ADD: the addend's registers do not fit twice)
            for (int mt = 0; mt < kTileRows / 16; ++mt) {
                const int r0 = trow + mt * 16 + g, r1 = r0 + 8;
                float4 x0a, x0b, x1a, x1b;
                x0a = x0b = x1a = x1b = make_float4(0.f, 0.f, 0.f, 0.f);
                if (use_resid) {
                    if (r0 < n) { if (o0) x0a = ldg4_stream(resid + (size_t)r0 * ldr + oc); if (o1) x0b = ldg4_stream(resid + (size_t)r0 * ldr + oc1); }
                    if (r1 < n) { if (o0) x1a = ldg4_stream(resid + (size_t)r1 * ldr + oc); if (o1) x1b = ldg4_stream(resid + (size_t)r1 * ldr + oc1); }
                }
                float acc[4][4];
#pragma unroll
                for (int j = 0; j < 4; ++j)
#pragma unroll
                    for (int i = 0; i < 4; ++i) acc[j][i] = 0.f;
#pragma unroll
                for (int ks = 0; ks < KS; ++ks) {
                    uint32_t ah[4], al[4];
                    const int hr = (mt * 16 + g) * RS + ks * 8 + t;
                    ah[0] = Hh[hr]; ah[1] = Hh[hr + 8 * RS]; ah[2] = Hh[hr + 4]; ah[3] = Hh[hr + 8 * RS + 4];
                    al[0] = Hl[hr]; al[1] = Hl[hr + 8 * RS]; al[2] = Hl[hr + 4]; al[3] = Hl[hr + 8 * RS + 4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        mma_tf32(acc[j], ah, wh[ks][j][0], wh[ks][j][1]);
                        mma_tf32(acc[j], al, wh[ks][j][0], wh[ks][j][1]);
                        mma_tf32(acc[j], ah, wl[ks][j][0], wl[ks][j][1]);
                    }
                }
                // acc[j][0] = (row g, col oc + j), [1] = (row g, col oc1 + j), [2] / [3] = row g + 8
                auto fin = [&](float a0, float a1, float a2, float a3, const float4& b4, const float4& x) {
                    float4 y = make_float4(alpha * (a0 + b4.x), alpha * (a1 + b4.y), alpha * (a2 + b4.z), alpha * (a3 + b4.w));
                    if (use_resid) {
                        y.x = fmaf(beta, x.x, y.x); y.y = fmaf(beta, x.y, y.y); y.z = fmaf(beta, x.z, y.z); y.w = fmaf(beta, x.w, y.w);
                    }
                    return y;
                };
                if constexpr (!ADD) {
                    if (r0 < n) {
                        if (o0) stg4_stream(Out + (size_t)r0 * ldo + oc, fin(acc[0][0], acc[1][0], acc[2][0], acc[3][0], b4a, x0a));
                        if (o1) stg4_stream(Out + (size_t)r0 * ldo + oc1, fin(acc[0][1], acc[1][1], acc[2][1], acc[3][1], b4b, x0b));
                    }
                    if (r1 < n) {
                        if (o0) stg4_stream(Out + (size_t)r1 * ldo + oc, fin(acc[0][2], acc[1][2], acc[2][2], acc[3][2], b4a, x1a));
                        if (o1) stg4_stream(Out + (size_t)r1 * ldo + oc1, fin(acc[0][3], acc[1][3], acc[2][3], acc[3][3], b4b, x1b));
                    }
                } else {
                    float4 a0a, a0b, a1a, a1b;
                    a0a = a0b = a1a = a1b = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (r0 < n) { if (o0) a0a = ld4_addend(addend + (size_t)r0 * lda + oc); if (o1) a0b = ld4_addend(addend + (size_t)r0 * lda + oc1); }
                    if (r1 < n) { if (o0) a1a = ld4_addend(addend + (size_t)r1 * lda + oc); if (o1) a1b = ld4_addend(addend + (size_t)r1 * lda + oc1); }
                    if (r0 < n) {
                        if (o0) stg4_stream(Out + (size_t)r0 * ldo + oc, f4_add_rn(fin(acc[0][0], acc[1][0], acc[2][0], acc[3][0], b4a, x0a), a0a));
                        if (o1) stg4_stream(Out + (size_t)r0 * ldo + oc1, f4_add_rn(fin(acc[0][1], acc[1][1], acc[2][1], acc[3][1], b4b, x0b), a0b));
                    }
                    if (r1 < n) {
                        if (o0) stg4_stream(Out + (size_t)r1 * ldo + oc, f4_add_rn(fin(acc[0][2], acc[1][2], acc[2][2], acc[3][2], b4a, x1a), a1a));
                        if (o1) stg4_stream(Out + (size_t)r1 * ldo + oc1, f4_add_rn(fin(acc[0][3], acc[1][3], acc[2][3], acc[3][3], b4b, x1b), a1b));
                    }
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// K3-tc: hop + expand with the expansion on the 5th-generation tensor core (tcgen05, accumulator in TMEM) and
// all d-wide traffic moved by the bulk-copy engine.  One persistent 512-thread CTA per SM, 128-row tiles:
//   warps 0-7   gather: the pipelined r-wide SpMM of tile k -> H tile (tf32 hi / lo, UMMA canonical K-major
//               core-matrix layout) in shared memory, double-buffered; H2 rows also go to global memory.
//   warp  8     one thread issues the 3 x (R/8) tcgen05.mma.kind::tf32 of a tile: D[128, d] = H_hi W_hi + H_lo W_hi
//               + H_hi W_lo with W resident in shared memory (K-major, split once per CTA), D in one of two
//               256-column TMEM stages; tcgen05.commit hands the H buffer back and the accumulator over.
//   warps 12-15 epilogue: warp q owns TMEM lanes / tile rows 32q..32q+31, lane = row.  Per 64-column chunk:
//               tcgen05.ld the accumulator, read the residual chunk from this warp's ring slot (filled by a
//               per-row cp.async.bulk, completion on an mbarrier), y = alpha (acc + b) + beta x in place,
//               fence.proxy.async, per-row cp.async.bulk store to Y, then refill the previous slot with the
//               chunk 4 items ahead once its store has drained (wait_group.read).
// The mma.sync variant spends ~3300 cycles of tensor pipe per 64 rows on the 3xTF32 expansion and as much again
// in its store phase, serialised per warp (profiles/README.md); here the tensor work is 6 instructions per tile
// and no d-wide byte passes through a register of a load/store instruction.
// ------------------------------------------------------------------------------------------
constexpr int kTcRows = 128;
constexpr int kTcChunk = 64;                    // columns per epilogue item = two 32-column TMA boxes
template <int R> __host__ __device__ constexpr int tc_slots() { return R <= 16 ? 4 : 3; }   // ring slots per epilogue warp (what fits next to W and H)
constexpr int kTcQ = 8;                         // entries of the per-CTA tile queue
constexpr int kTcBoxBytes = 32 * 32 * 4;        // one box: 32 rows x 128 bytes, SWIZZLE_128B (1 KB atoms)
constexpr int kTcSlotBytes = 2 * kTcBoxBytes;

template <int R>
constexpr size_t hop_expand_tc_smem(int d) {
    return (size_t)2 * R * d * 4 + (size_t)4 * R * kTcRows * 4 + (size_t)4 * tc_slots<R>() * kTcSlotBytes + (size_t)d * 4 + 64 * 8 + 64 + 1024;
}

template <int R, bool W_IS_DR, bool ADD>
__global__ void __launch_bounds__(512, 1)
k_hop_expand_tc(const int* __restrict__ rowptr, const int* __restrict__ colidx, const float* __restrict__ dis,
                const float* __restrict__ F, const float* __restrict__ W, const float* __restrict__ bias,
                const float* __restrict__ resid, int64_t ldr, const float* __restrict__ scalar,
                int alpha_is_scalar, int use_resid, float* __restrict__ Hout, float* __restrict__ Out, int64_t ldo,
                int n, int d, const int* __restrict__ hubitem, const float* __restrict__ hub_part,
                const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_y, int pregathered,
                const float* addend, int64_t lda) {
    constexpr int LPG = R / 4, GPW = 32 / LPG;
    constexpr int kTcSlots = tc_slots<R>();
    constexpr int SCA = (kTcRows >> 3) * 128;          // bytes between 4-column K chunks of the H tile
    constexpr int kHPart = R * kTcRows * 4;            // one of {hi, lo} of one H buffer
    extern __shared__ uint8_t smem_unaligned[];
    // (pointer arithmetic on the array, not an integer round trip, so the accesses stay LDS/STS instead of generic LD/ST)
    uint8_t* smem_raw = smem_unaligned + ((1024u - (smem_addr(smem_unaligned) & 1023u)) & 1023u);
    const int SCW = (d >> 3) * 128;                    // bytes between 4-column K chunks of W ([d, R], K-major)
    uint8_t* Wh = smem_raw;
    uint8_t* Wl = Wh + (size_t)R * d * 4;
    uint8_t* Hb = Wl + (size_t)R * d * 4;              // [2 buffers][hi, lo][kHPart]
    uint8_t* Xr = Hb + 4 * kHPart;                     // [4 warps][kTcSlots][2 boxes][32 rows][128 B swizzled]; 1 KB aligned
    float* bias_s = reinterpret_cast<float*>(Xr + 4 * kTcSlots * kTcSlotBytes);
    uint64_t* bars = reinterpret_cast<uint64_t*>(bias_s + d);
    const uint32_t bar0 = smem_addr(bars);
    auto hfull = [&](int b) { return bar0 + 8u * b; };
    auto hempty = [&](int b) { return bar0 + 8u * (2 + b); };
    auto tfull = [&](int a) { return bar0 + 8u * (4 + a); };
    auto tempty = [&](int a) { return bar0 + 8u * (6 + a); };
    auto xfull = [&](int q, int s_) { return bar0 + 8u * (8 + q * kTcSlots + s_); };
    // tile queue: the scheduler thread (warp 9) publishes the CTA's tile sequence, the 13 consumer warps read it
    auto qfull = [&](int i) { return bar0 + 8u * (8 + 4 * kTcSlots + i); };
    auto qempty = [&](int i) { return bar0 + 8u * (8 + 4 * kTcSlots + kTcQ + i); };
    int* tileq = reinterpret_cast<int*>(bars + 8 + 4 * kTcSlots + 2 * kTcQ);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tileq + kTcQ);

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
        for (int b = 0; b < 2; ++b) { mbar_init(hfull(b), 8); mbar_init(hempty(b), 1); mbar_init(tfull(b), 1); mbar_init(tempty(b), 4); }
        for (int i = 0; i < 4 * kTcSlots; ++i) mbar_init(bar0 + 8u * (8 + i), 1);
        for (int i = 0; i < kTcQ; ++i) { mbar_init(qfull(i), 1); mbar_init(qempty(i), 13); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 8) tc::tmem_alloc(smem_addr(tmem_slot), 512);
    // W -> shared, split, canonical K-major layout: element (c, k) -> (k/4) SCW + (c/8) 128 + (c%8) 16 + (k%4) 4
    // (128-bit loads, all of a thread's loads in flight together: the prologue is not hidden behind anything when
    // the previous kernel's CTA still owns the shared memory of this SM)
#pragma unroll 2
    for (int idx4 = threadIdx.x; idx4 < (d * R) / 4; idx4 += blockDim.x) {
        const int idx = idx4 * 4;
        const float4 w4 = ldg4(W + idx);
        const float wv[4] = {w4.x, w4.y, w4.z, w4.w};
        uint32_t hi[4], lo[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) split_tf32(wv[e], hi[e], lo[e]);
        if (W_IS_DR) {                                  // 4 consecutive k of one output column c: one 16-byte slot
            const int c = idx / R, k = idx - c * R;
            const uint32_t off = (uint32_t)((k >> 2) * SCW + (c >> 3) * 128 + (c & 7) * 16);
            *reinterpret_cast<uint4*>(Wh + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
            *reinterpret_cast<uint4*>(Wl + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        } else {                                        // 4 consecutive columns c of one k
            const int k = idx / d, c0 = idx - k * d;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int c = c0 + e;
                const uint32_t off = (uint32_t)((k >> 2) * SCW + (c >> 3) * 128 + (c & 7) * 16 + (k & 3) * 4);
                *reinterpret_cast<uint32_t*>(Wh + off) = hi[e];
                *reinterpret_cast<uint32_t*>(Wl + off) = lo[e];
            }
        }
    }
    for (int i = threadIdx.x; i < d; i += blockDim.x) bias_s[i] = bias ? bias[i] : 0.f;
    tc::fence_proxy_async();
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_wait();
    pdl_trigger();

    const int ntiles = (n + kTcRows - 1) / kTcRows;
    // i-th tile of this CTA (or -1 after the last one); every consumer warp calls this exactly once per i, in order
    auto get_tile = [&](int i) {
        mbar_wait(qfull(i % kTcQ), (uint32_t)((i / kTcQ) & 1));
        const int t_ = tileq[i % kTcQ];
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(qempty(i % kTcQ));
        return t_;
    };

    if (warp < 8) {
        // ===================== gather warps (same software pipeline as K3-ws) =====================
        const int sub = lane % LPG, grp = lane / LPG;
        constexpr int PASSES = kTcRows / (8 * GPW);
        constexpr int kPre = 16;
        static_assert(PASSES >= 2, "the look-ahead below assumes that steps s .. s+2 span at most two tiles");
        int tk = get_tile(0), tk1 = tk >= 0 ? get_tile(1) : -1;    // tiles of step s and of the tile after it
        auto row_in = [&](int tile, int ps) { return tile * kTcRows + ps * 8 * GPW + warp * GPW + grp; };
        struct Meta { int beg, end; float dis; };
        auto meta_load = [&](int tile, int ps) {
            Meta m{0, 0, 0.f};
            if (tile >= 0 && !pregathered) {
                const int row = row_in(tile, ps);
                if (row < n) { m.beg = __ldg(rowptr + row); m.end = __ldg(rowptr + row + 1); m.dis = __ldg(dis + row); }
            }
            return m;
        };
        auto idx_load = [&](const Meta& m, int (&j)[kPre]) {
            const bool fast = m.end - m.beg <= kLongRow;
#pragma unroll
            for (int u = 0; u < kPre; ++u) j[u] = (fast && m.beg + u < m.end) ? __ldg(colidx + m.beg + u) : -1;
        };
        // pregathered = 1 (second half of a split K3): H is already in global memory, the warps only stage their rows
        auto hrow_load = [&](int tile, int ps) {
            float4 h_ = make_float4(0.f, 0.f, 0.f, 0.f);
            if (pregathered && tile >= 0) {
                const int row = row_in(tile, ps);
                if (row < n) h_ = ldg4(Hout + (size_t)row * R + sub * 4);
            }
            return h_;
        };
        float4 hp0 = hrow_load(tk, 0), hp1 = hrow_load(tk, 1);
        Meta m0 = meta_load(tk, 0), m1 = meta_load(tk, 1);
        int j0[kPre], j1[kPre];
        idx_load(m0, j0);
        for (int s_ = 0; tk >= 0; ++s_) {
            const int k = s_ / PASSES, ps = s_ - k * PASSES, b = k & 1;
            const float4 hp2 = ps + 2 < PASSES ? hrow_load(tk, ps + 2) : hrow_load(tk1, ps + 2 - PASSES);
            // step s+2: pass ps+2 of this tile, or pass ps+2-PASSES of the next one
            const Meta m2 = ps + 2 < PASSES ? meta_load(tk, ps + 2) : meta_load(tk1, ps + 2 - PASSES);
            idx_load(m1, j1);
            float4 v[kPre];
#pragma unroll
            for (int u = 0; u < kPre; ++u)
                v[u] = (j0[u] >= 0) ? ldg4(F + (size_t)j0[u] * R + sub * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int u = 0; u < kPre; ++u) acc = f4_add(acc, v[u]);
            const int row = row_in(tk, ps);
            const bool valid = row < n;
            const int deg = m0.end - m0.beg;
            const bool is_hub = deg > kHubDeg;
            const bool is_long = deg > kLongRow && !is_hub;
            if (is_hub) {
                acc = hub_row_sum<R>(hub_part, __ldg(hubitem + row), (deg + kHubChunk - 1) / kHubChunk, sub);
            } else if (!is_long && deg > kPre) {
                const float4 rest = gather_rows<R>(F, colidx, m0.beg + kPre, m0.end, 1, sub);
                acc = f4_add(acc, rest);
            }
            unsigned longmask = __ballot_sync(0xffffffffu, is_long);
            while (longmask) {                                   // warp-uniform
                const int src = __ffs(longmask) - 1;
                const int g_ = src / LPG;
                const unsigned gm = (LPG >= 32) ? 0xffffffffu : (((1u << LPG) - 1u) << (g_ * LPG));
                longmask &= ~gm;
                const int lb = __shfl_sync(0xffffffffu, m0.beg, src), le = __shfl_sync(0xffffffffu, m0.end, src);
                float4 part = gather_rows<R>(F, colidx, lb + grp, le, GPW, sub);
#pragma unroll
                for (int off = LPG; off < 32; off <<= 1) part = f4_add(part, f4_shfl_xor(part, off));
                if (grp == g_) acc = part;
            }
            float4 h = make_float4(0.f, 0.f, 0.f, 0.f);
            if (pregathered) {
                h = hp0;
            } else if (valid) {
                h = f4_scale(acc, m0.dis);
                *reinterpret_cast<float4*>(Hout + (size_t)row * R + sub * 4) = h;
            }
            uint4 hi, lo;
            split_tf32(h.x, hi.x, lo.x); split_tf32(h.y, hi.y, lo.y); split_tf32(h.z, hi.z, lo.z); split_tf32(h.w, hi.w, lo.w);
            if (ps == 0 && k >= 2) mbar_wait(hempty(b), (uint32_t)(((k >> 1) - 1) & 1));   // MMAs of tile k-2 have retired
            const int hr = ps * 8 * GPW + warp * GPW + grp;
            const uint32_t off = (uint32_t)(sub * SCA + (hr >> 3) * 128 + (hr & 7) * 16);
            *reinterpret_cast<uint4*>(Hb + (size_t)(b * 2) * kHPart + off) = hi;
            *reinterpret_cast<uint4*>(Hb + (size_t)(b * 2 + 1) * kHPart + off) = lo;
            if (ps == PASSES - 1) {
                tc::fence_proxy_async();                          // generic-proxy writes -> visible to the tensor core
                __syncwarp();
                if (lane == 0) tc::mbar_arrive(hfull(b));
            }
            m0 = m1; m1 = m2;
            hp0 = hp1; hp1 = hp2;
#pragma unroll
            for (int u = 0; u < kPre; ++u) j0[u] = j1[u];
            if (ps == PASSES - 1) { tk = tk1; tk1 = tk >= 0 ? get_tile(k + 2) : -1; }
        }
    } else if (warp == 8) {
        // ===================== MMA issuer =====================
        if (lane == 0) {
            const uint32_t idesc = tc::make_idesc_tf32(kTcRows, d, 0, 0);
            const uint64_t stepA = (uint64_t)((2 * SCA) >> 4), stepB = (uint64_t)((2 * SCW) >> 4);
            const uint64_t b_hi = tc::make_desc(smem_addr(Wh), (uint32_t)SCW, 128), b_lo = tc::make_desc(smem_addr(Wl), (uint32_t)SCW, 128);
            for (int k = 0;; ++k) {
                // (lane 0 only: the queue hand-shake is done by hand instead of get_tile's warp-wide version)
                mbar_wait(qfull(k % kTcQ), (uint32_t)((k / kTcQ) & 1));
                const int tile_k = tileq[k % kTcQ];
                tc::mbar_arrive(qempty(k % kTcQ));
                if (tile_k < 0) break;
                const int b = k & 1;
                mbar_wait(hfull(b), (uint32_t)((k >> 1) & 1));
                mbar_wait(tempty(b), (uint32_t)(((k >> 1) & 1) ^ 1));
                tc::tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(b * 256);
                const uint64_t a_hi = tc::make_desc(smem_addr(Hb + (size_t)(b * 2) * kHPart), SCA, 128);
                const uint64_t a_lo = tc::make_desc(smem_addr(Hb + (size_t)(b * 2 + 1) * kHPart), SCA, 128);
#pragma unroll
                for (int ks = 0; ks < R / 8; ++ks) {
                    tc::umma_tf32(d_tmem, a_lo + ks * stepA, b_hi + ks * stepB, idesc, ks > 0 ? 1u : 0u);
                    tc::umma_tf32(d_tmem, a_hi + ks * stepA, b_lo + ks * stepB, idesc, 1u);
                    tc::umma_tf32(d_tmem, a_hi + ks * stepA, b_hi + ks * stepB, idesc, 1u);
                }
                tc::umma_commit(hempty(b));
                tc::umma_commit(tfull(b));
            }
        }
    } else if (warp == 9) {
        // ===================== tile scheduler =====================
        // static round-robin tile sequence (a global tile counter measured slower: 81 vs 76 us, profiles/README.md)
        if (lane == 0) {
            for (int i = 0;; ++i) {
                int t_ = (int)blockIdx.x + i * (int)gridDim.x;
                if (t_ >= ntiles) t_ = -1;
                if (i >= kTcQ) mbar_wait(qempty(i % kTcQ), (uint32_t)(((i / kTcQ) - 1) & 1));
                tileq[i % kTcQ] = t_;
                tc::mbar_arrive(qfull(i % kTcQ));                   // release: consumers acquire through their wait
                if (t_ < 0) break;
            }
        }
    } else if (warp >= 12) {
        // ===================== epilogue =====================
        const int q = warp & 3;
        const float s = scalar ? __ldg(scalar) : 1.f;
        const float alpha = alpha_is_scalar ? s : 1.f;
        const float beta = use_resid ? s : 0.f;
        const int nchunk = d / kTcChunk;
        const int lead = nchunk < kTcSlots - 1 ? nchunk : kTcSlots - 1;   // items between a chunk's load and its use
        const uint64_t pol = policy_evict_first();
        uint8_t* myslots = Xr + (size_t)q * kTcSlots * kTcSlotBytes;
        int tk = get_tile(0), tk1 = tk >= 0 ? get_tile(1) : -1;    // this tile and the next one (loads run ahead into it)
        auto issue_load = [&](int tile, int c_, int it_) {         // residual chunk c_ of `tile` = item it_ -> ring slot (lane 0)
            const int slot = it_ % kTcSlots;
            const int row0 = tile * kTcRows + q * 32;
            const uint32_t dst = smem_addr(myslots + (size_t)slot * kTcSlotBytes);
            mbar_arrive_expect_tx(xfull(q, slot), (uint32_t)kTcSlotBytes);
            tma_load_box(dst, &tm_x, c_ * kTcChunk, row0, xfull(q, slot), pol);
            tma_load_box(dst + kTcBoxBytes, &tm_x, c_ * kTcChunk + 32, row0, xfull(q, slot), pol);
        };
        if (use_resid && lane == 0 && tk >= 0)
            for (int c_ = 0; c_ < lead; ++c_) issue_load(tk, c_, c_);
        const int sw = lane & 7;                                   // 16-byte chunk j of row `lane` sits at chunk j ^ (lane % 8)
        // ADD: the addend's 32 columns from col0 of row `lane` of `tile` (zeros past the last row)
        auto load_half = [&](int tile, int col0, float4 (&dst)[8]) {
            const int row = tile * kTcRows + q * 32 + lane;
            const bool ok = row < n;
#pragma unroll
            for (int j = 0; j < 8; ++j)
                dst[j] = ok ? ld4_addend(addend + (size_t)row * lda + col0 + 4 * j) : make_float4(0.f, 0.f, 0.f, 0.f);
        };
        int it = 0;
        for (int k = 0; tk >= 0; ++k) {
            const int b = k & 1;
            const int row0 = tk * kTcRows + q * 32;
            mbar_wait(tfull(b), (uint32_t)((k >> 1) & 1));
            tc::tc_fence_after();
            const uint32_t tb = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(b * 256);
            for (int c = 0; c < nchunk; ++c, ++it) {
                const int slot = it % kTcSlots;
                if constexpr (!ADD) {
                    float acc[kTcChunk];
                    tmem_ld32(tb + (uint32_t)(c * kTcChunk), acc);
                    tmem_ld32(tb + (uint32_t)(c * kTcChunk + 32), acc + 32);
                    if (use_resid) mbar_wait(xfull(q, slot), (uint32_t)((it / kTcSlots) & 1));
                    tmem_ld_wait();
                    if (c == nchunk - 1) {                              // accumulator stage can be overwritten
                        tc::tc_fence_before();
                        __syncwarp();
                        if (lane == 0) tc::mbar_arrive(tempty(b));
                    }
                    uint8_t* slotp = myslots + (size_t)slot * kTcSlotBytes + (size_t)lane * 128;
                    const float4* bs = reinterpret_cast<const float4*>(bias_s + c * kTcChunk);
                    // all loads of a half chunk first, then the arithmetic, then the stores: the compiler cannot tell that
                    // the swizzled in-place stores do not alias the later loads and would otherwise serialise them
#pragma unroll
                    for (int h = 0; h < 4; ++h) {                       // quarter chunks of 16 columns
                        float4 xv[4], bv[4];
#pragma unroll
                        for (int jj = 0; jj < 4; ++jj) {
                            const int j = h * 4 + jj;
                            bv[jj] = bs[j];
                            xv[jj] = use_resid ? *reinterpret_cast<const float4*>(slotp + (j >> 3) * kTcBoxBytes + (((j & 7) ^ sw) << 4))
                                               : make_float4(0.f, 0.f, 0.f, 0.f);
                        }
#pragma unroll
                        for (int jj = 0; jj < 4; ++jj) {
                            const int j = h * 4 + jj;
                            float4 y = make_float4(alpha * (acc[4 * j] + bv[jj].x), alpha * (acc[4 * j + 1] + bv[jj].y),
                                                   alpha * (acc[4 * j + 2] + bv[jj].z), alpha * (acc[4 * j + 3] + bv[jj].w));
                            y.x = fmaf(beta, xv[jj].x, y.x); y.y = fmaf(beta, xv[jj].y, y.y);
                            y.z = fmaf(beta, xv[jj].z, y.z); y.w = fmaf(beta, xv[jj].w, y.w);
                            xv[jj] = y;
                        }
#pragma unroll
                        for (int jj = 0; jj < 4; ++jj) {
                            const int j = h * 4 + jj;
                            *reinterpret_cast<float4*>(slotp + (j >> 3) * kTcBoxBytes + (((j & 7) ^ sw) << 4)) = xv[jj];
                        }
                    }
                } else {
                    // Y = (...) + A.  Lane = row; A comes in 32-column halves of 128-bit loads into registers (the 128
                    // registers of the kernel leave no room for a whole chunk, or for the next half, next to the
                    // accumulator), issued before the half waits on TMEM and the residual.  The next chunk's bytes are
                    // prefetched into L2 one chunk ahead (no shared memory is left for a ring of A), so those loads hit L2.
                    // Every load of chunk c is consumed before chunk c's store is issued, which is what makes Y == A safe.
                    uint8_t* slotp = myslots + (size_t)slot * kTcSlotBytes + (size_t)lane * 128;
                    const float4* bs = reinterpret_cast<const float4*>(bias_s + c * kTcChunk);
                    {
                        const int cn = c + 1 < nchunk ? c + 1 : 0, tile_n = c + 1 < nchunk ? tk : tk1;
                        const int prow = tile_n * kTcRows + q * 32 + lane;
                        if (tile_n >= 0 && prow < n) prefetch_l2_bulk(addend + (size_t)prow * lda + cn * kTcChunk, kTcChunk * 4);
                    }
#pragma unroll
                    for (int hh = 0; hh < 2; ++hh) {
                        float4 cur[8];
                        load_half(tk, c * kTcChunk + hh * 32, cur);
                        float acc[32];
                        tmem_ld32(tb + (uint32_t)(c * kTcChunk + hh * 32), acc);
                        if (hh == 0 && use_resid) mbar_wait(xfull(q, slot), (uint32_t)((it / kTcSlots) & 1));
                        tmem_ld_wait();
                        if (hh == 1 && c == nchunk - 1) {                   // accumulator stage can be overwritten
                            tc::tc_fence_before();
                            __syncwarp();
                            if (lane == 0) tc::mbar_arrive(tempty(b));
                        }
#pragma unroll
                        for (int h2 = 0; h2 < 4; ++h2) {                   // batches of 2 float4 (registers are at the cap)
                            float4 xv[2], bv[2];
#pragma unroll
                            for (int jj = 0; jj < 2; ++jj) {
                                const int j = hh * 8 + h2 * 2 + jj;
                                bv[jj] = bs[j];
                                xv[jj] = use_resid ? *reinterpret_cast<const float4*>(slotp + (j >> 3) * kTcBoxBytes + (((j & 7) ^ sw) << 4))
                                                   : make_float4(0.f, 0.f, 0.f, 0.f);
                            }
#pragma unroll
                            for (int jj = 0; jj < 2; ++jj) {
                                const int e = h2 * 2 + jj;
                                float4 y = make_float4(alpha * (acc[4 * e] + bv[jj].x), alpha * (acc[4 * e + 1] + bv[jj].y),
                                                       alpha * (acc[4 * e + 2] + bv[jj].z), alpha * (acc[4 * e + 3] + bv[jj].w));
                                y.x = fmaf(beta, xv[jj].x, y.x); y.y = fmaf(beta, xv[jj].y, y.y);
                                y.z = fmaf(beta, xv[jj].z, y.z); y.w = fmaf(beta, xv[jj].w, y.w);
                                xv[jj] = f4_add_rn(y, cur[e]);
                            }
#pragma unroll
                            for (int jj = 0; jj < 2; ++jj) {
                                const int j = hh * 8 + h2 * 2 + jj;
                                *reinterpret_cast<float4*>(slotp + (j >> 3) * kTcBoxBytes + (((j & 7) ^ sw) << 4)) = xv[jj];
                            }
                        }
                    }
                }
                tc::fence_proxy_async();                           // generic-proxy writes -> visible to the bulk store
                __syncwarp();
                if (lane == 0) {
                    const uint32_t src = smem_addr(myslots + (size_t)slot * kTcSlotBytes);
                    tma_store_box(&tm_y, c * kTcChunk, row0, src, pol);
                    tma_store_box(&tm_y, c * kTcChunk + 32, row0, src + kTcBoxBytes, pol);
                    bulk_commit();
                    if (it >= 1) bulk_wait_read<1>();              // the store of item it-1 has left its slot ...
                    if (use_resid) {                               // ... which item it+lead may now be loaded into
                        int cn = c + lead;
                        const int tile_n = cn < nchunk ? tk : tk1;
                        if (cn >= nchunk) cn -= nchunk;
                        if (tile_n >= 0) issue_load(tile_n, cn, it + lead);
                    }
                }
                __syncwarp();                                       // nobody rewrites a slot before lane 0 saw it drained
            }
            tk = tk1;
            tk1 = tk >= 0 ? get_tile(k + 2) : -1;
        }
        bulk_wait_all();
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 8) {
        tc::tc_fence_after();
        tc::tmem_dealloc(tmem_base, 512);
    }
}

template <int R, bool W_IS_DR, bool ADD>
int launch_hop_expand_fused_t(const Csr& c, const float* F, const float* W,
                              const float* bias, const float* resid, int64_t ldr, const float* scalar, int alpha_is_scalar,
                              int use_resid, float* Hout, float* Out, int64_t ldo, int n, int d, const float* addend, int64_t lda,
                              cudaStream_t st) {
    GCA_TRY(launch_hub_partials(R, c, F, st));
    const int* rowptr = c.rowptr; const int* colidx = c.colidx; const float* dis = c.dis;
    if constexpr (R == 16 || R == 32) {
        if (tc_enabled()) {
            // tcgen05 + tensor-map TMA variant
            const bool tc_ok = Out && d <= 256 && n >= 4 * kTcRows && (d % kTcChunk) == 0 && (ldo % 4) == 0 &&
                               (reinterpret_cast<uintptr_t>(Out) % 16) == 0 && hop_expand_tc_smem<R>(d) <= 227 * 1024 &&
                               (!use_resid || (resid && (ldr % 4) == 0 && (reinterpret_cast<uintptr_t>(resid) % 16) == 0));
            CUtensorMap tm_x, tm_y;
            // (a driver without cuTensorMapEncodeTiled, or a tensor it refuses, leaves the mma.sync kernel below)
            if (tc_ok && get_box_map(&tm_y, Out, n, d, ldo, 32, 32, true) &&
                get_box_map(&tm_x, use_resid ? resid : Out, n, d, use_resid ? ldr : ldo, 32, 32, true)) {
                // When the gathered operand is far larger than L2 the neighbour rows come from HBM and the 8 gather warps of
                // the fused kernel cannot keep enough of them in flight: run the hop as its own high-occupancy kernel
                // (k_hop, plain mode: 64 warps per SM) and let the fused kernel only expand the H it left in global memory.
                const int pregathered = (long long)c.n_full * R * 4 > split_bytes() ? 1 : 0;
                if (pregathered)
                    GCA_TRY(launch_hop(R, false, c, F, nullptr, GCA_ACT_NONE, nullptr, nullptr, Hout, nullptr, nullptr, nullptr, n, st, 1,
                                       W_IS_DR ? "hop_plain_fwd" : "hop_plain_bwd"));
                const char* prof_k3 = pregathered ? (W_IS_DR ? "expand_fwd" : "expand_bwd") : (W_IS_DR ? "hop_expand_fwd" : "hop_expand_bwd");
                const size_t smem_tc = hop_expand_tc_smem<R>(d);
                GCA_TRY(set_smem(k_hop_expand_tc<R, W_IS_DR, ADD>, smem_tc));
                const int ntiles_t = (n + kTcRows - 1) / kTcRows;
                const int grid_t = ntiles_t < num_sms() ? ntiles_t : num_sms();
                {
                    ProfScope ps(prof_k3, st, "tcgen05");
                    GCA_CUDA(launch_pdl(k_hop_expand_tc<R, W_IS_DR, ADD>, dim3(grid_t), dim3(512), smem_tc, st, rowptr, colidx, dis, F, W,
                                        bias, resid, ldr, scalar, alpha_is_scalar, use_resid, Hout, Out, ldo, n, d, c.hubitem, c.hub_part,
                                        tm_x, tm_y, pregathered, addend, lda));
                }
                GCA_LAUNCH_OK();
                return GCA_OK;
            }
            const size_t smem_m = sizeof(uint32_t) * ((size_t)2 * R * (d + 1) + (size_t)2 * kTileRows * (R + 4));
            if (smem_m <= 200 * 1024) {
                GCA_TRY(set_smem(k_hop_expand_mma<R, W_IS_DR, ADD>, smem_m));
                const int ntiles_m = (n + kTileRows - 1) / kTileRows;
                const int per_sm = smem_m <= 100 * 1024 ? 2 : 1;
                const int grid_m = ntiles_m < per_sm * num_sms() ? ntiles_m : per_sm * num_sms();
                {
                    ProfScope ps(W_IS_DR ? "hop_expand_fwd" : "hop_expand_bwd", st, "mma");
                    k_hop_expand_mma<R, W_IS_DR, ADD><<<grid_m, 256, smem_m, st>>>(rowptr, colidx, dis, F, W, bias, resid, ldr, scalar,
                                                                                   alpha_is_scalar, use_resid, Hout, Out, ldo, n, d, c.hubitem,
                                                                                   c.hub_part, addend, lda);
                }
                GCA_LAUNCH_OK();
                return GCA_OK;
            }
        }
    }
    const size_t smem = sizeof(float) * ((size_t)R * d + (size_t)kTileRows * R);
    if (smem > 200 * 1024) return GCA_ERR_UNSUPPORTED;
    GCA_TRY(set_smem(k_hop_expand<R, W_IS_DR, ADD>, smem));
    const int ntiles = (n + kTileRows - 1) / kTileRows;
    const int grid = ntiles < 2 * num_sms() ? ntiles : 2 * num_sms();
    {
        ProfScope ps(W_IS_DR ? "hop_expand_fwd" : "hop_expand_bwd", st, "ffma");
        k_hop_expand<R, W_IS_DR, ADD><<<grid, 256, smem, st>>>(rowptr, colidx, dis, F, W, bias, resid, ldr, scalar,
                                                                alpha_is_scalar, use_resid, Hout, Out, ldo, n, d, c.hubitem, c.hub_part,
                                                                addend, lda);
    }
    GCA_LAUNCH_OK();
    return GCA_OK;
}

// r = 128: the hop as its own kernel (k_hop, plain mode: H -> Hout), then the FFMA expansion of H by column blocks of
// kPreCols (k_hop_expand<128, ., ., PRE>, blockIdx.y = block).  H has the bits of the fused kernels' H (the same gather).
template <bool W_IS_DR, bool ADD>
int launch_hop_expand_wide(const Csr& c, const float* F, const float* W, const float* bias, const float* resid, int64_t ldr,
                           const float* scalar, int alpha_is_scalar, int use_resid, float* Hout, float* Out, int64_t ldo, int n,
                           int d, const float* addend, int64_t lda, cudaStream_t st) {
    constexpr int R = 128;
    GCA_TRY(launch_hop(R, false, c, F, nullptr, GCA_ACT_NONE, nullptr, nullptr, Hout, nullptr, nullptr, nullptr, n, st, 1,
                       W_IS_DR ? "hop_plain_fwd" : "hop_plain_bwd"));
    if (!Out) return GCA_OK;
    const size_t smem = sizeof(float) * ((size_t)R * kPreCols + (size_t)kTileRows * R);   // 96 KB: two CTAs per SM
    GCA_TRY(set_smem(k_hop_expand<R, W_IS_DR, ADD, true>, smem));
    const int ncb = (d + kPreCols - 1) / kPreCols;
    const int ntiles = (n + kTileRows - 1) / kTileRows;
    int gx = (2 * num_sms() + ncb - 1) / ncb;
    if (gx > ntiles) gx = ntiles;
    {
        ProfScope ps(W_IS_DR ? "expand_fwd" : "expand_bwd", st, "ffma");
        k_hop_expand<R, W_IS_DR, ADD, true><<<dim3(gx, ncb), 256, smem, st>>>(c.rowptr, c.colidx, c.dis, F, W, bias, resid, ldr,
                                                                            scalar, alpha_is_scalar, use_resid, Hout, Out, ldo, n,
                                                                            d, c.hubitem, c.hub_part, addend, lda);
    }
    GCA_LAUNCH_OK();
    return GCA_OK;
}

template <int R, bool W_IS_DR, bool ADD>
int launch_hop_expand_t(const Csr& c, const float* F, const float* W,
                        const float* bias, const float* resid, int64_t ldr, const float* scalar, int alpha_is_scalar,
                        int use_resid, float* Hout, float* Out, int64_t ldo, int n, int d, const float* addend, int64_t lda,
                        cudaStream_t st) {
    if (n == 0) return GCA_OK;
    if constexpr (R == 128)
        return launch_hop_expand_wide<W_IS_DR, ADD>(c, F, W, bias, resid, ldr, scalar, alpha_is_scalar, use_resid, Hout, Out, ldo,
                                                    n, d, addend, lda, st);
    else
        return launch_hop_expand_fused_t<R, W_IS_DR, ADD>(c, F, W, bias, resid, ldr, scalar, alpha_is_scalar, use_resid, Hout, Out,
                                                          ldo, n, d, addend, lda, st);
}

}  // namespace

int launch_hop_expand(int r, bool w_is_dr, const Csr& c, const float* F, const float* W, const float* bias, const float* resid,
                      int64_t ldr, const float* scalar, int alpha_is_scalar, int use_resid, float* Hout, float* Out, int64_t ldo,
                      int n, int d, cudaStream_t st, const float* addend, int64_t lda) {
    // the addend is forward-only (Y = ... + A); the variant choice inside does not depend on it
    if (w_is_dr && addend) {
        GCA_DISPATCH_R(r, (launch_hop_expand_t<R_, true, true>(c, F, W, bias, resid, ldr, scalar, alpha_is_scalar, use_resid, Hout, Out, ldo,
                                                               n, d, addend, lda, st)));
    }
    if (addend) return GCA_ERR_UNSUPPORTED;
    if (w_is_dr) {
        GCA_DISPATCH_R(r, (launch_hop_expand_t<R_, true, false>(c, F, W, bias, resid, ldr, scalar, alpha_is_scalar, use_resid, Hout, Out,
                                                                ldo, n, d, nullptr, 0, st)));
    }
    GCA_DISPATCH_R(r, (launch_hop_expand_t<R_, false, false>(c, F, W, bias, resid, ldr, scalar, alpha_is_scalar, use_resid, Hout, Out, ldo,
                                                             n, d, nullptr, 0, st)));
}

}  // namespace gca
