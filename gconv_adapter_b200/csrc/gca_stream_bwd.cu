// Backward tail in ONE pass over the d-wide tensors:   gX = gP Wd + s gY ,  gWd partials = gP^T X ,  <gY, X>.
//
// Before this kernel the backward read gY four times (projection, weight gradient up, residual of K3-bwd, <gY, X> of
// wgrad_down) where the minimum is two (SURVEY.md section 8d).  bwd_up (gca_stream.cu) folded the first two; this kernel
// folds the last two and the X pass: after a plain r-wide hop produced gP (k_hop, gca_hop.cu), gY and X cross HBM once each
// and gX is written once - 12 N d bytes instead of 8 N d (K3-bwd) + 8 N d (wgrad_down).
//
// Structure = the TMA-fed ring of gca_stream.cu with 16-row tiles (a stage holds the X tile, the gY tile and the gP tile):
//   warp 0      producer (one thread issues the boxes of a stage once all box warps released it)
//   warps 1-8   box warp w owns the 32-column box w of every tile:
//     expansion   C[16 rows, 32 cols] = gP_tile[16, R] Wd[R, 32 cols]: A = gP rows (fp16 hi / lo, per-tile scale), B = this warp's
//                 Wd fragments (registers, split once);  gX = C + s gY is written IN PLACE over the gY box and leaves through a
//                 tensor-map TMA store; the stage is released one tile later, when that store has drained.
//     weight grad G[R, 32 cols] += gP_tile^T X_box: A = movmatrix.trans of the expansion's A fragments (the same 16 rows are the
//                 k dimension), B = the X box (fp16 hi / lo, per-box scale); accumulators in registers for the whole kernel,
//                 unscaled and folded every tile -> ONE partial per CTA.
//     <gY, X>     at the positions of the expansion's C fragments, where gY is read anyway.
// Row permutation rho (matrix row m of the 16-row m-tile -> tile row): rho(m) = 2 p(m) + 8 (m >> 2) for m < 8 with
// p(m) = (m & 3) ^ (m >> 2), rho(m + 8) = rho(m) + 1.  It makes every shared-memory access of a warp conflict-free under
// the 128-byte swizzle: the C-fragment float2s (rows rho(g): four different row pairs per half warp) and the float4 B-fragment
// loads (rows rho(2t), rho(2t+1), rho(2t+8), rho(2t+9): four different row pairs per quarter warp).
// The gP tile is read through a [n/2, 32]-float view at r = 16 (two nodes per 128-byte row, 128-byte swizzle): 2-way conflicts
// instead of the 8-way ones of 64-byte rows.
//
// Reference semantics: autograd of conv_down (/root/reference/src/finetune/gconv_adapter.py:92) + the skip (:94-95).
#include <cstdlib>
#include <initializer_list>

#include "gca_common.cuh"
#include "gca_device.cuh"
#include "gca_host.cuh"
#include "gca_stream.cuh"

namespace gca {
namespace {

constexpr int kXRows = 16;                 // rows per tile
constexpr int kXBox = 32 * kXRows * 4;     // one 32-column box of a tile: 2 KB, SWIZZLE_128B
constexpr int kXWarps = 8;                 // box warps = column boxes of a 256-wide tile

struct ExpandParams {
    const float* Wd; const float* scalar;
    float* partG; float* partDot; int* header; int slot;
    int n, d, nb, stages, want_dot;
    uint32_t stage_bytes, gy_off, h_off, tx_bytes, bar_off;
};

template <int R>
__global__ void __launch_bounds__(32 * (1 + kXWarps), 1)
k_expand_wgrad(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmG,
               const __grid_constant__ CUtensorMap tmH, const __grid_constant__ CUtensorMap tmO, const ExpandParams p) {
    constexpr int KS = R / 16;                             // k16 steps of the expansion = c m-tiles of the weight gradient
    extern __shared__ uint8_t smem_unaligned[];
    uint8_t* smem = smem_unaligned + ((1024u - (smem_addr(smem_unaligned) & 1023u)) & 1023u);
    const uint32_t bar0 = smem_addr(smem + p.bar_off);
    auto full = [&](int s) { return bar0 + 8u * (uint32_t)s; };
    auto empty = [&](int s) { return bar0 + 8u * (uint32_t)(p.stages + s); };
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
        for (int s = 0; s < p.stages; ++s) { mbar_init(full(s), 1); mbar_init(empty(s), kXWarps); }
        mbar_fence_init();
    }
    __syncthreads();
    pdl_wait();                                            // gP comes from the hop that precedes this kernel
    pdl_trigger();
    const int ntiles = (p.n + kXRows - 1) / kXRows;
    const int q = ntiles / (int)gridDim.x, rem = ntiles % (int)gridDim.x;
    const int bid = blockIdx.x;
    const int t0 = bid * q + min(bid, rem);
    const int my_tiles = q + (bid < rem ? 1 : 0);

    if (warp == 0) {
        // ===================== producer =====================
        if (lane == 0) {
            const uint64_t pol = policy_evict_first();
            int s = 0, use = 0;
            for (int k = 0; k < my_tiles; ++k) {
                if (use > 0) mbar_wait(empty(s), (uint32_t)((use - 1) & 1));
                const int row0 = (t0 + k) * kXRows;
                const uint32_t dst = smem_addr(smem + (size_t)s * p.stage_bytes);
                mbar_arrive_expect_tx(full(s), p.tx_bytes);
                for (int b = 0; b < p.nb; ++b) tma_load_box(dst + (uint32_t)(b * kXBox), &tmX, b * 32, row0, full(s), pol);
                for (int b = 0; b < p.nb; ++b) tma_load_box(dst + p.gy_off + (uint32_t)(b * kXBox), &tmG, b * 32, row0, full(s), pol);
                tma_load_box_nohint(dst + p.h_off, &tmH, 0, R == 16 ? row0 / 2 : row0, full(s));
                if (++s == p.stages) { s = 0; ++use; }
            }
        }
        return;
    }

    // ===================== box warps =====================
    const int bx = warp - 1;
    const bool active = bx < p.nb;
    const int g = lane >> 2, t = lane & 3;
    auto rho = [](int m) { const int m8 = m & 7; return 2 * ((m8 & 3) ^ (m8 >> 2)) + 8 * (m8 >> 2) + (m >> 3); };
    const int pr0 = rho(g), pr1 = pr0 + 1;                 // tile rows of matrix rows g and g + 8
    // byte offset of element (tile row i, channel c) inside the gP tile
    auto hoff = [](int i, int c) -> uint32_t {
        if (R == 16) { const int col = 16 * (i & 1) + c; return box_off(i >> 1, col >> 2) + (uint32_t)((col & 3) * 4); }
        return box_off(i, c >> 2) + (uint32_t)((c & 3) * 4);
    };
    // Wd fragments of this warp's 32 columns (expansion B operand): k = channel c, n = g -> column 32 bx + 8 j + g
    uint32_t wdh[KS][4][2], wdl[KS][4][2];
    float inv_w = 1.f;
    {
        float wv[KS][4][4];
        float m = 0.f;
#pragma unroll
        for (int ks = 0; ks < KS; ++ks)
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int c = 16 * ks + 2 * t + (e & 1) + 8 * (e >> 1), col = 32 * bx + 8 * j + g;
                    wv[ks][j][e] = active ? __ldg(p.Wd + (size_t)c * p.d + col) : 0.f;
                    m = fmaxf(m, fabsf(wv[ks][j][e]));
                }
        float sw;
        pow2_scale(warp_max(m), sw, inv_w);
#pragma unroll
        for (int ks = 0; ks < KS; ++ks)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                split_h2(wv[ks][j][0], wv[ks][j][1], sw, wdh[ks][j][0], wdl[ks][j][0]);
                split_h2(wv[ks][j][2], wv[ks][j][3], sw, wdh[ks][j][1], wdl[ks][j][1]);
            }
    }
    const float beta = p.scalar ? __ldg(p.scalar) : 1.f;
    const uint64_t pol = policy_evict_first();
    float run[KS][4][4];
#pragma unroll
    for (int cm = 0; cm < KS; ++cm)
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int i = 0; i < 4; ++i) run[cm][j][i] = 0.f;
    float dot = 0.f;
    int s = 0, prev_s = -1;
    uint32_t ph = 0;
    for (int k = 0; k < my_tiles; ++k) {
        mbar_wait(full(s), ph);
        uint8_t* stg = smem + (size_t)s * p.stage_bytes;
        if (active) {
            const uint8_t* boxX = stg + bx * kXBox;
            uint8_t* boxG = stg + p.gy_off + bx * kXBox;
            const uint8_t* ht = stg + p.h_off;
            const int row0 = (t0 + k) * kXRows;
            const bool ok0 = row0 + pr0 < p.n, ok1 = row0 + pr1 < p.n;   // (rows past n: gP is not zero-filled by a row count that
                                                                         //  ends inside a 128-byte row of the [n/2, 32] view)
            // ---- gP tile -> expansion A fragments (fp16 hi / lo, tile scale) ----
            float hv[KS][8];
            float mh = 0.f;
#pragma unroll
            for (int ks = 0; ks < KS; ++ks)
#pragma unroll
                for (int q2 = 0; q2 < 4; ++q2) {            // a0: (pr0, c0) a1: (pr1, c0) a2: (pr0, c0 + 8) a3: (pr1, c0 + 8)
                    const int row = (q2 & 1) ? pr1 : pr0, c0 = 16 * ks + 2 * t + 8 * (q2 >> 1);
                    const float2 v = *reinterpret_cast<const float2*>(ht + hoff(row, c0));
                    const bool ok = (q2 & 1) ? ok1 : ok0;
                    hv[ks][2 * q2] = ok ? v.x : 0.f;
                    hv[ks][2 * q2 + 1] = ok ? v.y : 0.f;
                    mh = fmaxf(mh, fmaxf(fabsf(hv[ks][2 * q2]), fabsf(hv[ks][2 * q2 + 1])));
                }
            float sh, inv_h;
            pow2_scale(warp_max(mh), sh, inv_h);
            uint32_t ah[KS][4], al[KS][4];
#pragma unroll
            for (int ks = 0; ks < KS; ++ks)
#pragma unroll
                for (int q2 = 0; q2 < 4; ++q2) split_h2(hv[ks][2 * q2], hv[ks][2 * q2 + 1], sh, ah[ks][q2], al[ks][q2]);
            // ---- expansion: C[16, 32] = gP_tile Wd_box ----
            float C[4][4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
#pragma unroll
                for (int i = 0; i < 4; ++i) C[j][i] = 0.f;
#pragma unroll
                for (int ks = 0; ks < KS; ++ks) {
                    mma_f16(C[j], ah[ks], wdh[ks][j][0], wdh[ks][j][1]);
                    mma_f16(C[j], al[ks], wdh[ks][j][0], wdh[ks][j][1]);
                    mma_f16(C[j], ah[ks], wdl[ks][j][0], wdl[ks][j][1]);
                }
            }
            // ---- X box -> weight-gradient B fragments (fp16 hi / lo, box scale): rows rho(2t), rho(2t+1), rho(2t+8), rho(2t+9) ----
            float4 xv[4];
            float mb = 0.f;
#pragma unroll
            for (int q2 = 0; q2 < 4; ++q2) {
                xv[q2] = lds4(boxX + box_off(rho(2 * t + (q2 & 1) + 8 * (q2 >> 1)), g));
                mb = absmax4(mb, xv[q2]);
            }
            float sb, inv_b;
            pow2_scale(warp_max(mb), sb, inv_b);
            uint32_t bh0[4], bl0[4], bh1[4], bl1[4];
            {
                const float e0[4] = {xv[0].x, xv[0].y, xv[0].z, xv[0].w}, e1[4] = {xv[1].x, xv[1].y, xv[1].z, xv[1].w};
                const float e2[4] = {xv[2].x, xv[2].y, xv[2].z, xv[2].w}, e3[4] = {xv[3].x, xv[3].y, xv[3].z, xv[3].w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    split_h2(e0[j], e1[j], sb, bh0[j], bl0[j]);          // k = 2t, 2t+1      (n-tile j: column 32 bx + 4 g + j)
                    split_h2(e2[j], e3[j], sb, bh1[j], bl1[j]);          // k = 2t+8, 2t+9
                }
            }
            const float fw = inv_b * inv_h;
#pragma unroll
            for (int cm = 0; cm < KS; ++cm) {
                // A = gP_tile^T: the expansion's fragment registers transposed ; (a0, a1, a2, a3) <- trans of (a0, a2, a1, a3)
                uint32_t th[4], tl[4];
                th[0] = movmatrix_trans(ah[cm][0]); th[1] = movmatrix_trans(ah[cm][2]);
                th[2] = movmatrix_trans(ah[cm][1]); th[3] = movmatrix_trans(ah[cm][3]);
                tl[0] = movmatrix_trans(al[cm][0]); tl[1] = movmatrix_trans(al[cm][2]);
                tl[2] = movmatrix_trans(al[cm][1]); tl[3] = movmatrix_trans(al[cm][3]);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float acc[4] = {0.f, 0.f, 0.f, 0.f};
                    mma_f16(acc, th, bh0[j], bh1[j]);
                    mma_f16(acc, tl, bh0[j], bh1[j]);
                    mma_f16(acc, th, bl0[j], bl1[j]);
#pragma unroll
                    for (int i = 0; i < 4; ++i) run[cm][j][i] = fmaf(acc[i], fw, run[cm][j][i]);
                }
            }
            // ---- gX = C + s gY in place over the gY box ; <gY, X> at the same positions ----
            const float fc = inv_h * inv_w;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint32_t o0 = box_off(pr0, 2 * j + (t >> 1)) + (uint32_t)((2 * t & 3) * 4);
                const uint32_t o1 = box_off(pr1, 2 * j + (t >> 1)) + (uint32_t)((2 * t & 3) * 4);
                const float2 g0 = *reinterpret_cast<const float2*>(boxG + o0), g1 = *reinterpret_cast<const float2*>(boxG + o1);
                if (p.want_dot) {
                    const float2 x0 = *reinterpret_cast<const float2*>(boxX + o0), x1 = *reinterpret_cast<const float2*>(boxX + o1);
                    dot = fmaf(g0.x, x0.x, fmaf(g0.y, x0.y, fmaf(g1.x, x1.x, fmaf(g1.y, x1.y, dot))));
                }
                *reinterpret_cast<float2*>(boxG + o0) = make_float2(fmaf(beta, g0.x, C[j][0] * fc), fmaf(beta, g0.y, C[j][1] * fc));
                *reinterpret_cast<float2*>(boxG + o1) = make_float2(fmaf(beta, g1.x, C[j][2] * fc), fmaf(beta, g1.y, C[j][3] * fc));
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");    // generic-proxy writes -> visible to the bulk store
        }
        __syncwarp();
        if (lane == 0) {
            // the store of the previous tile has had a whole tile to read its box: release that stage, then send this one
            if (prev_s >= 0) {
                if (active) bulk_wait_read<0>();
                mbar_arrive(empty(prev_s));
            }
            if (active) {
                tma_store_box(&tmO, bx * 32, (t0 + k) * kXRows, smem_addr(stg + p.gy_off + bx * kXBox), pol);
                bulk_commit();
            }
        }
        prev_s = s;
        if (++s == p.stages) { s = 0; ph ^= 1u; }
    }
    if (lane == 0 && active) bulk_wait_all();
    // ---- per-CTA partial: lane (g, t) owns rows c = g, g + 8 (+ 16 cm) and columns 32 bx + 8t .. + 7 ----
    if (active) {
        float* pgp = p.partG + (size_t)bid * R * p.d;
        const int oc = 32 * bx + 8 * t;
#pragma unroll
        for (int cm = 0; cm < KS; ++cm)
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int c = cm * 16 + g + 8 * half, i0 = 2 * half;
                *reinterpret_cast<float4*>(pgp + (size_t)c * p.d + oc) =
                    make_float4(run[cm][0][i0], run[cm][1][i0], run[cm][2][i0], run[cm][3][i0]);
                *reinterpret_cast<float4*>(pgp + (size_t)c * p.d + oc + 4) =
                    make_float4(run[cm][0][i0 + 1], run[cm][1][i0 + 1], run[cm][2][i0 + 1], run[cm][3][i0 + 1]);
            }
    }
    float* s_dot = reinterpret_cast<float*>(smem + p.bar_off + 192);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, off);
    if (lane == 0) s_dot[bx] = active ? dot : 0.f;
    named_sync(2, kXWarps * 32);
    if (bx == 0 && lane == 0) {
        if (p.partDot) {
            float tsum = 0.f;
            for (int w = 0; w < kXWarps; ++w) tsum += s_dot[w];
            p.partDot[bid] = tsum;
        }
        if (bid == 0) p.header[p.slot] = (int)gridDim.x;
    }
}

}  // namespace

int launch_expand_wgrad(int r, const float* X, int64_t ldx, const float* gY, int64_t ldg, const float* gP, const float* Wd,
                        const float* scalar, float* gX, int64_t ldgx, float* partG, float* partDot, int* header, int slot,
                        int n, int d, cudaStream_t st) {
    // r = 32 doubles the tensor-core and conversion work per streamed byte: measured 1.76 ms against 0.87 + 0.78 ms for
    // K3 + K4 at products size, so only r = 16 takes the one-pass kernel
    if (r != 16) return GCA_ERR_UNSUPPORTED;
    constexpr int R = 16;
    static const bool off = [] { const char* e = getenv("GCA_DISABLE_BWD_FUSE"); return e && e[0] == '1'; }();
    if (!tc_enabled() || !stream_enabled() || off) return GCA_ERR_UNSUPPORTED;
    if (!X || !gY || !gP || !gX || d % 32 != 0 || d > 32 * kXWarps || n < 128 * kXRows) return GCA_ERR_UNSUPPORTED;
    if ((ldx % 4) || (ldg % 4) || (ldgx % 4)) return GCA_ERR_UNSUPPORTED;
    for (const void* q : {(const void*)X, (const void*)gY, (const void*)gP, (const void*)gX})
        if (reinterpret_cast<uintptr_t>(q) % 16) return GCA_ERR_UNSUPPORTED;
    ExpandParams p{};
    p.Wd = Wd; p.scalar = scalar; p.partG = partG; p.partDot = partDot; p.header = header; p.slot = slot;
    p.n = n; p.d = d; p.nb = d / 32; p.want_dot = partDot ? 1 : 0;
    const uint32_t a_bytes = (uint32_t)p.nb * kXBox, h_bytes = (uint32_t)(kXRows * R * 4);
    p.gy_off = a_bytes;
    p.h_off = 2 * a_bytes;
    p.stage_bytes = (p.h_off + h_bytes + 1023u) & ~1023u;
    p.tx_bytes = 2 * a_bytes + h_bytes;
    int stages = (int)((227 * 1024 - 256 - 1024) / p.stage_bytes);
    if (stages > 8) stages = 8;
    if (stages < 3) return GCA_ERR_UNSUPPORTED;
    p.stages = stages;
    p.bar_off = (uint32_t)stages * p.stage_bytes;
    const size_t smem = (size_t)p.bar_off + 256 + 1024;
    CUtensorMap tmX, tmG, tmH, tmO;
    if (!get_box_map(&tmX, X, n, d, ldx, 32, kXRows, true) || !get_box_map(&tmG, gY, n, d, ldg, 32, kXRows, true) ||
        !get_box_map(&tmO, gX, n, d, ldgx, 32, kXRows, true))
        return GCA_ERR_UNSUPPORTED;
    // gP [n, 16] is read as [ceil(n / 2), 32]: two nodes per 128-byte row (the caller's buffer holds an even number of rows)
    if (!get_box_map(&tmH, gP, (n + 1) / 2, 32, 32, 32, kXRows / 2, true)) return GCA_ERR_UNSUPPORTED;
    auto kern = k_expand_wgrad<R>;
    GCA_TRY(set_smem(kern, smem));
    const int ntiles = (n + kXRows - 1) / kXRows;
    const int grid = ntiles < num_sms() ? ntiles : num_sms();
    {
        ProfScope ps("expand_wgrad_bwd", st, "stream_f16");
        GCA_CUDA(launch_pdl(kern, dim3(grid), dim3(32 * (1 + kXWarps)), smem, st, tmX, tmG, tmH, tmO, p));
    }
    GCA_LAUNCH_OK();
    return GCA_OK;
}

}  // namespace gca
