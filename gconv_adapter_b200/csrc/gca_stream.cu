// TMA-fed dense streaming family: every dense pass over a d-wide tensor of the adapter in ONE kernel template.
//
//   project_fwd   P'   = dis * (X Wd^T)                                   PROJ            (conv_down.lin)
//   bwd_up        gH2' = dis * s * (gY Wu)  AND  gWu/gbu partials         PROJ + WGRAD    gY crosses HBM ONCE
//   wgrad_down    gWd partials = gP^T X  AND  <gY, X>                     WGRAD + DOT
//
// Why: the register-fed mma.sync kernels (gca_project.cu, gca_wgrad.cu) reach 47-49 % of the HBM peak at 24 % warps
// active - every LDG of a warp shares one scoreboard, so a warp never overlaps its own loads with its tensor-core work
// (profiles/README.md section 2b) - and the backward read gY once for the projection and once more for the weight
// gradient.  Here the copy engine streams [32 rows x d] tiles into a shared-memory ring (tensor-map boxes of
// 32 x 32 fp32, SWIZZLE_128B, mbarrier hand-over) and warp-specialised consumers read every tile from shared memory.
// Warp 0 is the producer in every layout: one thread issues the boxes of tile k + stages - 1 as soon as all consumers
// released the stage.  The consumers come in three layouts:
//
//   projection (PROJ: project_fwd, project_bwd)                                     1 + 8 + 2 warps
//     warps 1-8     warp w owns the 32-column box w of every tile (W fragments for those 32 k's live in registers, split
//                   once), multiplies both 16-row m-tiles of the tile and leaves a [32, R] partial in one of two
//                   shared-memory buffers (mbarrier red_full / red_free).  The tile's 32 row scales arrive with the tile
//                   (1D bulk copy into the stage) and are applied here.
//     warps 9-10    epilogue: add the eight partials of a tile in box order and store the rows - the MMA warps never
//                   wait for it unless they run two tiles ahead.  (No global load anywhere in the consumers: a cold
//                   rowscale LDG per tile paced the whole kernel at one DRAM latency per tile.)
//   fused (PROJ + WGRAD: bwd_up at r = 16)                                          1 + 16 + 2 warps
//     warps 1-16    warp (w, mt) owns the 16-row m-tile mt of box w: the projection of those rows as above, and the
//                   weight gradient over the same rows from the same converted fragments (see the role below).
//     warps 17-18   the projection epilogue.
//   weight gradient (WGRAD, + DOT: wgrad_up, wgrad_down)                            1 + 8 warps
//     warps 1-8     warp w owns box w as the N dimension (32 columns = 4 n-tiles), K = the 32 rows of the tile (2 k16
//                   steps), M = R.  The H tile [32, R] arrives through its own tensor map in the same stage.
//                   Accumulators stay in registers for the whole kernel (unscaled into a running fp32 sum every tile)
//                   -> ONE partial per CTA.
//
// Fragment reads are bank-conflict free by construction (g = lane >> 2, t = lane & 3):
//   projection A-fragment: LDS.128 of chunk 4*kb2 + t of rows pg(g) and pg(g) + 8 with pg(g) = (g >> 1) + 4 (g & 1):
//       a quarter warp (g in {2q, 2q+1}) touches rows q and q + 4, whose swizzle XORs differ in bit 2.
//       One float4 feeds one k16 step through the K permutation  k = 2t, 2t+1 -> column 4t, 4t+1 ; k = 2t+8, 2t+9 -> 4t+2, 4t+3.
//   weight-gradient B-fragment: LDS.128 of chunk g of rows 16 ks2 + {0,3,4,7}[t] (+ 8) (k = 2t, k = 2t+8) and
//       16 ks2 + {1,2,5,6}[t] (+ 8) (k = 2t+1, 2t+9); the float4 feeds the four n-tiles through the column permutation
//       col = 32 w + 4 n + j  (n-tile j).
// Arithmetic: the scaled 2xFP16 split of gca_stream.cuh, three m16n8k16 per product.
//
// Reference semantics: the two Linear layers of /root/reference/src/finetune/gconv_adapter.py:92 and their autograd.
#include "gca_common.cuh"
#include "gca_device.cuh"
#include "gca_host.cuh"
#include "gca_stream.cuh"

namespace gca {
namespace {

constexpr int kSRows = 32;                 // rows per tile
constexpr int kSBox = 32 * kSRows * 4;     // one 32-column box of a tile: 4 KB, SWIZZLE_128B
constexpr int kSWarps = 8;                 // consumer warps per role = column boxes of a 256-wide tile
constexpr int kSEpi = 2;                   // epilogue warps of the projection role

// warps that read the stages: one per (box, m-tile) in the fused layout, else one per box
__host__ __device__ constexpr int stream_consumers(bool proj, bool wgrad) { return proj && wgrad ? 2 * kSWarps : kSWarps; }
// producer + consumers + the projection epilogue
__host__ __device__ constexpr int stream_threads(bool proj, bool wgrad) {
    return 32 * (1 + stream_consumers(proj, wgrad) + (proj ? kSEpi : 0));
}

// element (row, c) of the [32, R] H tile of a stage: 128-byte swizzled rows at r = 32, plain rows at r = 16
template <int R>
__device__ __forceinline__ float hload(const uint8_t* ht, int row, int c) {
    if (R == 32) return *reinterpret_cast<const float*>(ht + box_off(row, c >> 2) + (c & 3) * 4);
    return *reinterpret_cast<const float*>(ht + (row * R + c) * 4);
}

struct StreamParams {
    const float* W; const float* rowscale; const float* scalar; float* out;
    float* partG; float* partCol; float* partDot; int* header; int slot;
    int n, d, nb, stages;
    uint32_t stage_bytes, b_off, h_off, sc_off, tx_bytes, red_off, bar_off;
    gca_push push;   // peers that receive every projected row as well (count = 0: none)
};

template <int R, bool PROJ, bool WGRAD, bool DOT, bool W_IS_RD>
__global__ void __launch_bounds__(stream_threads(PROJ, WGRAD), 1)
k_dense_stream(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmH, const StreamParams p) {
    constexpr int NT = R / 8, MT = R / 16;
    constexpr bool FUSED = PROJ && WGRAD;
    constexpr int kConsumers = stream_consumers(PROJ, WGRAD);
    extern __shared__ uint8_t smem_unaligned[];
    uint8_t* smem = smem_unaligned + ((1024u - (smem_addr(smem_unaligned) & 1023u)) & 1023u);
    const uint32_t bar0 = smem_addr(smem + p.bar_off);
    auto full = [&](int s) { return bar0 + 8u * (uint32_t)s; };
    auto empty = [&](int s) { return bar0 + 8u * (uint32_t)(p.stages + s); };
    auto red_full = [&](int b) { return bar0 + 8u * (uint32_t)(2 * p.stages + b); };        // MMA warps -> epilogue
    auto red_free = [&](int b) { return bar0 + 8u * (uint32_t)(2 * p.stages + 2 + b); };    // epilogue -> MMA warps
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
        for (int s = 0; s < p.stages; ++s) { mbar_init(full(s), 1); mbar_init(empty(s), kConsumers); }
        for (int b = 0; b < 2; ++b) { mbar_init(red_full(b), kConsumers); mbar_init(red_free(b), kSEpi); }
        mbar_fence_init();
    }
    __syncthreads();
    // what precedes these kernels on the stream is either not ours (an optimizer step may just have written W) or
    // produced the H operand: wait before the first read of anything
    pdl_wait();
    pdl_trigger();

    // contiguous tile ranges: CTA b takes q (+1) consecutive tiles, so its partial covers one row range
    const int ntiles = (p.n + kSRows - 1) / kSRows;
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
                const int row0 = (t0 + k) * kSRows;
                const uint32_t dst = smem_addr(smem + (size_t)s * p.stage_bytes);
                mbar_arrive_expect_tx(full(s), p.tx_bytes);
                for (int b = 0; b < p.nb; ++b) tma_load_box(dst + (uint32_t)(b * kSBox), &tmA, b * 32, row0, full(s), pol);
                if (DOT)
                    for (int b = 0; b < p.nb; ++b) tma_load_box(dst + p.b_off + (uint32_t)(b * kSBox), &tmB, b * 32, row0, full(s), pol);
                if (WGRAD) tma_load_box_nohint(dst + p.h_off, &tmH, 0, row0, full(s));
                // the tile's 32 row scales travel with the tile (rows past n read padding of the same allocation and
                // are never used): no consumer ever waits on a cold global load
                if (PROJ && p.rowscale) bulk_load_1d(dst + p.sc_off, p.rowscale + row0, kSRows * 4, full(s));
                if (++s == p.stages) { s = 0; ++use; }
            }
        }
        return;
    }
    const int cw = warp - 1;
    const int g = lane >> 2, t = lane & 3;

    if (FUSED && cw < kConsumers) {
        // ===================== fused role (PROJ + WGRAD): one conversion serves both products =====================
        // Warp (w, mt) owns the 16-row m-tile mt of box w of every tile (16 warps: four per scheduler hide each other's
        // shuffle-max -> convert -> HMMA -> movmatrix -> HMMA chains; with 8 warps the same work ran at 27 % issue utilisation).
        // It converts its 16 x 32 half box ONCE into projection A-fragments (fp16 hi / lo, its own power-of-two scale),
        // multiplies them with its W fragments (-> [16, R] partial, as the projection role),
        // then transposes every fragment register with movmatrix: the 8 x 8 block (row pg(g), columns C(2t), C(2t+1)) turns
        // into (rows pg(2t), pg(2t+1) ; column C(g)) = the B-fragment of the weight gradient over the SAME 16 rows
        // (k = rows of m-tile mt, n-tiles 2 kb2 / 2 kb2 + 1 = the even / odd column pairs of the 16-column block kb2).
        // Through the permutations lane (g, t) ends up owning G[c = g (+8)][32 w + 16 kb2 + 4t .. + 3]: a float4.
        const int bx = cw % kSWarps, mt = cw / kSWarps;
        const bool active = bx < p.nb;
        uint32_t wf[2][NT][4];
        float inv_w = 1.f;
        {
            float wv[2][NT][4];
            float m = 0.f;
#pragma unroll
            for (int kb2 = 0; kb2 < 2; ++kb2)
#pragma unroll
                for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int k_ = 32 * bx + 16 * kb2 + 4 * t + e, c = nt * 8 + g;
                        wv[kb2][nt][e] = !active ? 0.f : (W_IS_RD ? __ldg(p.W + (size_t)c * p.d + k_) : __ldg(p.W + (size_t)k_ * R + c));
                        m = fmaxf(m, fabsf(wv[kb2][nt][e]));
                    }
            float sw;
            pow2_scale(warp_max(m), sw, inv_w);
#pragma unroll
            for (int kb2 = 0; kb2 < 2; ++kb2)
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    split_h2(wv[kb2][nt][0], wv[kb2][nt][1], sw, wf[kb2][nt][0], wf[kb2][nt][2]);
                    split_h2(wv[kb2][nt][2], wv[kb2][nt][3], sw, wf[kb2][nt][1], wf[kb2][nt][3]);
                }
        }
        const int pg = (g >> 1) + 4 * (g & 1);
        const float sc_s = p.scalar ? __ldg(p.scalar) : 1.f;
        float4* red = reinterpret_cast<float4*>(smem + p.red_off);
        constexpr int kSlots = 2 * NT * 32;
        float run[MT][2][2][4];                                              // [c m-tile][kb2][even / odd pair][c-fragment]
        float4 csum[2];                                                      // column sums of this lane's 8 columns (its rows)
#pragma unroll
        for (int m = 0; m < MT; ++m)
#pragma unroll
            for (int a_ = 0; a_ < 2; ++a_)
#pragma unroll
                for (int b_ = 0; b_ < 2; ++b_)
#pragma unroll
                    for (int i = 0; i < 4; ++i) run[m][a_][b_][i] = 0.f;
        csum[0] = csum[1] = make_float4(0.f, 0.f, 0.f, 0.f);
        int s = 0;
        uint32_t ph = 0;
        for (int k = 0; k < my_tiles; ++k) {
            float accp[2][NT][4];                                            // projection: [hi.hi / corrections][nt]
#pragma unroll
            for (int a_ = 0; a_ < 2; ++a_)
#pragma unroll
                for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                    for (int i = 0; i < 4; ++i) accp[a_][nt][i] = 0.f;
            float sc[2], inv_x = 1.f;
            mbar_wait(full(s), ph);
            const uint8_t* stg = smem + (size_t)s * p.stage_bytes;
            const uint8_t* box = stg + bx * kSBox;
            const uint8_t* ht = stg + p.h_off;
            const float* scs = reinterpret_cast<const float*>(stg + p.sc_off);
            sc[0] = (p.rowscale ? scs[16 * mt + pg] : 1.f) * sc_s * inv_w;
            sc[1] = (p.rowscale ? scs[16 * mt + pg + 8] : 1.f) * sc_s * inv_w;
            if (active) {
                {
                    // ---- this m-tile's 16 rows x 32 columns and its H rows: load, scale, split ----
                    float4 x[2][2];                                          // [kb2][row pg / pg + 8]
                    float m = 0.f;
#pragma unroll
                    for (int kb2 = 0; kb2 < 2; ++kb2) {
                        x[kb2][0] = lds4(box + box_off(16 * mt + pg, 4 * kb2 + t));
                        x[kb2][1] = lds4(box + box_off(16 * mt + pg + 8, 4 * kb2 + t));
                        m = absmax4(absmax4(m, x[kb2][0]), x[kb2][1]);
                        csum[kb2] = f4_add(csum[kb2], f4_add(x[kb2][0], x[kb2][1]));
                    }
                    float hv[MT][8];
                    float mh = 0.f;
#pragma unroll
                    for (int cm = 0; cm < MT; ++cm)
#pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            // q: bit 0 = row t / t + 4 (k = 2t / 2t+1), bit 1 = c + 8, bit 2 = rows + 8 (k + 8)
                            hv[cm][q] = hload<R>(ht, 16 * mt + 8 * (q >> 2) + t + 4 * (q & 1), 16 * cm + g + 8 * ((q >> 1) & 1));
                            mh = fmaxf(mh, fabsf(hv[cm][q]));
                        }
                    float sx, sh, inv_h;
                    pow2_scale(warp_max(m), sx, inv_x);
                    pow2_scale(warp_max(mh), sh, inv_h);
                    uint32_t ah[2][4], al[2][4];
#pragma unroll
                    for (int kb2 = 0; kb2 < 2; ++kb2) {
                        split_h2(x[kb2][0].x, x[kb2][0].y, sx, ah[kb2][0], al[kb2][0]);
                        split_h2(x[kb2][1].x, x[kb2][1].y, sx, ah[kb2][1], al[kb2][1]);
                        split_h2(x[kb2][0].z, x[kb2][0].w, sx, ah[kb2][2], al[kb2][2]);
                        split_h2(x[kb2][1].z, x[kb2][1].w, sx, ah[kb2][3], al[kb2][3]);
                    }
                    // ---- projection: [16 rows, R] += box[16, 32] W[32, R] ----
#pragma unroll
                    for (int kb2 = 0; kb2 < 2; ++kb2)
#pragma unroll
                        for (int nt = 0; nt < NT; ++nt) {
                            mma_f16(accp[0][nt], ah[kb2], wf[kb2][nt][0], wf[kb2][nt][1]);
                            mma_f16(accp[1][nt], al[kb2], wf[kb2][nt][0], wf[kb2][nt][1]);
                            mma_f16(accp[1][nt], ah[kb2], wf[kb2][nt][2], wf[kb2][nt][3]);
                        }
                    // ---- weight gradient over the same 16 rows: B = transposed fragments, A = H^T ----
                    uint32_t hh[MT][4], hl[MT][4];
#pragma unroll
                    for (int cm = 0; cm < MT; ++cm) {
                        split_h2(hv[cm][0], hv[cm][1], sh, hh[cm][0], hl[cm][0]);     // c = g,   k = 2t, 2t+1
                        split_h2(hv[cm][2], hv[cm][3], sh, hh[cm][1], hl[cm][1]);     // c = g+8
                        split_h2(hv[cm][4], hv[cm][5], sh, hh[cm][2], hl[cm][2]);     // c = g,   k = 2t+8, 2t+9
                        split_h2(hv[cm][6], hv[cm][7], sh, hh[cm][3], hl[cm][3]);     // c = g+8
                    }
                    const float f = inv_x * inv_h;
#pragma unroll
                    for (int kb2 = 0; kb2 < 2; ++kb2) {
                        uint32_t bh[4], bl[4];
#pragma unroll
                        for (int i = 0; i < 4; ++i) { bh[i] = movmatrix_trans(ah[kb2][i]); bl[i] = movmatrix_trans(al[kb2][i]); }
#pragma unroll
                        for (int pr = 0; pr < 2; ++pr) {                     // n-tile = even / odd column pairs: registers {0,1} / {2,3}
#pragma unroll
                            for (int cm = 0; cm < MT; ++cm) {
                                float accw[4] = {0.f, 0.f, 0.f, 0.f};
                                mma_f16(accw, hh[cm], bh[2 * pr], bh[2 * pr + 1]);
                                mma_f16(accw, hl[cm], bh[2 * pr], bh[2 * pr + 1]);
                                mma_f16(accw, hh[cm], bl[2 * pr], bl[2 * pr + 1]);
#pragma unroll
                                for (int i = 0; i < 4; ++i) run[cm][kb2][pr][i] = fmaf(accw[i], f, run[cm][kb2][pr][i]);
                            }
                        }
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(empty(s));
            const int rbuf = k & 1;
            if (k >= 2) mbar_wait(red_free(rbuf), (uint32_t)(((k >> 1) - 1) & 1));
            float4* mine = red + ((size_t)rbuf * kSWarps + bx) * kSlots;
#pragma unroll
            for (int nt = 0; nt < NT; ++nt)
                mine[(mt * NT + nt) * 32 + lane] =
                    make_float4((accp[0][nt][0] + accp[1][nt][0]) * inv_x * sc[0], (accp[0][nt][1] + accp[1][nt][1]) * inv_x * sc[0],
                                (accp[0][nt][2] + accp[1][nt][2]) * inv_x * sc[1], (accp[0][nt][3] + accp[1][nt][3]) * inv_x * sc[1]);
            __syncwarp();
            if (lane == 0) mbar_arrive(red_full(rbuf));
            if (++s == p.stages) { s = 0; ph ^= 1u; }
        }
        // ---- per-CTA partial.  c-fragment of n-tile (kb2, pr): c0 = (c = g, n = 2t) -> column 16 kb2 + 4t + 2 pr, c1 = (g, 2t+1) ->
        //      + 1, c2 / c3 = c + 8: lane (g, t) owns G[c][32 bx + 16 kb2 + 4t .. + 3] for c = g, g + 8 (+ 16 cm) ----
        //      Every CTA emits TWO partials (one per m-tile half): 2 * grid <= kMaxParts rows for k_finalize.
        const int pid = 2 * bid + mt;
        if (active) {
            float* pgp = p.partG + (size_t)pid * R * p.d;
#pragma unroll
            for (int cm = 0; cm < MT; ++cm)
#pragma unroll
                for (int kb2 = 0; kb2 < 2; ++kb2) {
                    const int col = 32 * bx + 16 * kb2 + 4 * t;
                    *reinterpret_cast<float4*>(pgp + (size_t)(16 * cm + g) * p.d + col) =
                        make_float4(run[cm][kb2][0][0], run[cm][kb2][0][1], run[cm][kb2][1][0], run[cm][kb2][1][1]);
                    *reinterpret_cast<float4*>(pgp + (size_t)(16 * cm + g + 8) * p.d + col) =
                        make_float4(run[cm][kb2][0][2], run[cm][kb2][0][3], run[cm][kb2][1][2], run[cm][kb2][1][3]);
                }
            if (p.partCol) {
                // this lane summed rows pg(g), pg(g) + 8 (+ 16) of its 8 columns: add the 8 row groups (lanes with equal t)
#pragma unroll
                for (int kb2 = 0; kb2 < 2; ++kb2) {
                    float4 c4 = csum[kb2];
                    c4 = f4_add(c4, f4_shfl_xor(c4, 4));
                    c4 = f4_add(c4, f4_shfl_xor(c4, 8));
                    c4 = f4_add(c4, f4_shfl_xor(c4, 16));
                    if (g == 0) *reinterpret_cast<float4*>(p.partCol + (size_t)pid * p.d + 32 * bx + 16 * kb2 + 4 * t) = c4;
                }
            }
        }
        if (bid == 0 && cw == 0 && lane == 0) p.header[p.slot] = 2 * (int)gridDim.x;
        return;
    }

    if (PROJ && !WGRAD && cw < kConsumers) {
        // ===================== projection warps =====================
        const int bx = cw % kSWarps;
        const bool active = bx < p.nb;
        // W fragments of this warp's 32 k's, in registers for the whole kernel: wf[kb2][nt] = {hi(c0,c0+1), hi(c0+2,c0+3),
        // lo(c0,c0+1), lo(c0+2,c0+3)} (packed pairs), c0 = 32 bx + 16 kb2 + 4 t, c = 8 nt + g, scaled by this warp's own power
        // of two (inv_w undoes it).  The fused role loads the same fragments with its own copy of this code: as one shared
        // helper, ptxas scheduled this role differently.
        uint32_t wf[2][NT][4];
        float inv_w = 1.f;
        auto wload = [&](int k_, int c) -> float {
            if (!active) return 0.f;
            return W_IS_RD ? __ldg(p.W + (size_t)c * p.d + k_) : __ldg(p.W + (size_t)k_ * R + c);
        };
        {
            float wv[2][NT][4];
            float m = 0.f;
#pragma unroll
            for (int kb2 = 0; kb2 < 2; ++kb2)
#pragma unroll
                for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        wv[kb2][nt][e] = wload(32 * bx + 16 * kb2 + 4 * t + e, nt * 8 + g);
                        m = fmaxf(m, fabsf(wv[kb2][nt][e]));
                    }
            float sw;
            pow2_scale(warp_max(m), sw, inv_w);
#pragma unroll
            for (int kb2 = 0; kb2 < 2; ++kb2)
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    split_h2(wv[kb2][nt][0], wv[kb2][nt][1], sw, wf[kb2][nt][0], wf[kb2][nt][2]);
                    split_h2(wv[kb2][nt][2], wv[kb2][nt][3], sw, wf[kb2][nt][1], wf[kb2][nt][3]);
                }
        }
        const int pg = (g >> 1) + 4 * (g & 1);
        const float sc_s = p.scalar ? __ldg(p.scalar) : 1.f;
        float4* red = reinterpret_cast<float4*>(smem + p.red_off);          // [2][kSWarps][2 NT][32]
        constexpr int kSlots = 2 * NT * 32;                                  // float4 per partial
        int s = 0;
        uint32_t ph = 0;
        for (int k = 0; k < my_tiles; ++k) {
            float acc[2][2][NT][4];
#pragma unroll
            for (int a_ = 0; a_ < 2; ++a_)
#pragma unroll
                for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                        for (int i = 0; i < 4; ++i) acc[a_][mt][nt][i] = 0.f;
            mbar_wait(full(s), ph);
            float inv_x = 1.f;                                               // undoes the box scale
            if (active) {
                const uint8_t* box = smem + (size_t)s * p.stage_bytes + bx * kSBox;
                // the whole box first: its largest magnitude fixes the scale
                float4 x[2][2][2];                                           // [kb2][mt][row g / g + 8]
                float m = 0.f;
#pragma unroll
                for (int kb2 = 0; kb2 < 2; ++kb2)
#pragma unroll
                    for (int mt = 0; mt < 2; ++mt) {
                        x[kb2][mt][0] = lds4(box + box_off(16 * mt + pg, 4 * kb2 + t));
                        x[kb2][mt][1] = lds4(box + box_off(16 * mt + pg + 8, 4 * kb2 + t));
                        m = absmax4(absmax4(m, x[kb2][mt][0]), x[kb2][mt][1]);
                    }
                float sx;
                pow2_scale(warp_max(m), sx, inv_x);
#pragma unroll
                for (int kb2 = 0; kb2 < 2; ++kb2)
#pragma unroll
                    for (int mt = 0; mt < 2; ++mt) {
                        // one float4 per row = one k16 step: k = 2t, 2t+1 -> columns 4t, 4t+1 ; k = 2t+8, 2t+9 -> 4t+2, 4t+3
                        uint32_t ah[4], al[4];
                        split_h2(x[kb2][mt][0].x, x[kb2][mt][0].y, sx, ah[0], al[0]);
                        split_h2(x[kb2][mt][1].x, x[kb2][mt][1].y, sx, ah[1], al[1]);
                        split_h2(x[kb2][mt][0].z, x[kb2][mt][0].w, sx, ah[2], al[2]);
                        split_h2(x[kb2][mt][1].z, x[kb2][mt][1].w, sx, ah[3], al[3]);
#pragma unroll
                        for (int nt = 0; nt < NT; ++nt) {
                            mma_f16(acc[0][mt][nt], ah, wf[kb2][nt][0], wf[kb2][nt][1]);
                            mma_f16(acc[1][mt][nt], al, wf[kb2][nt][0], wf[kb2][nt][1]);
                            mma_f16(acc[1][mt][nt], ah, wf[kb2][nt][2], wf[kb2][nt][3]);
                        }
                    }
            }
            // row scales of this lane's rows (16 mt + pg, + 8), read before the stage is released
            float sc[2][2];
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) {
                const float* scs = reinterpret_cast<const float*>(smem + (size_t)s * p.stage_bytes + p.sc_off);
                sc[mt][0] = (p.rowscale ? scs[16 * mt + pg] : 1.f) * sc_s * inv_w;
                sc[mt][1] = (p.rowscale ? scs[16 * mt + pg + 8] : 1.f) * sc_s * inv_w;
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(empty(s));                            // this warp is done with the stage
            // hand the scaled [32, R] partial of this warp's 32 k's to the epilogue warps (two buffers)
            const int rbuf = k & 1;
            if (k >= 2) mbar_wait(red_free(rbuf), (uint32_t)(((k >> 1) - 1) & 1));
            float4* mine = red + ((size_t)rbuf * kSWarps + bx) * kSlots;
#pragma unroll
            for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                for (int nt = 0; nt < NT; ++nt)
                    mine[(mt * NT + nt) * 32 + lane] =
                        make_float4((acc[0][mt][nt][0] + acc[1][mt][nt][0]) * inv_x * sc[mt][0], (acc[0][mt][nt][1] + acc[1][mt][nt][1]) * inv_x * sc[mt][0],
                                    (acc[0][mt][nt][2] + acc[1][mt][nt][2]) * inv_x * sc[mt][1], (acc[0][mt][nt][3] + acc[1][mt][nt][3]) * inv_x * sc[mt][1]);
            __syncwarp();
            if (lane == 0) mbar_arrive(red_full(rbuf));                      // release: the epilogue acquires through its wait
            if (++s == p.stages) { s = 0; ph ^= 1u; }
        }
        return;
    }

    if (PROJ && cw < kConsumers + kSEpi) {
        // ===================== projection epilogue warps =====================
        constexpr int kSlots = 2 * NT * 32;
        constexpr int kPer = kSlots / (kSEpi * 32);                          // fragment slots per thread (2 at r = 16)
        const float4* red = reinterpret_cast<const float4*>(smem + p.red_off);
        const int th = (cw - kConsumers) * 32 + lane;
        // The summed tile is staged as [32][R] floats (two buffers) so that it leaves as whole rows: the tile is ONE
        // contiguous block of 32 R floats in `out` and in every peer's gathered buffer, written with 512 contiguous bytes
        // per warp instruction (8-byte fragment stores ran the NVLink pushes at a third of that).
        float* outs = reinterpret_cast<float*>(smem + p.bar_off + 256);     // [2][kSRows][R]
        constexpr int kF4 = kSRows * R / 4;                                  // float4 per tile
        for (int k = 0; k < my_tiles; ++k) {
            const int rbuf = k & 1;
            mbar_wait(red_full(rbuf), (uint32_t)((k >> 1) & 1));
            const float4* rb = red + (size_t)rbuf * kSWarps * kSlots;
            float* ot = outs + (size_t)rbuf * kSRows * R;
#pragma unroll
            for (int u = 0; u < kPer; ++u) {
                const int idx = th + u * kSEpi * 32;
                float4 v = rb[idx];
#pragma unroll
                for (int w = 1; w < kSWarps; ++w) v = f4_add(v, rb[w * kSlots + idx]);   // box order: fixed
                const int slot = idx >> 5, g2 = (idx & 31) >> 2, t2 = idx & 3;
                const int mt = slot / NT, nt = slot - mt * NT;
                const int lr = 16 * mt + (g2 >> 1) + 4 * (g2 & 1);
                *reinterpret_cast<float2*>(ot + lr * R + nt * 8 + 2 * t2) = make_float2(v.x, v.y);
                *reinterpret_cast<float2*>(ot + (lr + 8) * R + nt * 8 + 2 * t2) = make_float2(v.z, v.w);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(red_free(rbuf));                      // the partial buffers are free again
            named_sync(3, kSEpi * 32);                                       // tile staged by both epilogue warps
            const size_t base4 = (size_t)(t0 + k) * kF4;
            const int rows_left = p.n - (t0 + k) * kSRows;
            const int lim4 = (rows_left >= kSRows ? kSRows : (rows_left > 0 ? rows_left : 0)) * (R / 4);
            for (int q = th; q < lim4; q += kSEpi * 32) {
                const float4 v = reinterpret_cast<const float4*>(ot)[q];
                reinterpret_cast<float4*>(p.out)[base4 + q] = v;
                for (int hp = 0; hp < p.push.count; ++hp) reinterpret_cast<float4*>(p.push.dst[hp])[base4 + q] = v;
            }
            // (two staging buffers: tile k+1 is staged into the other one; the barrier of tile k+1 orders these reads
            //  before anybody stages tile k+2 into this one)
        }
        return;
    }

    if (WGRAD && !PROJ) {
        // ===================== weight-gradient warps =====================
        const int bx = cw;
        const bool active = bx < p.nb;
        float acc[MT][4][4], run[MT][4][4];
#pragma unroll
        for (int m = 0; m < MT; ++m)
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int i = 0; i < 4; ++i) { acc[m][j][i] = 0.f; run[m][j][i] = 0.f; }
        float4 csum = make_float4(0.f, 0.f, 0.f, 0.f);
        float dot = 0.f;
        const int rA = 4 * (t >> 1) + 3 * (t & 1);          // {0, 3, 4, 7}[t]  -> k = 2t (+ 8)
        const int rB = 4 * (t >> 1) + 1 + (t & 1);          // {1, 2, 5, 6}[t]  -> k = 2t + 1 (+ 8)
        int s = 0;
        uint32_t ph = 0;
        for (int k = 0; k < my_tiles; ++k) {
            mbar_wait(full(s), ph);
            if (active) {
                const uint8_t* stg = smem + (size_t)s * p.stage_bytes;
                const uint8_t* boxA = stg + bx * kSBox;
                const uint8_t* boxB = stg + p.b_off + bx * kSBox;
                const uint8_t* ht = stg + p.h_off;
                // the whole box first (its largest magnitude fixes the scale): k16 step ks2 covers rows 16 ks2 .. + 15,
                // k = 2t, 2t+1, 2t+8, 2t+9 -> rows rA, rB, 8 + rA, 8 + rB
                float4 v[2][4];
                float mb = 0.f;
#pragma unroll
                for (int ks2 = 0; ks2 < 2; ++ks2)
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int row = 16 * ks2 + 8 * (q >> 1) + ((q & 1) ? rB : rA);
                        v[ks2][q] = lds4(boxA + box_off(row, g));
                        mb = absmax4(mb, v[ks2][q]);
                        if (DOT) {
                            const float4 w = lds4(boxB + box_off(row, g));
                            dot = fmaf(v[ks2][q].x, w.x, fmaf(v[ks2][q].y, w.y, fmaf(v[ks2][q].z, w.z, fmaf(v[ks2][q].w, w.w, dot))));
                        } else {
                            csum = f4_add(csum, v[ks2][q]);
                        }
                    }
                float hv[2][MT][8];
                float mh = 0.f;
#pragma unroll
                for (int ks2 = 0; ks2 < 2; ++ks2)
#pragma unroll
                    for (int m = 0; m < MT; ++m)
#pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            const int row = 16 * ks2 + 8 * (q >> 2) + ((q & 1) ? rB : rA);
                            hv[ks2][m][q] = hload<R>(ht, row, 16 * m + g + 8 * ((q >> 1) & 1));
                            mh = fmaxf(mh, fabsf(hv[ks2][m][q]));
                        }
                float sb, inv_b, sh, inv_h;
                pow2_scale(warp_max(mb), sb, inv_b);
                pow2_scale(warp_max(mh), sh, inv_h);
#pragma unroll
                for (int ks2 = 0; ks2 < 2; ++ks2) {
                    uint32_t bh0[4], bl0[4], bh1[4], bl1[4];
                    const float e0[4] = {v[ks2][0].x, v[ks2][0].y, v[ks2][0].z, v[ks2][0].w};
                    const float e1[4] = {v[ks2][1].x, v[ks2][1].y, v[ks2][1].z, v[ks2][1].w};
                    const float e2[4] = {v[ks2][2].x, v[ks2][2].y, v[ks2][2].z, v[ks2][2].w};
                    const float e3[4] = {v[ks2][3].x, v[ks2][3].y, v[ks2][3].z, v[ks2][3].w};
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        split_h2(e0[j], e1[j], sb, bh0[j], bl0[j]);          // k = 2t, 2t+1   (n-tile j)
                        split_h2(e2[j], e3[j], sb, bh1[j], bl1[j]);          // k = 2t+8, 2t+9
                    }
#pragma unroll
                    for (int m = 0; m < MT; ++m) {
                        uint32_t ah[4], al[4];
                        split_h2(hv[ks2][m][0], hv[ks2][m][1], sh, ah[0], al[0]);   // c = g,   k = 2t, 2t+1
                        split_h2(hv[ks2][m][2], hv[ks2][m][3], sh, ah[1], al[1]);   // c = g+8
                        split_h2(hv[ks2][m][4], hv[ks2][m][5], sh, ah[2], al[2]);   // c = g,   k = 2t+8, 2t+9
                        split_h2(hv[ks2][m][6], hv[ks2][m][7], sh, ah[3], al[3]);   // c = g+8
#pragma unroll
                        for (int j = 0; j < 4; ++j) mma_f16(acc[m][j], ah, bh0[j], bh1[j]);
#pragma unroll
                        for (int j = 0; j < 4; ++j) mma_f16(acc[m][j], al, bh0[j], bh1[j]);
#pragma unroll
                        for (int j = 0; j < 4; ++j) mma_f16(acc[m][j], ah, bl0[j], bl1[j]);
                    }
                }
                // the accumulators hold box-scaled x tile-scaled values: unscale and fold every tile
                const float f = inv_b * inv_h;
#pragma unroll
                for (int m = 0; m < MT; ++m)
#pragma unroll
                    for (int j = 0; j < 4; ++j)
#pragma unroll
                        for (int i = 0; i < 4; ++i) { run[m][j][i] = fmaf(acc[m][j][i], f, run[m][j][i]); acc[m][j][i] = 0.f; }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(empty(s));
            if (++s == p.stages) { s = 0; ph ^= 1u; }
        }
        // ---- per-CTA partial: lane (g, t) owns rows c = g, g+8 (+16 m) and columns 32 bx + 8t .. + 7 ----
        if (active) {
            float* pgp = p.partG + (size_t)bid * R * p.d;
            const int oc = 32 * bx + 8 * t;
#pragma unroll
            for (int m = 0; m < MT; ++m) {
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    const int c = m * 16 + g + 8 * half;
                    const int i0 = 2 * half;
                    *reinterpret_cast<float4*>(pgp + (size_t)c * p.d + oc) =
                        make_float4(run[m][0][i0], run[m][1][i0], run[m][2][i0], run[m][3][i0]);
                    *reinterpret_cast<float4*>(pgp + (size_t)c * p.d + oc + 4) =
                        make_float4(run[m][0][i0 + 1], run[m][1][i0 + 1], run[m][2][i0 + 1], run[m][3][i0 + 1]);
                }
            }
            if (!DOT && p.partCol) {
                csum = f4_add(csum, f4_shfl_xor(csum, 1));
                csum = f4_add(csum, f4_shfl_xor(csum, 2));
                if (t == 0) *reinterpret_cast<float4*>(p.partCol + (size_t)bid * p.d + 32 * bx + 4 * g) = csum;
            }
        }
        if (DOT) {
            float* s_dot = reinterpret_cast<float*>(smem + p.bar_off + 192);
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, off);
            if (lane == 0) s_dot[bx] = active ? dot : 0.f;
            named_sync(2, kSWarps * 32);
            if (bx == 0 && lane == 0 && p.partDot) {
                float tsum = 0.f;
                for (int w = 0; w < kSWarps; ++w) tsum += s_dot[w];
                p.partDot[bid] = tsum;
            }
        }
        if (bid == 0 && bx == 0 && lane == 0) p.header[p.slot] = (int)gridDim.x;
    }
}

template <int R, bool PROJ, bool WGRAD, bool DOT, bool W_IS_RD>
int launch_one(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmH, const StreamParams& p, size_t smem,
               int grid, const char* name, cudaStream_t st) {
    ProfScope ps(name, st, "stream_f16");
    auto kern = k_dense_stream<R, PROJ, WGRAD, DOT, W_IS_RD>;
    GCA_TRY(set_smem(kern, smem));
    GCA_CUDA(launch_pdl(kern, dim3(grid), dim3(stream_threads(PROJ, WGRAD)), smem, st, tmA, tmB, tmH, p));
    GCA_LAUNCH_OK();
    return GCA_OK;
}

template <int R>
int launch_dense_stream_t(const DenseStreamArgs& a, cudaStream_t st) {
    if constexpr (R != 16 && R != 32) {
        return GCA_ERR_UNSUPPORTED;
    } else {
        const bool proj = a.W != nullptr, wgrad = a.H != nullptr, dot = wgrad && a.B != nullptr;
        if (!tc_enabled() || !stream_enabled() || (!proj && !wgrad)) return GCA_ERR_UNSUPPORTED;
        // small inputs are launch-bound: the register-fed kernels (no tensor maps, 2 CTAs per SM) serve them
        if (a.d % 32 != 0 || a.d > 32 * kSWarps || a.n < 64 * kSRows) return GCA_ERR_UNSUPPORTED;
        if ((a.lda % 4) != 0 || (reinterpret_cast<uintptr_t>(a.A) % 16) != 0) return GCA_ERR_UNSUPPORTED;
        if (dot && ((a.ldb % 4) != 0 || (reinterpret_cast<uintptr_t>(a.B) % 16) != 0)) return GCA_ERR_UNSUPPORTED;
        if (wgrad && (reinterpret_cast<uintptr_t>(a.H) % 16) != 0) return GCA_ERR_UNSUPPORTED;
        // r = 32: projection + weight gradient in one CTA would need more than the 120 registers 17 warps leave a
        // thread; the caller issues the two halves as separate launches
        if (R == 32 && proj && wgrad) return GCA_ERR_UNSUPPORTED;
        constexpr int NT = R / 8;
        StreamParams p{};
        p.W = a.W; p.rowscale = a.rowscale; p.scalar = a.scalar; p.out = a.out;
        p.partG = a.partG; p.partCol = a.partCol; p.partDot = a.partDot; p.header = a.header; p.slot = a.slot;
        p.n = a.n; p.d = a.d; p.nb = a.d / 32;
        if (proj && a.push) {
            if (a.push->count < 0 || a.push->count > GCA_MAX_PEERS) return GCA_ERR_INVALID_ARG;
            p.push = *a.push;
        }
        const uint32_t a_bytes = (uint32_t)p.nb * kSBox;
        const uint32_t h_bytes = wgrad ? (uint32_t)(kSRows * R * 4) : 0u;
        p.b_off = dot ? a_bytes : 0u;
        p.h_off = a_bytes * (dot ? 2u : 1u);
        p.sc_off = p.h_off + h_bytes;
        const uint32_t sc_bytes = proj && a.rowscale ? (uint32_t)(kSRows * 4) : 0u;
        p.stage_bytes = (p.sc_off + sc_bytes + 1023u) & ~1023u;
        p.tx_bytes = p.sc_off + sc_bytes;
        const size_t red_bytes = proj ? (size_t)2 * kSWarps * (2 * NT * 32) * 16 : 0;
        const size_t out_bytes = proj ? (size_t)2 * kSRows * R * 4 : 0;       // staged output tiles of the projection epilogue
        const size_t fixed = red_bytes + 256 + out_bytes + 1024;     // partials + barriers / dot scratch + staging + alignment slack
        int stages = (int)((227 * 1024 - fixed) / p.stage_bytes);
        if (stages > 8) stages = 8;
        if (stages < 2) return GCA_ERR_UNSUPPORTED;
        p.stages = stages;
        p.red_off = (uint32_t)stages * p.stage_bytes;
        p.bar_off = p.red_off + (uint32_t)red_bytes;
        const size_t smem = (size_t)p.bar_off + 256 + out_bytes + 1024;
        CUtensorMap tmA, tmB, tmH;
        if (!get_box_map(&tmA, a.A, a.n, a.d, a.lda, 32, kSRows, true)) return GCA_ERR_UNSUPPORTED;
        tmB = tmA; tmH = tmA;
        if (dot && !get_box_map(&tmB, a.B, a.n, a.d, a.ldb, 32, kSRows, true)) return GCA_ERR_UNSUPPORTED;
        if (wgrad && !get_box_map(&tmH, a.H, a.n, R, R, R, kSRows, R == 32)) return GCA_ERR_UNSUPPORTED;
        const int ntiles = (a.n + kSRows - 1) / kSRows;
        const int grid = ntiles < num_sms() ? ntiles : num_sms();
        if (proj && wgrad) {                                         // R == 16: r = 32 was turned away above
            if (a.w_is_rd) return GCA_ERR_UNSUPPORTED;               // only the backward pairs the two (W = Wu [d, r])
            return launch_one<16, true, true, false, false>(tmA, tmB, tmH, p, smem, grid, a.prof_name, st);
        }
        if (proj)
            return a.w_is_rd ? launch_one<R, true, false, false, true>(tmA, tmB, tmH, p, smem, grid, a.prof_name, st)
                             : launch_one<R, true, false, false, false>(tmA, tmB, tmH, p, smem, grid, a.prof_name, st);
        return dot ? launch_one<R, false, true, true, false>(tmA, tmB, tmH, p, smem, grid, a.prof_name, st)
                   : launch_one<R, false, true, false, false>(tmA, tmB, tmH, p, smem, grid, a.prof_name, st);
    }
}

}  // namespace

int launch_dense_stream(int r, const DenseStreamArgs& a, cudaStream_t st) {
    GCA_DISPATCH_R(r, (launch_dense_stream_t<R_>(a, st)));
}

}  // namespace gca
