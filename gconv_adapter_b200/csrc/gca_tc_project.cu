// K1-tc: out[i, 0:R] = rowscale[i] * s * sum_k A[i,k] W[k, 0:R]  on tcgen05 (3xTF32, fp32 TMEM accumulators).
// The r = 32 projection whenever the streaming family (gca_stream.cu) does not run: n < 2048, d > 256, tensor maps
// refused, or the family switched off.  r = 16 takes the mma.sync kernel of gca_project.cu instead.
//
// Persistent, warp-specialised CTA (one per SM, 21 warps):
//   warps 0-15  producers : LDG.128 a [128 rows x 64 cols] chunk of A (4 rows x 128 B per warp instruction,
//                           four independent groups of 4 warps), split every value into tf32 hi / lo,
//                           STS both into a pipeline stage
//   warp  20    MMA issuer: per K-step (8 columns)  A_hi x [W_hi | W_lo]  (M=128, N=2R)  and
//                           A_lo x W_hi (N=R): every A byte is read from shared memory once;
//                           tcgen05.commit frees the stage / publishes the accumulators
//   warps 16-19 epilogue  : tcgen05.ld the accumulators (lane = row), add, scale, STG.128
// Stages and accumulators are handed over with mbarriers; accumulators are double-buffered in TMEM
// so the epilogue of tile t overlaps the loads and MMAs of tile t+1.
//
// Accuracy: the tensor core adds into its fp32 accumulator with truncation, a one-sided error that
// grows with the number of sequential updates (measured 2.2e-6 of max|out| with a single accumulator
// at K = 256, 2e-7 when spread).  The hi*hi (and hi*lo) products of K-step ks therefore go to
// accumulator group ks % NG, the lo*hi corrections to a separate one, and the epilogue adds them with
// round-to-nearest.
#include "gca_common.cuh"
#include "gca_host.cuh"
#include "gca_tc.cuh"

namespace gca {
namespace tc {

constexpr int kRows = 128;                 // rows per tile  (UMMA M)
constexpr int kCols = 64;                  // columns per pipeline stage
// S_C: bytes between 4-column chunks.  Padded by 16 B so that the 8 lanes of a quarter warp, which hold
// 8 consecutive column quads of ONE row (a full 128-byte line per global load), store to 8 distinct
// 16-byte bank groups.
constexpr int kColChunk = (kRows / 8) * 128 + 16;
constexpr int kHalfBytes = (kCols / 4) * kColChunk;   // ~32 KB: hi part of a stage; lo part follows
constexpr int kStageBytes = 2 * kHalfBytes;           // ~64 KB
constexpr int kProdWarps = 16;
constexpr int kThreads = 32 * (kProdWarps + 4 + 1);
constexpr int kPerThread = (kRows * kCols / 4) / 128;   // float4 per producer thread per chunk (16)

template <int R, bool W_IS_RD>
__global__ void __launch_bounds__(kThreads, 1)
k_project_tc(const float* __restrict__ A, int64_t lda, const float* __restrict__ W, const float* __restrict__ rowscale,
             const float* __restrict__ scalar, float* __restrict__ out, int n, int d, int nstage) {
    constexpr int NG = R == 16 ? 4 : 2;                 // accumulator groups
    constexpr int kAccCols = NG * 2 * R + R;            // TMEM columns per tile buffer
    constexpr uint32_t kTmemCols = 2 * kAccCols <= 256 ? 256 : 512;
    static_assert(2 * kAccCols <= 512, "TMEM budget");
    constexpr int SCW = (2 * R / 8) * 128;              // bytes between 4-k chunks of [W_hi | W_lo]

    extern __shared__ __align__(128) uint8_t smem_raw[];
    // layout: [stages][Wcat = rows 0..R-1 hi, rows R..2R-1 lo][barriers]
    uint8_t* stages = smem_raw;
    uint8_t* wcat = stages + (size_t)nstage * kStageBytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(wcat + (size_t)2 * R * d * 4);
    const uint32_t bar0 = smem_u32(bars);
    auto full_bar = [&](int s) { return bar0 + 8u * s; };
    auto empty_bar = [&](int s) { return bar0 + 8u * (nstage + s); };
    auto tfull_bar = [&](int a) { return bar0 + 8u * (2 * nstage + a); };
    auto tempty_bar = [&](int a) { return bar0 + 8u * (2 * nstage + 2 + a); };
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * nstage + 4);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    // ---- one-time setup ----
    if (threadIdx.x == 0) {
        for (int s = 0; s < nstage; ++s) { mbar_init(full_bar(s), 4); mbar_init(empty_bar(s), 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 4); }
        fence_barrier_init();
    }
    if (warp == kProdWarps + 4) tmem_alloc(smem_u32(tmem_slot), kTmemCols);
    // W -> shared, split, canonical K-major layout: element (n, k) -> (k/4) * SCW + (n/8)*128 + (n%8)*16 + (k%4)*4
    for (int idx = threadIdx.x; idx < d * R; idx += blockDim.x) {
        int k, c;
        if (W_IS_RD) { c = idx / d; k = idx - c * d; } else { k = idx / R; c = idx - k * R; }
        const float w = W[idx];
        const float hi = to_tf32(w), lo = to_tf32(w - hi);
        const int nl = c + R;
        *reinterpret_cast<float*>(wcat + (k >> 2) * SCW + (c >> 3) * 128 + (c & 7) * 16 + (k & 3) * 4) = hi;
        *reinterpret_cast<float*>(wcat + (k >> 2) * SCW + (nl >> 3) * 128 + (nl & 7) * 16 + (k & 3) * 4) = lo;
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const int ntiles = (n + kRows - 1) / kRows;
    const int nchunks = d / kCols;
    const int my_tiles = blockIdx.x < ntiles ? (ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

    if (warp < kProdWarps) {
        // ================= producers =================
        // Group g (4 warps) owns ring stage g for the whole kernel and fills chunks g, g + nstage, ...: one
        // producer per stage keeps the mbarrier phases in lock step (a parity wait cannot tell "two uses
        // ago" from "now").  A thread never has loads of a later chunk in flight when it executes
        // fence.proxy.async (which waits for the thread's outstanding memory operations); the other groups
        // keep HBM busy meanwhile.
        const int k4i = lane & 7, ri = lane >> 3;          // 8 lanes = one 128-byte line of a row
        const int grp = warp >> 2, wq = warp & 3;
        const int total = grp < nstage ? my_tiles * nchunks : 0;
        const int kGroups = nstage;
        int ltile = blockIdx.x, lch = grp;                 // (tile, chunk) of this group's next item
        while (lch >= nchunks) { lch -= nchunks; ltile += gridDim.x; }
        const int ps = grp;                                // this group's stage
        int pq = 0;                                        // how many times it has been filled
        for (int it = grp; it < total; it += kGroups) {
            float4 v[kPerThread];
#pragma unroll
            for (int j = 0; j < kPerThread; ++j) {
                // j -> (column half jc, row quad jr): rows wq*32 + jr*4 + ri, column quads jc*8 + k4i
                const int jc = j & 1, jr = j >> 1;
                const int row = min(ltile * kRows + wq * 32 + jr * 4 + ri, n - 1);
                v[j] = ldg4_stream(A + (size_t)row * lda + lch * kCols + jc * 32 + k4i * 4);
            }
            mbar_wait(empty_bar(ps), (uint32_t)((pq & 1) ^ 1));
            uint8_t* st = stages + (size_t)ps * kStageBytes;
#pragma unroll
            for (int j = 0; j < kPerThread; ++j) {
                const int jc = j & 1, jr = j >> 1;
                const int rl = wq * 32 + jr * 4 + ri;              // row inside the tile
                const uint32_t off = (uint32_t)((jc * 8 + k4i) * kColChunk + (rl >> 3) * 128 + (rl & 7) * 16);
                float4 hi, lo;
                split_tf32(v[j], hi, lo);
                *reinterpret_cast<float4*>(st + off) = hi;
                *reinterpret_cast<float4*>(st + kHalfBytes + off) = lo;
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(full_bar(ps));
            lch += kGroups;
            while (lch >= nchunks) { lch -= nchunks; ltile += gridDim.x; }
            ++pq;
        }
    } else if (warp == kProdWarps + 4) {
        // ================= MMA issuer =================
        // One thread feeds the tensor core, so its instruction stream is kept minimal: descriptors are
        // built once and advanced by adding constants to their low word (the 14-bit address field never
        // carries: shared memory is < 256 KB), stage / phase are counters, not divisions.
        if (lane == 0) {
            constexpr uint32_t idesc_cat = make_idesc_tf32(kRows, 2 * R, 0, 0);
            constexpr uint32_t idesc_r = make_idesc_tf32(kRows, R, 0, 0);
            constexpr uint64_t kStepA = (uint64_t)((2 * kColChunk) >> 4);     // one K-step = two 4-column chunks of A
            constexpr uint64_t kStepB = (uint64_t)((2 * SCW) >> 4);
            constexpr uint64_t kLoOff = (uint64_t)(kHalfBytes >> 4);
            const uint64_t a_desc0 = make_desc(smem_u32(stages), kColChunk, 128);
            const uint64_t b_desc0 = make_desc(smem_u32(wcat), SCW, 128);
            int s = 0;
            uint32_t ph = 0;
            for (int t = 0; t < my_tiles; ++t) {
                const int a = t & 1;
                mbar_wait(tempty_bar(a), (uint32_t)(((t >> 1) & 1) ^ 1));
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(a * kAccCols);
                uint64_t bd = b_desc0;
                for (int ch = 0; ch < nchunks; ++ch) {
                    mbar_wait(full_bar(s), ph);
                    tc_fence_after();
                    const uint64_t ad = a_desc0 + (uint64_t)s * (uint64_t)(kStageBytes >> 4);
                    const uint32_t later = ch != 0;
#pragma unroll
                    for (int ks = 0; ks < kCols / 8; ++ks) {
                        // group g = ks % NG: columns [g*2R, g*2R+R) = hi*hi, [g*2R+R, (g+1)*2R) = hi*lo
                        umma_tf32(d_tmem + (uint32_t)((ks % NG) * 2 * R), ad + ks * kStepA, bd + ks * kStepB, idesc_cat,
                                  ks >= NG ? 1u : later);
                        umma_tf32(d_tmem + (uint32_t)(NG * 2 * R), ad + kLoOff + ks * kStepA, bd + ks * kStepB, idesc_r,
                                  ks > 0 ? 1u : later);
                    }
                    bd += (kCols / 8) * kStepB;
                    umma_commit(empty_bar(s));                       // stage reusable once these MMAs retire
                    if (ch == nchunks - 1) umma_commit(tfull_bar(a)); // accumulators complete
                    if (++s == nstage) { s = 0; ph ^= 1u; }
                }
            }
        }
    } else {
        // ================= epilogue (warps 16-19 <-> TMEM lanes 32*(warp%4) ..) =================
        const int q = warp & 3;
        const float s = scalar ? __ldg(scalar) : 1.f;
        for (int t = 0; t < my_tiles; ++t) {
            const int a = t & 1;
            const int tile = blockIdx.x + t * gridDim.x;
            mbar_wait(tfull_bar(a), (uint32_t)((t >> 1) & 1));
            tc_fence_after();
            const uint32_t tb = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(a * kAccCols);
            float v[R];
#pragma unroll
            for (int c0 = 0; c0 < R; c0 += 16) {
                float big[16], small[16], t16[16];
                tmem_ld16(tb + (uint32_t)c0, big);                     // group 0: hi*hi
                tmem_ld16(tb + (uint32_t)(R + c0), small);             // group 0: hi*lo
#pragma unroll
                for (int g = 1; g < NG; ++g) {
                    tmem_ld16(tb + (uint32_t)(g * 2 * R + c0), t16);
#pragma unroll
                    for (int i = 0; i < 16; ++i) big[i] += t16[i];
                    tmem_ld16(tb + (uint32_t)(g * 2 * R + R + c0), t16);
#pragma unroll
                    for (int i = 0; i < 16; ++i) small[i] += t16[i];
                }
                tmem_ld16(tb + (uint32_t)(NG * 2 * R + c0), t16);      // lo*hi
#pragma unroll
                for (int i = 0; i < 16; ++i) v[c0 + i] = big[i] + (small[i] + t16[i]);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty_bar(a));
            const int row = tile * kRows + q * 32 + lane;
            if (row < n) {
                const float sc = (rowscale ? __ldg(rowscale + row) : 1.f) * s;
                float* o = out + (size_t)row * R;
#pragma unroll
                for (int c = 0; c < R; c += 4)
                    *reinterpret_cast<float4*>(o + c) = make_float4(v[c] * sc, v[c + 1] * sc, v[c + 2] * sc, v[c + 3] * sc);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == kProdWarps + 4) {
        tc_fence_after();
        tmem_dealloc(tmem_base, kTmemCols);
    }
}

template <int R, bool W_IS_RD>
int launch_project_tc_impl(const float* A, int64_t lda, const float* W, const float* rowscale, const float* scalar,
                           float* out, int n, int d, cudaStream_t st) {
    const size_t fixed = (size_t)2 * R * d * 4 + 256;
    const size_t budget = 227 * 1024;
    if (fixed + 2 * (size_t)kStageBytes > budget) return GCA_ERR_UNSUPPORTED;
    int nstage = (int)((budget - fixed) / kStageBytes);
    if (nstage > 4) nstage = 4;
    const size_t smem = fixed + (size_t)nstage * kStageBytes;
    GCA_TRY(set_smem(k_project_tc<R, W_IS_RD>, smem));
    const int ntiles = (n + kRows - 1) / kRows;
    const int grid = ntiles < num_sms() ? ntiles : num_sms();
    {
        ProfScope ps(W_IS_RD ? "project_fwd" : "project_bwd", st, "tcgen05");
        k_project_tc<R, W_IS_RD><<<grid, kThreads, smem, st>>>(A, lda, W, rowscale, scalar, out, n, d, nstage);
    }
    GCA_LAUNCH_OK();
    return GCA_OK;
}

}  // namespace tc

// Returns GCA_ERR_UNSUPPORTED when the shape is not on the tensor-core path (caller falls back to K1).
int launch_project_tc(int r, bool w_is_rd, const float* A, int64_t lda, const float* W, const float* rowscale,
                      const float* scalar, float* out, int n, int d, cudaStream_t st) {
    if (r != 32 || d % tc::kCols != 0 || n < 1) return GCA_ERR_UNSUPPORTED;
    return w_is_rd ? tc::launch_project_tc_impl<32, true>(A, lda, W, rowscale, scalar, out, n, d, st)
                   : tc::launch_project_tc_impl<32, false>(A, lda, W, rowscale, scalar, out, n, d, st);
}

}  // namespace gca
