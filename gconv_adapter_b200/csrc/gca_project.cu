// K1 projection  [n,d] x [d,R] -> [n,R]   (conv_down.lin ; gH2' = gY Wu), register-fed variants:
//   k_project_mma   3xTF32 mma.sync, A fragments straight from global memory            (r = 16 / 32, d % 16 == 0)
//   k_project       FFMA, register-tiled                                                 (every other shape; r = 128
//                   as two 64-column blocks, k_project<64, W_IS_RD, 128>)
// The default for large inputs is the TMA-fed family in gca_stream.cu; tc::k_project_tc (gca_tc_project.cu) is the
// tcgen05 / TMEM variant used at r = 32.
// Reference semantics: /root/reference/src/finetune/gconv_adapter.py:92 (the Linear inside each GCNConv).
#include "gca_common.cuh"
#include "gca_device.cuh"
#include "gca_host.cuh"

namespace gca {
namespace {

// ------------------------------------------------------------------------------------------
// K1: out[i, 0:R] = rowscale[i] * s * sum_k A[i,k] W[k, 0:R]
// Thread (kq = lane & 7, rg = lane >> 3) of warp w owns RT rows and the k-quads kq, kq+8, ...:
// a quarter warp reads 128 contiguous bytes of one row; W sits in shared memory, padded so the
// eight k-quads of a quarter warp hit distinct banks.  Partial sums are combined over the eight
// kq lanes with a transposing butterfly (56 shuffles for 64 values).
// ------------------------------------------------------------------------------------------
//
// RW > R (k_project<64, W_IS_RD, 128>, the r = 128 projection): blockIdx.y picks the R-column block of W and of out that
// the CTA computes; out's rows are RW floats apart, and so are W's when it is stored [d, RW].  Every block reads all of
// A: at r = 128 the projection is FFMA-bound (2 r = 256 flop per 4-byte element of A against ~9 flop/B of machine
// balance), so the second read of A costs bandwidth that is spare.
template <int R, bool W_IS_RD, int RW = R>
__global__ void __launch_bounds__(256, 2)
k_project(const float* __restrict__ A, int64_t lda, const float* __restrict__ W, const float* __restrict__ rowscale,
          const float* __restrict__ scalar, float* __restrict__ out, int n, int d) {
    constexpr int RT = 64 / R;            // rows per thread
    constexpr int TILE = 32 * RT;         // rows per CTA tile (8 warps x 4 row groups x RT)
    constexpr int KS = 4 * R + 4;         // padded floats per k-quad of W
    extern __shared__ __align__(16) float smem[];
    float* Ws = smem;
    const int nk4 = d >> 2;
    if constexpr (RW != R) {
        const int cb = blockIdx.y * R;
        W += W_IS_RD ? (size_t)cb * d : (size_t)cb;
        out += cb;
    }
    for (int idx = threadIdx.x; idx < d * R; idx += blockDim.x) {
        int k, c;
        if (W_IS_RD) { c = idx / d; k = idx - c * d; } else { k = idx / R; c = idx - k * R; }
        if constexpr (RW == R || W_IS_RD) Ws[(k >> 2) * KS + (k & 3) * R + c] = W[idx];
        else Ws[(k >> 2) * KS + (k & 3) * R + c] = W[(size_t)k * RW + c];
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int kq = lane & 7, rg = lane >> 3;
    const float s = scalar ? __ldg(scalar) : 1.f;
    const int ntiles = (n + TILE - 1) / TILE;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int row0 = tile * TILE + (warp * 4 + rg) * RT;
        const float* arow[RT];
#pragma unroll
        for (int t = 0; t < RT; ++t) arow[t] = A + (size_t)min(row0 + t, n - 1) * lda;
        float v[RT * R];
#pragma unroll
        for (int i = 0; i < RT * R; ++i) v[i] = 0.f;
        float4 a[RT];
        if (kq < nk4) {
#pragma unroll
            for (int t = 0; t < RT; ++t) a[t] = ldg4_stream(arow[t] + kq * 4);
        }
        for (int k4 = kq; k4 < nk4; k4 += 8) {
            float4 an[RT];
            const int k4n = k4 + 8;
            if (k4n < nk4) {
#pragma unroll
                for (int t = 0; t < RT; ++t) an[t] = ldg4_stream(arow[t] + k4n * 4);
            }
            const float* w = Ws + k4 * KS;
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
#pragma unroll
                for (int c4 = 0; c4 < R / 4; ++c4) {
                    const float4 wv = *reinterpret_cast<const float4*>(w + kk * R + c4 * 4);
#pragma unroll
                    for (int t = 0; t < RT; ++t) {
                        const float av = kk == 0 ? a[t].x : kk == 1 ? a[t].y : kk == 2 ? a[t].z : a[t].w;
                        v[t * R + c4 * 4 + 0] = fmaf(av, wv.x, v[t * R + c4 * 4 + 0]);
                        v[t * R + c4 * 4 + 1] = fmaf(av, wv.y, v[t * R + c4 * 4 + 1]);
                        v[t * R + c4 * 4 + 2] = fmaf(av, wv.z, v[t * R + c4 * 4 + 2]);
                        v[t * R + c4 * 4 + 3] = fmaf(av, wv.w, v[t * R + c4 * 4 + 3]);
                    }
                }
            }
            if (k4n < nk4) {
#pragma unroll
                for (int t = 0; t < RT; ++t) a[t] = an[t];
            }
        }
        // transposing butterfly over lane bits 2,1,0: 64 -> 32 -> 16 -> 8 values per lane
#pragma unroll
        for (int half = 32, bit = 4; half >= 8; half >>= 1, bit >>= 1) {
            const bool up = (lane & bit) != 0;
#pragma unroll
            for (int i = 0; i < half; ++i) {
                const float send = up ? v[i] : v[i + half];
                const float keep = up ? v[i + half] : v[i];
                v[i] = keep + __shfl_xor_sync(0xffffffffu, send, bit);
            }
        }
        const int base = ((lane >> 2) & 1) * 32 + ((lane >> 1) & 1) * 16 + (lane & 1) * 8;
        const int row = row0 + base / R, c0 = base % R;
        if (row < n) {
            const float sc = (rowscale ? __ldg(rowscale + row) : 1.f) * s;
            float* o = out + (size_t)row * RW + c0;
            *reinterpret_cast<float4*>(o) = make_float4(v[0] * sc, v[1] * sc, v[2] * sc, v[3] * sc);
            *reinterpret_cast<float4*>(o + 4) = make_float4(v[4] * sc, v[5] * sc, v[6] * sc, v[7] * sc);
        }
    }
}

// ------------------------------------------------------------------------------------------
// K1-mma: out[i, 0:R] = rowscale[i] * s * sum_k A[i,k] W[k, 0:R] with M = rows, N = R, K = columns of A.
// A-fragments come straight from global memory: lane (g, t) loads the float4 A[row g (+8)][kb + 4t .. +3] of a
// 16-column block kb (8 rows x 64 contiguous bytes per warp instruction) and uses it for two k-steps through
// the K permutation  k-step s: logical k = t -> column kb+4t+2s, logical k = t+4 -> column kb+4t+2s+1.
// W sits in shared memory as {b0_hi, b1_hi, b0_lo, b1_lo} quads in exactly that order, one LDS.128 per
// (k-step, n-tile).  Products go to 2 accumulator sets (alternating 16-column blocks) + 1 for the lo terms.
// ------------------------------------------------------------------------------------------
template <int R, bool W_IS_RD>
__device__ __forceinline__ void project_mma_body(const float* __restrict__ A, int64_t lda, const float* __restrict__ W,
                                                 const float* __restrict__ rowscale, const float* __restrict__ scalar,
                                                 float* __restrict__ out, int n, int d, int bid, int nblocks,
                                                 uint32_t* smem_u) {
    constexpr int NT = R / 8;                       // n-tiles
    // The projections are the first kernels of gca_forward / gca_backward: what precedes them on the stream is
    // not ours (an optimizer step may just have written W), so they wait before touching anything.
    pdl_wait();
    // Wq[kb][s][nt][g][t] = uint4 {hi(k0,c), hi(k1,c), lo(k0,c), lo(k1,c)}, k0 = kb*16+4t+2s, k1 = k0+1, c = nt*8+g
    // (lane = 4g + t reads consecutive 16-byte slots: conflict-free LDS.128)
    uint4* Wq = reinterpret_cast<uint4*>(smem_u);
    const int nkb = d >> 4;                         // 16-column blocks (d % 16 == 0)
    for (int idx = threadIdx.x; idx < nkb * 2 * 4 * NT * 8; idx += blockDim.x) {
        int r_ = idx;
        const int t_ = r_ & 3; r_ >>= 2;
        const int g_ = r_ & 7; r_ >>= 3;
        const int nt_ = r_ % NT; r_ /= NT;
        const int s_ = r_ & 1; const int kb_ = r_ >> 1;
        const int k0 = kb_ * 16 + 4 * t_ + 2 * s_, c = nt_ * 8 + g_;
        const float w0 = W_IS_RD ? W[(size_t)c * d + k0] : W[(size_t)k0 * R + c];
        const float w1 = W_IS_RD ? W[(size_t)c * d + k0 + 1] : W[(size_t)(k0 + 1) * R + c];
        uint4 q;
        split_tf32(w0, q.x, q.z);
        split_tf32(w1, q.y, q.w);
        Wq[idx] = q;
    }
    __syncthreads();
    pdl_trigger();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, t = lane & 3;
    const float sc_s = scalar ? __ldg(scalar) : 1.f;
    const int nmt = (n + 15) / 16;                  // 16-row m-tiles
    const int wglobal = bid * 8 + warp, wtotal = nblocks * 8;
    // m-tiles are handed out round-robin (static): the kernel keeps no state outside its own outputs
    for (int mt = wglobal; mt < nmt; mt += wtotal) {
        const int r0 = mt * 16 + g, r1 = r0 + 8;
        const float* p0 = A + (size_t)min(r0, n - 1) * lda + 4 * t;
        const float* p1 = A + (size_t)min(r1, n - 1) * lda + 4 * t;
        float acc[3][NT][4];
#pragma unroll
        for (int a_ = 0; a_ < 3; ++a_)
#pragma unroll
            for (int j = 0; j < NT; ++j)
#pragma unroll
                for (int i = 0; i < 4; ++i) acc[a_][j][i] = 0.f;
        // software pipeline over batches of 4 column blocks: the 8 loads of batch b+1 are issued before the
        // tensor-core work of batch b, so 8-16 loads per lane are in flight at all times
        float4 xa0[4], xa1[4], xb0[4], xb1[4];
        auto load = [&](float4 (&x0)[4], float4 (&x1)[4], int kb0) {
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (kb0 + u < nkb) {
                    x0[u] = ldg4_stream(p0 + (kb0 + u) * 16);
                    x1[u] = ldg4_stream(p1 + (kb0 + u) * 16);
                }
            }
        };
        auto compute = [&](const float4 (&x0)[4], const float4 (&x1)[4], int kb0) {
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (kb0 + u >= nkb) break;
                const float e0[4] = {x0[u].x, x0[u].y, x0[u].z, x0[u].w};
                const float e1[4] = {x1[u].x, x1[u].y, x1[u].z, x1[u].w};
#pragma unroll
                for (int s_ = 0; s_ < 2; ++s_) {
                    uint32_t ah[4], al[4];
                    split_tf32(e0[2 * s_], ah[0], al[0]);        // (row g,   k = t)
                    split_tf32(e1[2 * s_], ah[1], al[1]);        // (row g+8, k = t)
                    split_tf32(e0[2 * s_ + 1], ah[2], al[2]);    // (row g,   k = t+4)
                    split_tf32(e1[2 * s_ + 1], ah[3], al[3]);    // (row g+8, k = t+4)
                    const uint4* wq = Wq + (((kb0 + u) * 2 + s_) * NT) * 32 + lane;
#pragma unroll
                    for (int j = 0; j < NT; ++j) {
                        const uint4 q = wq[j * 32];
                        mma_tf32(acc[u & 1][j], ah, q.x, q.y);
                        mma_tf32(acc[2][j], al, q.x, q.y);
                        mma_tf32(acc[2][j], ah, q.z, q.w);
                    }
                }
            }
        };
        load(xa0, xa1, 0);
        for (int kb0 = 0; kb0 < nkb; kb0 += 8) {
            if (kb0 + 4 < nkb) load(xb0, xb1, kb0 + 4);
            compute(xa0, xa1, kb0);
            if (kb0 + 4 < nkb) {
                if (kb0 + 8 < nkb) load(xa0, xa1, kb0 + 8);
                compute(xb0, xb1, kb0 + 4);
            }
        }
        const float sc0 = (r0 < n ? (rowscale ? __ldg(rowscale + r0) : 1.f) : 0.f) * sc_s;
        const float sc1 = (r1 < n ? (rowscale ? __ldg(rowscale + r1) : 1.f) : 0.f) * sc_s;
#pragma unroll
        for (int j = 0; j < NT; ++j) {
            float v[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) v[i] = (acc[0][j][i] + acc[1][j][i]) + acc[2][j][i];
            if (r0 < n) *reinterpret_cast<float2*>(out + (size_t)r0 * R + j * 8 + 2 * t) = make_float2(v[0] * sc0, v[1] * sc0);
            if (r1 < n) *reinterpret_cast<float2*>(out + (size_t)r1 * R + j * 8 + 2 * t) = make_float2(v[2] * sc1, v[3] * sc1);
        }
    }
}

template <int R, bool W_IS_RD>
__global__ void __launch_bounds__(256, 2)
k_project_mma(const float* __restrict__ A, int64_t lda, const float* __restrict__ W, const float* __restrict__ rowscale,
              const float* __restrict__ scalar, float* __restrict__ out, int n, int d) {
    extern __shared__ __align__(16) uint32_t smem_dyn[];
    project_mma_body<R, W_IS_RD>(A, lda, W, rowscale, scalar, out, n, d, blockIdx.x, gridDim.x, smem_dyn);
}

template <int R, bool W_IS_RD>
int launch_project_narrow_t(const float* A, int64_t lda, const float* W, const float* rowscale, const float* scalar,
                            float* out, int n, int d, cudaStream_t st) {
    if (tc_enabled()) {
        // Register-fed tensor-core variants (the TMA-fed family of gca_stream.cu is tried first by the callers):
        // r = 32 -> tcgen05 / TMEM kernel (r = 32 doubles the 3xTF32 mma.sync work; 0.69 vs 0.84 ms at products size),
        // r = 16 -> mma.sync with fragments straight from global memory.
        if (R == 32) {
            const int st_first = launch_project_tc(R, W_IS_RD, A, lda, W, rowscale, scalar, out, n, d, st);
            if (st_first != GCA_ERR_UNSUPPORTED) return st_first;
        }
        if constexpr (R == 16 || R == 32) {
            if (d % 16 == 0) {
                const size_t smem_m = sizeof(uint4) * (size_t)(d / 16) * 2 * 4 * (R / 8) * 8;
                if (smem_m <= 100 * 1024) {
                    GCA_TRY(set_smem(k_project_mma<R, W_IS_RD>, smem_m));
                    const int nmt = (n + 15) / 16;
                    int grid_m = (nmt + 7) / 8;
                    if (grid_m > 2 * num_sms()) grid_m = 2 * num_sms();
                    {
                        ProfScope ps(W_IS_RD ? "project_fwd" : "project_bwd", st, "mma");
                        GCA_CUDA(launch_pdl(k_project_mma<R, W_IS_RD>, dim3(grid_m), dim3(256), smem_m, st, A, lda, W, rowscale, scalar, out, n, d));
                    }
                    GCA_LAUNCH_OK();
                    return GCA_OK;
                }
            }
        }
    }
    constexpr int TILE = 32 * (64 / R);
    const size_t smem = sizeof(float) * (size_t)(d / 4) * (4 * R + 4);
    if (smem > 200 * 1024) return GCA_ERR_UNSUPPORTED;
    GCA_TRY(set_smem(k_project<R, W_IS_RD>, smem));
    const int ntiles = (n + TILE - 1) / TILE;
    const int grid = ntiles < 2 * num_sms() ? ntiles : 2 * num_sms();
    {
        ProfScope ps(W_IS_RD ? "project_fwd" : "project_bwd", st, "ffma");
        k_project<R, W_IS_RD><<<grid, 256, smem, st>>>(A, lda, W, rowscale, scalar, out, n, d);
    }
    GCA_LAUNCH_OK();
    return GCA_OK;
}

// r = 128: the 64-column blocks of k_project<64, W_IS_RD, 128> as blockIdx.y = 0 / 1
template <bool W_IS_RD>
int launch_project_wide(const float* A, int64_t lda, const float* W, const float* rowscale, const float* scalar,
                        float* out, int n, int d, cudaStream_t st) {
    constexpr int TILE = 32;                                  // rows per CTA tile of the R = 64 body
    const size_t smem = sizeof(float) * (size_t)(d / 4) * (4 * 64 + 4);
    if (smem > 200 * 1024) return GCA_ERR_UNSUPPORTED;
    GCA_TRY(set_smem(k_project<64, W_IS_RD, 128>, smem));
    const int ntiles = (n + TILE - 1) / TILE;
    const int grid = ntiles < num_sms() ? ntiles : num_sms();   // x 2 halves: two CTAs per SM as for R = 64
    {
        ProfScope ps(W_IS_RD ? "project_fwd" : "project_bwd", st, "ffma");
        k_project<64, W_IS_RD, 128><<<dim3(grid, 2), 256, smem, st>>>(A, lda, W, rowscale, scalar, out, n, d);
    }
    GCA_LAUNCH_OK();
    return GCA_OK;
}

template <int R, bool W_IS_RD>
int launch_project_t(const float* A, int64_t lda, const float* W, const float* rowscale, const float* scalar,
                     float* out, int n, int d, cudaStream_t st) {
    if (n == 0) return GCA_OK;
    if constexpr (R == 128) {
        return launch_project_wide<W_IS_RD>(A, lda, W, rowscale, scalar, out, n, d, st);
    } else {
        return launch_project_narrow_t<R, W_IS_RD>(A, lda, W, rowscale, scalar, out, n, d, st);
    }
}

}  // namespace

int launch_project(int r, bool w_is_rd, const float* A, int64_t lda, const float* W, const float* rowscale, const float* scalar,
                   float* out, int n, int d, cudaStream_t st) {
    if (w_is_rd) { GCA_DISPATCH_R(r, (launch_project_t<R_, true>(A, lda, W, rowscale, scalar, out, n, d, st))); }
    GCA_DISPATCH_R(r, (launch_project_t<R_, false>(A, lda, W, rowscale, scalar, out, n, d, st)));
}

}  // namespace gca
