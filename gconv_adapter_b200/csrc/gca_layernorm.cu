// normalization = 'layer_norm' (src/finetune/gconv_adapter.py:54-61, applied at :98-106): the adapter's tail
//     out = LayerNorm(out) ; out = out * scalar
// as ONE pass forward (read the pre-norm rows, write the result) and ONE pass backward (read gY and the pre-norm rows,
// write the gradient) instead of the two elementwise kernels forward / four backward of the stock ops (SURVEY.md 8f rank 2).
// Row statistics need the finished skip sum, so this runs after the fused hop + expand kernel on its output; a warp owns
// a row (d <= 1024: the row lives in registers), the per-column sums for the LayerNorm weight / bias gradients and the
// scalar's gradient are per-CTA partials combined in a fixed order by a second small kernel - no atomics.
//
//   forward   mean, rstd per row (two-pass in registers) ; Y = s * (gamma * (x - mean) * rstd + beta)
//   backward  xh = (x - mean) * rstd ; a = s * gY * gamma ; gX = rstd * (a - mean_c(a) - xh * mean_c(a * xh))
//             ggamma = sum_rows s * gY * xh ; gbeta = sum_rows s * gY ; gscalar = sum gY * (gamma * xh + beta)
#include "gca_common.cuh"
#include "gca_host.cuh"
#include "gca_norm.cuh"     // kLnThreads (8 warps, a row per warp here), warp_sum, k_ln_bwd_finalize

namespace gca {
namespace {

template <int VPL, bool ADD>   // float4s per lane: d <= 128 * VPL ; ADD: Y = ... + A (gca_layernorm_scale_add_fwd)
__global__ void __launch_bounds__(kLnThreads)
k_ln_fwd(const float* __restrict__ X, int64_t ldx, const float* __restrict__ gamma, const float* __restrict__ beta,
         const float* __restrict__ scalar, float eps, float* __restrict__ Y, int64_t ldy, float* __restrict__ mean_out,
         float* __restrict__ rstd_out, int n, int d, const float* A, int64_t lda) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nq = d >> 2;
    const float s = scalar ? __ldg(scalar) : 1.f;
    const float inv_d = 1.f / (float)d;
    float4 gm[VPL], bt[VPL];
#pragma unroll
    for (int v = 0; v < VPL; ++v) {
        const int q = lane + 32 * v;
        gm[v] = (gamma && q < nq) ? ldg4(gamma + 4 * q) : make_float4(1.f, 1.f, 1.f, 1.f);
        bt[v] = (beta && q < nq) ? ldg4(beta + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    pdl_wait();
    pdl_trigger();
    for (int row = blockIdx.x * kLnWarps + warp; row < n; row += gridDim.x * kLnWarps) {
        float4 x[VPL];
        float sum = 0.f;
#pragma unroll
        for (int v = 0; v < VPL; ++v) {
            const int q = lane + 32 * v;
            x[v] = q < nq ? ldg4_stream(X + (size_t)row * ldx + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
            sum += (x[v].x + x[v].y) + (x[v].z + x[v].w);
        }
        float4 av[ADD ? VPL : 1];
        if constexpr (ADD) {
#pragma unroll
            for (int v = 0; v < VPL; ++v) {
                const int q = lane + 32 * v;
                av[v] = q < nq ? ld4_addend(A + (size_t)row * lda + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
        const float mean = warp_sum(sum) * inv_d;
        float sq = 0.f;
#pragma unroll
        for (int v = 0; v < VPL; ++v) {
            if (lane + 32 * v < nq) {
                const float a = x[v].x - mean, b = x[v].y - mean, c = x[v].z - mean, e = x[v].w - mean;
                sq += (a * a + b * b) + (c * c + e * e);
            }
        }
        const float rstd = 1.f / sqrtf(warp_sum(sq) * inv_d + eps);
        if (lane == 0) { mean_out[row] = mean; rstd_out[row] = rstd; }
#pragma unroll
        for (int v = 0; v < VPL; ++v) {
            const int q = lane + 32 * v;
            if (q < nq) {
                float4 y;
                y.x = s * fmaf((x[v].x - mean) * rstd, gm[v].x, bt[v].x);
                y.y = s * fmaf((x[v].y - mean) * rstd, gm[v].y, bt[v].y);
                y.z = s * fmaf((x[v].z - mean) * rstd, gm[v].z, bt[v].z);
                y.w = s * fmaf((x[v].w - mean) * rstd, gm[v].w, bt[v].w);
                if constexpr (ADD) y = f4_add_rn(y, av[v]);
                stg4_stream(Y + (size_t)row * ldy + 4 * q, y);
            }
        }
    }
}

template <int VPL>
__global__ void __launch_bounds__(kLnThreads)
k_ln_bwd(const float* __restrict__ gY, int64_t ldg, const float* __restrict__ X, int64_t ldx,
         const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ scalar,
         const float* __restrict__ mean_in, const float* __restrict__ rstd_in, float* __restrict__ gX, int64_t ldgx,
         float* __restrict__ partG /*[grid][2][d]*/, float* __restrict__ partS /*[grid]*/, int n, int d, int rows_per_cta) {
    extern __shared__ float sm[];                     // [warps][2][d] + [warps]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nq = d >> 2;
    const float s = scalar ? __ldg(scalar) : 1.f;
    const float inv_d = 1.f / (float)d;
    float4 gm[VPL], bt[VPL], agm[VPL], abt[VPL];
#pragma unroll
    for (int v = 0; v < VPL; ++v) {
        const int q = lane + 32 * v;
        gm[v] = (gamma && q < nq) ? ldg4(gamma + 4 * q) : make_float4(1.f, 1.f, 1.f, 1.f);
        bt[v] = (beta && q < nq) ? ldg4(beta + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
        agm[v] = make_float4(0.f, 0.f, 0.f, 0.f);
        abt[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    float gs = 0.f;
    pdl_wait();
    pdl_trigger();
    const int r0 = blockIdx.x * rows_per_cta, r1 = min(n, r0 + rows_per_cta);
    for (int row = r0 + warp; row < r1; row += kLnWarps) {
        const float mean = __ldg(mean_in + row), rstd = __ldg(rstd_in + row);
        float4 xh[VPL], a[VPL];
        float m1 = 0.f, m2 = 0.f;
#pragma unroll
        for (int v = 0; v < VPL; ++v) {
            const int q = lane + 32 * v;
            if (q < nq) {
                const float4 x = ldg4_stream(X + (size_t)row * ldx + 4 * q);
                const float4 g = ldg4_stream(gY + (size_t)row * ldg + 4 * q);
                xh[v] = make_float4((x.x - mean) * rstd, (x.y - mean) * rstd, (x.z - mean) * rstd, (x.w - mean) * rstd);
                gs = fmaf(g.x, fmaf(gm[v].x, xh[v].x, bt[v].x), gs);
                gs = fmaf(g.y, fmaf(gm[v].y, xh[v].y, bt[v].y), gs);
                gs = fmaf(g.z, fmaf(gm[v].z, xh[v].z, bt[v].z), gs);
                gs = fmaf(g.w, fmaf(gm[v].w, xh[v].w, bt[v].w), gs);
                const float4 gl = make_float4(s * g.x, s * g.y, s * g.z, s * g.w);      // gradient w.r.t. the LayerNorm output
                agm[v].x = fmaf(gl.x, xh[v].x, agm[v].x); agm[v].y = fmaf(gl.y, xh[v].y, agm[v].y);
                agm[v].z = fmaf(gl.z, xh[v].z, agm[v].z); agm[v].w = fmaf(gl.w, xh[v].w, agm[v].w);
                abt[v].x += gl.x; abt[v].y += gl.y; abt[v].z += gl.z; abt[v].w += gl.w;
                a[v] = make_float4(gl.x * gm[v].x, gl.y * gm[v].y, gl.z * gm[v].z, gl.w * gm[v].w);
                m1 += (a[v].x + a[v].y) + (a[v].z + a[v].w);
                m2 += (a[v].x * xh[v].x + a[v].y * xh[v].y) + (a[v].z * xh[v].z + a[v].w * xh[v].w);
            } else {
                xh[v] = make_float4(0.f, 0.f, 0.f, 0.f);
                a[v] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
        m1 = warp_sum(m1) * inv_d;
        m2 = warp_sum(m2) * inv_d;
        if (gX) {
#pragma unroll
            for (int v = 0; v < VPL; ++v) {
                const int q = lane + 32 * v;
                if (q < nq) {
                    float4 o;
                    o.x = rstd * (a[v].x - m1 - xh[v].x * m2);
                    o.y = rstd * (a[v].y - m1 - xh[v].y * m2);
                    o.z = rstd * (a[v].z - m1 - xh[v].z * m2);
                    o.w = rstd * (a[v].w - m1 - xh[v].w * m2);
                    stg4_stream(gX + (size_t)row * ldgx + 4 * q, o);
                }
            }
        }
    }
    // ---- per-CTA partials: the warps' column sums are added in warp order ----
    float* s_col = sm;                                // [warps][2][d]
    float* s_gs = sm + kLnWarps * 2 * d;              // [warps]
#pragma unroll
    for (int v = 0; v < VPL; ++v) {
        const int q = lane + 32 * v;
        if (q < nq) {
            *reinterpret_cast<float4*>(s_col + (size_t)(warp * 2 + 0) * d + 4 * q) = agm[v];
            *reinterpret_cast<float4*>(s_col + (size_t)(warp * 2 + 1) * d + 4 * q) = abt[v];
        }
    }
    gs = warp_sum(gs);
    if (lane == 0) s_gs[warp] = gs;
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * d; i += kLnThreads) {
        const int which = i / d, c = i - which * d;
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < kLnWarps; ++w) t += s_col[(size_t)(w * 2 + which) * d + c];
        partG[((size_t)blockIdx.x * 2 + which) * d + c] = t;
    }
    if (threadIdx.x == 0) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < kLnWarps; ++w) t += s_gs[w];
        partS[blockIdx.x] = t;
    }
}

inline size_t ln_scratch_bytes(int d) { return align_up(sizeof(float) * ((size_t)kLnMaxParts * 2 * d + kLnMaxParts)); }

template <int VPL, bool ADD>
int ln_fwd_t(const float* X, int64_t ldx, const float* gamma, const float* beta, const float* scalar, float eps, float* Y,
             int64_t ldy, float* mean, float* rstd, int n, int d, const float* A, int64_t lda, cudaStream_t st) {
    int grid = (n + kLnWarps - 1) / kLnWarps;
    if (grid > 8 * num_sms()) grid = 8 * num_sms();
    {
        ProfScope ps("layernorm_fwd", st);
        GCA_CUDA(launch_pdl(k_ln_fwd<VPL, ADD>, dim3(grid), dim3(kLnThreads), 0, st, X, ldx, gamma, beta, scalar, eps, Y, ldy, mean, rstd,
                            n, d, A, lda));
    }
    GCA_LAUNCH_OK();
    return GCA_OK;
}

template <int VPL>
int ln_bwd_t(const float* gY, int64_t ldg, const float* X, int64_t ldx, const float* gamma, const float* beta,
             const float* scalar, const float* mean, const float* rstd, float* gX, int64_t ldgx, float* ggamma, float* gbeta,
             float* gscalar, void* scratch, int n, int d, cudaStream_t st) {
    int grid = (n + kLnWarps - 1) / kLnWarps;
    const int cap = 2 * num_sms() < kLnMaxParts ? 2 * num_sms() : kLnMaxParts;
    if (grid > cap) grid = cap;
    const int rows_per_cta = (n + grid - 1) / grid;
    float* partG = static_cast<float*>(scratch);
    float* partS = partG + (size_t)kLnMaxParts * 2 * d;
    const size_t smem = sizeof(float) * ((size_t)kLnWarps * 2 * d + kLnWarps);
    GCA_TRY(set_smem(k_ln_bwd<VPL>, smem));
    {
        ProfScope ps("layernorm_bwd", st);
        GCA_CUDA(launch_pdl(k_ln_bwd<VPL>, dim3(grid), dim3(kLnThreads), smem, st, gY, ldg, X, ldx, gamma, beta, scalar, mean, rstd,
                            gX, ldgx, partG, partS, n, d, rows_per_cta));
    }
    GCA_LAUNCH_OK();
    const int fgrid = (2 * d + 1 + kLnWarps - 1) / kLnWarps;
    {
        ProfScope ps("layernorm_bwd_finalize", st);
        GCA_CUDA(launch_pdl(k_ln_bwd_finalize, dim3(fgrid), dim3(kLnThreads), 0, st, (const float*)partG, (const float*)partS,
                            grid, d, ggamma, gbeta, gscalar));
    }
    GCA_LAUNCH_OK();
    return GCA_OK;
}

#define GCA_DISPATCH_VPL(d, CALL)                                   \
    if ((d) <= 128) { constexpr int V_ = 1; return CALL; }          \
    if ((d) <= 256) { constexpr int V_ = 2; return CALL; }          \
    if ((d) <= 512) { constexpr int V_ = 4; return CALL; }          \
    { constexpr int V_ = 8; return CALL; }

inline bool ln_args_ok(const void* a, const void* b, int64_t lda, int64_t ldb, int n, int d) {
    return a && b && n >= 0 && d > 0 && (d % 4) == 0 && d <= 1024 && lda >= d && ldb >= d && (lda % 4) == 0 && (ldb % 4) == 0 &&
           (reinterpret_cast<uintptr_t>(a) % 16) == 0 && (reinterpret_cast<uintptr_t>(b) % 16) == 0;
}

}  // namespace
}  // namespace gca

using namespace gca;

extern "C" size_t gca_layernorm_scratch_bytes(int32_t d) { return d > 0 ? ln_scratch_bytes(d) : 0; }

extern "C" int gca_layernorm_scale_fwd(const float* X, int64_t ldx, const float* gamma, const float* beta, const float* scalar,
                                       float eps, float* Y, int64_t ldy, float* mean, float* rstd, int32_t n, int32_t d,
                                       gca_stream_t stream) {
    if (!mean || !rstd || !(eps >= 0.f)) return GCA_ERR_INVALID_ARG;
    if (!X || !Y || n < 0 || d <= 0) return GCA_ERR_INVALID_ARG;
    if (!ln_args_ok(X, Y, ldx, ldy, n, d)) return GCA_ERR_UNSUPPORTED;
    if (n == 0) return GCA_OK;
    const PdlHint pdl_hint(n);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    GCA_DISPATCH_VPL(d, (ln_fwd_t<V_, false>(X, ldx, gamma, beta, scalar, eps, Y, ldy, mean, rstd, n, d, nullptr, 0, st)));
}

extern "C" int gca_layernorm_scale_add_fwd(const float* X, int64_t ldx, const float* gamma, const float* beta,
                                           const float* scalar, float eps, const float* A, int64_t lda, float* Y, int64_t ldy,
                                           float* mean, float* rstd, int32_t n, int32_t d, gca_stream_t stream) {
    if (!mean || !rstd || !(eps >= 0.f)) return GCA_ERR_INVALID_ARG;
    if (!X || !A || !Y || n < 0 || d <= 0) return GCA_ERR_INVALID_ARG;
    if (!ln_args_ok(X, Y, ldx, ldy, n, d) || !ln_args_ok(A, Y, lda, ldy, n, d)) return GCA_ERR_UNSUPPORTED;
    if (n == 0) return GCA_OK;
    const PdlHint pdl_hint(n);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    GCA_DISPATCH_VPL(d, (ln_fwd_t<V_, true>(X, ldx, gamma, beta, scalar, eps, Y, ldy, mean, rstd, n, d, A, lda, st)));
}

extern "C" int gca_layernorm_scale_bwd(const float* gY, int64_t ldg, const float* X, int64_t ldx, const float* gamma,
                                       const float* beta, const float* scalar, const float* mean, const float* rstd, float* gX,
                                       int64_t ldgx, float* ggamma, float* gbeta, float* gscalar, void* scratch, int32_t n,
                                       int32_t d, gca_stream_t stream) {
    if (!gY || !X || !mean || !rstd || !scratch || n < 0 || d <= 0) return GCA_ERR_INVALID_ARG;
    if ((reinterpret_cast<uintptr_t>(scratch) % kAlign) != 0) return GCA_ERR_WORKSPACE;
    if (!ln_args_ok(gY, X, ldg, ldx, n, d)) return GCA_ERR_UNSUPPORTED;
    if (gX && (ldgx < d || (ldgx % 4) != 0 || (reinterpret_cast<uintptr_t>(gX) % 16) != 0)) return GCA_ERR_UNSUPPORTED;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (n == 0) {       // empty input: the parameter gradients are zero
        if (ggamma) GCA_CUDA(cudaMemsetAsync(ggamma, 0, sizeof(float) * d, st));
        if (gbeta) GCA_CUDA(cudaMemsetAsync(gbeta, 0, sizeof(float) * d, st));
        if (gscalar) GCA_CUDA(cudaMemsetAsync(gscalar, 0, sizeof(float), st));
        return GCA_OK;
    }
    const PdlHint pdl_hint(n);
    GCA_DISPATCH_VPL(d, (ln_bwd_t<V_>(gY, ldg, X, ldx, gamma, beta, scalar, mean, rstd, gX, ldgx, ggamma, gbeta, gscalar, scratch,
                                      n, d, st)));
}
