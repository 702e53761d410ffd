// normalization = 'batch_norm' (src/finetune/gconv_adapter.py:54-61, applied at :98-106): the adapter's tail
//     out = BatchNorm1d(out) ; out = out * scalar
// with torch.nn.BatchNorm1d's semantics for a 2-D input: batch statistics (biased variance) and the running-buffer update
// in training, the running statistics in eval.  Column statistics over all n rows, so unlike the LayerNorm tail any
// d % 4 == 0 works: columns go in chunks of 128 (a warp reads 512 contiguous bytes of a row), one chunk per CTA in the
// statistics and elementwise passes, all chunks in turn in the backward's reduce pass (one scalar partial per CTA).
//
//   statistics  per-CTA sums of (x - K_c) and (x - K_c)^2 over contiguous row ranges, K_c = X[0, c] for every CTA (the shift
//               keeps the second sum from cancelling when |mean| >> std); fp32 over kBnFold rows, then fp64; a second kernel
//               adds the CTAs' sums in a fixed order in fp64 -> mean, rstd and the running buffers
//   forward     Y = s * (gamma * (x - mean) * rstd + beta)                                      one read, one write
//   backward    xh = (x - mean) * rstd ; a = s * gamma * gY
//               ggamma = sum_rows s * gY * xh ; gbeta = sum_rows s * gY ; gscalar = sum gY * (gamma * xh + beta)
//               training: gX = rstd * (a - mean_rows(a) - xh * mean_rows(a * xh)), the row means being gamma * gbeta / n
//               and gamma * ggamma / n: one reduce pass over gY and X, k_ln_bwd_finalize, one pass that writes gX
//               eval: gX = s * gamma * rstd * gY, written by the reduce pass itself
// No atomics: every sum has a fixed order, so results are bitwise reproducible.
#include "gca_common.cuh"
#include "gca_host.cuh"
#include "gca_norm.cuh"     // kLnThreads, kLnWarps, kLnMaxParts, warp_sum, k_ln_bwd_finalize

namespace gca {
namespace {

constexpr int kBnChunk = 32;      // float4 columns per chunk: one per lane
constexpr int kBnFold = 16;       // rows a thread sums in fp32 before it folds the sums into wider accumulators
constexpr int kBnUnroll = 4;      // rows whose loads a thread has in flight at once (twice that in k_bn_stats)

__device__ __forceinline__ float4 f4_ld(const float* p) { return make_float4(__ldg(p), __ldg(p + 1), __ldg(p + 2), __ldg(p + 3)); }
__device__ __forceinline__ float4 f4_ld_or(const float* p, float v) { return p ? f4_ld(p) : make_float4(v, v, v, v); }
__device__ __forceinline__ float4 f4_sub(float4 a, float4 b) { return make_float4(a.x - b.x, a.y - b.y, a.z - b.z, a.w - b.w); }
__device__ __forceinline__ float4 f4_mul(float4 a, float4 b) { return make_float4(a.x * b.x, a.y * b.y, a.z * b.z, a.w * b.w); }
__device__ __forceinline__ float4 f4_fma(float4 a, float4 b, float4 c) {
    return make_float4(fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y), fmaf(a.z, b.z, c.z), fmaf(a.w, b.w, c.w));
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}

// ---- statistics, stage 1: part[cta][0][c] = sum (x - K_c), part[cta][1][c] = sum (x - K_c)^2 over the CTA's rows;
// grid (row ranges, column chunks) ----
__global__ void __launch_bounds__(kLnThreads)
k_bn_stats(const float* __restrict__ X, int64_t ldx, double* __restrict__ part, int n, int d, int rows_per_cta) {
    __shared__ double s_col[kLnWarps][2][4 * kBnChunk];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c0 = blockIdx.y * kBnChunk, q = c0 + lane;
    pdl_wait();
    pdl_trigger();
    const int r0 = blockIdx.x * rows_per_cta, r1 = min(n, r0 + rows_per_cta);
    if (q < (d >> 2)) {
        double s1[4] = {0., 0., 0., 0.}, s2[4] = {0., 0., 0., 0.};
        const float4 k = ldg4(X + 4 * q);
        for (int row = r0 + warp; row < r1; row += kBnFold * kLnWarps) {
            float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
#pragma unroll
            for (int u = 0; u < kBnFold; u += 2 * kBnUnroll) {
                float4 x[2 * kBnUnroll];
#pragma unroll
                for (int j = 0; j < 2 * kBnUnroll; ++j) {
                    const int rr = row + (u + j) * kLnWarps;
                    x[j] = rr < r1 ? ldg4_stream(X + (size_t)rr * ldx + 4 * q) : k;
                }
#pragma unroll
                for (int j = 0; j < 2 * kBnUnroll; ++j) {
                    const float4 t = f4_sub(x[j], k);
                    a = f4_add(a, t);
                    b = f4_fma(t, t, b);
                }
            }
            s1[0] += a.x; s1[1] += a.y; s1[2] += a.z; s1[3] += a.w;
            s2[0] += b.x; s2[1] += b.y; s2[2] += b.z; s2[3] += b.w;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            s_col[warp][0][4 * lane + j] = s1[j];
            s_col[warp][1][4 * lane + j] = s2[j];
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * 4 * kBnChunk; i += kLnThreads) {
        const int which = i / (4 * kBnChunk), cc = i - which * 4 * kBnChunk, c = 4 * c0 + cc;
        if (c < d) {
            double t = 0.;
#pragma unroll
            for (int w = 0; w < kLnWarps; ++w) t += s_col[w][which][cc];
            part[((size_t)blockIdx.x * 2 + which) * d + c] = t;
        }
    }
}

// ---- statistics, stage 2: one warp per column.  training: the CTAs' sums in a fixed order -> mean, rstd, running
// buffers (when given); eval: mean, rstd of the running buffers ----
__global__ void __launch_bounds__(kLnThreads)
k_bn_stats_finalize(const double* __restrict__ part, int nparts, const float* __restrict__ X, int training, float momentum,
                    float eps, float* running_mean, float* running_var, float* __restrict__ mean, float* __restrict__ rstd,
                    int n, int d) {
    pdl_wait();
    pdl_trigger();
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * kLnWarps + (threadIdx.x >> 5);
    if (c >= d) return;
    if (!training) {
        if (lane == 0) {
            mean[c] = running_mean[c];
            rstd[c] = (float)(1.0 / sqrt((double)running_var[c] + (double)eps));
        }
        return;
    }
    double s1 = 0., s2 = 0.;
    for (int p = lane; p < nparts; p += 32) {
        s1 += part[((size_t)p * 2 + 0) * d + c];
        s2 += part[((size_t)p * 2 + 1) * d + c];
    }
    s1 = warp_sum_d(s1);
    s2 = warp_sum_d(s2);
    if (lane == 0) {
        const double m = s1 / n;                              // mean - K_c
        const double var = fmax(s2 / n - m * m, 0.);          // biased
        const double mu = (double)__ldg(X + c) + m;
        mean[c] = (float)mu;
        rstd[c] = (float)(1.0 / sqrt(var + (double)eps));
        if (running_mean && running_var) {
            const double f = momentum;
            running_mean[c] = (float)((1. - f) * (double)running_mean[c] + f * mu);
            running_var[c] = (float)((1. - f) * (double)running_var[c] + f * var * ((double)n / (double)(n - 1)));
        }
    }
}

// ---- forward: Y = s * (gamma * (x - mean) * rstd + beta); grid (row ranges, column chunks) ----
__global__ void __launch_bounds__(kLnThreads)
k_bn_fwd(const float* __restrict__ X, int64_t ldx, const float* __restrict__ gamma, const float* __restrict__ beta,
         const float* __restrict__ scalar, const float* __restrict__ mean, const float* __restrict__ rstd,
         float* __restrict__ Y, int64_t ldy, int n, int d, int rows_per_cta) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int q = blockIdx.y * kBnChunk + lane;
    pdl_wait();
    pdl_trigger();
    if (q >= (d >> 2)) return;
    const float s = scalar ? __ldg(scalar) : 1.f;
    const float4 gm = f4_ld_or(gamma ? gamma + 4 * q : nullptr, 1.f), bt = f4_ld_or(beta ? beta + 4 * q : nullptr, 0.f);
    const float4 mu = f4_ld(mean + 4 * q), rs = f4_ld(rstd + 4 * q);
    const int r0 = blockIdx.x * rows_per_cta, r1 = min(n, r0 + rows_per_cta);
    for (int row = r0 + warp; row < r1; row += kBnUnroll * kLnWarps) {
        float4 x[kBnUnroll];
#pragma unroll
        for (int j = 0; j < kBnUnroll; ++j) {
            const int rr = row + j * kLnWarps;
            x[j] = rr < r1 ? ldg4_stream(X + (size_t)rr * ldx + 4 * q) : mu;
        }
#pragma unroll
        for (int j = 0; j < kBnUnroll; ++j) {
            const int rr = row + j * kLnWarps;
            if (rr < r1) {
                float4 y;
                y.x = s * fmaf((x[j].x - mu.x) * rs.x, gm.x, bt.x);
                y.y = s * fmaf((x[j].y - mu.y) * rs.y, gm.y, bt.y);
                y.z = s * fmaf((x[j].z - mu.z) * rs.z, gm.z, bt.z);
                y.w = s * fmaf((x[j].w - mu.w) * rs.w, gm.w, bt.w);
                stg4_stream(Y + (size_t)rr * ldy + 4 * q, y);
            }
        }
    }
}

// ---- backward reduce pass: partG[cta][0][c] = sum s * gY * xh, partG[cta][1][c] = sum s * gY, partS[cta] =
// sum gY * (gamma * xh + beta) over the CTA's rows (k_ln_bwd's layout, for k_ln_bwd_finalize).  EVAL: also
// gX = s * gamma * rstd * gY (gX may be NULL) ----
template <bool EVAL>
__global__ void __launch_bounds__(kLnThreads)
k_bn_bwd(const float* __restrict__ gY, int64_t ldg, const float* __restrict__ X, int64_t ldx, const float* __restrict__ gamma,
         const float* __restrict__ beta, const float* __restrict__ scalar, const float* __restrict__ mean,
         const float* __restrict__ rstd, float* __restrict__ gX, int64_t ldgx, float* __restrict__ partG,
         float* __restrict__ partS, int n, int d, int rows_per_cta) {
    __shared__ __align__(16) float s_col[kLnWarps][2][4 * kBnChunk];
    __shared__ float s_gs[kLnWarps];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nq = d >> 2;
    pdl_wait();
    pdl_trigger();
    const float s = scalar ? __ldg(scalar) : 1.f;
    const int r0 = blockIdx.x * rows_per_cta, r1 = min(n, r0 + rows_per_cta);
    float gs = 0.f;
    for (int c0 = 0; c0 < nq; c0 += kBnChunk) {
        const int q = c0 + lane;
        if (q < nq) {
            const float4 gm = f4_ld_or(gamma ? gamma + 4 * q : nullptr, 1.f), bt = f4_ld_or(beta ? beta + 4 * q : nullptr, 0.f);
            const float4 mu = f4_ld(mean + 4 * q), rs = f4_ld(rstd + 4 * q);
            const float4 k = f4_scale(f4_mul(gm, rs), s);          // eval: gX = k * gY
            float4 agm = make_float4(0.f, 0.f, 0.f, 0.f), abt = agm;
            for (int row = r0 + warp; row < r1; row += kBnFold * kLnWarps) {
                float4 ia = make_float4(0.f, 0.f, 0.f, 0.f), ib = ia;
                float igs = 0.f;
#pragma unroll 1
                for (int u = 0; u < kBnFold; u += kBnUnroll) {
                    float4 x[kBnUnroll], g[kBnUnroll];
#pragma unroll
                    for (int j = 0; j < kBnUnroll; ++j) {      // rows past the range read as gY = 0: they add nothing
                        const int rr = row + (u + j) * kLnWarps;
                        x[j] = rr < r1 ? ldg4_stream(X + (size_t)rr * ldx + 4 * q) : mu;
                        g[j] = rr < r1 ? ldg4_stream(gY + (size_t)rr * ldg + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
                    }
#pragma unroll
                    for (int j = 0; j < kBnUnroll; ++j) {
                        const float4 xh = f4_mul(f4_sub(x[j], mu), rs);
                        const float4 yb = f4_fma(gm, xh, bt);
                        igs = fmaf(g[j].x, yb.x, igs); igs = fmaf(g[j].y, yb.y, igs);
                        igs = fmaf(g[j].z, yb.z, igs); igs = fmaf(g[j].w, yb.w, igs);
                        const float4 gl = f4_scale(g[j], s);        // gradient w.r.t. the BatchNorm output
                        ia = f4_fma(gl, xh, ia);
                        ib = f4_add(ib, gl);
                        if constexpr (EVAL) {
                            const int rr = row + (u + j) * kLnWarps;
                            if (gX && rr < r1) stg4_stream(gX + (size_t)rr * ldgx + 4 * q, f4_mul(k, g[j]));
                        }
                    }
                }
                agm = f4_add(agm, ia);
                abt = f4_add(abt, ib);
                gs += igs;
            }
            *reinterpret_cast<float4*>(&s_col[warp][0][4 * lane]) = agm;
            *reinterpret_cast<float4*>(&s_col[warp][1][4 * lane]) = abt;
        }
        __syncthreads();
        for (int i = threadIdx.x; i < 2 * 4 * kBnChunk; i += kLnThreads) {
            const int which = i / (4 * kBnChunk), cc = i - which * 4 * kBnChunk, c = 4 * c0 + cc;
            if (c < d) {
                float t = 0.f;
#pragma unroll
                for (int w = 0; w < kLnWarps; ++w) t += s_col[w][which][cc];
                partG[((size_t)blockIdx.x * 2 + which) * d + c] = t;
            }
        }
        __syncthreads();
    }
    gs = warp_sum(gs);
    if (lane == 0) s_gs[warp] = gs;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < kLnWarps; ++w) t += s_gs[w];
        partS[blockIdx.x] = t;
    }
}

// ---- backward, training: gX = rstd * (a - gamma * gbeta / n - xh * gamma * ggamma / n), a = s * gamma * gY ----
__global__ void __launch_bounds__(kLnThreads)
k_bn_bwd_dx(const float* __restrict__ gY, int64_t ldg, const float* __restrict__ X, int64_t ldx, const float* __restrict__ gamma,
            const float* __restrict__ scalar, const float* __restrict__ mean, const float* __restrict__ rstd,
            const float* __restrict__ ggamma, const float* __restrict__ gbeta, float* __restrict__ gX, int64_t ldgx, int n, int d,
            int rows_per_cta) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int q = blockIdx.y * kBnChunk + lane;
    pdl_wait();
    pdl_trigger();
    if (q >= (d >> 2)) return;
    const float s = scalar ? __ldg(scalar) : 1.f;
    const float inv_n = 1.f / (float)n;
    const float4 gm = f4_ld_or(gamma ? gamma + 4 * q : nullptr, 1.f);
    const float4 mu = f4_ld(mean + 4 * q), rs = f4_ld(rstd + 4 * q);
    const float4 cs = f4_scale(gm, s);
    const float4 m1 = f4_scale(f4_mul(gm, f4_ld(gbeta + 4 * q)), inv_n);    // mean_rows(a)
    const float4 m2 = f4_scale(f4_mul(gm, f4_ld(ggamma + 4 * q)), inv_n);   // mean_rows(a * xh)
    const int r0 = blockIdx.x * rows_per_cta, r1 = min(n, r0 + rows_per_cta);
    for (int row = r0 + warp; row < r1; row += kBnUnroll * kLnWarps) {
        float4 x[kBnUnroll], g[kBnUnroll];
#pragma unroll
        for (int j = 0; j < kBnUnroll; ++j) {
            const int rr = row + j * kLnWarps;
            x[j] = rr < r1 ? ldg4_stream(X + (size_t)rr * ldx + 4 * q) : mu;
            g[j] = rr < r1 ? ldg4_stream(gY + (size_t)rr * ldg + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int j = 0; j < kBnUnroll; ++j) {
            const int rr = row + j * kLnWarps;
            if (rr < r1) {
                const float4 xh = f4_mul(f4_sub(x[j], mu), rs);
                const float4 a = f4_mul(cs, g[j]);
                float4 o;
                o.x = rs.x * (a.x - m1.x - xh.x * m2.x);
                o.y = rs.y * (a.y - m1.y - xh.y * m2.y);
                o.z = rs.z * (a.z - m1.z - xh.z * m2.z);
                o.w = rs.w * (a.w - m1.w - xh.w * m2.w);
                stg4_stream(gX + (size_t)rr * ldgx + 4 * q, o);
            }
        }
    }
}

// CTAs of the passes that write per-CTA partials: contiguous row ranges, at most 2 per SM (and kLnMaxParts)
inline int bn_parts(int n) {
    int grid = (n + kLnWarps - 1) / kLnWarps;
    const int cap = 2 * num_sms() < kLnMaxParts ? 2 * num_sms() : kLnMaxParts;
    return grid < cap ? (grid > 0 ? grid : 1) : cap;
}
// row ranges of the elementwise passes (grid.y = column chunks): about 8 CTAs per SM in all
inline int bn_rows_grid(int n, int nchunks) {
    const int cap = 8 * num_sms() / nchunks > 0 ? 8 * num_sms() / nchunks : 1;
    const int want = (n + kLnWarps * kBnUnroll - 1) / (kLnWarps * kBnUnroll);
    return want < cap ? want : cap;
}

// scratch: the statistics' fp64 partials, or the backward's fp32 partials + [2][d] for ggamma / gbeta the caller did not ask for
inline size_t bn_stats_bytes(int d) { return align_up(sizeof(double) * (size_t)kLnMaxParts * 2 * d); }
inline size_t bn_bwd_part_bytes(int d) { return align_up(sizeof(float) * ((size_t)kLnMaxParts * 2 * d + kLnMaxParts)); }
inline size_t bn_scratch_bytes(int d) {
    const size_t bwd = bn_bwd_part_bytes(d) + align_up(sizeof(float) * 2 * (size_t)d);
    return bn_stats_bytes(d) > bwd ? bn_stats_bytes(d) : bwd;
}

inline bool bn_pitch_ok(const void* p, int64_t ld, int d) {
    return ld >= d && (ld % 4) == 0 && (reinterpret_cast<uintptr_t>(p) % 16) == 0;
}

}  // namespace
}  // namespace gca

using namespace gca;

extern "C" size_t gca_batchnorm_scratch_bytes(int32_t d) { return d > 0 ? bn_scratch_bytes(d) : 0; }

extern "C" int gca_batchnorm_scale_fwd(const float* X, int64_t ldx, const float* gamma, const float* beta, const float* scalar,
                                       float eps, int training, float momentum, float* running_mean, float* running_var,
                                       float* Y, int64_t ldy, float* mean, float* rstd, void* scratch, int32_t n, int32_t d,
                                       gca_stream_t stream) {
    if (!X || !Y || !mean || !rstd || !scratch || n < 0 || d <= 0 || !(eps >= 0.f)) return GCA_ERR_INVALID_ARG;
    if (training ? n < 2 : (!running_mean || !running_var)) return GCA_ERR_INVALID_ARG;
    if ((reinterpret_cast<uintptr_t>(scratch) % kAlign) != 0) return GCA_ERR_WORKSPACE;
    if ((d % 4) != 0 || !bn_pitch_ok(X, ldx, d) || !bn_pitch_ok(Y, ldy, d)) return GCA_ERR_UNSUPPORTED;
    if (n == 0) return GCA_OK;
    const PdlHint pdl_hint(n);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int parts = 0;
    double* part = static_cast<double*>(scratch);
    if (training) {
        parts = bn_parts(n);
        const int rows_per_cta = (n + parts - 1) / parts;
        {
            ProfScope ps("batchnorm_stats", st);
            GCA_CUDA(launch_pdl(k_bn_stats, dim3(parts, (d / 4 + kBnChunk - 1) / kBnChunk), dim3(kLnThreads), 0, st, X, ldx, part,
                                n, d, rows_per_cta));
        }
        GCA_LAUNCH_OK();
    }
    {
        ProfScope ps("batchnorm_stats", st);
        GCA_CUDA(launch_pdl(k_bn_stats_finalize, dim3((d + kLnWarps - 1) / kLnWarps), dim3(kLnThreads), 0, st, (const double*)part,
                            parts, X, training, momentum, eps, running_mean, running_var, mean, rstd, n, d));
    }
    GCA_LAUNCH_OK();
    const int nchunks = (d / 4 + kBnChunk - 1) / kBnChunk;
    const int gx = bn_rows_grid(n, nchunks);
    {
        ProfScope ps("batchnorm_fwd", st);
        GCA_CUDA(launch_pdl(k_bn_fwd, dim3(gx, nchunks), dim3(kLnThreads), 0, st, X, ldx, gamma, beta, scalar, (const float*)mean,
                            (const float*)rstd, Y, ldy, n, d, (n + gx - 1) / gx));
    }
    GCA_LAUNCH_OK();
    return GCA_OK;
}

extern "C" int gca_batchnorm_scale_bwd(const float* gY, int64_t ldg, const float* X, int64_t ldx, const float* gamma,
                                       const float* beta, const float* scalar, const float* mean, const float* rstd, int training,
                                       float* gX, int64_t ldgx, float* ggamma, float* gbeta, float* gscalar, void* scratch,
                                       int32_t n, int32_t d, gca_stream_t stream) {
    if (!gY || !X || !mean || !rstd || !scratch || n < 0 || d <= 0 || (training && n == 1)) return GCA_ERR_INVALID_ARG;
    if ((reinterpret_cast<uintptr_t>(scratch) % kAlign) != 0) return GCA_ERR_WORKSPACE;
    if ((d % 4) != 0 || !bn_pitch_ok(gY, ldg, d) || !bn_pitch_ok(X, ldx, d) || (gX && !bn_pitch_ok(gX, ldgx, d)))
        return GCA_ERR_UNSUPPORTED;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (n == 0) {       // empty input: the parameter gradients are zero
        if (ggamma) GCA_CUDA(cudaMemsetAsync(ggamma, 0, sizeof(float) * d, st));
        if (gbeta) GCA_CUDA(cudaMemsetAsync(gbeta, 0, sizeof(float) * d, st));
        if (gscalar) GCA_CUDA(cudaMemsetAsync(gscalar, 0, sizeof(float), st));
        return GCA_OK;
    }
    const PdlHint pdl_hint(n);
    const int parts = bn_parts(n);
    const int rows_per_cta = (n + parts - 1) / parts;
    float* partG = static_cast<float*>(scratch);
    float* partS = partG + (size_t)kLnMaxParts * 2 * d;
    // the gX pass needs both column sums: they go to scratch when the caller does not want them
    float* sums = reinterpret_cast<float*>(static_cast<char*>(scratch) + bn_bwd_part_bytes(d));
    const bool dx_pass = training && gX;
    float* gg = ggamma ? ggamma : (dx_pass ? sums : nullptr);
    float* gb = gbeta ? gbeta : (dx_pass ? sums + d : nullptr);
    {
        ProfScope ps("batchnorm_bwd", st, training ? "train" : "eval");
        if (training)
            GCA_CUDA(launch_pdl(k_bn_bwd<false>, dim3(parts), dim3(kLnThreads), 0, st, gY, ldg, X, ldx, gamma, beta, scalar, mean, rstd,
                                (float*)nullptr, ldgx, partG, partS, n, d, rows_per_cta));
        else
            GCA_CUDA(launch_pdl(k_bn_bwd<true>, dim3(parts), dim3(kLnThreads), 0, st, gY, ldg, X, ldx, gamma, beta, scalar, mean, rstd,
                                gX, ldgx, partG, partS, n, d, rows_per_cta));
    }
    GCA_LAUNCH_OK();
    const int fgrid = (2 * d + 1 + kLnWarps - 1) / kLnWarps;
    {
        ProfScope ps("batchnorm_bwd_finalize", st);
        GCA_CUDA(launch_pdl(k_ln_bwd_finalize, dim3(fgrid), dim3(kLnThreads), 0, st, (const float*)partG, (const float*)partS, parts, d,
                            gg, gb, gscalar));
    }
    GCA_LAUNCH_OK();
    if (dx_pass) {
        const int nchunks = (d / 4 + kBnChunk - 1) / kBnChunk;
        const int gx = bn_rows_grid(n, nchunks);
        {
            ProfScope ps("batchnorm_bwd_dx", st);
            GCA_CUDA(launch_pdl(k_bn_bwd_dx, dim3(gx, nchunks), dim3(kLnThreads), 0, st, gY, ldg, X, ldx, gamma, scalar, mean, rstd,
                                (const float*)gg, (const float*)gb, gX, ldgx, n, d, (n + gx - 1) / gx));
        }
        GCA_LAUNCH_OK();
    }
    return GCA_OK;
}
