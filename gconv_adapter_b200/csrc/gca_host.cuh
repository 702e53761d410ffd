// Host-side pieces shared by the translation units of libgca: scratch layouts, the CSR view handed to the
// launchers, shared-memory opt-in, the tensor-map cache, and the launcher entry points each kernel family exports.
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "gca_common.cuh"

namespace gca {

constexpr int kMaxParts = 320;    // per-CTA weight-gradient partials (>= 2 * 148)
constexpr int kMaxPartsBd = 1280; // per-CTA bias-gradient partials of the transpose hop
constexpr int kMaxFin = 256;      // CTAs of the finalize kernel

// Backward scratch (caller-owned): header ints + per-CTA partial sums, reduced by k_finalize in a fixed order.
// header ints: [0] #partials gu/col, [1] #partials gd/dot, [2] #partials bd, [3] finalize ticket
struct ScratchLayout {
    size_t header, gu, col, gd, dot, bd, gsp, total;   // byte offsets
};
__host__ __device__ inline ScratchLayout scratch_layout(int d, int r) {
    ScratchLayout L;
    size_t off = 0;
    auto up = [](size_t x) { return (x + 255) / 256 * 256; };
    L.header = off; off += 256;
    // blocks whose offsets depend on r only come first (gca_bwd_hop2 does not know d)
    L.bd = off;  off += up(sizeof(float) * (size_t)kMaxPartsBd * r);
    L.gsp = off; off += up(sizeof(float) * (size_t)kMaxFin);
    L.dot = off; off += up(sizeof(float) * (size_t)kMaxParts);
    L.gu = off;  off += up(sizeof(float) * (size_t)kMaxParts * r * d);
    L.col = off; off += up(sizeof(float) * (size_t)kMaxParts * d);
    L.gd = off;  off += up(sizeof(float) * (size_t)kMaxParts * r * d);
    L.total = off;
    return L;
}
struct Scratch {
    int* header;
    float *gu, *col, *gd, *dot, *bd, *gsp;
};
inline Scratch scratch_ptrs(void* scratch, int d, int r) {
    const ScratchLayout L = scratch_layout(d, r);
    char* b = static_cast<char*>(scratch);
    return Scratch{reinterpret_cast<int*>(b + L.header), reinterpret_cast<float*>(b + L.gu),
                   reinterpret_cast<float*>(b + L.col), reinterpret_cast<float*>(b + L.gd),
                   reinterpret_cast<float*>(b + L.dot), reinterpret_cast<float*>(b + L.bd),
                   reinterpret_cast<float*>(b + L.gsp)};
}

// CSR view of one direction of a graph handle (+ its hub work items).  hub_part is per-CALL scratch supplied by the
// caller (gca_hub_scratch_bytes), never state of the handle: a handle can be used from several streams at once.
struct Csr {
    const int* rowptr; const int* colidx; const float* dis;
    const int* hubitem; const int* item_row; const int* nitems_ptr; float* hub_part; int nitems_host;
    int n_full;   // rows of the gathered operand (all N nodes)
};
inline Csr csr_of(const gca_graph* g, bool transpose, void* hub_scratch) {
    float* hp = static_cast<float*>(hub_scratch);
    return transpose ? Csr{g->rowptr_t, g->colidx_t, g->dis, g->hubitem_t, g->item_row_t, g->flags + 4, hp, g->nitems_t, g->N}
                     : Csr{g->rowptr, g->colidx, g->dis, g->hubitem, g->item_row, g->flags + 3, hp, g->nitems, g->N};
}
// Bytes of hub scratch one call on this handle needs (0 when the validated build found no hub row).
inline size_t hub_scratch_bytes(const gca_graph* g) {
    if (g->nitems == 0 && g->nitems_t == 0) return 0;
    return align_up(sizeof(float) * (size_t)g->hub_cap * 64);
}

inline bool shape_ok(int d, int r) { return d > 0 && (d % 4) == 0 && (r == 8 || r == 16 || r == 32 || r == 64); }

bool tc_enabled();        // GCA_DISABLE_TC=1 -> CUDA-core (FFMA) kernels everywhere
bool stream_enabled();    // GCA_DISABLE_STREAM=1 -> register-fed mma.sync kernels instead of the TMA-fed family
long long split_bytes();  // GCA_SPLIT_MB (default 160): gathered operand above this -> K3 runs as plain hop + expand-only

// Opt in to > 48 KB of dynamic shared memory, remembered per (device, kernel): cudaFuncSetAttribute applies to the
// current device only.
int set_smem_impl(const void* kernel, size_t bytes, bool has_static_smem);
template <typename K>
int set_smem(K kernel, size_t bytes, bool has_static_smem = false) {
    return set_smem_impl(reinterpret_cast<const void*>(kernel), bytes, has_static_smem);
}

// Tensor map of a row-major fp32 [rows, cols] matrix (leading dimension ld), box = box_cols x box_rows, 128-byte swizzle
// (swizzle = true; box_cols must then be 32) or none.  Encoded maps are cached (LRU) per (base, rows, cols, ld, box).
// Returns false when the driver entry point is missing or the encode is refused (callers fall back to kernels
// that do not need tensor maps).
bool get_box_map(CUtensorMap* tm, const float* base, int rows, int cols, int64_t ld, int box_cols, int box_rows, bool swizzle);

// ---- launchers (one per kernel family; each dispatches on r and picks the variant) ----
// K1: out[i, 0:r] = rowscale[i] * s * sum_k A[i,k] W[k, 0:r]    (w_is_rd: W stored [r, d], else [d, r])
int launch_project(int r, bool w_is_rd, const float* A, int64_t lda, const float* W, const float* rowscale, const float* scalar,
                   float* out, int n, int d, cudaStream_t st);
// K1 on tcgen05 / TMEM (gca_tc_project.cu): r = 32 only, GCA_ERR_UNSUPPORTED otherwise
int launch_project_tc(int r, bool w_is_rd, const float* A, int64_t lda, const float* W, const float* rowscale,
                      const float* scalar, float* out, int n, int d, cudaStream_t st);
// K2: r-wide hop (forward: bias + act ; backward: act' + bias-gradient partials ; plain: just the hop)
int launch_hop(int r, bool bwd, const Csr& c, const float* F, const float* bias, int act, const float* Zp, const float* H1s,
               float* out, float* H1o, float* part_bd, int* header, int n, cudaStream_t st, int plain, const char* prof_name,
               const gca_push* push = nullptr);
// copy a finished local shard to the peers (producers without a fused push)
int launch_push_rows(const float* src, size_t nfloats, const gca_push* push, cudaStream_t st);
// K3: hop + expansion  Out = alpha (H W + bias) + beta Resid   (w_is_dr: W stored [d, r], else [r, d])
int launch_hop_expand(int r, bool w_is_dr, const Csr& c, const float* F, const float* W, const float* bias, const float* resid,
                      int64_t ldr, const float* scalar, int alpha_is_scalar, int use_resid, float* Hout, float* Out, int64_t ldo,
                      int n, int d, cudaStream_t st);
// K4: per-CTA partials of G[r, d] = H^T A (+ column sums of A, <A, B>)
int launch_wgrad(int r, const float* A, int64_t lda, const float* H, const float* B, int64_t ldb, float* partG, float* partCol,
                 float* partDot, int* header, int slot, int n, int d, cudaStream_t st);
// TMA-fed dense streaming family (gca_stream.cu): any combination of the projection of A and the weight gradient
// over A in ONE pass over A.  Returns GCA_ERR_UNSUPPORTED for shapes it does not cover (callers fall back).
struct DenseStreamArgs {
    const float* A; int64_t lda;                 // streamed [n, d]
    const float* B; int64_t ldb;                 // second stream for <A, B> (wgrad only), or null
    // projection (null W = no projection)
    const float* W; bool w_is_rd; const float* rowscale; const float* scalar; float* out;
    const gca_push* push;                        // peers that receive every output row as well (or null)
    // weight gradient (null H = none)
    const float* H; float* partG; float* partCol; float* partDot; int* header; int slot;
    int n, d;
    const char* prof_name;
};
int launch_dense_stream(int r, const DenseStreamArgs& a, cudaStream_t st);
// Fused small-graph path (gca_small.cu): the whole forward / backward of a full-graph handle as ONE cooperative kernel
// each, for n <= 4096, n d <= 2^19, r d <= 8192, on a stream that is not being captured (GCA_DISABLE_SMALL=1 switches it off).
bool small_path_ok(const gca_graph* g, int d, int r, cudaStream_t st);
int small_forward(const gca_graph* g, const float* X, int64_t ldx, const float* Wd, const float* bd, const float* Wu,
                  const float* bu, const float* scalar, int act, int skip, float* P, float* Zp, float* H1, float* H2, float* Y,
                  int64_t ldy, int d, int r, cudaStream_t st);
int small_backward(const gca_graph* g, const float* gY, int64_t ldg, const float* X, int64_t ldx, const float* Zp,
                   const float* H1, const float* H2, const float* Wd, const float* Wu, const float* bu, const float* scalar,
                   int act, int skip, float* gH2, float* gH1, float* gP, float* gX, int64_t ldgx, const Scratch& S, float* gWd,
                   float* gbd, float* gWu, float* gbu, float* gscalar, int d, int r, cudaStream_t st);
// gX = gP Wd + s gY, gWd partials = gP^T X and <gY, X> in one pass over gY and X (gca_stream_bwd.cu; gP from a plain hop).
// Returns GCA_ERR_UNSUPPORTED for shapes it does not cover (callers fall back to K3 + K4).
int launch_expand_wgrad(int r, const float* X, int64_t ldx, const float* gY, int64_t ldg, const float* gP, const float* Wd,
                        const float* scalar, float* gX, int64_t ldgx, float* partG, float* partDot, int* header, int slot,
                        int n, int d, cudaStream_t st);
// K6
int launch_finalize(const Scratch& S, const float* Wu, const float* bu, const float* scalar, int skip, float* gWd, float* gbd,
                    float* gWu, float* gbu, float* gscalar, int d, int r, cudaStream_t st);

#define GCA_DISPATCH_R(r, CALL)                         \
    switch (r) {                                        \
        case 8:  { constexpr int R_ = 8;  return CALL; }  \
        case 16: { constexpr int R_ = 16; return CALL; }  \
        case 32: { constexpr int R_ = 32; return CALL; }  \
        case 64: { constexpr int R_ = 64; return CALL; }  \
        default: return GCA_ERR_UNSUPPORTED;            \
    }

}  // namespace gca
