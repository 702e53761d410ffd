// extern "C" entry points of include/gca.h for the forward / backward phases: argument checks, the choice between
// the TMA-fed streaming family (gca_stream.cu) and the register-fed kernels, and the single-GPU conveniences.
// Nothing here (or below) keeps per-launch state in the graph handle: every scratch byte comes from the caller.
#include "gca_common.cuh"
#include "gca_host.cuh"

using namespace gca;

extern "C" int gca_shape_is_fast(int32_t d, int32_t r) { return shape_ok(d, r) ? 1 : 0; }

extern "C" size_t gca_hub_scratch_bytes(const gca_graph* g) { return g ? hub_scratch_bytes(g) : 0; }

extern "C" size_t gca_hub_scratch_bytes_r(const gca_graph* g, int32_t r) {
    return g && r > 0 && r <= 128 ? hub_scratch_bytes(g, r) : 0;
}

namespace {
inline bool hub_scratch_ok(const gca_graph* g, const void* hub_scratch) {
    return hub_scratch_bytes(g) == 0 || (hub_scratch && (reinterpret_cast<uintptr_t>(hub_scratch) % kAlign) == 0);
}

// K1 through the streaming family when the shape allows, else the register-fed kernels.
int project_any(int r, bool w_is_rd, const float* A, int64_t lda, const float* W, const float* rowscale, const float* scalar,
                float* out, int n, int d, const gca_push* push, cudaStream_t st) {
    DenseStreamArgs a{};
    a.A = A; a.lda = lda; a.W = W; a.w_is_rd = w_is_rd; a.rowscale = rowscale; a.scalar = scalar; a.out = out; a.push = push;
    a.n = n; a.d = d; a.prof_name = w_is_rd ? "project_fwd" : "project_bwd";
    const int s = launch_dense_stream(r, a, st);
    if (s != GCA_ERR_UNSUPPORTED) return s;
    // register-fed kernels have no fused push: copy the finished shard to the peers
    GCA_TRY(launch_project(r, w_is_rd, A, lda, W, rowscale, scalar, out, n, d, st));
    return launch_push_rows(out, (size_t)n * r, push, st);
}

// K4 through the streaming family when the shape allows, else the register-fed kernels.
int wgrad_any(int r, const float* A, int64_t lda, const float* H, const float* B, int64_t ldb, float* partG, float* partCol,
              float* partDot, int* header, int slot, int n, int d, cudaStream_t st) {
    DenseStreamArgs a{};
    a.A = A; a.lda = lda; a.B = B; a.ldb = ldb; a.H = H; a.partG = partG; a.partCol = partCol; a.partDot = partDot;
    a.header = header; a.slot = slot; a.n = n; a.d = d; a.prof_name = slot == 0 ? "wgrad_up" : "wgrad_down";
    const int s = launch_dense_stream(r, a, st);
    if (s != GCA_ERR_UNSUPPORTED) return s;
    return launch_wgrad(r, A, lda, H, B, ldb, partG, partCol, partDot, header, slot, n, d, st);
}
}  // namespace

extern "C" int gca_fwd_project(const gca_graph* g, const float* X, int64_t ldx, const float* Wd, float* Pp_local,
                               const gca_push* push, int32_t d, int32_t r, gca_stream_t stream) {
    if (!g || !X || !Wd || !Pp_local || ldx < d) return GCA_ERR_INVALID_ARG;
    if (!shape_ok(d, r) || (ldx % 4) != 0) return GCA_ERR_UNSUPPORTED;
    const int n = g->row_end - g->row_begin;
    const PdlHint pdl_hint(n);
    if (n == 0) return GCA_OK;
    return project_any(r, true, X, ldx, Wd, g->dis, nullptr, Pp_local, n, d, push, static_cast<cudaStream_t>(stream));
}

extern "C" int gca_fwd_hop1(const gca_graph* g, const float* Pp_full, const float* bd, int act, float* Zp_local,
                            float* H1_local, void* hub_scratch, const gca_push* push, int32_t r, gca_stream_t stream) {
    if (!g || !Pp_full || !bd || !Zp_local) return GCA_ERR_INVALID_ARG;
    if (act < GCA_ACT_NONE || act > GCA_ACT_SILU) return GCA_ERR_INVALID_ARG;
    if (act == GCA_ACT_SILU && !H1_local) return GCA_ERR_INVALID_ARG;
    if (!hub_scratch_ok(g, hub_scratch)) return GCA_ERR_WORKSPACE;
    const int n = g->row_end - g->row_begin;
    const PdlHint pdl_hint(n);
    return launch_hop(r, false, csr_of(g, false, hub_scratch), Pp_full, bd, act, nullptr, nullptr, Zp_local, H1_local, nullptr,
                      nullptr, n, static_cast<cudaStream_t>(stream), 0, nullptr, push);
}

namespace {
// gca_fwd_hop2_up (A = NULL) and gca_fwd_hop2_up_add (A = the addend, checked by the caller)
int fwd_hop2_up(const gca_graph* g, const float* Zp_full, const float* X, int64_t ldx, const float* Wu, const float* bu,
                const float* scalar, int skip, float* H2_local, const float* A, int64_t lda, float* Y, int64_t ldy,
                void* hub_scratch, int32_t d, int32_t r, gca_stream_t stream) {
    if (!g || !Zp_full || !Wu || !bu || !H2_local || !Y || ldy < d) return GCA_ERR_INVALID_ARG;
    if (skip && (!X || ldx < d)) return GCA_ERR_INVALID_ARG;
    if (!shape_ok(d, r) || (ldy % 4) != 0 || (skip && (ldx % 4) != 0)) return GCA_ERR_UNSUPPORTED;
    if (!hub_scratch_ok(g, hub_scratch)) return GCA_ERR_WORKSPACE;
    const int n = g->row_end - g->row_begin;
    const PdlHint pdl_hint(n);
    return launch_hop_expand(r, true, csr_of(g, false, hub_scratch), Zp_full, Wu, bu, X, ldx, scalar, 1, skip ? 1 : 0, H2_local,
                             Y, ldy, n, d, static_cast<cudaStream_t>(stream), A, lda);
}
inline bool addend_ok(const float* A, int64_t lda, int32_t d) { return A && lda >= d; }
}  // namespace

extern "C" int gca_fwd_hop2_up(const gca_graph* g, const float* Zp_full, const float* X, int64_t ldx, const float* Wu,
                               const float* bu, const float* scalar, int skip, float* H2_local, float* Y, int64_t ldy,
                               void* hub_scratch, int32_t d, int32_t r, gca_stream_t stream) {
    return fwd_hop2_up(g, Zp_full, X, ldx, Wu, bu, scalar, skip, H2_local, nullptr, 0, Y, ldy, hub_scratch, d, r, stream);
}

extern "C" int gca_fwd_hop2_up_add(const gca_graph* g, const float* Zp_full, const float* X, int64_t ldx, const float* Wu,
                                   const float* bu, const float* scalar, int skip, float* H2_local, const float* A, int64_t lda,
                                   float* Y, int64_t ldy, void* hub_scratch, int32_t d, int32_t r, gca_stream_t stream) {
    if (!addend_ok(A, lda, d)) return GCA_ERR_INVALID_ARG;
    if ((lda % 4) != 0) return GCA_ERR_UNSUPPORTED;
    return fwd_hop2_up(g, Zp_full, X, ldx, Wu, bu, scalar, skip, H2_local, A, lda, Y, ldy, hub_scratch, d, r, stream);
}

extern "C" size_t gca_bwd_scratch_bytes(int32_t d, int32_t r) {
    if (d <= 0 || r <= 0) return 0;
    return scratch_layout(d, r).total;
}

extern "C" int gca_bwd_up(const gca_graph* g, const float* gY, int64_t ldg, const float* H2_local, const float* Wu,
                          const float* scalar, float* gH2p_local, void* scratch, const gca_push* push, int32_t d, int32_t r,
                          gca_stream_t stream) {
    if (!g || !gY || !H2_local || !Wu || !gH2p_local || !scratch || ldg < d) return GCA_ERR_INVALID_ARG;
    if (!shape_ok(d, r) || (ldg % 4) != 0) return GCA_ERR_UNSUPPORTED;
    if ((reinterpret_cast<uintptr_t>(scratch) % kAlign) != 0) return GCA_ERR_WORKSPACE;
    const int n = g->row_end - g->row_begin;
    const PdlHint pdl_hint(n);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const Scratch S = scratch_ptrs(scratch, d, r);
    GCA_CUDA(cudaMemsetAsync(S.header, 0, 256, st));
    if (n == 0) return GCA_OK;
    // one pass over gY for both the projection and the weight gradient (r = 16) ...
    DenseStreamArgs a{};
    a.A = gY; a.lda = ldg; a.W = Wu; a.w_is_rd = false; a.rowscale = g->dis; a.scalar = scalar; a.out = gH2p_local; a.push = push;
    a.H = H2_local; a.partG = S.gu; a.partCol = S.col; a.header = S.header; a.slot = 0; a.n = n; a.d = d;
    a.prof_name = "bwd_up";
    const int s = launch_dense_stream(r, a, st);
    if (s != GCA_ERR_UNSUPPORTED) return s;
    // ... else two passes
    GCA_TRY(project_any(r, false, gY, ldg, Wu, g->dis, scalar, gH2p_local, n, d, push, st));
    return wgrad_any(r, gY, ldg, H2_local, nullptr, 0, S.gu, S.col, nullptr, S.header, 0, n, d, st);
}

extern "C" int gca_bwd_up_project(const gca_graph* g, const float* gY, int64_t ldg, const float* Wu, const float* scalar,
                                  float* gH2p_local, void* scratch, const gca_push* push, int32_t d, int32_t r, gca_stream_t stream) {
    if (!g || !gY || !Wu || !gH2p_local || !scratch || ldg < d) return GCA_ERR_INVALID_ARG;
    if (!shape_ok(d, r) || (ldg % 4) != 0) return GCA_ERR_UNSUPPORTED;
    if ((reinterpret_cast<uintptr_t>(scratch) % kAlign) != 0) return GCA_ERR_WORKSPACE;
    const int n = g->row_end - g->row_begin;
    const PdlHint pdl_hint(n);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const Scratch S = scratch_ptrs(scratch, d, r);
    GCA_CUDA(cudaMemsetAsync(S.header, 0, 256, st));
    if (n == 0) return GCA_OK;
    return project_any(r, false, gY, ldg, Wu, g->dis, scalar, gH2p_local, n, d, push, st);
}

extern "C" int gca_bwd_up_wgrad(const gca_graph* g, const float* gY, int64_t ldg, const float* H2_local, void* scratch,
                                int32_t d, int32_t r, gca_stream_t stream) {
    if (!g || !gY || !H2_local || !scratch || ldg < d) return GCA_ERR_INVALID_ARG;
    if (!shape_ok(d, r) || (ldg % 4) != 0) return GCA_ERR_UNSUPPORTED;
    const int n = g->row_end - g->row_begin;
    const PdlHint pdl_hint(n);
    if (n == 0) return GCA_OK;
    const Scratch S = scratch_ptrs(scratch, d, r);
    return wgrad_any(r, gY, ldg, H2_local, nullptr, 0, S.gu, S.col, nullptr, S.header, 0, n, d, static_cast<cudaStream_t>(stream));
}

extern "C" int gca_bwd_hop2(const gca_graph* g, const float* gH2p_full, const float* Zp_local, const float* H1_local,
                            int act, float* gH1p_local, void* scratch, void* hub_scratch, const gca_push* push, int32_t r,
                            gca_stream_t stream) {
    if (!g || !gH2p_full || !gH1p_local || !scratch) return GCA_ERR_INVALID_ARG;
    if (act < GCA_ACT_NONE || act > GCA_ACT_SILU) return GCA_ERR_INVALID_ARG;
    if ((act == GCA_ACT_RELU && !Zp_local) || (act == GCA_ACT_SILU && !H1_local)) return GCA_ERR_INVALID_ARG;
    if ((reinterpret_cast<uintptr_t>(scratch) % kAlign) != 0 || !hub_scratch_ok(g, hub_scratch)) return GCA_ERR_WORKSPACE;
    const int n = g->row_end - g->row_begin;
    const PdlHint pdl_hint(n);
    const Scratch S = scratch_ptrs(scratch, 4, r);      // header / bd offsets do not depend on d
    return launch_hop(r, true, csr_of(g, true, hub_scratch), gH2p_full, nullptr, act, Zp_local, H1_local, gH1p_local, nullptr,
                      S.bd, S.header, n, static_cast<cudaStream_t>(stream), 0, nullptr, push);
}

extern "C" int gca_bwd_hop1_down(const gca_graph* g, const float* gH1p_full, const float* X, int64_t ldx,
                                 const float* gY, int64_t ldg, const float* Wd, const float* scalar, int skip,
                                 float* gP_local, float* gX, int64_t ldgx, void* scratch, void* hub_scratch,
                                 int32_t d, int32_t r, gca_stream_t stream) {
    if (!g || !gH1p_full || !X || !Wd || !gP_local || !scratch || ldx < d) return GCA_ERR_INVALID_ARG;
    if (skip && (!gY || ldg < d)) return GCA_ERR_INVALID_ARG;
    if (gX && ldgx < d) return GCA_ERR_INVALID_ARG;
    if (!shape_ok(d, r) || (ldx % 4) != 0 || (skip && (ldg % 4) != 0) || (gX && (ldgx % 4) != 0)) return GCA_ERR_UNSUPPORTED;
    if ((reinterpret_cast<uintptr_t>(scratch) % kAlign) != 0 || !hub_scratch_ok(g, hub_scratch)) return GCA_ERR_WORKSPACE;
    const int n = g->row_end - g->row_begin;
    const PdlHint pdl_hint(n);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const Scratch S = scratch_ptrs(scratch, d, r);
    const bool want_dot = skip && scalar;
    if (n > 0 && skip && gX && r == 16 && d % 32 == 0 && d <= 256 && n >= 2048) {
        // One pass over gY and X: plain r-wide hop for gP, then gX = gP Wd + s gY, the gWd partials and <gY, X> together
        // (gY and X cross HBM once each instead of twice).  Falls through to K3 + K4 when the streaming kernel declines.
        const Csr c = csr_of(g, true, hub_scratch);
        GCA_TRY(launch_hop(r, false, c, gH1p_full, nullptr, GCA_ACT_NONE, nullptr, nullptr, gP_local, nullptr, nullptr, nullptr, n, st,
                           1, "hop_plain_bwd"));
        const int s2 = launch_expand_wgrad(r, X, ldx, gY, ldg, gP_local, Wd, scalar, gX, ldgx, S.gd, want_dot ? S.dot : nullptr,
                                           S.header, 1, n, d, st);
        if (s2 == GCA_OK) return GCA_OK;
        if (s2 != GCA_ERR_UNSUPPORTED) return s2;
        // (gP is already in place; the register-fed path below recomputes it inside K3 - correct, only slower)
    }
    GCA_TRY(launch_hop_expand(r, false, csr_of(g, true, hub_scratch), gH1p_full, Wd, nullptr, gY, ldg, scalar, 0, skip ? 1 : 0,
                              gP_local, gX, ldgx, n, d, st));
    if (n == 0) return GCA_OK;
    return wgrad_any(r, X, ldx, gP_local, want_dot ? gY : nullptr, ldg, S.gd, nullptr, want_dot ? S.dot : nullptr, S.header, 1,
                     n, d, st);
}

extern "C" int gca_bwd_finalize(const void* scratch, const float* Wu, const float* bu, const float* scalar, int skip,
                                float* gWd, float* gbd, float* gWu, float* gbu, float* gscalar, int32_t d, int32_t r,
                                gca_stream_t stream) {
    if (!scratch || !Wu || !bu || d <= 0 || r <= 0) return GCA_ERR_INVALID_ARG;
    const Scratch S = scratch_ptrs(const_cast<void*>(scratch), d, r);
    return launch_finalize(S, Wu, bu, scalar, skip, gWd, gbd, gWu, gbu, gscalar, d, r, static_cast<cudaStream_t>(stream));
}

// ---------------- single-GPU conveniences ----------------
// forward workspace: [P' scratch | hub scratch]; backward workspace: [gH2' | gH1' | gP | partial-sum scratch | hub scratch]
namespace {
inline size_t rw_bytes(int n, int r) { return align_up(sizeof(float) * (size_t)(n > 0 ? n + (n & 1) : 2) * r); }   // even row count
}

extern "C" size_t gca_forward_workspace_bytes(const gca_graph* g, int32_t d, int32_t r) {
    (void)d;
    if (!g || r <= 0) return 0;
    return rw_bytes(g->row_end - g->row_begin, r) + hub_scratch_bytes(g, r);
}

namespace {
// gca_forward (A = NULL) and gca_forward_add: the same kernels and the same choice between them, A only changes the store
int forward(const gca_graph* g, const float* X, int64_t ldx, const float* Wd, const float* bd, const float* Wu, const float* bu,
            const float* scalar, int act, int skip, void* workspace, float* Zp_save, float* H1_save, float* H2_save,
            const float* A, int64_t lda, float* Y, int64_t ldy, int32_t d, int32_t r, gca_stream_t stream) {
    if (!g || !workspace) return GCA_ERR_INVALID_ARG;
    if (g->row_begin != 0 || g->row_end != g->N) return GCA_ERR_INVALID_ARG;   // partitioned graphs use the phases
    if ((reinterpret_cast<uintptr_t>(workspace) % kAlign) != 0) return GCA_ERR_WORKSPACE;
    char* b = static_cast<char*>(workspace);
    float* Pp = reinterpret_cast<float*>(b);
    void* hub = hub_scratch_bytes(g, r) ? b + rw_bytes(g->N, r) : nullptr;
    // small graphs: one cooperative kernel for the whole forward (anything it cannot take goes through the phases,
    // which also report argument errors)
    if (X && Wd && bd && Wu && bu && Zp_save && H2_save && Y && ldx >= d && ldy >= d && act >= GCA_ACT_NONE &&
        act <= GCA_ACT_SILU && (act != GCA_ACT_SILU || H1_save) && small_path_ok(g, d, r, static_cast<cudaStream_t>(stream)))
        return small_forward(g, X, ldx, Wd, bd, Wu, bu, scalar, act, skip, Pp, Zp_save, H1_save, H2_save, Y, ldy, d, r,
                             static_cast<cudaStream_t>(stream), A, lda);
    GCA_TRY(gca_fwd_project(g, X, ldx, Wd, Pp, nullptr, d, r, stream));
    GCA_TRY(gca_fwd_hop1(g, Pp, bd, act, Zp_save, H1_save, hub, nullptr, r, stream));
    return fwd_hop2_up(g, Zp_save, X, ldx, Wu, bu, scalar, skip, H2_save, A, lda, Y, ldy, hub, d, r, stream);
}
}  // namespace

extern "C" int gca_forward(const gca_graph* g, const float* X, int64_t ldx, const float* Wd, const float* bd,
                           const float* Wu, const float* bu, const float* scalar, int act, int skip, void* workspace,
                           float* Zp_save, float* H1_save, float* H2_save, float* Y, int64_t ldy, int32_t d, int32_t r,
                           gca_stream_t stream) {
    return forward(g, X, ldx, Wd, bd, Wu, bu, scalar, act, skip, workspace, Zp_save, H1_save, H2_save, nullptr, 0, Y, ldy, d, r,
                   stream);
}

extern "C" int gca_forward_add(const gca_graph* g, const float* X, int64_t ldx, const float* Wd, const float* bd,
                               const float* Wu, const float* bu, const float* scalar, int act, int skip, void* workspace,
                               float* Zp_save, float* H1_save, float* H2_save, const float* A, int64_t lda, float* Y, int64_t ldy,
                               int32_t d, int32_t r, gca_stream_t stream) {
    if (!addend_ok(A, lda, d)) return GCA_ERR_INVALID_ARG;
    if ((lda % 4) != 0) return GCA_ERR_UNSUPPORTED;
    return forward(g, X, ldx, Wd, bd, Wu, bu, scalar, act, skip, workspace, Zp_save, H1_save, H2_save, A, lda, Y, ldy, d, r, stream);
}

extern "C" size_t gca_backward_workspace_bytes(const gca_graph* g, int32_t d, int32_t r) {
    if (!g || d <= 0 || r <= 0) return 0;
    return 3 * rw_bytes(g->row_end - g->row_begin, r) + gca_bwd_scratch_bytes(d, r) + hub_scratch_bytes(g, r);
}

extern "C" int gca_backward(const gca_graph* g, const float* gY, int64_t ldg, const float* X, int64_t ldx,
                            const float* Zp_save, const float* H1_save, const float* H2_save, const float* Wd,
                            const float* Wu, const float* bu, const float* scalar, int act, int skip, void* workspace,
                            float* gX, int64_t ldgx, float* gWd, float* gbd, float* gWu, float* gbu, float* gscalar,
                            int32_t d, int32_t r, gca_stream_t stream) {
    if (!g || !workspace) return GCA_ERR_INVALID_ARG;
    if (g->row_begin != 0 || g->row_end != g->N) return GCA_ERR_INVALID_ARG;
    if ((reinterpret_cast<uintptr_t>(workspace) % kAlign) != 0) return GCA_ERR_WORKSPACE;
    const size_t rw = rw_bytes(g->N, r);
    char* b = static_cast<char*>(workspace);
    float* gH2p = reinterpret_cast<float*>(b);
    float* gH1p = reinterpret_cast<float*>(b + rw);
    float* gP = reinterpret_cast<float*>(b + 2 * rw);
    void* scratch = b + 3 * rw;
    void* hub = hub_scratch_bytes(g, r) ? b + 3 * rw + gca_bwd_scratch_bytes(d, r) : nullptr;
    if (gY && X && Zp_save && H2_save && Wd && Wu && bu && ldg >= d && ldx >= d && (!gX || ldgx >= d) && act >= GCA_ACT_NONE &&
        act <= GCA_ACT_SILU && (act != GCA_ACT_SILU || H1_save) && small_path_ok(g, d, r, static_cast<cudaStream_t>(stream)))
        return small_backward(g, gY, ldg, X, ldx, Zp_save, H1_save, H2_save, Wd, Wu, bu, scalar, act, skip, gH2p, gH1p, gP, gX,
                              ldgx, scratch_ptrs(scratch, d, r), gWd, gbd, gWu, gbu, gscalar, d, r,
                              static_cast<cudaStream_t>(stream));
    GCA_TRY(gca_bwd_up(g, gY, ldg, H2_save, Wu, scalar, gH2p, scratch, nullptr, d, r, stream));
    GCA_TRY(gca_bwd_hop2(g, gH2p, Zp_save, H1_save, act, gH1p, scratch, hub, nullptr, r, stream));
    GCA_TRY(gca_bwd_hop1_down(g, gH1p, X, ldx, gY, ldg, Wd, scalar, skip, gP, gX, ldgx, scratch, hub, d, r, stream));
    return gca_bwd_finalize(scratch, Wu, bu, scalar, skip, gWd, gbd, gWu, gbu, gscalar, d, r, stream);
}
