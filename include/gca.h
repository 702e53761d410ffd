/*
 * gca.h -- C ABI of the B200-native GConv-Adapter hot path (libgca.so).
 *
 * The reference is pure Python: its "FFI" for this path is the torch.nn.Module
 *   src/finetune/gconv_adapter.py:5   class GConvAdapter
 *   src/finetune/gconv_adapter.py:80  forward(x, edge_index, edge_attr=None)
 * which bottoms out in two torch_geometric GCNConv calls (:40-41, :92) and autograd.
 * Every entry point below cites the piece of that interface it replaces.  The Python
 * mirror (gconv_adapter_b200/finetune/gconv_adapter.py) binds them with ctypes; the stub a
 * reference maintainer would add is shown in INTEGRATION.md.
 *
 * Conventions
 *  - plain pointers and sizes only; every pointer is a DEVICE pointer unless it says host.
 *  - every call is asynchronous on `stream` (a cudaStream_t) except where noted; nothing
 *    is allocated by the library: the caller passes workspaces sized by the *_bytes calls.
 *  - return value: GCA_OK (0) or a negative gca_status; no exceptions cross the ABI.
 *  - fp32 row-major tensors; `ld*` is the row pitch in elements (>= d, multiple of 4).  X / Y / gY / gX pointers
 *    (and every other pitched operand) are 16 B aligned: the kernels load and store them as float4 and through tensor
 *    maps, and do not check.  A column window of a wider tensor qualifies when its first column is.
 *  - re-entrant per (graph handle, stream): a built handle is read-only; every byte a call scribbles on (projection
 *    scratch, partial sums, the partial sums of hub rows) comes from the caller's per-call workspaces, so one handle
 *    may serve several streams / threads / adapters at once (SURVEY.md section 8b "Threading").
 *  - node rows are partitioned: a graph handle covers rows [row_begin, row_end) of an
 *    N-node graph ("local rows", n = row_end - row_begin); neighbour ids stay global.
 *    A single-GPU run uses row_begin = 0, row_end = N.
 *
 * Arithmetic (normalize = 1; dis = (in_degree + 1)^-1/2, A' = A without loops + I):
 *   P'  = dis * (X Wd^T)                    gca_fwd_project
 *   Z'  = dis * act(dis * (A' P') + bd)     gca_fwd_hop1          (all-gather P' before)
 *   H2  = dis * (A' Z')                     gca_fwd_hop2_up       (all-gather Z' before)
 *   Y   = s * (H2 Wu^T + bu [+ X])
 * which equals the reference's  s * (Ahat(act(Ahat X Wd^T + bd)) Wu^T + bu + X)  with
 * Ahat = D^-1/2 A' D^-1/2 applied at width r instead of width d (SURVEY.md section 7).
 * normalize = 0: dis = 1, A' = A exactly as given (no loops added or removed).
 */
#ifndef GCA_H_
#define GCA_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GCA_ABI_VERSION 2

typedef void* gca_stream_t;               /* cudaStream_t */
typedef struct gca_graph gca_graph;       /* opaque, host-side descriptor of device arrays */

typedef enum gca_status {
    GCA_OK = 0,
    GCA_ERR_INVALID_ARG = -1,    /* null pointer, negative size, bad enum */
    GCA_ERR_WORKSPACE = -2,      /* workspace too small or misaligned (256 B) */
    GCA_ERR_CUDA = -3,           /* a CUDA runtime call / launch failed (see gca_last_cuda_error) */
    GCA_ERR_INDEX_RANGE = -4,    /* edge_index holds an id outside [0, N) */
    GCA_ERR_UNSUPPORTED = -5,    /* shape outside what the kernels implement */
    GCA_ERR_NO_DEVICE = -6       /* no sm_100 device */
} gca_status;

typedef enum gca_act { GCA_ACT_NONE = 0, GCA_ACT_RELU = 1, GCA_ACT_SILU = 2 } gca_act;

/* -------- multi-GPU (one process per GPU, rows partitioned; SURVEY.md section 8e) --------
 * The r-wide operand of every sparse hop is needed in full on every GPU.  The phase that PRODUCES it takes a gca_push:
 * peer-mapped device pointers (CUDA IPC, see gca_peer_*) to the caller's OWN rows inside each peer's gathered buffer,
 * i.e. peer_full[h] + row_begin * r.  The producing kernel stores every finished row there as well (plain stores over
 * NVLink / NVSwitch, overlapped with its own streaming), so no collective call sits between two phases - only
 * gca_peer_barrier.  NULL or count = 0: single GPU, nothing is pushed. */
#define GCA_MAX_PEERS 8
#define GCA_IPC_HANDLE_BYTES 64
typedef struct gca_push {
    int32_t count;                    /* destinations, 0 .. GCA_MAX_PEERS */
    int32_t reserved;
    float*  dst[GCA_MAX_PEERS];
} gca_push;
typedef struct gca_peer_sync {
    int32_t   world, rank;
    uint32_t* flags[GCA_MAX_PEERS];   /* flags[h]: GPU h's flag array (world x uint32, zero-initialised), peer-mapped; [rank] = local */
    uint32_t* seq;                    /* local device counter (zero-initialised), bumped by every barrier / all-reduce */
} gca_peer_sync;

/* -------- library -------- */
int         gca_abi_version(void);
const char* gca_status_string(int status);
/* cudaGetErrorString of the last CUDA error this library saw on the calling thread (host string). */
const char* gca_last_cuda_error(void);
/* 1 if (d, r) is on the vectorised kernels (d % 4 == 0, r in {8,16,32}); 0 = generic kernels. */
int         gca_shape_is_fast(int32_t d, int32_t r);

/* -------- graph structure (K0) --------
 * Replaces torch_geometric gcn_norm + add_remaining_self_loops, which the reference
 * re-runs inside both GCNConv calls of every forward (src/finetune/gconv_adapter.py:92;
 * PyG default cached=False).  Built once per edge_index and reused by both hops, by the
 * backward, and by every adapter that sees the same graph.
 *
 * src/dst: edge_index[0] / edge_index[1], int64, E entries each (PyG source_to_target).
 * Produces, for local rows: CSR by target (forward gathers), CSR by source (backward
 * gathers), neighbour ids ascending inside every row (deterministic sums), and dis.
 */
size_t gca_graph_workspace_bytes(int64_t E, int32_t N, int32_t row_begin, int32_t row_end);
int    gca_graph_build(const int64_t* src, const int64_t* dst, int64_t E, int32_t N,
                       int32_t row_begin, int32_t row_end, int normalize,
                       void* workspace, size_t workspace_bytes, gca_stream_t stream,
                       gca_graph** out);
/* Synchronises `stream`; returns GCA_ERR_INDEX_RANGE if an id was out of range, else GCA_OK,
 * and fills nnz / nnz_t (entries of the two CSRs) when the pointers are non-null (host). */
int    gca_graph_validate(gca_graph* g, gca_stream_t stream, int64_t* nnz, int64_t* nnz_t);
/* The same without a host synchronisation: _async copies the five flag words into PINNED host memory on `stream`; once an
 * event the caller recorded after it has completed, _finish (host only) returns what gca_graph_validate would have.
 * Until then the handle is usable with "hub items unknown": the hop phases then need hub_scratch (gca_hub_scratch_bytes > 0). */
int    gca_graph_validate_async(const gca_graph* g, int32_t* pinned_host_flags5, gca_stream_t stream);
int    gca_graph_validate_finish(gca_graph* g, const int32_t* pinned_host_flags5, int64_t* nnz, int64_t* nnz_t);
void   gca_graph_destroy(gca_graph* g);   /* frees the host descriptor only */

typedef struct gca_graph_view {          /* device pointers into the caller's workspace */
    int32_t  N, row_begin, row_end, normalize;
    int64_t  capacity;                   /* allocated entries per CSR */
    const int32_t* rowptr;               /* [n+1]  CSR by target */
    const int32_t* colidx;               /* [nnz]  source ids, ascending per row */
    const int32_t* rowptr_t;             /* [n+1]  CSR by source (transpose) */
    const int32_t* colidx_t;             /* [nnz_t] target ids, ascending per row */
    const float*   dis;                  /* [n]    (deg+1)^-1/2, or 1 when normalize = 0 */
} gca_graph_view;
int    gca_graph_get_view(const gca_graph* g, gca_graph_view* out /* host */);
/* coef[e] = dis[row(e)] * dis[colidx[e]] for the forward CSR, in CSR order: the fp32
 * edge weights gcn_norm would produce.  Only valid for a full-graph handle (n == N). */
int    gca_graph_edge_coef(const gca_graph* g, float* coef, gca_stream_t stream);
/* Rows with more than 512 neighbours ("hubs") are pre-reduced per work item into per-CALL scratch of this many bytes
 * (256 B aligned), passed as `hub_scratch` to every phase that walks the graph.  0 when the validated build
 * (gca_graph_validate) found no hub row: hub_scratch may then be NULL. */
size_t gca_hub_scratch_bytes(const gca_graph* g);

/* -------- backbone propagation over the same handle (SURVEY section 8f, rank 3) --------
 * out[i, 0:D] = dst_scale[i] * sum_{j in N(i)} src_scale[j] * X[j, 0:D]  for the handle's rows; transpose = 1 is the adjoint
 * (walks the CSR by source; the backward of transpose = 0).  NULL scales mean the handle's dis = (in-degree)^-1/2, which for a
 * graph that already contains exactly one self loop per node is DIFFormer's gcn_conv
 * (src/models/transductive/difformer.py:63-79, edge_weight = None: both factors use the IN-degree).  NodeFormer's
 * add_conv_relational_bias (src/models/transductive/nodeformer.py:202-224) scales the source end by the OUT-degree:
 * pass src_scale[j] = out_degree(j)^-1/2 (they coincide on undirected graphs).  Heads are flattened into D; coefficients
 * differ from the reference's sqrt(1/d) products by <= 2 ULP.  D % 4 == 0; full-graph handles only. */
int gca_propagate(const gca_graph* g, int transpose, const float* X_full /*[N,D]*/, int64_t ldx,
                  float* out_local /*[n,D]*/, int64_t ldo, const float* src_scale /*[N] or NULL*/,
                  const float* dst_scale /*[n] or NULL*/, int32_t D, gca_stream_t stream);

/* -------- forward phases (src/finetune/gconv_adapter.py:92-106) --------
 * n = local rows.  *_full buffers hold all N rows (after the caller's all-gather);
 * *_local buffers hold the n local rows.  On one GPU they are the same buffer.
 */
/* conv_down.lin (d -> r) with the source-side D^-1/2 folded in: P'[i] = dis[i] * X[i] Wd^T */
int gca_fwd_project(const gca_graph* g, const float* X, int64_t ldx, const float* Wd /*[r,d]*/,
                    float* Pp_local /*[n,r]*/, const gca_push* push, int32_t d, int32_t r, gca_stream_t stream);
/* conv_down.propagate + bias + act_fn, result pre-scaled for the next hop.
 * H1_local may be NULL unless act == GCA_ACT_SILU (backward needs the pre-activation). */
int gca_fwd_hop1(const gca_graph* g, const float* Pp_full /*[N,r]*/, const float* bd /*[r]*/, int act,
                 float* Zp_local /*[n,r]*/, float* H1_local /*[n,r] or NULL*/, void* hub_scratch, const gca_push* push,
                 int32_t r, gca_stream_t stream);
/* conv_up (propagate at width r, then lin r -> d, + bias) + skip + scalar.
 * scalar may be NULL (= 1).  H2_local is saved for the backward. */
int gca_fwd_hop2_up(const gca_graph* g, const float* Zp_full /*[N,r]*/, const float* X, int64_t ldx,
                    const float* Wu /*[d,r]*/, const float* bu /*[d]*/, const float* scalar /*[1] or NULL*/,
                    int skip, float* H2_local /*[n,r]*/, float* Y, int64_t ldy, void* hub_scratch,
                    int32_t d, int32_t r, gca_stream_t stream);

/* -------- backward phases (autograd of the above) -------- */
size_t gca_bwd_scratch_bytes(int32_t d, int32_t r);
/* gH2'[i] = dis[i] * s * gY[i] Wu ; partial sums for gWu = s * gY^T H2 and gbu = s * sum_i gY[i].
 * One pass over gY serves both (gca_stream.cu) when d % 32 == 0, d <= 256, r = 16. */
int gca_bwd_up(const gca_graph* g, const float* gY, int64_t ldg, const float* H2_local,
               const float* Wu, const float* scalar, float* gH2p_local /*[n,r]*/,
               void* scratch, const gca_push* push, int32_t d, int32_t r, gca_stream_t stream);
/* The two halves of gca_bwd_up as separate calls, so that a multi-GPU caller can start the all-gather of gH2'
 * between them (the weight-gradient half does not depend on it): _project clears the scratch header and writes
 * gH2', _wgrad accumulates the gWu / gbu partials. */
int gca_bwd_up_project(const gca_graph* g, const float* gY, int64_t ldg, const float* Wu, const float* scalar,
                       float* gH2p_local, void* scratch, const gca_push* push, int32_t d, int32_t r, gca_stream_t stream);
int gca_bwd_up_wgrad(const gca_graph* g, const float* gY, int64_t ldg, const float* H2_local, void* scratch,
                     int32_t d, int32_t r, gca_stream_t stream);
/* gH1'[j] = dis[j] * act'(.) * dis[j] * sum_{i in out(j)} gH2'[i] ; partial sums for gbd */
int gca_bwd_hop2(const gca_graph* g, const float* gH2p_full /*[N,r]*/, const float* Zp_local,
                 const float* H1_local /*NULL unless silu*/, int act, float* gH1p_local /*[n,r]*/,
                 void* scratch, void* hub_scratch, const gca_push* push, int32_t r, gca_stream_t stream);
/* gP[j] = dis[j] * sum_{i in out(j)} gH1'[i] ; gX = gP Wd [+ s * gY] ; partials for gWd = gP^T X
 * and for <gY, X> (needed by gscalar).  gX may be NULL (x does not require grad).
 * With skip, gX, r = 16, d % 32 == 0, d <= 256, n >= 2048 this is a plain hop + ONE streaming pass over gY and X
 * (gca_stream_bwd.cu).  gP_local must be readable for an EVEN number of rows (n rounded up; contents of the pad row are
 * ignored): at r = 16 the pass reads it through a [ceil(n / 2), 32]-float tensor map. */
int gca_bwd_hop1_down(const gca_graph* g, const float* gH1p_full /*[N,r]*/, const float* X, int64_t ldx,
                      const float* gY, int64_t ldg, const float* Wd, const float* scalar, int skip,
                      float* gP_local /*[n,r] workspace*/, float* gX, int64_t ldgx,
                      void* scratch, void* hub_scratch, int32_t d, int32_t r, gca_stream_t stream);
/* Deterministic second-stage reduction of the partial sums into the parameter gradients.
 * Any output pointer may be NULL.  gscalar = <gY, X>(if skip) + <gY^T H2, Wu> + <sum gY, bu>. */
int gca_bwd_finalize(const void* scratch, const float* Wu, const float* bu, const float* scalar, int skip,
                     float* gWd /*[r,d]*/, float* gbd /*[r]*/, float* gWu /*[d,r]*/, float* gbu /*[d]*/,
                     float* gscalar /*[1]*/, int32_t d, int32_t r, gca_stream_t stream);

/* -------- single-GPU conveniences: the whole forward / backward on one stream -------- */
size_t gca_forward_workspace_bytes(const gca_graph* g, int32_t d, int32_t r);   /* P' scratch + hub scratch */
int gca_forward(const gca_graph* g, const float* X, int64_t ldx,
                const float* Wd, const float* bd, const float* Wu, const float* bu, const float* scalar,
                int act, int skip, void* workspace,
                float* Zp_save, float* H1_save /*NULL unless silu*/, float* H2_save,
                float* Y, int64_t ldy, int32_t d, int32_t r, gca_stream_t stream);
size_t gca_backward_workspace_bytes(const gca_graph* g, int32_t d, int32_t r);  /* gH2', gH1', gP + partial sums + hub scratch */
int gca_backward(const gca_graph* g, const float* gY, int64_t ldg, const float* X, int64_t ldx,
                 const float* Zp_save, const float* H1_save, const float* H2_save,
                 const float* Wd, const float* Wu, const float* bu, const float* scalar,
                 int act, int skip, void* workspace,
                 float* gX, int64_t ldgx, float* gWd, float* gbd, float* gWu, float* gbu, float* gscalar,
                 int32_t d, int32_t r, gca_stream_t stream);

/* -------- multi-GPU plumbing over peer memory --------
 * gca_peer_barrier: returns (on the stream) once every GPU of the group has reached the same barrier in ITS stream: all
 * rows pushed by kernels that precede it on any GPU are then visible locally.  Every rank issues the same sequence of
 * barriers / all-reduces.  One warp; no host synchronisation; capturable in a CUDA graph.
 * gca_peer_allreduce: out[i] = sum over ranks (in rank order: bitwise identical everywhere) of src[i]; slots->dst[h] is
 * GPU h's slot array ([world][len] floats, peer-mapped), slots->count = world.
 * gca_push_rows: copy nfloats (multiple of 4) floats of a finished local shard to the peers (for producers without a fused push).
 * gca_peer_alloc / export / open / close / free: zero-initialised device memory that other processes of the node can map
 * (cudaIpcGetMemHandle / cudaIpcOpenMemHandle with lazy peer access); handles are GCA_IPC_HANDLE_BYTES bytes (host). */
int gca_peer_barrier(const gca_peer_sync* sync, gca_stream_t stream);
int gca_peer_allreduce(const gca_peer_sync* sync, const gca_push* slots, const float* src, float* out, int32_t len,
                       gca_stream_t stream);
int gca_push_rows(const float* src, int64_t nfloats, const gca_push* push, gca_stream_t stream);
int gca_peer_alloc(size_t bytes, void** ptr /* host out */);
int gca_peer_free(void* ptr);
int gca_peer_export(void* ptr, void* handle64 /* host out */);
int gca_peer_open(const void* handle64 /* host */, void** ptr /* host out */);
int gca_peer_close(void* ptr);

/* -------- normalization = 'layer_norm' tail (src/finetune/gconv_adapter.py:54-61, 98-106; SURVEY.md 8f rank 2) --------
 * Y = s * (gamma * (X - mean_row) * rstd_row + beta): torch.nn.LayerNorm over the last dimension (biased variance, eps inside
 * the square root) followed by the adapter's learnable scalar, one pass forward and one pass backward over [n, d].
 * gamma / beta / scalar may be NULL (= 1 / 0 / 1).  mean, rstd: [n] floats written by the forward and read by the backward.
 * X is the forward's input (the output of gca_fwd_hop2_up without scalar).  d % 4 == 0, d <= 1024.
 * Backward: gX (may be NULL), ggamma / gbeta [d] and gscalar [1] (any may be NULL); scratch of gca_layernorm_scratch_bytes(d)
 * bytes (256 B aligned) holds the per-CTA partial sums, combined in a fixed order (no atomics). */
size_t gca_layernorm_scratch_bytes(int32_t d);
int    gca_layernorm_scale_fwd(const float* X, int64_t ldx, const float* gamma, const float* beta, const float* scalar,
                               float eps, float* Y, int64_t ldy, float* mean, float* rstd, int32_t n, int32_t d,
                               gca_stream_t stream);
int    gca_layernorm_scale_bwd(const float* gY, int64_t ldg, const float* X, int64_t ldx, const float* gamma, const float* beta,
                               const float* scalar, const float* mean, const float* rstd, float* gX, int64_t ldgx,
                               float* ggamma, float* gbeta, float* gscalar, void* scratch, int32_t n, int32_t d,
                               gca_stream_t stream);

/* -------- multi-GPU for a client that owns an NCCL communicator (SURVEY.md section 8b) --------
 * The whole partitioned forward / backward of ONE rank: the phases above with an in-place ncclAllGather of each r-wide
 * operand between them and an ncclAllReduce (sum) of the parameter gradients at the end, all on `stream`.
 * nccl_comm is the caller's ncclComm_t (as void*), world / rank its size and this caller's rank; g must cover this rank's
 * block of ceil(N / world) rows (row_begin = rank * ceil(N / world)).  X, Y, gY, gX, Zp_save, H1_save, H2_save are the
 * LOCAL rows.  libgca does not link NCCL: ncclAllGather / ncclAllReduce / ncclGroupStart / ncclGroupEnd are resolved at
 * first use from the NCCL already loaded in the process ("libnccl.so.2" by soname, or the file named by GCA_NCCL_LIB);
 * gca_nccl_available() tells whether that worked (GCA_ERR_UNSUPPORTED otherwise; world = 1 never needs it).
 * On an NVLink box the peer-memory exchange above (gca_push + gca_peer_barrier) is the faster path. */
int    gca_nccl_available(void);
size_t gca_forward_nccl_workspace_bytes(const gca_graph* g, int32_t world, int32_t d, int32_t r);
int    gca_forward_nccl(const gca_graph* g, void* nccl_comm, int32_t world, int32_t rank, const float* X, int64_t ldx,
                        const float* Wd, const float* bd, const float* Wu, const float* bu, const float* scalar,
                        int act, int skip, void* workspace, float* Zp_save, float* H1_save /*NULL unless silu*/,
                        float* H2_save, float* Y, int64_t ldy, int32_t d, int32_t r, gca_stream_t stream);
size_t gca_backward_nccl_workspace_bytes(const gca_graph* g, int32_t world, int32_t d, int32_t r);
int    gca_backward_nccl(const gca_graph* g, void* nccl_comm, int32_t world, int32_t rank, const float* gY, int64_t ldg,
                         const float* X, int64_t ldx, const float* Zp_save, const float* H1_save, const float* H2_save,
                         const float* Wd, const float* Wu, const float* bu, const float* scalar, int act, int skip,
                         void* workspace, float* gX, int64_t ldgx, float* gWd, float* gbd, float* gWu, float* gbu,
                         float* gscalar, int32_t d, int32_t r, gca_stream_t stream);

/* Number of kernels this library has launched since load (bench.py's gpu_launches). */
int64_t gca_launch_count(void);
/* Per-kernel device timing for bench.py's roofline: while enabled, every launch is bracketed by
 * cudaEvents on its own stream.  enable(0|1) also clears what was recorded.  report synchronises
 * and writes JSON {"kernel": {"launches": n, "ms": total}, ...} into buf (host). */
int gca_profile_enable(int on);
int gca_profile_report(char* buf, size_t buf_bytes);

#ifdef __cplusplus
}
#endif
#endif /* GCA_H_ */
