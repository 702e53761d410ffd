// Partitioned forward / backward for a client that already owns an NCCL communicator (SURVEY.md section 8b: "multi-GPU
// variants taking ncclComm_t").  One process (or thread) per GPU calls these with its row block's graph handle; the four
// r-wide operands are exchanged with in-place ncclAllGather on the caller's stream, the parameter gradients with
// ncclAllReduce.  The peer-memory exchange of gca_peer.cu (pushes fused into the producing kernels) is the faster path on
// an NVLink box; this one needs nothing but the communicator.
//
// libgca has no link-time dependency on NCCL: the four functions used are resolved at first use from the NCCL the
// process has already loaded (dlopen by soname returns that copy - the communicator must be used with the library that
// created it), or from GCA_NCCL_LIB.
#include <dlfcn.h>

#include <cstdlib>
#include <mutex>

#include "gca_common.cuh"
#include "gca_host.cuh"

using namespace gca;

namespace {

typedef int (*AllGatherFn)(const void*, void*, size_t, int, void*, cudaStream_t);
typedef int (*AllReduceFn)(const void*, void*, size_t, int, int, void*, cudaStream_t);
typedef int (*GroupFn)(void);
constexpr int kNcclFloat = 7, kNcclSum = 0;   // ncclFloat32, ncclSum (stable since NCCL 2.0)

struct Nccl {
    AllGatherFn all_gather = nullptr;
    AllReduceFn all_reduce = nullptr;
    GroupFn group_start = nullptr, group_end = nullptr;
    bool ok = false;
};

const Nccl& nccl() {
    static Nccl n;
    static std::once_flag once;
    std::call_once(once, [] {
        void* h = RTLD_DEFAULT;                                    // symbols already global in the process?
        if (!dlsym(RTLD_DEFAULT, "ncclAllGather")) {
            const char* path = getenv("GCA_NCCL_LIB");
            h = dlopen(path && path[0] ? path : "libnccl.so.2", RTLD_NOW | RTLD_LOCAL);
            if (!h) return;
        }
        n.all_gather = reinterpret_cast<AllGatherFn>(dlsym(h, "ncclAllGather"));
        n.all_reduce = reinterpret_cast<AllReduceFn>(dlsym(h, "ncclAllReduce"));
        n.group_start = reinterpret_cast<GroupFn>(dlsym(h, "ncclGroupStart"));
        n.group_end = reinterpret_cast<GroupFn>(dlsym(h, "ncclGroupEnd"));
        n.ok = n.all_gather && n.all_reduce && n.group_start && n.group_end;
    });
    return n;
}

inline size_t full_bytes(int32_t N, int32_t world, int32_t r) {
    const size_t s = ((size_t)N + world - 1) / world;
    return align_up(sizeof(float) * s * world * r + sizeof(float) * r);   // + one pad row (even-row reads of the last shard)
}

// rows [row_begin, row_end) must be this rank's block of ceil(N / world) rows
inline bool block_ok(const gca_graph* g, int32_t world, int32_t rank) {
    if (world < 1 || rank < 0 || rank >= world) return false;
    const int64_t s = ((int64_t)g->N + world - 1) / world;
    const int64_t lo = s * rank < g->N ? s * rank : g->N, hi = s * (rank + 1) < g->N ? s * (rank + 1) : g->N;
    return g->row_begin == lo && g->row_end == hi;
}

int gather_rows_inplace(void* comm, float* full, int32_t N, int32_t world, int32_t rank, int32_t r, cudaStream_t st) {
    if (world == 1) return GCA_OK;
    const size_t count = (((size_t)N + world - 1) / world) * r;
    if (nccl().all_gather(full + count * rank, full, count, kNcclFloat, comm, st) != 0) return GCA_ERR_CUDA;
    return GCA_OK;
}

}  // namespace

extern "C" int gca_nccl_available(void) { return nccl().ok ? 1 : 0; }

extern "C" size_t gca_forward_nccl_workspace_bytes(const gca_graph* g, int32_t world, int32_t d, int32_t r) {
    if (!g || world < 1 || d <= 0 || r <= 0) return 0;
    return 2 * full_bytes(g->N, world, r) + hub_scratch_bytes(g, r);
}

extern "C" int gca_forward_nccl(const gca_graph* g, void* nccl_comm, int32_t world, int32_t rank, const float* X, int64_t ldx,
                                const float* Wd, const float* bd, const float* Wu, const float* bu, const float* scalar,
                                int act, int skip, void* workspace, float* Zp_save, float* H1_save, float* H2_save, float* Y,
                                int64_t ldy, int32_t d, int32_t r, gca_stream_t stream) {
    if (!g || !workspace || !Zp_save || (!nccl_comm && world > 1)) return GCA_ERR_INVALID_ARG;
    if (!block_ok(g, world, rank)) return GCA_ERR_INVALID_ARG;
    if ((reinterpret_cast<uintptr_t>(workspace) % kAlign) != 0) return GCA_ERR_WORKSPACE;
    if (world > 1 && !nccl().ok) return GCA_ERR_UNSUPPORTED;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t fb = full_bytes(g->N, world, r);
    const size_t shard = (((size_t)g->N + world - 1) / world) * r;          // floats per rank
    const int n = g->row_end - g->row_begin;
    char* b = static_cast<char*>(workspace);
    float* Pfull = reinterpret_cast<float*>(b);
    float* Zfull = reinterpret_cast<float*>(b + fb);
    void* hub = hub_scratch_bytes(g, r) ? b + 2 * fb : nullptr;
    GCA_TRY(gca_fwd_project(g, X, ldx, Wd, Pfull + shard * rank, nullptr, d, r, stream));
    GCA_TRY(gather_rows_inplace(nccl_comm, Pfull, g->N, world, rank, r, st));
    GCA_TRY(gca_fwd_hop1(g, Pfull, bd, act, Zfull + shard * rank, H1_save, hub, nullptr, r, stream));
    if (n > 0) GCA_CUDA(cudaMemcpyAsync(Zp_save, Zfull + shard * rank, sizeof(float) * (size_t)n * r, cudaMemcpyDeviceToDevice, st));
    GCA_TRY(gather_rows_inplace(nccl_comm, Zfull, g->N, world, rank, r, st));
    return gca_fwd_hop2_up(g, Zfull, X, ldx, Wu, bu, scalar, skip, H2_save, Y, ldy, hub, d, r, stream);
}

extern "C" size_t gca_backward_nccl_workspace_bytes(const gca_graph* g, int32_t world, int32_t d, int32_t r) {
    if (!g || world < 1 || d <= 0 || r <= 0) return 0;
    const int n = g->row_end - g->row_begin;
    const size_t gp = align_up(sizeof(float) * (size_t)(n > 0 ? n + (n & 1) : 2) * r);
    return 2 * full_bytes(g->N, world, r) + gp + gca_bwd_scratch_bytes(d, r) + hub_scratch_bytes(g, r);
}

extern "C" int gca_backward_nccl(const gca_graph* g, void* nccl_comm, int32_t world, int32_t rank, const float* gY, int64_t ldg,
                                 const float* X, int64_t ldx, const float* Zp_save, const float* H1_save, const float* H2_save,
                                 const float* Wd, const float* Wu, const float* bu, const float* scalar, int act, int skip,
                                 void* workspace, float* gX, int64_t ldgx, float* gWd, float* gbd, float* gWu, float* gbu,
                                 float* gscalar, int32_t d, int32_t r, gca_stream_t stream) {
    if (!g || !workspace || (!nccl_comm && world > 1)) return GCA_ERR_INVALID_ARG;
    if (!block_ok(g, world, rank)) return GCA_ERR_INVALID_ARG;
    if ((reinterpret_cast<uintptr_t>(workspace) % kAlign) != 0) return GCA_ERR_WORKSPACE;
    if (world > 1 && !nccl().ok) return GCA_ERR_UNSUPPORTED;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t fb = full_bytes(g->N, world, r);
    const size_t shard = (((size_t)g->N + world - 1) / world) * r;
    const int n = g->row_end - g->row_begin;
    const size_t gpb = align_up(sizeof(float) * (size_t)(n > 0 ? n + (n & 1) : 2) * r);
    char* b = static_cast<char*>(workspace);
    float* gH2full = reinterpret_cast<float*>(b);
    float* gH1full = reinterpret_cast<float*>(b + fb);
    float* gP = reinterpret_cast<float*>(b + 2 * fb);
    void* scratch = b + 2 * fb + gpb;
    void* hub = hub_scratch_bytes(g, r) ? b + 2 * fb + gpb + gca_bwd_scratch_bytes(d, r) : nullptr;
    GCA_TRY(gca_bwd_up(g, gY, ldg, H2_save, Wu, scalar, gH2full + shard * rank, scratch, nullptr, d, r, stream));
    GCA_TRY(gather_rows_inplace(nccl_comm, gH2full, g->N, world, rank, r, st));
    GCA_TRY(gca_bwd_hop2(g, gH2full, Zp_save, H1_save, act, gH1full + shard * rank, scratch, hub, nullptr, r, stream));
    GCA_TRY(gather_rows_inplace(nccl_comm, gH1full, g->N, world, rank, r, st));
    GCA_TRY(gca_bwd_hop1_down(g, gH1full, X, ldx, gY, ldg, Wd, scalar, skip, gP, gX, ldgx, scratch, hub, d, r, stream));
    GCA_TRY(gca_bwd_finalize(scratch, Wu, bu, scalar, skip, gWd, gbd, gWu, gbu, gscalar, d, r, stream));
    if (world == 1) return GCA_OK;
    // every replica ends up with the same (summed) parameter gradients
    const Nccl& nc = nccl();
    int bad = nc.group_start();
    if (gWd) bad |= nc.all_reduce(gWd, gWd, (size_t)r * d, kNcclFloat, kNcclSum, nccl_comm, st);
    if (gbd) bad |= nc.all_reduce(gbd, gbd, (size_t)r, kNcclFloat, kNcclSum, nccl_comm, st);
    if (gWu) bad |= nc.all_reduce(gWu, gWu, (size_t)r * d, kNcclFloat, kNcclSum, nccl_comm, st);
    if (gbu) bad |= nc.all_reduce(gbu, gbu, (size_t)d, kNcclFloat, kNcclSum, nccl_comm, st);
    if (gscalar) bad |= nc.all_reduce(gscalar, gscalar, 1, kNcclFloat, kNcclSum, nccl_comm, st);
    bad |= nc.group_end();
    return bad ? GCA_ERR_CUDA : GCA_OK;
}
