// Shared host/device helpers for libgca (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "gca.h"

// Host-side descriptor handed out by gca_graph_build.  All pointers are device pointers
// into the caller's workspace; the struct itself lives on the host heap.
struct gca_graph {
    int32_t N, row_begin, row_end, normalize;
    int64_t E;
    int64_t capacity;
    int32_t* rowptr;
    int32_t* colidx;
    int32_t* rowptr_t;
    int32_t* colidx_t;
    float* dis;
    int32_t* cnt;      // [n] counters / fill cursors (forward CSR)
    int32_t* cnt_t;    // [n] counters / fill cursors (transposed CSR)
    int32_t* flags;    // [0] index-range error, [1] nnz, [2] nnz_t, [3] hub items, [4] hub items (transpose); written by the
                       // build only: the handle carries NO per-launch mutable state (re-entrant per (handle, stream))
    // Hub rows (degree > kHubDeg) are cut into work items of kHubChunk neighbours (see gca_graph.cu / k_hub_partials)
    int32_t* hubitem;      // [n]  first item of a hub row, -1 otherwise          (forward CSR)
    int32_t* hubitem_t;    // [n]                                                 (transposed CSR)
    int32_t* item_row;     // [hub_cap] local row of an item
    int32_t* item_row_t;
    int64_t hub_cap;       // capacity of the item lists; the items' partial sums live in per-call scratch of
                           // hub_cap * 64 floats supplied by the caller (gca_hub_scratch_bytes)
    int32_t nitems, nitems_t;   // host copies after gca_graph_validate; -1 = unknown
};

namespace gca {
constexpr int kHubDeg = 512;      // rows longer than this take the hub path
constexpr int kHubChunk = 512;    // neighbours per hub work item (one warp each)
}

namespace gca {

extern thread_local cudaError_t tl_last_cuda_error;
void count_launch(int n = 1);
int num_sms();

// Optional per-kernel timing with CUDA events recorded on the launching stream
// (gca_profile_enable / gca_profile_report); off by default and free when off.
bool prof_enabled();
void prof_begin(const char* name, const char* variant, cudaStream_t st);
void prof_end(cudaStream_t st);
// `variant` names the kernel implementation that was picked (reported by gca_profile_report, so that the tests can
// assert which code path a run-time switch really selected).
struct ProfScope {
    cudaStream_t st;
    bool on;
    ProfScope(const char* name, cudaStream_t s, const char* variant = "") : st(s), on(prof_enabled()) { if (on) prof_begin(name, variant, s); }
    ~ProfScope() { if (on) prof_end(st); }
};

inline int record(cudaError_t e) {
    if (e != cudaSuccess) { tl_last_cuda_error = e; return GCA_ERR_CUDA; }
    return GCA_OK;
}

#define GCA_TRY(expr)                                   \
    do {                                                \
        int _st = (expr);                               \
        if (_st != GCA_OK) return _st;                  \
    } while (0)

#define GCA_CUDA(call) GCA_TRY(::gca::record((call)))

// Check the launch that was just issued (asynchronous: configuration errors only).
#define GCA_LAUNCH_OK()                                 \
    do {                                                \
        ::gca::count_launch();                          \
        GCA_CUDA(cudaGetLastError());                   \
    } while (0)

// Programmatic dependent launch (PDL): kernels of one forward / backward are chained on a stream; with the
// launch attribute below the next kernel's CTAs may start (and run their prologue: weight staging into shared
// memory) while the previous kernel drains.  pdl_wait() blocks until the previous kernel has completed and its
// writes are visible - it MUST precede the first access to anything a neighbouring kernel reads or writes;
// pdl_trigger() lets the dependent kernel start launching (kernels trigger right after their own prologue).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
bool pdl_enabled();
// Programmatic launches hide ~1 us of launch gap per kernel boundary: worth 4 us on the 0.36 ms arxiv-shaped step, noise on
// kernels that run for a millisecond - where they measured HARMFUL (products-shaped step 9.4 ms without, 12.0 ms with,
// wherever the trigger sits).  Each entry point states its problem size; launches above kPdlMaxRows are plain.
constexpr int64_t kPdlMaxRows = 1 << 20;
extern thread_local bool tl_pdl_size_ok;
struct PdlHint {
    bool prev;
    explicit PdlHint(int64_t rows) : prev(tl_pdl_size_ok) { tl_pdl_size_ok = rows <= kPdlMaxRows; }
    ~PdlHint() { tl_pdl_size_ok = prev; }
};

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = (pdl_enabled() && tl_pdl_size_ok) ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

constexpr int kWarp = 32;
constexpr size_t kAlign = 256;
inline size_t align_up(size_t x, size_t a = kAlign) { return (x + a - 1) / a * a; }

// ---- device helpers -------------------------------------------------------------
__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
// Streaming (read-once / write-once) 128-bit accesses to the d-wide tensors: no L1 allocation, and an L2
// evict-first policy so that the streams do not push the r-wide activations, the CSR and the weight-gradient
// partials (all re-read by later kernels) out of the 126 MB L2.
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
    uint64_t pol;
    asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ float4 ldg4_stream(const float* p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(l2_evict_first_policy()));
    return v;
}
__device__ __forceinline__ void stg4_stream(float* p, float4 v) {
    asm volatile("st.global.L1::no_allocate.L2::cache_hint.v4.f32 [%0], {%1,%2,%3,%4}, %5;"
                 :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(l2_evict_first_policy()) : "memory");
}
// The addend A of the *_add entries (Y = ... + A).  Y == A is allowed, so A is read through the coherent path (not .nc,
// whose data must stay unchanged for the kernel's lifetime), still without L1 allocation and L2 evict-first.
__device__ __forceinline__ float4 ld4_addend(const float* p) {
    float4 v;
    asm volatile("ld.global.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(l2_evict_first_policy()));
    return v;
}
// y + a as one round-to-nearest add per element (never contracted into an FMA with the product that formed y), so the
// fused sum has the bits of the separate `y + a`.
__device__ __forceinline__ float4 f4_add_rn(float4 y, float4 a) {
    return make_float4(__fadd_rn(y.x, a.x), __fadd_rn(y.y, a.y), __fadd_rn(y.z, a.z), __fadd_rn(y.w, a.w));
}
__device__ __forceinline__ float4 f4_add(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
__device__ __forceinline__ float4 f4_scale(float4 a, float s) { return make_float4(a.x * s, a.y * s, a.z * s, a.w * s); }
__device__ __forceinline__ float4 f4_shfl_xor(float4 v, int m) {
    v.x = __shfl_xor_sync(0xffffffffu, v.x, m);
    v.y = __shfl_xor_sync(0xffffffffu, v.y, m);
    v.z = __shfl_xor_sync(0xffffffffu, v.z, m);
    v.w = __shfl_xor_sync(0xffffffffu, v.w, m);
    return v;
}

}  // namespace gca
