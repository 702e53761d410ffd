// Library-level entry points of libgca: version, status strings, device probe, launch counter.
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include <cuda.h>

#include "gca_common.cuh"
#include "gca_host.cuh"

namespace gca {

static std::atomic<int64_t> g_launches{0};
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

int num_sms() {
    // cached per device: one process may drive several GPUs (torch.cuda.set_device between calls)
    static std::mutex mu;
    static std::map<int, int> cache;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    std::lock_guard<std::mutex> lk(mu);
    auto it = cache.find(dev);
    if (it != cache.end()) return it->second;
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;   // B200
    cache[dev] = sms;
    return sms;
}

static bool env_flag(const char* name) {
    const char* e = getenv(name);
    return e && e[0] == '1';
}
// Run-time switches (diagnostics / A-B runs; every one of them is exercised by tests/test_gpu_switches.py):
//   GCA_DISABLE_TC=1      CUDA-core (FFMA) kernels everywhere
//   GCA_DISABLE_STREAM=1  register-fed mma.sync projection / weight gradient instead of the TMA-fed family
//   GCA_DISABLE_TMA=1     behave as if the driver refused every tensor map (kernels that need none take over)
//   GCA_DISABLE_PDL=1     every kernel fully serialised (no programmatic dependent launch)
//   GCA_SPLIT_MB=<n>      gathered operand above n MB: K3 = plain hop + expand-only (default 160)
//   GCA_DISABLE_BWD_FUSE=1  backward tail as K3 (hop + expand) + K4 (weight gradient) instead of the one-pass kernel
bool tc_enabled() { static const bool on = !env_flag("GCA_DISABLE_TC"); return on; }
bool stream_enabled() { static const bool on = !env_flag("GCA_DISABLE_STREAM"); return on; }
thread_local bool tl_pdl_size_ok = true;
bool pdl_enabled() { static const bool on = !env_flag("GCA_DISABLE_PDL"); return on; }
long long split_bytes() {
    static const long long v = [] { const char* e = getenv("GCA_SPLIT_MB"); return (e ? atoll(e) : 160LL) << 20; }();
    return v;
}

int set_smem_impl(const void* kernel, size_t bytes, bool has_static_smem) {
    if (bytes <= 48 * 1024 && !has_static_smem) return GCA_OK;   // static + dynamic > 48 KB needs the opt-in too
    static std::mutex mu;
    static std::map<std::pair<int, const void*>, size_t> done;
    int dev = 0;
    GCA_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(mu);
    const auto key = std::make_pair(dev, kernel);
    auto it = done.find(key);
    if (it != done.end() && it->second >= bytes) return GCA_OK;
    GCA_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    done[key] = bytes;
    return GCA_OK;
}

// cuTensorMapEncodeTiled is fetched through the runtime (no link-time dependency on libcuda).
bool get_box_map(CUtensorMap* tm, const float* base, int rows, int cols, int64_t ld, int box_cols, int box_rows, bool swizzle) {
    typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static const EncodeFn enc = [] {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
            fn = nullptr;
        return reinterpret_cast<EncodeFn>(fn);
    }();
    static const bool disabled = env_flag("GCA_DISABLE_TMA");
    if (!enc || disabled) return false;
    // A map depends only on (address, shape, pitch, box), not on the data: the training loop presents the same few
    // tensors every step, so a small per-thread cache removes the host-side encode from the launch path.
    struct Key { const float* base; int rows, cols; int64_t ld; int bc, br, sw; };
    struct Entry { Key k; CUtensorMap tm; uint64_t stamp; };
    constexpr int kCap = 32;
    static thread_local Entry cache[kCap];
    static thread_local int used = 0;
    static thread_local uint64_t clock_ = 0;
    const Key k{base, rows, cols, ld, box_cols, box_rows, swizzle ? 1 : 0};
    int victim = 0;
    for (int i = 0; i < used; ++i) {
        const Key& c = cache[i].k;
        if (c.base == k.base && c.rows == k.rows && c.cols == k.cols && c.ld == k.ld && c.bc == k.bc && c.br == k.br && c.sw == k.sw) {
            cache[i].stamp = ++clock_;
            *tm = cache[i].tm;
            return true;
        }
        if (cache[i].stamp < cache[victim].stamp) victim = i;
    }
    const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
    const cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    if (enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            swizzle ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
        return false;
    const int slot = used < kCap ? used++ : victim;
    cache[slot] = Entry{k, *tm, ++clock_};
    return true;
}

struct ProfEntry { const char* name; const char* variant; cudaEvent_t a, b; };
static std::atomic<bool> g_prof_on{false};
static std::mutex g_prof_mu;
static std::vector<ProfEntry> g_prof;

bool prof_enabled() { return g_prof_on.load(std::memory_order_relaxed); }
void prof_begin(const char* name, const char* variant, cudaStream_t st) {
    ProfEntry e{name, variant ? variant : "", nullptr, nullptr};
    if (cudaEventCreate(&e.a) != cudaSuccess || cudaEventCreate(&e.b) != cudaSuccess) return;
    cudaEventRecord(e.a, st);
    std::lock_guard<std::mutex> lk(g_prof_mu);
    g_prof.push_back(e);
}
void prof_end(cudaStream_t st) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    if (!g_prof.empty() && g_prof.back().b) cudaEventRecord(g_prof.back().b, st);
}

}  // namespace gca

extern "C" int gca_profile_enable(int on) {
    std::lock_guard<std::mutex> lk(gca::g_prof_mu);
    for (auto& e : gca::g_prof) { cudaEventDestroy(e.a); cudaEventDestroy(e.b); }
    gca::g_prof.clear();
    gca::g_prof_on.store(on != 0);
    return GCA_OK;
}

// Synchronises the recorded events and writes {"name": {"launches": n, "ms": total, "variant": "..."}, ...} (JSON).
extern "C" int gca_profile_report(char* buf, size_t n) {
    if (!buf || n == 0) return GCA_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(gca::g_prof_mu);
    std::map<std::string, std::pair<long, double>> acc;
    std::map<std::string, std::string> variant;
    std::vector<std::string> order;
    for (auto& e : gca::g_prof) {
        if (cudaEventSynchronize(e.b) != cudaSuccess) continue;
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, e.a, e.b) != cudaSuccess) continue;
        auto it = acc.find(e.name);
        if (it == acc.end()) { order.push_back(e.name); acc[e.name] = {1, ms}; variant[e.name] = e.variant; }
        else { it->second.first++; it->second.second += ms; }
    }
    std::string out = "{";
    for (size_t i = 0; i < order.size(); ++i) {
        char tmp[256];
        snprintf(tmp, sizeof(tmp), "%s\"%s\": {\"launches\": %ld, \"ms\": %.6f, \"variant\": \"%s\"}", i ? ", " : "", order[i].c_str(),
                 acc[order[i]].first, acc[order[i]].second, variant[order[i]].c_str());
        out += tmp;
    }
    out += "}";
    if (out.size() + 1 > n) return GCA_ERR_WORKSPACE;
    memcpy(buf, out.c_str(), out.size() + 1);
    return GCA_OK;
}

extern "C" int gca_abi_version(void) { return GCA_ABI_VERSION; }

extern "C" const char* gca_status_string(int status) {
    switch (status) {
        case GCA_OK: return "ok";
        case GCA_ERR_INVALID_ARG: return "invalid argument";
        case GCA_ERR_WORKSPACE: return "workspace too small or misaligned";
        case GCA_ERR_CUDA: return "CUDA error";
        case GCA_ERR_INDEX_RANGE: return "edge_index holds a node id outside [0, N)";
        case GCA_ERR_UNSUPPORTED: return "unsupported shape";
        case GCA_ERR_NO_DEVICE: return "no sm_100 CUDA device";
        default: return "unknown status";
    }
}

extern "C" const char* gca_last_cuda_error(void) { return cudaGetErrorString(gca::tl_last_cuda_error); }

extern "C" int64_t gca_launch_count(void) { return gca::g_launches.load(std::memory_order_relaxed); }
