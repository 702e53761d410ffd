// K2: one r-wide hop (conv_down.propagate and its transpose), plus the partial sums of hub rows.
//   k_hop           gather-SpMM + bias, act | act' + bias-gradient partials | plain hop (first half of a split K3)
//   k_hub_partials  work items of rows with more than kHubDeg neighbours
// Sparse rows are processed by lane groups (R/4 lanes x 128-bit loads per neighbour row), see gca_device.cuh.
// Reference semantics: PyG GCNConv.propagate as called from /root/reference/src/finetune/gconv_adapter.py:92.
#include "gca_common.cuh"
#include "gca_device.cuh"
#include "gca_host.cuh"

namespace gca {
namespace {

// Partial sums of the hub work items: one warp per item (kHubChunk consecutive neighbours of a hub row), the
// lane groups stride over the neighbours, a fixed shuffle tree combines them.  Runs before every hop over the
// operand that hop gathers; grid-stride over the item count the build left in flags.
template <int R>
__global__ void __launch_bounds__(256)
k_hub_partials(const int* __restrict__ rowptr, const int* __restrict__ colidx, const int* __restrict__ hubitem,
               const int* __restrict__ item_row, const int* __restrict__ nitems_ptr, const float* __restrict__ F,
               float* __restrict__ hub_part) {
    constexpr int LPG = R / 4, GPW = 32 / LPG;
    pdl_wait();
    pdl_trigger();
    const int nitems = *nitems_ptr;
    const int lane = threadIdx.x & 31;
    const int sub = lane % LPG, grp = lane / LPG;
    const int wglobal = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), wtotal = gridDim.x * (blockDim.x >> 5);
    for (int item = wglobal; item < nitems; item += wtotal) {
        const int row = __ldg(item_row + item);
        const int chunk = item - __ldg(hubitem + row);
        const int rbeg = __ldg(rowptr + row), rend = __ldg(rowptr + row + 1);
        const int b = rbeg + chunk * kHubChunk;
        const int e = min(rend, b + kHubChunk);
        float4 part = gather_rows<R>(F, colidx, b + grp, e, GPW, sub);
#pragma unroll
        for (int off = LPG; off < 32; off <<= 1) part = f4_add(part, f4_shfl_xor(part, off));
        if (grp == 0) *reinterpret_cast<float4*>(hub_part + (size_t)item * R + sub * 4) = part;
    }
}

// ------------------------------------------------------------------------------------------
// K2: one r-wide hop.  FWD:  Z'[i] = dis[i] * act(dis[i] * sum_j F[j] + b)      (H1 saved for silu)
//                      BWD:  gH1'[j] = dis[j] * act'(.) * dis[j] * sum_i F[i]   (+ per-CTA sum for gbd)
// ------------------------------------------------------------------------------------------
template <int R, bool BWD>
__global__ void __launch_bounds__(256, 5)   // 5 CTAs / SM = 48 registers: the gather wants warps, not registers
k_hop(const int* __restrict__ rowptr, const int* __restrict__ colidx, const float* __restrict__ dis,
      const float* __restrict__ F, const float* __restrict__ bias, int act,
      const float* __restrict__ Zp_saved, const float* __restrict__ H1_saved,
      float* __restrict__ out, float* __restrict__ H1_out, float* __restrict__ part_bd, int* header, int n,
      const int* __restrict__ hubitem, const float* __restrict__ hub_part, int plain, const gca_push push) {
    constexpr int LPG = R / 4, GPW = 32 / LPG;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int sub = lane % LPG, grp = lane / LPG;
    const int wglobal = blockIdx.x * (blockDim.x >> 5) + warp, wtotal = gridDim.x * (blockDim.x >> 5);
    // row header (rowptr pair + dis) of the NEXT batch is fetched while the current one gathers: two of the four dependent
    // memory round trips of a batch leave the critical path.  The first header is read before the dependency wait: the
    // graph arrays were written by the build, which completed before the kernel preceding this one started.
    int nbeg = 0, nend = 0;
    float ndi = 0.f;
    {
        const int row0 = wglobal * GPW + grp;
        if (row0 < n) { nbeg = __ldg(rowptr + row0); nend = __ldg(rowptr + row0 + 1); ndi = __ldg(dis + row0); }
    }
    pdl_wait();
    pdl_trigger();
    float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!BWD && bias) b4 = ldg4(bias + sub * 4);
    float4 gb = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int rowbase = wglobal * GPW; rowbase < n; rowbase += wtotal * GPW) {
        const int row = rowbase + grp;
        const bool valid = row < n;
        const int beg = nbeg, end = nend;
        const float di = ndi;
        {
            const int nrow = row + wtotal * GPW;
            nbeg = nend = 0;
            if (nrow < n) { nbeg = __ldg(rowptr + nrow); nend = __ldg(rowptr + nrow + 1); ndi = __ldg(dis + nrow); }
        }
        const float4 acc = warp_spmm_range<R>(colidx, F, row, beg, end, lane, hubitem, hub_part);
        if (!valid) continue;
        const size_t o = (size_t)row * R + sub * 4;
        if (!BWD) {
            if (plain) {                                   // just the hop: out = dis * (A' F)  (first half of a split K3)
                *reinterpret_cast<float4*>(out + o) = f4_scale(acc, di);
                continue;
            }
            float4 h = make_float4(fmaf(di, acc.x, b4.x), fmaf(di, acc.y, b4.y), fmaf(di, acc.z, b4.z), fmaf(di, acc.w, b4.w));
            if (H1_out) *reinterpret_cast<float4*>(H1_out + o) = h;
            h = make_float4(act_apply(h.x, act), act_apply(h.y, act), act_apply(h.z, act), act_apply(h.w, act));
            const float4 zo = f4_scale(h, di);
            *reinterpret_cast<float4*>(out + o) = zo;
            for (int hp = 0; hp < push.count; ++hp) *reinterpret_cast<float4*>(push.dst[hp] + o) = zo;   // peers' gathered buffers
        } else {
            float4 g = f4_scale(acc, di);
            if (act == GCA_ACT_RELU) {
                const float4 z = ldg4(Zp_saved + o);
                g = make_float4(z.x > 0.f ? g.x : 0.f, z.y > 0.f ? g.y : 0.f, z.z > 0.f ? g.z : 0.f, z.w > 0.f ? g.w : 0.f);
            } else if (act == GCA_ACT_SILU) {
                const float4 h = ldg4(H1_saved + o);
                g = make_float4(g.x * silu_grad(h.x), g.y * silu_grad(h.y), g.z * silu_grad(h.z), g.w * silu_grad(h.w));
            }
            gb = f4_add(gb, g);
            const float4 go = f4_scale(g, di);
            *reinterpret_cast<float4*>(out + o) = go;
            for (int hp = 0; hp < push.count; ++hp) *reinterpret_cast<float4*>(push.dst[hp] + o) = go;
        }
    }
    if (BWD) {
        __shared__ float s_gb[8][R];
#pragma unroll
        for (int off = LPG; off < 32; off <<= 1) gb = f4_add(gb, f4_shfl_xor(gb, off));
        if (grp == 0) *reinterpret_cast<float4*>(&s_gb[warp][sub * 4]) = gb;
        __syncthreads();
        if (threadIdx.x < R) {
            float t = 0.f;
#pragma unroll
            for (int w = 0; w < 8; ++w) t += s_gb[w][threadIdx.x];
            part_bd[(size_t)blockIdx.x * R + threadIdx.x] = t;
        }
        if (blockIdx.x == 0 && threadIdx.x == 0) header[2] = gridDim.x;
    }
}

// Partial sums of the hub rows over operand F (skipped when the validated build found no hub row).
template <int R>
int launch_hub_partials_t(const Csr& c, const float* F, cudaStream_t st) {
    if (c.nitems_host != 0 && !c.hub_part) return GCA_ERR_WORKSPACE;   // hub rows (or unknown) need the caller's hub scratch
    if (c.nitems_host == 0) return GCA_OK;
    int grid = c.nitems_host > 0 ? (c.nitems_host + 7) / 8 : 2 * num_sms();
    if (grid > 8 * num_sms()) grid = 8 * num_sms();
    {
        ProfScope ps("hub_partials", st);
        GCA_CUDA(launch_pdl(k_hub_partials<R>, dim3(grid), dim3(256), 0, st, c.rowptr, c.colidx, c.hubitem, c.item_row, c.nitems_ptr, F, c.hub_part));
    }
    GCA_LAUNCH_OK();
    return GCA_OK;
}

template <int R, bool BWD>
int launch_hop_t(const Csr& c, const float* F, const float* bias, int act,
                 const float* Zp, const float* H1s, float* out, float* H1o, float* part_bd, int* header, int n, cudaStream_t st,
                 int plain, const char* prof_name, const gca_push* push) {
    constexpr int GPW = 32 / (R / 4);
    gca_push pv{};
    if (push && !plain) pv = *push;
    if (pv.count < 0 || pv.count > GCA_MAX_PEERS) return GCA_ERR_INVALID_ARG;
    GCA_TRY(launch_hub_partials_t<R>(c, F, st));
    const int* rowptr = c.rowptr; const int* colidx = c.colidx; const float* dis = c.dis;
    int grid = (n + 8 * GPW - 1) / (8 * GPW);
    // one resident wave: the warps loop over their row batches; a second, partially filled wave of CTAs only adds a tail
    static const int per_sm = [] {
        int v = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, k_hop<R, BWD>, 256, 0) != cudaSuccess) v = 0;
        return v > 0 && v <= 16 ? v : 8;
    }();
    const int cap = BWD ? (kMaxPartsBd < per_sm * num_sms() ? kMaxPartsBd : per_sm * num_sms()) : per_sm * num_sms();
    if (grid > cap) grid = cap;
    if (grid < 1) grid = 1;
    {
        ProfScope ps(prof_name ? prof_name : (BWD ? "hop_bwd" : "hop_fwd"), st);
        GCA_CUDA(launch_pdl(k_hop<R, BWD>, dim3(grid), dim3(256), 0, st, rowptr, colidx, dis, F, bias, act, Zp, H1s, out, H1o, part_bd, header, n, c.hubitem, c.hub_part, plain, pv));
    }
    GCA_LAUNCH_OK();
    return GCA_OK;
}

}  // namespace

int launch_hop(int r, bool bwd, const Csr& c, const float* F, const float* bias, int act, const float* Zp, const float* H1s,
               float* out, float* H1o, float* part_bd, int* header, int n, cudaStream_t st, int plain, const char* prof_name,
               const gca_push* push) {
    if (bwd) { GCA_DISPATCH_R(r, (launch_hop_t<R_, true>(c, F, bias, act, Zp, H1s, out, H1o, part_bd, header, n, st, plain, prof_name, push))); }
    GCA_DISPATCH_R(r, (launch_hop_t<R_, false>(c, F, bias, act, Zp, H1s, out, H1o, part_bd, header, n, st, plain, prof_name, push)));
}
int launch_hub_partials(int r, const Csr& c, const float* F, cudaStream_t st) {
    GCA_DISPATCH_R(r, (launch_hub_partials_t<R_>(c, F, st)));
}

}  // namespace gca
