// pd_shard.cu -- sample sharding of one cohort over several contexts (SURVEY.md 8e, BASELINE.json configs[4]): every
// rank holds N/world samples of the SAME window range and the scan exchanges
//   * the tile flags of the screen (all-gather + OR),
//   * the per-(window, sample) Q3 values (all-gather; every rank then derives the same candidate lengths),
//   * the last-window summary of the pushed read pairs and the unify settings (all-gather of 64 bytes),
//   * the per-iteration EM sufficient statistics, inside the EM kernels through peer memory (pd_em_common.cuh),
//   * with pd_set_unify: the number of merged variants and one allele count per variant (pd_unify.cu).
// Two transports for the all-gathers and for mapping the peers' exchange slots:
//   NCCL  one process per GPU; the caller hands over an ncclUniqueId (pd_shard_unique_id on rank 0, distributed by
//         whatever the launcher offers, e.g. torch.distributed); slots are mapped with CUDA IPC over NVLink. libnccl
//         is opened with dlopen so that the library itself has no link-time dependency on it.
//   group several contexts of ONE process (any devices, also all on one GPU): plain device pointers, host barrier.
//         pd_shard_group_scan runs one host thread per context. Used by the single-GPU tests.
#include <dlfcn.h>

#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <cstring>
#include <mutex>
#include <thread>
#include <vector>

#include "pd_device.cuh"
#include "pd_shard.h"

namespace {

// ---- NCCL through dlopen ----------------------------------------------------------------------------------------
struct NcclId { char internal[128]; };
typedef void * NcclComm;
struct NcclApi {
    void * lib = nullptr;
    int (*GetUniqueId)(NcclId *) = nullptr;
    int (*CommInitRank)(NcclComm *, int, NcclId, int) = nullptr;
    int (*AllGather)(const void *, void *, size_t, int, NcclComm, cudaStream_t) = nullptr;
    int (*CommDestroy)(NcclComm) = nullptr;
    const char * (*GetErrorString)(int) = nullptr;
    std::string err;
};
NcclApi & nccl()
{
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        const char * names[] = {getenv("PD_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
        for (const char * n : names) {
            if (!n) continue;
            api.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
            if (api.lib) break;
        }
        if (!api.lib) { api.err = std::string("cannot open libnccl: ") + dlerror(); return; }
        api.GetUniqueId = (int (*)(NcclId *))dlsym(api.lib, "ncclGetUniqueId");
        api.CommInitRank = (int (*)(NcclComm *, int, NcclId, int))dlsym(api.lib, "ncclCommInitRank");
        api.AllGather = (int (*)(const void *, void *, size_t, int, NcclComm, cudaStream_t))dlsym(api.lib, "ncclAllGather");
        api.CommDestroy = (int (*)(NcclComm))dlsym(api.lib, "ncclCommDestroy");
        api.GetErrorString = (const char * (*)(int))dlsym(api.lib, "ncclGetErrorString");
        if (!api.GetUniqueId || !api.CommInitRank || !api.AllGather || !api.CommDestroy) api.err = "libnccl lacks the expected symbols";
    });
    return api;
}
constexpr int NCCL_UINT8 = 1;

__global__ void k_or_flags(uint32_t * __restrict__ dst, const uint32_t * __restrict__ parts, uint32_t n, uint32_t world)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t v = 0;
    for (uint32_t r = 0; r < world; ++r) v |= parts[(size_t)r * n + i];
    dst[i] = v;
}

}  // namespace

// ---- in-process group --------------------------------------------------------------------------------------------
struct PdGroup {
    std::mutex m; std::condition_variable cv;
    uint32_t n = 0, arrived = 0; uint64_t gen = 0;
    std::vector<pd_ctx *> ctxs;
    std::vector<const void *> send;
    int refs = 0;
    bool broken = false;
    bool barrier()                       // false: a rank did not arrive within two minutes (it failed) -> the group is unusable
    {
        std::unique_lock<std::mutex> lk(m);
        if (broken) return false;
        const uint64_t g = gen;
        if (++arrived == n) { arrived = 0; ++gen; cv.notify_all(); return true; }
        if (!cv.wait_for(lk, std::chrono::seconds(120), [&] { return gen != g || broken; }) || broken) { broken = true; cv.notify_all(); return false; }
        return true;
    }
};

static int shard_alloc_common(pd_ctx * c, const pd_shard_info * info)
{
    if (info->world < 2 || info->world > PD_MAX_WORLD || info->rank >= info->world || !info->min_init_global || !info->samples_per_rank)
        return pd_fail(c, PD_ERR_ARG, "pd_shard_attach: world must be 2..8, rank < world, min_init_global and samples_per_rank set");
    if (c->device < 0) return pd_fail(c, PD_ERR_CUDA, "pd_shard_attach: host-only context");
    if (c->shard) return pd_fail(c, PD_ERR_ARG, "pd_shard_attach: context is already attached");
    uint64_t tot = 0, off = 0;
    for (uint32_t r = 0; r < info->world; ++r) { if (r < info->rank) off += info->samples_per_rank[r]; tot += info->samples_per_rank[r]; }
    if (tot != info->n_samples_global || info->samples_per_rank[info->rank] != c->N || info->n_rg_global < info->n_samples_global)
        return pd_fail(c, PD_ERR_ARG, "pd_shard_attach: samples_per_rank does not match the contexts / the cohort");
    PD_CUDA(c, cudaSetDevice(c->device));
    PdShard * s = new PdShard();
    s->rank = info->rank; s->world = info->world; s->n_global = info->n_samples_global; s->r_global = info->n_rg_global;
    s->sample_offset = (uint32_t)off;
    for (uint32_t r = 0; r < info->world; ++r) { s->part_n[r] = info->samples_per_rank[r]; s->n_local_max = std::max(s->n_local_max, s->part_n[r]); }
    c->shard = s;
    // thresholds of the whole cohort: rank-indexed in initialize_deletion_lengths, and their minimum drives the screen
    cudaFree(c->d_min_init); c->d_min_init = nullptr;
    PD_CUDA(c, cudaMalloc(&c->d_min_init, (size_t)info->n_rg_global * 4));
    PD_CUDA(c, cudaMemcpy(c->d_min_init, info->min_init_global, (size_t)info->n_rg_global * 4, cudaMemcpyHostToDevice));
    int64_t tmin = INT32_MAX;
    for (uint32_t g = 0; g < info->n_rg_global; ++g) tmin = std::min<int64_t>(tmin, info->min_init_global[g]);
    c->t_min = (int32_t)std::min<int64_t>(tmin, PD_DEV_MAX - 1);
    // exchange slots: [2 launches][pairs][2 reductions][world]
    s->xr_pairs_cap = PD_XR_PAIRS;
    const size_t slots = (size_t)2 * s->xr_pairs_cap * 2 * s->world;
    PD_CUDA(c, cudaMalloc(&s->xr_mine, slots * sizeof(XrSlot)));
    PD_CUDA(c, cudaMemset(s->xr_mine, 0, slots * sizeof(XrSlot)));
    PD_CUDA(c, cudaMalloc(&s->d_ticket, 16));
    PD_CUDA(c, cudaMemset(s->d_ticket, 0, 16));
    s->d_err = s->d_ticket + 2;
    PD_CUDA(c, cudaMalloc(&s->d_small, 4096));
    return pd_em_preload_xr(c);
}

void pd_shard_release(pd_ctx * c)
{
    PdShard * s = c->shard;
    if (!s) return;
    cudaSetDevice(c->device);
    if (s->mode == 2) {
        for (uint32_t r = 0; r < s->world; ++r)
            if (r != s->rank && s->xr_peer[r]) cudaIpcCloseMemHandle(s->xr_peer[r]);
        if (s->nccl_comm) nccl().CommDestroy((NcclComm)s->nccl_comm);
    }
    if (s->group) {
        bool last;
        { std::lock_guard<std::mutex> lk(s->group->m); last = --s->group->refs == 0; }
        if (last) delete s->group;
    }
    cudaFree(s->xr_mine); cudaFree(s->d_ticket); cudaFree(s->d_small); cudaFree(s->d_send); cudaFree(s->d_recv);
    delete s;
    c->shard = nullptr;
}

// recv = [world][bytes]; every rank contributes `bytes` from `send` (device memory). Ordered on `st`.
int pd_shard_allgather(pd_ctx * c, const void * send, void * recv, size_t bytes, cudaStream_t st)
{
    PdShard * s = c->shard;
    if (s->mode == 2) {
        const int rc = nccl().AllGather(send, recv, bytes, NCCL_UINT8, (NcclComm)s->nccl_comm, st);
        if (rc != 0) return pd_fail(c, PD_ERR_CUDA, std::string("ncclAllGather: ") + (nccl().GetErrorString ? nccl().GetErrorString(rc) : "error"));
        return 0;
    }
    PdGroup * g = s->group;
    PD_CUDA(c, cudaStreamSynchronize(st));                          // my contribution is complete
    g->send[s->rank] = send;
    if (!g->barrier()) return pd_fail(c, PD_ERR_CUDA, "sample-sharded scan: a rank of the group did not reach the exchange");
    for (uint32_t r = 0; r < s->world; ++r)
        PD_CUDA(c, cudaMemcpyAsync((char *)recv + (size_t)r * bytes, g->send[r], bytes, cudaMemcpyDefault, st));
    PD_CUDA(c, cudaStreamSynchronize(st));
    if (!g->barrier()) return pd_fail(c, PD_ERR_CUDA, "sample-sharded scan: a rank of the group did not reach the exchange");   // all have read: send buffers reusable
    return 0;
}

// In-process groups on ONE GPU: a host call that implicitly synchronises the device (cudaFree, cudaHostAlloc) between a
// peer's EM launch and mine would wait for the peer's blocks, which spin until MY blocks answer. All ranks therefore
// meet here right before launching, with every allocation of the chunk done.
int pd_shard_prelaunch(pd_ctx * c)
{
    PdShard * s = c->shard;
    if (s->mode != 1) return 0;
    if (!s->group->barrier()) return pd_fail(c, PD_ERR_CUDA, "sample-sharded scan: a rank of the group did not reach the EM launch");
    return 0;
}

int pd_shard_or_flags(pd_ctx * c, uint32_t * flags, uint32_t n, cudaStream_t st)
{
    PdShard * s = c->shard;
    const size_t need = (size_t)n * 4 * s->world;
    if (need > s->cap_recv) { cudaFree(s->d_recv); s->d_recv = nullptr; s->cap_recv = 0; PD_CUDA(c, cudaMalloc(&s->d_recv, need + need / 4)); s->cap_recv = need + need / 4; }
    if (pd_shard_allgather(c, flags, s->d_recv, (size_t)n * 4, st)) return c->status;
    k_or_flags<<<(n + 255) / 256, 256, 0, st>>>(flags, (const uint32_t *)s->d_recv, n, s->world);
    PD_CUDA(c, cudaGetLastError());
    return 0;
}

// number of windows the reference scans for the COHORT's contig: combines the ranks' tail summaries. The same exchange
// carries every rank's unify settings (the first collective of a sharded scan): the unify stage has collectives of its
// own, so a rank that merged while another did not would wait for it forever. On a difference every rank fails here,
// before any kernel of the scan runs.
int pd_shard_window_total(pd_ctx * c, uint64_t * total)
{
    PdShard * s = c->shard;
    int64_t mine[8] = {c->tail.kf, c->tail.S, c->tail.E, c->tail.E_spill, c->unify_on, 0, 0, 0};
    if (c->unify_on) {
        memcpy(&mine[5], &c->unify.mean_stddev, 8); memcpy(&mine[6], &c->unify.min_relative_window_cover, 8);
        mine[7] = c->unify.output_failed != 0;
    }
    int64_t all[8 * PD_MAX_WORLD];
    PD_CUDA(c, cudaMemcpyAsync(s->d_small, mine, 64, cudaMemcpyHostToDevice, c->stream));
    if (pd_shard_allgather(c, s->d_small, (char *)s->d_small + 1024, 64, c->stream)) return c->status;
    PD_CUDA(c, cudaMemcpyAsync(all, (char *)s->d_small + 1024, 64 * s->world, cudaMemcpyDeviceToHost, c->stream));
    PD_CUDA(c, cudaStreamSynchronize(c->stream));
    for (uint32_t r = 1; r < s->world; ++r)
        if (memcmp(all + 4, all + 8 * r + 4, 32) != 0) return pd_fail(c, PD_ERR_ARG, "sample-sharded scan: unify settings differ between ranks (pd_set_unify)");
    PdTail t;
    for (uint32_t r = 0; r < s->world; ++r) t.kf = std::max(t.kf, all[8 * r]);
    for (uint32_t r = 0; r < s->world; ++r) {
        const int64_t * a = all + 8 * r;
        if (a[0] < 0) continue;
        if (a[0] == t.kf) { t.S = std::max(t.S, a[1]); t.E = std::max(t.E, a[2]); }
        else if (a[0] == t.kf - 1) t.E = std::max(t.E, a[3]);
    }
    *total = pd_tail_windows(t, c->grid.window_buffer);
    return 0;
}

// ---- attach ------------------------------------------------------------------------------------------------------
extern "C" int pd_shard_unique_id(uint8_t * out128)
{
    if (!out128) return PD_ERR_ARG;
    NcclApi & n = nccl();
    if (!n.err.empty()) return PD_ERR_CUDA;
    NcclId id;
    if (n.GetUniqueId(&id) != 0) return PD_ERR_CUDA;
    memcpy(out128, id.internal, 128);
    return 0;
}

extern "C" int pd_shard_attach_nccl(pd_ctx * c, const pd_shard_info * info, const uint8_t * id128)
{
    if (!c || !info || !id128) return PD_ERR_ARG;
    if (c->status) return c->status;
    NcclApi & n = nccl();
    if (!n.err.empty()) return pd_fail(c, PD_ERR_CUDA, "pd_shard_attach_nccl: " + n.err);
    if (shard_alloc_common(c, info)) return c->status;
    PdShard * s = c->shard;
    s->mode = 2;
    NcclId id;
    memcpy(id.internal, id128, 128);
    NcclComm comm = nullptr;
    const int rc = n.CommInitRank(&comm, (int)s->world, id, (int)s->rank);
    if (rc != 0) return pd_fail(c, PD_ERR_CUDA, std::string("ncclCommInitRank: ") + (n.GetErrorString ? n.GetErrorString(rc) : "error"));
    s->nccl_comm = comm;
    // map every peer's exchange slots (CUDA IPC; NVLink peer access is enabled lazily by the open call)
    cudaIpcMemHandle_t mine, all[PD_MAX_WORLD];
    PD_CUDA(c, cudaIpcGetMemHandle(&mine, s->xr_mine));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    PD_CUDA(c, cudaMemcpyAsync(s->d_small, &mine, 64, cudaMemcpyHostToDevice, c->stream));
    if (pd_shard_allgather(c, s->d_small, (char *)s->d_small + 1024, 64, c->stream)) return c->status;
    PD_CUDA(c, cudaMemcpyAsync(all, (char *)s->d_small + 1024, 64 * s->world, cudaMemcpyDeviceToHost, c->stream));
    PD_CUDA(c, cudaStreamSynchronize(c->stream));
    for (uint32_t r = 0; r < s->world; ++r) {
        if (r == s->rank) { s->xr_peer[r] = s->xr_mine; continue; }
        void * p = nullptr;
        PD_CUDA(c, cudaIpcOpenMemHandle(&p, all[r], cudaIpcMemLazyEnablePeerAccess));
        s->xr_peer[r] = (XrSlot *)p;
    }
    int sms = 0;
    PD_CUDA(c, cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device));
    s->grid_cap = (uint32_t)sms * 2 - 12;           // persistent EM blocks, two per SM; 12 half-SMs stay free for the result emitter
    // nobody may post into a peer before that peer's slots are zeroed and mapped everywhere: one more collective
    if (pd_shard_allgather(c, s->d_small, (char *)s->d_small + 1024, 64, c->stream)) return c->status;
    PD_CUDA(c, cudaStreamSynchronize(c->stream));
    return 0;
}

extern "C" int pd_shard_attach_group(pd_ctx ** ctxs, uint32_t n, const pd_shard_info * infos)
{
    if (!ctxs || !infos || n < 2 || n > PD_MAX_WORLD) return PD_ERR_ARG;
    for (uint32_t r = 0; r < n; ++r) {
        if (!ctxs[r]) return PD_ERR_ARG;
        if (ctxs[r]->status) return ctxs[r]->status;
        if (infos[r].rank != r || infos[r].world != n) return pd_fail(ctxs[r], PD_ERR_ARG, "pd_shard_attach_group: infos[r] must describe rank r of n");
    }
    PdGroup * g = new PdGroup();
    g->n = n; g->ctxs.assign(ctxs, ctxs + n); g->send.assign(n, nullptr); g->refs = 0;
    for (uint32_t r = 0; r < n; ++r) {
        if (shard_alloc_common(ctxs[r], &infos[r])) { if (g->refs == 0) delete g; return ctxs[r]->status; }
        ctxs[r]->shard->mode = 1; ctxs[r]->shard->group = g; ++g->refs;
    }
    for (uint32_t r = 0; r < n; ++r) {
        pd_ctx * c = ctxs[r];
        PdShard * s = c->shard;
        uint32_t share = 0;
        PD_CUDA(c, cudaSetDevice(c->device));
        for (uint32_t q = 0; q < n; ++q) {
            s->xr_peer[q] = ctxs[q]->shard->xr_mine;
            if (ctxs[q]->device == c->device) { ++share; continue; }
            int can = 0;
            PD_CUDA(c, cudaDeviceCanAccessPeer(&can, c->device, ctxs[q]->device));
            if (!can) return pd_fail(c, PD_ERR_CUDA, "pd_shard_attach_group: no peer access between the devices of the group");
            const cudaError_t e = cudaDeviceEnablePeerAccess(ctxs[q]->device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return pd_fail(c, PD_ERR_CUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
            cudaGetLastError();
        }
        int sms = 0;
        PD_CUDA(c, cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device));
        // contexts sharing one GPU split it: all their persistent blocks must be resident at the same time
        s->grid_cap = share > 1 ? std::max<uint32_t>(1, (uint32_t)sms / share) : (uint32_t)sms * 2 - 12;
    }
    return 0;
}

extern "C" int pd_shard_group_scan(pd_ctx ** ctxs, uint32_t n, uint64_t first_window, uint64_t n_windows, pd_result * outs)
{
    if (!ctxs || !outs || n < 2 || n > PD_MAX_WORLD) return PD_ERR_ARG;
    for (uint32_t r = 0; r < n; ++r)
        if (!ctxs[r] || !ctxs[r]->shard || ctxs[r]->shard->mode != 1 || ctxs[r]->shard->world != n || ctxs[r]->shard->rank != r) return PD_ERR_ARG;
    std::vector<int> rc(n, 0);
    std::vector<std::thread> th;
    for (uint32_t r = 0; r < n; ++r)
        th.emplace_back([&, r] { rc[r] = pd_contig_scan(ctxs[r], first_window, n_windows, &outs[r]); });
    for (auto & t : th) t.join();
    for (uint32_t r = 0; r < n; ++r) if (rc[r]) return rc[r];
    return 0;
}
