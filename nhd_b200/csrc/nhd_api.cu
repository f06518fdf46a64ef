/*
 * nhd_api.cu — the C-ABI of include/nhd_b200.h on top of the sm_100a kernels.
 *
 * Host side of the drop-in boundary: owns the device mirror of the cluster (tiled node
 * records in HBM), de-duplicates the pod descriptors of a batch into pod types, launches
 * the snapshot predicate kernel and the select+assign sweep, and (when the node set is
 * sharded over several GPUs) merges the per-rank feasibility bitmaps with one NCCL
 * all-reduce.  There is no CPU fallback: every entry point that computes fails with
 * NHD_ERR_CUDA when no device is usable.
 */
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/nhd_b200.h"
#include "nhd_kernels.cuh"

using namespace nhd;

/* ------------------------------------------------------------------ NCCL, resolved at run time */

typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId_;
typedef int ncclResult_t_;
enum { NCCL_INT8 = 0 };                       /* ncclInt8 / ncclChar (nccl.h, stable since 2.0) */

struct NcclApi {
    void* lib = nullptr;
    ncclResult_t_ (*GetUniqueId)(ncclUniqueId_*) = nullptr;
    ncclResult_t_ (*CommInitRank)(ncclComm_t*, int, ncclUniqueId_, int) = nullptr;
    ncclResult_t_ (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t_ (*AllGather)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t_) = nullptr;
    bool load()
    {
        if (lib) return true;
        /* reuse the copy already mapped into the process (e.g. PyTorch's) before opening the system one */
        lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);
        if (!lib) lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_LOCAL);
        if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_LOCAL);
        if (!lib) return false;
        GetUniqueId = (decltype(GetUniqueId))dlsym(lib, "ncclGetUniqueId");
        CommInitRank = (decltype(CommInitRank))dlsym(lib, "ncclCommInitRank");
        CommDestroy = (decltype(CommDestroy))dlsym(lib, "ncclCommDestroy");
        AllGather = (decltype(AllGather))dlsym(lib, "ncclAllGather");
        GetErrorString = (decltype(GetErrorString))dlsym(lib, "ncclGetErrorString");
        return GetUniqueId && CommInitRank && CommDestroy && AllGather;
    }
};
static NcclApi g_nccl;

/* ------------------------------------------------------------------ handle */

struct nhd_handle {
    nhd_params params;
    double cap[NHD_MAX_SPEED_CLASSES];
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    int sm_count = 148;
    int smem_optin = 48 * 1024;
    ncclComm_t comm = nullptr;

    /* cluster mirror */
    int n_nodes = 0, n_super = 0, words = 0, max_numa = 1;
    /* NUMA count of every node the filter could accept (active, not in maintenance; 0 otherwise): the mapping stage's
       tuple limits are judged against the largest of these, and follow updates in both directions */
    std::vector<uint8_t> node_numa;
    int numa_hist[NHD_MAX_NUMA + 1] = {0, 0, 0, 0, 0};
    uint8_t* d_nodes = nullptr;
    uint8_t* d_snapshot = nullptr;
    size_t nodes_bytes = 0;
    bool loaded = false, have_snapshot = false;

    /* staging for records (AoS) */
    void* d_stage = nullptr;  size_t d_stage_cap = 0;
    void* h_stage = nullptr;  size_t h_stage_cap = 0;
    int32_t* d_idx = nullptr; size_t d_idx_cap = 0;

    /* batch */
    int n_pods = 0, n_types = 0;
    bool staged = false, solved = false;
    PodType* d_types = nullptr;     size_t types_cap = 0;
    int32_t* d_pod_type = nullptr;  double* d_now = nullptr;  nhd_binding* d_out = nullptr;  size_t pods_cap = 0;
    uint8_t* h_batch = nullptr;     size_t h_batch_cap = 0;     /* pinned: types | pod_type | now */
    nhd_binding* h_out = nullptr;   size_t h_out_cap = 0;       /* pinned */
    uint64_t* d_bitmaps = nullptr;  size_t bitmaps_cap = 0;
    int32_t* d_cursors = nullptr;   size_t cursors_cap = 0;
    int32_t* d_busy_list = nullptr;
    int32_t* d_pend = nullptr;
    uint4* d_dyn = nullptr;
    uint16_t* d_class = nullptr;
    ClassSlot* d_class_slots = nullptr;
    unsigned long long* d_prof = nullptr;
    int* d_vresult = nullptr;
    uint64_t* d_memo = nullptr;
    uint8_t* d_xchg = nullptr;  size_t xchg_cap = 0;     /* node-sharded ranks: one slot per rank (summaries + bitmap columns) */
    uint8_t* d_ftab = nullptr;            /* direct-path tables of the staged batch's pod types */
    uint8_t* d_mapt = nullptr;            /* GetNumaGroupIdx table of the direct path */
    uint8_t* d_mapt2 = nullptr;           /* ... with the GPU stage (resolve_kernel); the device's shared copy, not owned */
    uint32_t* d_sigs = nullptr;           /* per-NUMA NIC signatures */
    ClsFast* d_cls_fast = nullptr;        /* per hardware class */
    double now0 = 0.0;
    bool const_clock = true;
    long long shard_min_pairs = 1LL << 21;   /* nhd_shard_min_pairs() when the handle was created */
    int n_names = 0;
    uint64_t names_used = 0;
    uint64_t* d_pod_groups = nullptr; size_t pod_groups_cap = 0;
    std::vector<int32_t> pod_type_host;

    /* nhd_explain's own buffers: the call leaves everything above as it was */
    PodType* d_x_types = nullptr;   size_t x_types_cap = 0;
    double* d_x_now = nullptr;      size_t x_now_cap = 0;
    int32_t* d_x_out = nullptr;     size_t x_out_cap = 0;       /* counts [T][NHD_WHY_COUNT] | first [T][2] */
    uint8_t* d_x_reasons = nullptr; size_t x_reasons_cap = 0;   /* [T][n_nodes] */

    nhd_timing timing;
    std::string err;
};

static int32_t fail(nhd_handle* h, int32_t code, const char* fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (h) h->err = buf;
    return code;
}

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(h, NHD_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_),   \
                        __FILE__, __LINE__);                                                       \
    } while (0)

template <typename T>
static cudaError_t grow_dev(T*& p, size_t& cap, size_t need)
{
    if (need <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = std::max(need, (size_t)256);
    cudaError_t e = cudaMalloc((void**)&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
}

template <typename T>
static cudaError_t grow_pinned(T*& p, size_t& cap, size_t need)
{
    if (need <= cap) return cudaSuccess;
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
    size_t want = std::max(need, (size_t)256);
    cudaError_t e = cudaMallocHost((void**)&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
}

/* ------------------------------------------------------------------ validation */

extern "C" int32_t nhd_validate_node(const nhd_node_rec* r)
{
    if (!r) return NHD_ERR_INVALID;
    return validate_node_rec(*r);          /* same routine the upload path runs on the device */
}

extern "C" int32_t nhd_validate_pod(const nhd_pod* p)
{
    if (!p) return NHD_ERR_INVALID;
    if (p->n_groups < 1) return NHD_ERR_INVALID;             /* zero groups crashes the reference (Matcher.py:346) */
    if (p->n_groups > NHD_MAX_GROUPS) return NHD_ERR_UNSUPPORTED;
    int cores = p->n_misc, gpus = 0;
    for (int g = 0; g < p->n_groups; g++) {
        const nhd_pod_group& pg = p->groups[g];
        if (pg.n_gpus > NHD_MAX_GROUP_GPUS) return NHD_ERR_UNSUPPORTED;
        cores += pg.n_proc + pg.n_helpers;
        for (int j = 0; j < pg.n_gpus; j++) cores += pg.gpu_feeders[j];
        gpus += pg.n_gpus;
        if (!(pg.rx_gbps >= 0.0) || !(pg.tx_gbps >= 0.0) || !std::isfinite(pg.rx_gbps) || !std::isfinite(pg.tx_gbps))
            return NHD_ERR_INVALID;
    }
    if (cores > NHD_MAX_POD_CORES || gpus > NHD_MAX_POD_GPUS) return NHD_ERR_UNSUPPORTED;
    return NHD_OK;
}

/* numa^(groups+1) enumeration limits of the mapping stage */
static bool tuple_limits_ok(int K, int G)
{
    long nq = 1, np = 1;
    for (int i = 0; i < G + 1; i++) nq *= K;
    for (int i = 0; i < G; i++) np *= K;
    return nq <= NHD_MAX_TUPLES && np <= 64;
}

static inline uint8_t schedulable_numa(const nhd_node_rec& r)
{
    /* (a record not validated yet may say anything: counts beyond the limit are not counted — the load is rejected) */
    return ((r.flags & NHD_NODE_ACTIVE) && !(r.flags & NHD_NODE_MAINTENANCE) && r.n_numa <= NHD_MAX_NUMA) ? (uint8_t)r.n_numa : (uint8_t)0;
}

static void track_numa(nhd_handle* h, int n, const nhd_node_rec* recs, const int32_t* idx)
{
    for (int i = 0; i < n; i++) {
        const int node = idx ? idx[i] : i;
        const uint8_t k = schedulable_numa(recs[i]);
        h->numa_hist[h->node_numa[node]]--;
        h->numa_hist[k]++;
        h->node_numa[node] = k;
    }
    h->max_numa = 1;
    for (int k = 2; k <= NHD_MAX_NUMA; k++) if (h->numa_hist[k] > 0) h->max_numa = k;
}

/* ------------------------------------------------------------------ lifecycle */

extern "C" void nhd_default_params(nhd_params* p)
{
    if (!p) return;
    memset(p, 0, sizeof(*p));
    p->nic_bw_avail_percent = 0.9;       /* Node.py:18 */
    p->min_busy_secs = 30.0;             /* Node.py:107 */
    p->enable_sharing = 0;               /* Node.py:20 */
    p->world_size = 1;
}

/*
 * Node-sharding threshold: (nodes x distinct pod types) from which the snapshot filter is split over the ranks.
 * Below it the exchange costs more than the shard saves — measured on B200s over NVSwitch: the whole filter of
 * 65 536 nodes x 16 types takes 0.047 ms on one GPU, the all-gather + unpack of its bitmaps 0.026 / 0.029 / 0.070 ms
 * on 2 / 4 / 8 ranks — so every rank filters the whole cluster and no collective runs.  Every rank must use the same
 * value (it decides whether the collective is entered): NHD_SHARD_MIN_PAIRS in the environment of all ranks, read
 * when a handle is created; default 2^21.
 */
static long long shard_min_pairs_now()
{
    const char* e = getenv("NHD_SHARD_MIN_PAIRS");
    if (e && *e) {
        char* end = nullptr;
        const long long v = strtoll(e, &end, 10);
        if (end && *end == 0 && v >= 0) return v;
    }
    return 1LL << 21;
}
extern "C" int64_t nhd_shard_min_pairs(void) { return (int64_t)shard_min_pairs_now(); }

extern "C" int32_t nhd_nccl_unique_id(uint8_t out[128])
{
    if (!out) return NHD_ERR_INVALID;
    if (!g_nccl.load()) return NHD_ERR_NCCL;
    ncclUniqueId_ id;
    if (g_nccl.GetUniqueId(&id) != 0) return NHD_ERR_NCCL;
    memcpy(out, id.internal, 128);
    return NHD_OK;
}

/* MAPT2 (mapt2_kernel) is a constant of the CPython set model, 64 KB: one copy per device for the life of the process,
 * shared by every handle on that device and never freed.  Published only after the kernel that fills it has finished. */
static std::mutex g_mapt2_mu;
static uint8_t* g_mapt2[64];
static cudaError_t shared_mapt2(int device, cudaStream_t st, uint8_t** out)
{
    std::lock_guard<std::mutex> lk(g_mapt2_mu);
    if (device < 0 || device >= 64) return cudaErrorInvalidValue;
    if (!g_mapt2[device]) {
        uint8_t* t = nullptr;
        cudaError_t e = cudaMalloc((void**)&t, (size_t)MAPT2_BYTES);
        if (e != cudaSuccess) return e;
        mapt2_kernel<<<(MAPT2_BYTES + 127) / 128, 128, 0, st>>>(t);
        e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) { cudaFree(t); return e; }
        g_mapt2[device] = t;
    }
    *out = g_mapt2[device];
    return cudaSuccess;
}

extern "C" int32_t nhd_destroy(nhd_handle* h)
{
    if (!h) return NHD_OK;
    if (h->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm);
    cudaSetDevice(h->params.device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    cudaFree(h->d_nodes); cudaFree(h->d_snapshot); cudaFree(h->d_stage); cudaFree(h->d_idx);
    cudaFree(h->d_types); cudaFree(h->d_pod_type); cudaFree(h->d_now); cudaFree(h->d_out);
    cudaFree(h->d_bitmaps); cudaFree(h->d_cursors); cudaFree(h->d_busy_list); cudaFree(h->d_memo); cudaFree(h->d_dyn); cudaFree(h->d_class); cudaFree(h->d_class_slots); cudaFree(h->d_mapt); cudaFree(h->d_ftab); cudaFree(h->d_xchg); cudaFree(h->d_sigs); cudaFree(h->d_cls_fast); 
#ifdef NHD_CHECKS
    cudaFreeHost(h->d_prof);
#else
    cudaFree(h->d_prof);
#endif
    cudaFree(h->d_pend); cudaFree(h->d_vresult); cudaFree(h->d_pod_groups);
    cudaFree(h->d_x_types); cudaFree(h->d_x_now); cudaFree(h->d_x_out); cudaFree(h->d_x_reasons);
    if (h->h_stage) cudaFreeHost(h->h_stage);
    if (h->h_batch) cudaFreeHost(h->h_batch);
    if (h->h_out) cudaFreeHost(h->h_out);
    for (auto& e : h->ev) if (e) cudaEventDestroy(e);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return NHD_OK;
}

extern "C" int32_t nhd_create(const nhd_params* p, nhd_handle** out)
{
    if (!p || !out) return NHD_ERR_INVALID;
    *out = nullptr;
    if (p->enable_sharing) return NHD_ERR_UNSUPPORTED;        /* the reference ships with sharing off (Node.py:20) */
    if (p->n_speed_classes < 0 || p->n_speed_classes > NHD_MAX_SPEED_CLASSES) return NHD_ERR_INVALID;
    if (p->world_size < 1 || p->rank < 0 || p->rank >= p->world_size) return NHD_ERR_INVALID;
    nhd_handle* h = new nhd_handle();
    h->params = *p;
    memset(&h->timing, 0, sizeof(h->timing));
    for (int i = 0; i < NHD_MAX_SPEED_CLASSES; i++)
        h->cap[i] = p->speed_gbps[i] * p->nic_bw_avail_percent;   /* n.speed*NIC_BW_AVAIL_PERCENT, Node.py:292 */
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0 || p->device < 0 || p->device >= ndev) {
        delete h;
        return NHD_ERR_CUDA;                                    /* no CPU fallback */
    }
    *out = h;
    h->shard_min_pairs = shard_min_pairs_now();
    CK(cudaSetDevice(p->device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, p->device));
    h->sm_count = prop.multiProcessorCount;
    h->smem_optin = (int)prop.sharedMemPerBlockOptin;
    CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    for (auto& ev : h->ev) CK(cudaEventCreate(&ev));
    CK(cudaMalloc((void**)&h->d_memo, (size_t)MEMO_SLOTS * 16));
    CK(cudaMemsetAsync(h->d_memo, 0, (size_t)MEMO_SLOTS * 16, h->stream));
    CK(cudaMalloc((void**)&h->d_vresult, 16));
#ifdef NHD_CHECKS
    CK(cudaHostAlloc((void**)&h->d_prof, 64 * 8, cudaHostAllocMapped));      /* readable after a device fault */
    memset(h->d_prof, 0, 64 * 8);
#else
    CK(cudaMalloc((void**)&h->d_prof, 64 * 8));
    CK(cudaMemsetAsync(h->d_prof, 0, 64 * 8, h->stream));
#endif
    CK(cudaMalloc((void**)&h->d_class_slots, (size_t)CLASS_SLOTS * sizeof(ClassSlot)));
    CK(cudaMemsetAsync(h->d_class_slots, 0, (size_t)CLASS_SLOTS * sizeof(ClassSlot), h->stream));
    CK(cudaMalloc((void**)&h->d_mapt, (size_t)((MAPT_BYTES + 15) & ~15)));
    CK(cudaMalloc((void**)&h->d_ftab, ftab_bytes(FAST_MAX_TYPES)));
    CK(cudaMalloc((void**)&h->d_sigs, (size_t)FAST_NSIG * 4));
    CK(cudaMemsetAsync(h->d_sigs, 0, (size_t)FAST_NSIG * 4, h->stream));
    CK(cudaMalloc((void**)&h->d_cls_fast, (size_t)CLASS_SLOTS * sizeof(ClsFast)));
    CK(cudaMemsetAsync(h->d_cls_fast, 0, (size_t)CLASS_SLOTS * sizeof(ClsFast), h->stream));
    mapt_kernel<<<(MAPT_BYTES + 127) / 128, 128, 0, h->stream>>>(h->d_mapt);
    CK(cudaGetLastError());
    CK(shared_mapt2(p->device, h->stream, &h->d_mapt2));
    CK(cudaFuncSetAttribute(filter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            FILTER_STAGES * SUPER_BYTES + TYPES_SMEM_MAX * (int)sizeof(PodType)));
    CK(cudaFuncSetAttribute(sweep_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->smem_optin));
    CK(cudaFuncSetAttribute(sweep_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 1024));
    {
        /* one empty launch of the big kernel: its code is loaded (lazy module loading) and resident before the first
         * real batch instead of inside it (a first sweep used to take tens of milliseconds) */
        SweepArgs sa;
        memset(&sa, 0, sizeof(sa));
        sa.prof = h->d_prof;                               /* (profile builds flush their counters) */
        const size_t smem = (size_t)SMEMO_SLOTS * 16 + (size_t)DMEMO_SLOTS * 48 + (size_t)DCACHE_SLOTS * 36 + 16 +
                            (size_t)CLSNIC_SLOTS * 48 + (size_t)SPMEMO_SLOTS * 16 + ((MAPT_BYTES + 15) & ~15) + 4096;
        sweep_kernel<true><<<1, SWEEP_THREADS, smem, h->stream>>>(sa);
        sweep_kernel<false><<<1, SWEEP_THREADS, smem, h->stream>>>(sa);
        CK(cudaGetLastError());
    }
    if (p->world_size > 1) {
        if (!g_nccl.load()) return fail(h, NHD_ERR_NCCL, "libnccl.so.2 not loadable");
        ncclUniqueId_ id;
        memcpy(id.internal, p->nccl_unique_id, 128);
        ncclResult_t_ r = g_nccl.CommInitRank(&h->comm, p->world_size, id, p->rank);
        if (r != 0) return fail(h, NHD_ERR_NCCL, "ncclCommInitRank: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?");
    }
    CK(cudaStreamSynchronize(h->stream));
    return NHD_OK;
}

extern "C" const char* nhd_last_error(const nhd_handle* h) { return h ? h->err.c_str() : "null handle"; }

/* ------------------------------------------------------------------ cluster mirror */

static bool is_pinned_host(const void* p)
{
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost;
}

/* host -> device, ingest into the tiled layout, validate on the device, classify.  Records that
 * already sit in pinned memory (nhd_alloc_pinned) are copied straight from the caller's buffer. */
static int32_t upload_records(nhd_handle* h, int n, const nhd_node_rec* recs, const int32_t* idx, int* max_numa,
                              bool track_while_copying = false)
{
    const size_t bytes = (size_t)n * sizeof(nhd_node_rec);
    CK(grow_dev(h->d_stage, h->d_stage_cap, bytes));
    const void* src = recs;
    if (!is_pinned_host(recs)) {
        CK(grow_pinned(h->h_stage, h->h_stage_cap, bytes));
        memcpy(h->h_stage, recs, bytes);
        src = h->h_stage;
    }
    CK(cudaMemcpyAsync(h->d_stage, src, bytes, cudaMemcpyHostToDevice, h->stream));
    const int32_t* d_idx = nullptr;
    if (idx) {
        CK(grow_dev(h->d_idx, h->d_idx_cap, (size_t)n * 4));
        CK(cudaMemcpyAsync(h->d_idx, idx, (size_t)n * 4, cudaMemcpyHostToDevice, h->stream));
        d_idx = h->d_idx;
    }
    const int threads = 256;
    int vinit[4] = {0x7FFFFFFF, 0, 1, 0};
    CK(cudaMemcpyAsync(h->d_vresult, vinit, 16, cudaMemcpyHostToDevice, h->stream));
    validate_kernel<<<(n + threads - 1) / threads, threads, 0, h->stream>>>((const nhd_node_rec*)h->d_stage, n, h->d_vresult);
    CK(cudaGetLastError());
    int vres[4];
    CK(cudaMemcpyAsync(vres, h->d_vresult, 16, cudaMemcpyDeviceToHost, h->stream));
    /* full load: the host's own walk over the records (NUMA bookkeeping) runs while the copy and the validation are in
     * flight; a rejected load leaves the handle unloaded, and the next load starts that bookkeeping afresh */
    if (track_while_copying) track_numa(h, n, recs, idx);
    CK(cudaStreamSynchronize(h->stream));
    if (vres[0] != 0x7FFFFFFF) {
        const int32_t v = nhd_validate_node(&recs[vres[0]]);
        return fail(h, v != NHD_OK ? v : NHD_ERR_INVALID, "node record %d rejected by nhd_validate_node", vres[0]);
    }
    *max_numa = vres[2];
    const int total = n * REC_CHUNKS;
    ingest_kernel<<<(total + threads - 1) / threads, threads, 0, h->stream>>>(
        (const uint4*)h->d_stage, d_idx, n, h->d_nodes);
    CK(cudaGetLastError());
    /* hardware classes of the (re)written nodes */
    classify_claim_kernel<<<(n + threads - 1) / threads, threads, 0, h->stream>>>(h->d_nodes, d_idx, n, h->d_class_slots, h->d_class);
    CK(cudaGetLastError());
    classify_verify_kernel<<<(n + threads - 1) / threads, threads, 0, h->stream>>>(h->d_nodes, d_idx, n, h->d_class_slots, h->d_class);
    cls_fast_kernel<<<(CLASS_SLOTS + 255) / 256, 256, 0, h->stream>>>(h->d_class_slots, h->d_cls_fast, h->d_sigs);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(h->stream));
    return NHD_OK;
}

extern "C" int32_t nhd_load_nodes(nhd_handle* h, int32_t n_nodes, const nhd_node_rec* recs)
{
    if (!h || n_nodes < 0 || (n_nodes > 0 && !recs)) return NHD_ERR_INVALID;
    CK(cudaSetDevice(h->params.device));
    const int n_super = std::max(1, (n_nodes + SUPER_NODES - 1) / SUPER_NODES);
    const size_t bytes = (size_t)n_super * SUPER_BYTES;
    if (bytes != h->nodes_bytes) {
        cudaFree(h->d_nodes); cudaFree(h->d_snapshot); cudaFree(h->d_busy_list); cudaFree(h->d_dyn); cudaFree(h->d_class); cudaFree(h->d_pend);
        h->d_nodes = h->d_snapshot = nullptr; h->d_busy_list = nullptr; h->d_dyn = nullptr; h->d_class = nullptr; h->d_pend = nullptr;
        h->nodes_bytes = 0;
        CK(cudaMalloc((void**)&h->d_nodes, bytes));
        CK(cudaMalloc((void**)&h->d_snapshot, bytes));
        CK(cudaMalloc((void**)&h->d_busy_list, ((size_t)n_super * SUPER_NODES + 64) * 4));
        CK(cudaMalloc((void**)&h->d_dyn, (size_t)n_super * SUPER_NODES * sizeof(NodeDyn)));
        CK(cudaMalloc((void**)&h->d_class, (size_t)n_super * SUPER_NODES * sizeof(uint16_t)));
        CK(cudaMalloc((void**)&h->d_pend, (size_t)n_super * SUPER_NODES * sizeof(int32_t)));
        h->nodes_bytes = bytes;
    }
    h->n_nodes = n_nodes;
    h->n_super = n_super;
    h->words = n_super * SUPER_NODES / 64;
    CK(cudaMemsetAsync(h->d_nodes, 0, bytes, h->stream));     /* padding nodes: inactive */
    CK(cudaMemsetAsync(h->d_class, 0xFF, (size_t)n_super * SUPER_NODES * sizeof(uint16_t), h->stream));
    h->loaded = true;
    h->have_snapshot = false;
    h->staged = h->solved = false;
    h->max_numa = 1;
    h->node_numa.assign((size_t)n_nodes, 0);
    for (int k = 0; k <= NHD_MAX_NUMA; k++) h->numa_hist[k] = 0;
    h->numa_hist[0] = n_nodes;
    if (n_nodes == 0) { CK(cudaStreamSynchronize(h->stream)); return NHD_OK; }
    int mx = 1;
    const int32_t rc = upload_records(h, n_nodes, recs, nullptr, &mx, true);
    if (rc != NHD_OK) { h->loaded = false; return rc; }
    return NHD_OK;
}

extern "C" int32_t nhd_update_nodes(nhd_handle* h, int32_t n, const int32_t* idx, const nhd_node_rec* recs)
{
    if (!h || n < 0 || (n > 0 && (!idx || !recs))) return NHD_ERR_INVALID;
    if (!h->loaded) return fail(h, NHD_ERR_STATE, "nhd_update_nodes before nhd_load_nodes");
    CK(cudaSetDevice(h->params.device));
    {
        std::vector<uint8_t> seen((size_t)h->n_nodes, 0);            /* the device applies the records in parallel: one per node */
        for (int i = 0; i < n; i++) {
            if (idx[i] < 0 || idx[i] >= h->n_nodes) return fail(h, NHD_ERR_INVALID, "node index %d out of range", idx[i]);
            if (seen[idx[i]]) return fail(h, NHD_ERR_INVALID, "node index %d appears twice in one update", idx[i]);
            seen[idx[i]] = 1;
            int32_t v = nhd_validate_node(&recs[i]);      /* before anything is written: an update must not half-apply */
            if (v != NHD_OK) return fail(h, v, "update %d: record rejected", i);
        }
    }
    if (n == 0) return NHD_OK;
    int mx = 1;
    const int32_t rc = upload_records(h, n, recs, idx, &mx);
    if (rc == NHD_OK) track_numa(h, n, recs, idx);
    return rc;
}

extern "C" int32_t nhd_read_nodes(nhd_handle* h, int32_t first, int32_t n, nhd_node_rec* out)
{
    if (!h || first < 0 || n < 0 || (n > 0 && !out)) return NHD_ERR_INVALID;
    if (!h->loaded || (long long)first + (long long)n > (long long)h->n_nodes) return fail(h, NHD_ERR_STATE, "range outside the loaded cluster");
    if (n == 0) return NHD_OK;
    CK(cudaSetDevice(h->params.device));
    const size_t bytes = (size_t)n * sizeof(nhd_node_rec);
    CK(grow_dev(h->d_stage, h->d_stage_cap, bytes));
    CK(grow_pinned(h->h_stage, h->h_stage_cap, bytes));
    const int threads = 256, total = n * REC_CHUNKS;
    export_kernel<<<(total + threads - 1) / threads, threads, 0, h->stream>>>(h->d_nodes, first, n, (uint4*)h->d_stage);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(h->h_stage, h->d_stage, bytes, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    memcpy(out, h->h_stage, bytes);
    return NHD_OK;
}

extern "C" int32_t nhd_snapshot(nhd_handle* h)
{
    if (!h || !h->loaded) return NHD_ERR_STATE;
    CK(cudaSetDevice(h->params.device));
    CK(cudaMemcpyAsync(h->d_snapshot, h->d_nodes, h->nodes_bytes, cudaMemcpyDeviceToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->have_snapshot = true;
    return NHD_OK;
}

extern "C" int32_t nhd_restore(nhd_handle* h)
{
    if (!h || !h->loaded || !h->have_snapshot) return NHD_ERR_STATE;
    CK(cudaSetDevice(h->params.device));
    CK(cudaMemcpyAsync(h->d_nodes, h->d_snapshot, h->nodes_bytes, cudaMemcpyDeviceToDevice, h->stream));
    return NHD_OK;
}

/* ------------------------------------------------------------------ batch: stage / solve / fetch */

extern "C" int32_t nhd_sync(nhd_handle* h);

struct PodKey {
    nhd_pod p;
    bool operator==(const PodKey& o) const { return memcmp(&p, &o.p, sizeof(nhd_pod)) == 0; }
};
struct PodKeyHash {
    size_t operator()(const PodKey& k) const
    {
        const uint64_t* w = reinterpret_cast<const uint64_t*>(&k.p);
        uint64_t h = 0x9E3779B97F4A7C15ULL;
        for (size_t i = 0; i < sizeof(nhd_pod) / 8; i++) { h ^= w[i]; h *= 0xff51afd7ed558ccdULL; h ^= h >> 29; }
        return (size_t)h;
    }
};

/* normalise a descriptor so that equal requests compare equal bytewise */
static nhd_pod canonical_pod(const nhd_pod& in)
{
    nhd_pod p;
    memset(&p, 0, sizeof(p));
    p.n_groups = in.n_groups; p.map_type = in.map_type; p.n_misc = in.n_misc;
    p.flags = in.flags & NHD_POD_MISC_SMT;
    p.hugepages_gb = in.hugepages_gb; p.group_mask = in.group_mask;
    for (int g = 0; g < in.n_groups && g < NHD_MAX_GROUPS; g++) {
        nhd_pod_group& o = p.groups[g];
        const nhd_pod_group& i = in.groups[g];
        o.n_gpus = i.n_gpus; o.n_proc = i.n_proc; o.n_helpers = i.n_helpers;
        o.flags = i.flags & (NHD_GRP_PROC_SMT | NHD_GRP_HELPER_SMT | NHD_GRP_HAS_NIC_CORES);
        for (int j = 0; j < i.n_gpus && j < NHD_MAX_GROUP_GPUS; j++) o.gpu_feeders[j] = i.gpu_feeders[j];
        o.rx_gbps = i.rx_gbps + 0.0; o.tx_gbps = i.tx_gbps + 0.0;     /* -0.0 -> +0.0 */
    }
    return p;
}

/* The checks every call that takes a batch of pods runs (nhd_stage_batch, nhd_explain): the arguments and the call
 * order first, then each pod in order — its descriptor, its clock, the tuple limits of the loaded cluster. */
static int32_t check_batch_args(nhd_handle* h, int32_t n_pods, const nhd_pod* pods, const double* now, const char* fn)
{
    if (!h || n_pods < 0 || (n_pods > 0 && (!pods || !now))) return NHD_ERR_INVALID;
    if (!h->loaded) return fail(h, NHD_ERR_STATE, "%s before nhd_load_nodes", fn);
    return NHD_OK;
}

static int32_t check_pod_clock(nhd_handle* h, int i, double now)
{
    if (!std::isfinite(now)) return fail(h, NHD_ERR_INVALID, "pod %d: non-finite clock", i);
    return NHD_OK;
}

static int32_t check_pod(nhd_handle* h, int i, const nhd_pod& pod, double now)
{
    int32_t v = nhd_validate_pod(&pod);
    if (v != NHD_OK) return fail(h, v, "pod %d: descriptor rejected by nhd_validate_pod", i);
    v = check_pod_clock(h, i, now);
    if (v != NHD_OK) return v;
    if (!tuple_limits_ok(h->max_numa, pod.n_groups))
        return fail(h, NHD_ERR_UNSUPPORTED, "pod %d: %d groups on %d-NUMA nodes exceeds the tuple limits", i,
                    (int)pod.n_groups, h->max_numa);
    return NHD_OK;
}

extern "C" int32_t nhd_stage_batch(nhd_handle* h, int32_t n_pods, const nhd_pod* pods, const double* now)
{
    {
        const int32_t v = check_batch_args(h, n_pods, pods, now, "nhd_stage_batch");
        if (v != NHD_OK) return v;
    }
    CK(cudaSetDevice(h->params.device));
    h->staged = h->solved = false;

    /* node-group gate (NHDScheduler.py:235-247): one distinct pod group list -> folded into the pod
     * types; several -> types are group-agnostic and the sweep applies per-name node bitmaps */
    bool multi_group = false;
    uint64_t names_used = 0;
    for (int i = 0; i < n_pods; i++) {
        names_used |= pods[i].group_mask;
        if (pods[i].group_mask != pods[0].group_mask) multi_group = true;
    }
    h->n_names = 0;
    h->names_used = 0;
    if (multi_group) {
        h->names_used = names_used;
        h->n_names = __builtin_popcountll(names_used);
    }
    /* pod types = distinct descriptors (the reference re-derives everything per pod) */
    std::unordered_map<PodKey, int32_t, PodKeyHash> index;
    index.reserve(64);
    std::vector<PodType> types;
    h->pod_type_host.resize(n_pods);
    /* pending sets repeat a few descriptors thousands of times: a descriptor seen before (byte for byte) skips
     * validation, normalisation and the map */
    struct RawSlot { uint64_t hash; int32_t type; nhd_pod raw; };
    static thread_local std::vector<RawSlot> raw_cache;
    raw_cache.assign(256, RawSlot{0, -1, {}});
    for (int i = 0; i < n_pods; i++) {
        uint64_t rh = 0x9E3779B97F4A7C15ULL;
        {
            const uint64_t* w = reinterpret_cast<const uint64_t*>(&pods[i]);
            for (size_t q = 0; q < sizeof(nhd_pod) / 8; q++) { rh ^= w[q]; rh *= 0xff51afd7ed558ccdULL; rh ^= rh >> 29; }
        }
        RawSlot& rs = raw_cache[rh & 255];
        if (rs.type >= 0 && rs.hash == rh && memcmp(&rs.raw, &pods[i], sizeof(nhd_pod)) == 0) {
            const int32_t v = check_pod_clock(h, i, now[i]);
            if (v != NHD_OK) return v;
            h->pod_type_host[i] = rs.type;
            continue;
        }
        const int32_t v = check_pod(h, i, pods[i], now[i]);
        if (v != NHD_OK) return v;
        PodKey k{canonical_pod(pods[i])};
        if (multi_group) k.p.group_mask = ~0ULL;
        auto it = index.find(k);
        if (it == index.end()) {
            PodType t;
            memset(&t, 0, sizeof(t));
            make_pod_type(k.p, t);
            it = index.emplace(k, (int32_t)types.size()).first;
            types.push_back(t);
        }
        h->pod_type_host[i] = it->second;
        rs.hash = rh; rs.type = it->second; rs.raw = pods[i];
    }
    const int T = (int)types.size();
    const size_t types_bytes = (size_t)T * sizeof(PodType);
    const size_t off_pt = (types_bytes + 15) & ~(size_t)15;
    const size_t off_now = (off_pt + (size_t)n_pods * 4 + 15) & ~(size_t)15;
    const size_t total = off_now + (size_t)n_pods * 8;
    CK(grow_pinned(h->h_batch, h->h_batch_cap, total));
    if (T) memcpy(h->h_batch, types.data(), types_bytes);
    if (n_pods) {
        memcpy(h->h_batch + off_pt, h->pod_type_host.data(), (size_t)n_pods * 4);
        memcpy(h->h_batch + off_now, now, (size_t)n_pods * 8);
    }
    CK(grow_dev(h->d_types, h->types_cap, types_bytes));
    if ((size_t)n_pods > h->pods_cap) {
        cudaFree(h->d_pod_type); cudaFree(h->d_now); cudaFree(h->d_out);
        h->d_pod_type = nullptr; h->d_now = nullptr; h->d_out = nullptr; h->pods_cap = 0;
        CK(cudaMalloc((void**)&h->d_pod_type, (size_t)n_pods * 4));
        CK(cudaMalloc((void**)&h->d_now, (size_t)n_pods * 8));
        CK(cudaMalloc((void**)&h->d_out, ((size_t)n_pods + 8) * sizeof(nhd_binding)));      /* + spare records for check builds */
        h->pods_cap = n_pods;
    }
    CK(grow_dev(h->d_bitmaps, h->bitmaps_cap, (size_t)(T + 2 + h->n_names) * h->words * 8));
    if (multi_group) {
        CK(grow_dev(h->d_pod_groups, h->pod_groups_cap, (size_t)n_pods * 8));
        std::vector<uint64_t> gm(n_pods);
        for (int i = 0; i < n_pods; i++) gm[i] = pods[i].group_mask;
        CK(cudaMemcpyAsync(h->d_pod_groups, gm.data(), (size_t)n_pods * 8, cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    CK(grow_dev(h->d_cursors, h->cursors_cap, (size_t)std::max(T, 1) * 3 * 4));
    if (T) CK(cudaMemcpyAsync(h->d_types, h->h_batch, types_bytes, cudaMemcpyHostToDevice, h->stream));
    if (n_pods) {
        CK(cudaMemcpyAsync(h->d_pod_type, h->h_batch + off_pt, (size_t)n_pods * 4, cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(h->d_now, h->h_batch + off_now, (size_t)n_pods * 8, cudaMemcpyHostToDevice, h->stream));
    }
    h->n_pods = n_pods;
    h->n_types = T;
    h->now0 = n_pods ? now[0] : 0.0;
    h->const_clock = true;
    for (int i = 1; i < n_pods; i++) if (now[i] != now[0]) { h->const_clock = false; break; }
    h->staged = true;
    return NHD_OK;
}

static int32_t solve_staged(nhd_handle* h, bool filter_only);
extern "C" int32_t nhd_solve_staged(nhd_handle* h) { return solve_staged(h, false); }
extern "C" int32_t nhd_run_filter_only(nhd_handle* h)
{
    int32_t r = solve_staged(h, true);
    if (r != NHD_OK) return r;
    return nhd_sync(h);
}

static int32_t solve_staged(nhd_handle* h, bool filter_only)
{
    if (!h) return NHD_ERR_INVALID;
    if (!h->staged) return fail(h, NHD_ERR_STATE, "nhd_solve_staged without a staged batch");
    CK(cudaSetDevice(h->params.device));
    const int T = h->n_types, W = h->words;
    int launches = 0;
    CK(cudaEventRecord(h->ev[0], h->stream));

    /* 1. snapshot predicate kernel over this rank's node shard.  With several ranks every rank filters the nodes
     * of S consecutive super-tiles into its slot of an exchange buffer (their NodeDyn summaries, then their
     * columns of every bitmap row); one all-gather hands every rank all slots, and a small kernel lays them out
     * as the arrays the (replicated) sweep reads.  Clusters too small for that to pay (nhd_shard_min_pairs) are
     * filtered whole by every rank, without any exchange. */
    const int ws = h->params.world_size, rk = h->params.rank;
    const int rows = T + 2 + h->n_names;
    const size_t bm_bytes = (size_t)rows * W * 8;
    const bool sharded = ws > 1 && h->n_pods > 0 && (long long)h->n_nodes * T >= h->shard_min_pairs;
    const int S = sharded ? (h->n_super + ws - 1) / ws : h->n_super;
    const int super_lo = sharded ? std::min(rk * S, h->n_super) : 0;
    const int super_hi = sharded ? std::min(super_lo + S, h->n_super) : h->n_super;
    const size_t slot_bytes = (size_t)S * 32 * (SUPER_NODES + rows);
    if (sharded) CK(grow_dev(h->d_xchg, h->xchg_cap, slot_bytes * ws));
    const bool have_ftab = T > 0 && T <= FAST_MAX_TYPES;
    if (h->n_pods > 0 && have_ftab) {
        /* 0. the direct-path tables of this batch's pod types (filter and sweep both read them) */
        TablesArgs ta;
        ta.types = h->d_types; ta.n_types = T; ta.sigs = h->d_sigs; ta.out = h->d_ftab;
        memcpy(ta.cap, h->cap, sizeof(ta.cap));
        fast_tables_kernel<<<dim3(T, FAST_NSIG * 16 / 256), 256, 0, h->stream>>>(ta);
        CK(cudaGetLastError());
        launches++;
    }
    if (h->n_pods > 0 && super_hi > super_lo) {
        FilterArgs fa;
        fa.ftab = have_ftab ? h->d_ftab : nullptr; fa.mapt = h->d_mapt; fa.cls = h->d_cls_fast;
        fa.nodes = h->d_nodes; fa.types = h->d_types; fa.n_types = T; fa.n_nodes = h->n_nodes;
        fa.super_lo = super_lo; fa.super_hi = super_hi;
        if (sharded) {
            uint8_t* slot = h->d_xchg + slot_bytes * rk;
            fa.dyn = reinterpret_cast<uint4*>(slot);
            fa.bitmaps = reinterpret_cast<uint64_t*>(slot + (size_t)S * SUPER_NODES * 32);
            fa.words = S * 4; fa.word_base = super_lo * 4;
        } else {
            fa.dyn = h->d_dyn; fa.bitmaps = h->d_bitmaps; fa.words = W; fa.word_base = 0;
        }
        fa.class_id = h->d_class; fa.names_used = h->names_used;
        fa.now0 = h->now0; fa.min_busy = h->params.min_busy_secs;
        memcpy(fa.cap, h->cap, sizeof(fa.cap));
        /* few super-tiles (small cluster, or a rank's shard): deal the pod types over several CTAs per super-tile */
        const int n_sh = super_hi - super_lo;
        fa.type_split = std::max(1, std::min(T, (h->sm_count * 2) / n_sh));
        const int grid = std::min(n_sh, h->sm_count * 2) * fa.type_split;
        const size_t smem = FILTER_STAGES * SUPER_BYTES + (T <= TYPES_SMEM_MAX ? (size_t)T * sizeof(PodType) : 0);
        filter_kernel<<<grid, FILTER_THREADS, smem, h->stream>>>(fa);
        CK(cudaGetLastError());
        launches++;
    }
    CK(cudaEventRecord(h->ev[1], h->stream));

    /* 2. one collective per batch: every rank contributes its slot */
    if (sharded) {
        ncclResult_t_ r = g_nccl.AllGather(h->d_xchg + slot_bytes * rk, h->d_xchg, slot_bytes, NCCL_INT8, h->comm, h->stream);
        if (r != 0) return fail(h, NHD_ERR_NCCL, "ncclAllGather: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?");
        const size_t n16 = slot_bytes / 16 * ws;
        unpack_slots_kernel<<<(unsigned)((n16 + 255) / 256), 256, 0, h->stream>>>(reinterpret_cast<const uint4*>(h->d_xchg), ws, S, h->n_super,
                                                                              rows, W, h->d_dyn, h->d_bitmaps);
        CK(cudaGetLastError());
        launches += 2;
    }
    CK(cudaEventRecord(h->ev[2], h->stream));

    /* 3. sequential select + assign sweep (replicated on every rank) */
    if (h->n_pods > 0 && !filter_only) {
        SweepArgs sa;
        sa.nodes = h->d_nodes; sa.types = h->d_types; sa.pod_type = h->d_pod_type; sa.now = h->d_now; sa.out = h->d_out;
        sa.n_pods = h->n_pods; sa.n_types = T; sa.n_nodes = h->n_nodes; sa.words = W;
        sa.n_names = h->n_names; sa.names_used = h->names_used; sa.pod_groups = h->d_pod_groups;
        /* reserved_ (test knobs; every setting gives the same bindings): low byte 0 = default, 1 = the general one-warp
         * sweep only (no standing decisions), 2 = standing decisions but never the two pod classes side by side;
         * bits 8.. = debug switches of sweep_kernel */
        sa.dual = (h->const_clock && (h->params.reserved_ & 0xFF) != 1) ? 1 : 0;
        sa.sweep_flags = ((h->params.reserved_ & 0xFF) == 2 ? 1 : 0) | ((h->params.reserved_ >> 8) << 8);
        sa.bitmaps = h->d_bitmaps; sa.dyn = h->d_dyn; sa.cursors = h->d_cursors; sa.busy_list = h->d_busy_list;
        sa.memo = h->d_memo; sa.prof = h->d_prof; sa.pend_pod = h->d_pend;
        sa.mapt = h->d_mapt; sa.mapt2 = h->d_mapt2; sa.sigs = h->d_sigs; sa.cls_fast = h->d_cls_fast;
        sa.ftab = (T > 0 && T <= FAST_MAX_TYPES) ? h->d_ftab : nullptr;
        sa.min_busy = h->params.min_busy_secs;
        memcpy(sa.cap, h->cap, sizeof(sa.cap));
        /* shared memory: memo front | pod types | cursors | (bitmaps when they fit) */
        size_t smem = (size_t)SMEMO_SLOTS * 16 + (size_t)DMEMO_SLOTS * 48 + (size_t)DCACHE_SLOTS * 36 + 16 +
                      (size_t)CLSNIC_SLOTS * 48 + (size_t)SPMEMO_SLOTS * 16;
        if (T <= SWEEP_TYPES_SMEM_MAX) smem += (((size_t)T * sizeof(PodType) + 15) & ~(size_t)15) + (size_t)T * 256;
        smem += (((size_t)T * 3 * 4 + 15) & ~(size_t)15) + (size_t)W * 8;
        if (T <= FAST_MAX_TYPES)                /* standing decisions + their tables */
            smem += ftab_small_bytes(T) + (size_t)T * FAST_NSIG_SMEM * 128 + ((MAPT_BYTES + 15) & ~15) +
                    (((size_t)(T + 2) * 4 + 15) & ~(size_t)15);
        const size_t with_bitmaps = smem + bm_bytes;
        /* a second CTA takes the GPU pods when the two pod classes cannot meet (decided on the device, see sweep_kernel) */
        const int sweep_ctas = sa.dual ? 2 : 1;
        if (with_bitmaps <= (size_t)h->smem_optin) {
            sweep_kernel<true><<<sweep_ctas, SWEEP_THREADS, with_bitmaps, h->stream>>>(sa);
        } else {
            sweep_kernel<false><<<sweep_ctas, SWEEP_THREADS, smem, h->stream>>>(sa);
        }
        CK(cudaGetLastError());
        FinishArgs fin;
        fin.nodes = h->d_nodes; fin.types = h->d_types; fin.pod_type = h->d_pod_type; fin.out = h->d_out;
        fin.dyn = h->d_dyn; fin.n_pods = h->n_pods;
        const int fthreads = 128, fgrid = (h->n_pods + fthreads - 1) / fthreads;
        resolve_kernel<<<(h->n_pods + 63) / 64, 64, 0, h->stream>>>(sa);
        CK(cudaGetLastError());
        assign_cores_kernel<<<fgrid, fthreads, 0, h->stream>>>(fin);
        CK(cudaGetLastError());
        commit_kernel<<<fgrid, fthreads, 0, h->stream>>>(fin);
        CK(cudaGetLastError());
        launches += 4;
    }
    CK(cudaEventRecord(h->ev[3], h->stream));
    h->timing.n_launches = launches;
    h->timing.n_types = T;
    h->solved = true;
    return NHD_OK;
}

extern "C" int32_t nhd_fetch_bindings(nhd_handle* h, nhd_binding* out)
{
    if (!h) return NHD_ERR_INVALID;
    if (!h->solved) return fail(h, NHD_ERR_STATE, "nhd_fetch_bindings without a solved batch");
    CK(cudaSetDevice(h->params.device));
    const size_t bytes = (size_t)h->n_pods * sizeof(nhd_binding);
    bool direct = false;
    if (bytes) {
        if (!out) return NHD_ERR_INVALID;
        direct = is_pinned_host(out);
        if (!direct) CK(grow_pinned(h->h_out, h->h_out_cap, bytes));
        CK(cudaMemcpyAsync(direct ? (void*)out : (void*)h->h_out, h->d_out, bytes, cudaMemcpyDeviceToHost, h->stream));
    }
    CK(cudaStreamSynchronize(h->stream));
    if (bytes && !direct) memcpy(out, h->h_out, bytes);
    cudaEventElapsedTime(&h->timing.filter_ms, h->ev[0], h->ev[1]);
    cudaEventElapsedTime(&h->timing.exchange_ms, h->ev[1], h->ev[2]);
    cudaEventElapsedTime(&h->timing.sweep_ms, h->ev[2], h->ev[3]);
    cudaEventElapsedTime(&h->timing.total_ms, h->ev[0], h->ev[3]);
    return NHD_OK;
}

extern "C" int32_t nhd_sync(nhd_handle* h)
{
    if (!h) return NHD_ERR_INVALID;
    CK(cudaSetDevice(h->params.device));
    CK(cudaStreamSynchronize(h->stream));
    if (h->solved) {
        cudaEventElapsedTime(&h->timing.filter_ms, h->ev[0], h->ev[1]);
        cudaEventElapsedTime(&h->timing.exchange_ms, h->ev[1], h->ev[2]);
        cudaEventElapsedTime(&h->timing.sweep_ms, h->ev[2], h->ev[3]);
        cudaEventElapsedTime(&h->timing.total_ms, h->ev[0], h->ev[3]);
    }
    return NHD_OK;
}

extern "C" int32_t nhd_solve_batch(nhd_handle* h, int32_t n_pods, const nhd_pod* pods, const double* now, nhd_binding* out)
{
    int32_t r = nhd_stage_batch(h, n_pods, pods, now);
    if (r != NHD_OK) return r;
    r = nhd_solve_staged(h);
    if (r != NHD_OK) return r;
    return nhd_fetch_bindings(h, out);
}

extern "C" int32_t nhd_last_timing(const nhd_handle* h, nhd_timing* out)
{
    if (!h || !out) return NHD_ERR_INVALID;
    *out = h->timing;
    return NHD_OK;
}

extern "C" int32_t nhd_read_filter(nhd_handle* h, int32_t* n_types, int32_t* words_per_type, uint64_t* words,
                                   int64_t capacity_words, int32_t* pod_type, int32_t n_pods)
{
    if (!h || !h->solved) return NHD_ERR_STATE;
    CK(cudaSetDevice(h->params.device));
    if (n_types) *n_types = h->n_types;
    if (words_per_type) *words_per_type = h->words;
    const int64_t need = (int64_t)(h->n_types + 2) * h->words;   /* group-name bitmaps are not exported */
    if (words) {
        if (capacity_words < need) return NHD_ERR_INVALID;
        CK(cudaMemcpyAsync(words, h->d_bitmaps, (size_t)need * 8, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    if (pod_type) {
        if (n_pods < h->n_pods) return NHD_ERR_INVALID;
        memcpy(pod_type, h->pod_type_host.data(), (size_t)h->n_pods * 4);
    }
    return NHD_OK;
}

/* ------------------------------------------------------------------ explanation */

/* Explain types: pods with the same canonical descriptor, group mask and clock get the same answer.  Unlike a batch
 * with several group lists, the group gate is always part of the type (it is the first reason a node can have). */
struct ExplainKey {
    nhd_pod p;
    double now;
    bool operator==(const ExplainKey& o) const { return memcmp(this, &o, sizeof(ExplainKey)) == 0; }
};
struct ExplainKeyHash {
    size_t operator()(const ExplainKey& k) const
    {
        uint64_t x;
        memcpy(&x, &k.now, 8);
        return PodKeyHash()(PodKey{k.p}) ^ (x * 0x9E3779B97F4A7C15ULL);
    }
};

extern "C" int32_t nhd_explain(nhd_handle* h, int32_t n_pods, const nhd_pod* pods, const double* now,
                               int32_t* counts, int32_t* first_fit, uint8_t* reasons)
{
    {
        const int32_t v = check_batch_args(h, n_pods, pods, now, "nhd_explain");
        if (v != NHD_OK) return v;
    }
    if (n_pods > 0 && !counts) return NHD_ERR_INVALID;
    CK(cudaSetDevice(h->params.device));
    std::unordered_map<ExplainKey, int32_t, ExplainKeyHash> index;
    std::vector<PodType> types;
    std::vector<double> tnow;
    std::vector<int32_t> pod_type((size_t)n_pods);
    for (int i = 0; i < n_pods; i++) {
        const int32_t v = check_pod(h, i, pods[i], now[i]);
        if (v != NHD_OK) return v;
        ExplainKey k;
        memset(&k, 0, sizeof(k));
        k.p = canonical_pod(pods[i]);
        k.now = now[i] + 0.0;                                    /* -0.0 -> +0.0 */
        auto it = index.find(k);
        if (it == index.end()) {
            PodType t;
            memset(&t, 0, sizeof(t));
            make_pod_type(k.p, t);
            it = index.emplace(k, (int32_t)types.size()).first;
            types.push_back(t);
            tnow.push_back(k.now);
        }
        pod_type[i] = it->second;
    }
    const int T = (int)types.size(), N = h->n_nodes;
    if (T == 0) return NHD_OK;
    std::vector<int32_t> out((size_t)T * (NHD_WHY_COUNT + 2));
    std::vector<uint8_t> why;
    if (N > 0) {
        const size_t out_bytes = out.size() * 4;
        CK(grow_dev(h->d_x_types, h->x_types_cap, (size_t)T * sizeof(PodType)));
        CK(grow_dev(h->d_x_now, h->x_now_cap, (size_t)T * 8));
        CK(grow_dev(h->d_x_out, h->x_out_cap, out_bytes));
        if (reasons) CK(grow_dev(h->d_x_reasons, h->x_reasons_cap, (size_t)T * N));
        int32_t* d_counts = h->d_x_out;
        int32_t* d_first = h->d_x_out + (size_t)T * NHD_WHY_COUNT;
        CK(cudaMemcpyAsync(h->d_x_types, types.data(), (size_t)T * sizeof(PodType), cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(h->d_x_now, tnow.data(), (size_t)T * 8, cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemsetAsync(d_counts, 0, (size_t)T * NHD_WHY_COUNT * 4, h->stream));
        CK(cudaMemsetAsync(d_first, 0x7F, (size_t)T * 2 * 4, h->stream));     /* 0x7F7F7F7F > any node: none yet */
        ExplainArgs xa;
        xa.nodes = h->d_nodes; xa.types = h->d_x_types; xa.now = h->d_x_now;
        xa.n_types = T; xa.n_nodes = N;
        xa.counts = d_counts; xa.first = d_first;
        xa.reasons = reasons ? h->d_x_reasons : nullptr;
        xa.min_busy = h->params.min_busy_secs;
        memcpy(xa.cap, h->cap, sizeof(xa.cap));
        for (int t0 = 0; t0 < T; t0 += 65535) {                  /* gridDim.y limit */
            ExplainArgs xc = xa;
            xc.types += t0; xc.now += t0; xc.counts += (size_t)t0 * NHD_WHY_COUNT; xc.first += (size_t)t0 * 2;
            if (xc.reasons) xc.reasons += (size_t)t0 * N;
            xc.n_types = std::min(T - t0, 65535);
            explain_kernel<<<dim3((N + EXPLAIN_THREADS - 1) / EXPLAIN_THREADS, xc.n_types), EXPLAIN_THREADS, 0, h->stream>>>(xc);
            CK(cudaGetLastError());
        }
        CK(cudaMemcpyAsync(out.data(), h->d_x_out, out_bytes, cudaMemcpyDeviceToHost, h->stream));
        if (reasons) {
            why.resize((size_t)T * N);
            CK(cudaMemcpyAsync(why.data(), h->d_x_reasons, why.size(), cudaMemcpyDeviceToHost, h->stream));
        }
    }
    CK(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < n_pods; i++) {
        const int t = pod_type[i];
        memcpy(counts + (size_t)i * NHD_WHY_COUNT, &out[(size_t)t * NHD_WHY_COUNT], NHD_WHY_COUNT * 4);
        if (first_fit) {
            /* Matcher.SelectNode (Matcher.py:412-420): a pod without GPUs prefers the first node without GPUs */
            const int32_t any = out[(size_t)T * NHD_WHY_COUNT + 2 * t], nogpu = out[(size_t)T * NHD_WHY_COUNT + 2 * t + 1];
            const int32_t pick = (!types[t].needs_gpu && nogpu < N) ? nogpu : any;
            first_fit[i] = (N > 0 && pick < N) ? pick : -1;
        }
        if (reasons && N > 0) memcpy(reasons + (size_t)i * N, &why[(size_t)t * N], (size_t)N);
    }
    return NHD_OK;
}

/* debug: 16 cycle accumulators + 16 counters of the last sweep (only filled by NHD_PROFILE builds) */
extern "C" int32_t nhd_debug_counters(nhd_handle* h, uint64_t* out32)
{
    if (!h || !out32) return NHD_ERR_INVALID;
#ifdef NHD_CHECKS
    cudaStreamSynchronize(h->stream);
    memcpy(out32, h->d_prof, 64 * 8);
    memset(h->d_prof, 0, 64 * 8);
    return NHD_OK;
#endif
    CK(cudaSetDevice(h->params.device));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(out32, h->d_prof, 64 * 8, cudaMemcpyDeviceToHost));
    CK(cudaMemset(h->d_prof, 0, 64 * 8));
    return NHD_OK;
}

/* Page-locked host memory for records / pods / bindings: buffers from here are copied to and
 * from the device without an intermediate staging copy. */
extern "C" int32_t nhd_alloc_pinned(uint64_t bytes, void** out)
{
    if (!out) return NHD_ERR_INVALID;
    *out = nullptr;
    return cudaMallocHost(out, bytes ? bytes : 1) == cudaSuccess ? NHD_OK : NHD_ERR_CUDA;
}

extern "C" int32_t nhd_free_pinned(void* p)
{
    if (!p) return NHD_OK;
    return cudaFreeHost(p) == cudaSuccess ? NHD_OK : NHD_ERR_CUDA;
}
