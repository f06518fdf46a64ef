/*
 * nhd_kernels.cuh — sm_100a kernels of the NHD placement solver (one batch = 5 launches).
 *
 *   ingest / validate / classify / export   layout conversion of uploaded wire records, device-side
 *                   record validation, exact hardware-class ids of the nodes' static descriptions
 *   filter_kernel   snapshot predicate: F[type][node] bitmaps, NOGPU / BUSY / per-group-name bitmaps
 *                   and the 32-byte NodeDyn summaries.  Node tiles are staged into shared memory
 *                   with 1-D TMA bulk copies (cp.async.bulk + mbarrier, double buffered); one
 *                   thread per node, warp ballots produce the bitmap words.  Replaces the per-node
 *                   loops of Matcher.FilterPodResources / FilterNumaTopology / IntersectResources
 *                   (nhd/Matcher.py:65-391) and NHDScheduler.InitialNodeFilter
 *                   (nhd/NHDScheduler.py:235-247).
 *   sweep_kernel    the sequential part (1 CTA, one or two sweeping warps): for every pod in order,
 *                   first fit over the bitmaps, live re-validation on the node's summary, NUMA
 *                   mapping choice (CPython set order), GPU / NIC / hugepage / busy bookkeeping and
 *                   the binding header.  Replaces Matcher.SelectNode / GetNumaGroupIdx
 *                   (nhd/Matcher.py:393-452), everything of Node.SetPhysicalIdsFromMapping but the
 *                   core ids (nhd/Node.py:663-841) and the SetBusy / ClaimPodNICResources calls of
 *                   NHDScheduler.AttemptScheduling (nhd/NHDScheduler.py:289,302-304).
 *   resolve_kernel  pods the sweep bound to an untouched node without working out the mapping
 *   assign_cores_kernel   Node.GetFreeCpuBatch (nhd/Node.py:502-519) for every placed pod, in
 *                   parallel, from the snapshot core masks and per-socket prefix offsets
 *   commit_kernel   folds the batch into the node records
 *
 * Device layout of the node array ("tiled AoSoA"): tiles of 32 nodes, 4 KB each:
 *     byte offset(node n, 16-byte chunk c) = (n / 32) * 4096 + c * 512 + (n % 32) * 16
 * so a warp reading chunk c of 32 consecutive nodes touches 512 contiguous bytes both in
 * global memory (coalesced, TMA-friendly) and in shared memory (bank-conflict free).
 * DESIGN.md section 4 explains why the sweep is exact.
 */
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "nhd_core.cuh"

namespace nhd {

constexpr int TILE_NODES = 32;
constexpr int TILE_BYTES = 4096;
constexpr int REC_CHUNKS = 8;
constexpr int SUPER_TILES = 8;                       /* tiles per CTA stage */
constexpr int SUPER_NODES = TILE_NODES * SUPER_TILES;  /* 256 */
constexpr int SUPER_BYTES = TILE_BYTES * SUPER_TILES;  /* 32 KB */
constexpr int FILTER_THREADS = SUPER_NODES;
constexpr int FILTER_STAGES = 2;
constexpr int TYPES_SMEM_MAX = 128;                  /* pod types cached in shared memory */

constexpr int MEMO_SLOTS = 1 << 16;

union RecU {
    nhd_node_rec r;
    uint4 q[REC_CHUNKS];
    __device__ RecU() {}
};

__device__ __forceinline__ size_t chunk_off(int node, int c)
{
    return (size_t)(node >> 5) * TILE_BYTES + (size_t)c * 512 + (size_t)(node & 31) * 16;
}

__device__ __forceinline__ void load_rec(const uint8_t* nodes, int node, RecU& u)
{
#pragma unroll
    for (int c = 0; c < REC_CHUNKS; c++)
        u.q[c] = *reinterpret_cast<const uint4*>(nodes + chunk_off(node, c));
}

/* only chunks 0-3 hold mutable state (used mask, gpu/nic/hugepage words, busy_time) */
__device__ __forceinline__ void store_rec_mutable(uint8_t* nodes, int node, const RecU& u)
{
#pragma unroll
    for (int c = 0; c < 4; c++)
        *reinterpret_cast<uint4*>(nodes + chunk_off(node, c)) = u.q[c];
}

/* ------------------------------------------------------------------ layout conversion */

__global__ void ingest_kernel(const uint4* __restrict__ aos, const int32_t* __restrict__ idx, int n,
                              uint8_t* __restrict__ tiled)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;          /* one thread per (record, chunk) */
    if (i >= n * REC_CHUNKS) return;
    int rec = i >> 3, c = i & 7;
    int node = idx ? idx[rec] : rec;
    *reinterpret_cast<uint4*>(tiled + chunk_off(node, c)) = aos[i];
}

/* validation of freshly uploaded AoS records on the device: result[0] = lowest bad record index
 * (INT_MAX if none), result[1] = its error code, result[2] = max n_numa seen */
__global__ void validate_kernel(const nhd_node_rec* __restrict__ aos, int n, int* result)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const nhd_node_rec r = aos[i];
    const int v = validate_node_rec(r);
    if (v != 0) {
        const int prev = atomicMin(&result[0], i);
        if (i < prev) result[1] = v;          /* last writer with the smallest index wins (re-checked on host) */
    } else {
        atomicMax(&result[2], (int)r.n_numa);
    }
}

__global__ void export_kernel(const uint8_t* __restrict__ tiled, int first, int n, uint4* __restrict__ aos)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * REC_CHUNKS) return;
    int rec = i >> 3, c = i & 7;
    aos[i] = *reinterpret_cast<const uint4*>(tiled + chunk_off(first + rec, c));
}

/* ------------------------------------------------------------------ hardware classes */

/*
 * Nodes with the same static hardware description (NUMA count, SMT, GPU / NIC placement,
 * switches, link speeds) get the same small class id, so that decisions can be memoised per
 * (pod type, class, free counts).  Ids are exact: a slot is claimed by 64-bit hash and every
 * node then verifies the full 68-byte key against its slot; a mismatch (hash collision) or a
 * full table just leaves the node without a class (NHD_NO_CLASS), which only bypasses the memo.
 */
constexpr int CLASS_SLOTS = 4096;
constexpr int CLASS_KEY_WORDS = 17;
struct ClassSlot { unsigned long long hash; uint32_t key[CLASS_KEY_WORDS]; uint32_t pad; };

__device__ __forceinline__ unsigned long long static_key(const uint8_t* nodes, int node, uint32_t* key)
{
#pragma unroll
    for (int c = 0; c < 4; c++) {
        const uint4 q = *reinterpret_cast<const uint4*>(nodes + chunk_off(node, 4 + c));
        key[4 * c] = q.x; key[4 * c + 1] = q.y; key[4 * c + 2] = q.z; key[4 * c + 3] = q.w;
    }
    const uint4 c2 = *reinterpret_cast<const uint4*>(nodes + chunk_off(node, 2));
    /* n_gpus, n_nics (bytes 2,3 of word 0), n_numa and the SMT flag (bytes 0,1 of word 3) */
    key[16] = (c2.x >> 16) | ((c2.w & 0xFF) << 16) | (((c2.w >> 8) & NHD_NODE_SMT) << 24);
    unsigned long long h = 0x9E3779B97F4A7C15ULL;
#pragma unroll
    for (int i = 0; i < CLASS_KEY_WORDS; i++) { h ^= key[i]; h *= 0xff51afd7ed558ccdULL; h ^= h >> 29; }
    return h | 1ULL;                                   /* 0 marks an empty slot */
}

__global__ void classify_claim_kernel(const uint8_t* __restrict__ nodes, const int32_t* __restrict__ idx, int n,
                                      ClassSlot* slots, uint16_t* class_id)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int node = idx ? idx[i] : i;
    uint32_t key[CLASS_KEY_WORDS];
    const unsigned long long h = static_key(nodes, node, key);
    uint16_t cid = NHD_NO_CLASS;
    for (int probe = 0; probe < 64; probe++) {
        const int s = (int)((h + (unsigned long long)probe * 0x9E37ULL) & (CLASS_SLOTS - 1));
        const unsigned long long old = atomicCAS(&slots[s].hash, 0ULL, h);
        if (old == 0ULL) {
            for (int w = 0; w < CLASS_KEY_WORDS; w++) slots[s].key[w] = key[w];
            cid = (uint16_t)s;
            break;
        }
        if (old == h) { cid = (uint16_t)s; break; }
    }
    class_id[node] = cid;
}

__global__ void classify_verify_kernel(const uint8_t* __restrict__ nodes, const int32_t* __restrict__ idx, int n,
                                       const ClassSlot* __restrict__ slots, uint16_t* class_id)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int node = idx ? idx[i] : i;
    const uint16_t cid = class_id[node];
    if (cid == NHD_NO_CLASS) return;
    uint32_t key[CLASS_KEY_WORDS];
    static_key(nodes, node, key);
    bool same = true;
    for (int w = 0; w < CLASS_KEY_WORDS; w++) same = same && (slots[cid].key[w] == key[w]);
    if (!same) class_id[node] = NHD_NO_CLASS;
}

/* ------------------------------------------------------------------ direct-path tables */

#define NHD_SLOT_SLOW   0
#define NHD_SLOT_FAST   1
#define NHD_SLOT_DEFER  2
#define NHD_SLOT_NONE   3

#define NHD_PENDING_FAST 101          /* internal binding status: node and packed mapping known, header not formatted yet */

constexpr int FAST_MAX_TYPES = 32;    /* one lane per type */
constexpr int FAST_NSIG = 128;        /* distinct per-NUMA NIC signatures (count + speeds) the tables hold */
constexpr int FAST_NSIG_SMEM = 4;     /* ... of which the first few (ids are handed out in order of appearance) sit in shared memory */
constexpr int MAPT_BYTES = 4096 + 64;

struct ClsFast {             /* per hardware class, 16 bytes */
    uint32_t li0, li1;       /* byte j = index in Node.nics of the j-th NIC of NUMA 0 / 1 */
    uint8_t sig0, sig1;      /* signature ids of the two NUMA nodes */
    uint8_t n0, n1;          /* NICs per NUMA node */
    uint32_t ok;             /* 1: covered by the direct path */
};

struct TyFast {              /* per pod type, 16 bytes */
    uint8_t G, n_misc, misc_smt, nic_groups;
    uint8_t direct;          /* CPU-only, NUMA mode, G <= 2 */
    uint8_t pad_[3];
    int32_t hugepages_gb;
    uint32_t pad2_;
};

struct FastTables {
    const uint8_t* tb;       /* [T][2][2][64] */
    const uint32_t* sub0;    /* [T][FAST_NSIG][16], byte p = tuple p; global memory, read through L1 (filter) */
    const uint32_t* sub0s;   /* [T][FAST_NSIG_SMEM][16]: the rows of the first signatures, in shared memory (sweep) */
    const uint32_t* sub1s;
    const uint32_t* sub1;
    const uint8_t* mapt;     /* MAPT_BYTES */
    const uint16_t* gd;      /* [T][2][4] */
    const TyFast* ty;        /* [T] */
    const ClsFast* cls;      /* global, [CLASS_SLOTS] */
};

/* GetNumaGroupIdx for CPU-only pods on 2-NUMA nodes as a table (every GPU tuple passes the GPU stage):
 * [0, 4096): G = 2, index = CPU mask (8 bits, q = 2p + m) << 4 | NIC mask (4 bits, p); [4096, 4160): G = 1,
 * index = CPU mask (4 bits) << 2 | NIC mask (2 bits).  Value: 0x80 | tuple | misc NUMA << 2, or 0. */
__global__ void mapt_kernel(uint8_t* mapt)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= MAPT_BYTES) return;
    const int G = i < 4096 ? 2 : 1;
    const int j = i < 4096 ? i : i - 4096;
    TMask ma = tm_zero(), mb = tm_zero(), mc = tm_zero();
    ma.w[0] = (1u << (1 << G)) - 1;
    mb.w[0] = G == 2 ? (uint32_t)(j >> 4) : (uint32_t)(j >> 2);
    mc.w[0] = G == 2 ? (uint32_t)(j & 15) : (uint32_t)(j & 3);
    int ps = 0, ms = 0;
    mapt[i] = choose_mapping(2, G, ma, mb, mc, &ps, &ms) ? (uint8_t)(0x80 | ps | (ms << 2)) : (uint8_t)0;
}

/* The same function with the GPU stage as a third input (GPU pods; resolve_kernel): [0, 65536): G = 2, index =
 * GPU mask (4 bits, p) << 12 | CPU mask (8 bits) << 4 | NIC mask (4 bits); [65536, 65792): G = 1, index =
 * GPU mask (2 bits) << 6 | CPU mask (4 bits) << 2 | NIC mask (2 bits).  Same value format.  Once per handle. */
constexpr int MAPT2_BYTES = 65536 + 256;
__global__ void mapt2_kernel(uint8_t* mapt2)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= MAPT2_BYTES) return;
    const int G = i < 65536 ? 2 : 1;
    const int j = i < 65536 ? i : i - 65536;
    TMask ma = tm_zero(), mb = tm_zero(), mc = tm_zero();
    ma.w[0] = G == 2 ? (uint32_t)(j >> 12) : (uint32_t)(j >> 6);
    mb.w[0] = G == 2 ? (uint32_t)((j >> 4) & 0xFF) : (uint32_t)((j >> 2) & 15);
    mc.w[0] = G == 2 ? (uint32_t)(j & 15) : (uint32_t)(j & 3);
    int ps = 0, ms = 0;
    mapt2[i] = choose_mapping(2, G, ma, mb, mc, &ps, &ms) ? (uint8_t)(0x80 | ps | (ms << 2)) : (uint8_t)0;
}

/*
 * Per hardware class (ClassSlot key = the static description of its nodes): the NIC list indices of each NUMA
 * node in NodeNic.idx order and the signature ids (NIC count + speed classes in that order) of the two NUMA
 * nodes.  Runs after classification (load / update); signatures are only ever added.
 */
__global__ void cls_fast_kernel(const ClassSlot* __restrict__ slots, ClsFast* cls, uint32_t* sigs)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= CLASS_SLOTS) return;
    ClsFast cf;
    cf.li0 = cf.li1 = 0; cf.sig0 = cf.sig1 = 0; cf.n0 = cf.n1 = 0; cf.ok = 0;
    if (slots[s].hash != 0ULL) {
        const uint32_t* key = slots[s].key;
        const int n_numa = (int)((key[16] >> 16) & 0xFF);
        const uint32_t m[2] = {key[4], key[5]};
        const unsigned long long sp0 = (unsigned long long)key[12] | ((unsigned long long)key[13] << 32);
        const unsigned long long sp1 = (unsigned long long)key[14] | ((unsigned long long)key[15] << 32);
        const int n0 = popc32(m[0]), n1 = popc32(m[1]);
        bool ok = n_numa == 2 && n0 <= 4 && n1 <= 4;
        uint32_t li[2] = {0, 0};
        uint8_t sg[2] = {0, 0};
        for (int k = 0; k < 2 && ok; k++) {
            uint32_t sv = 0x80000000u | (uint32_t)(k ? n1 : n0);
            int j = 0;
            for (uint32_t f = m[k]; f; f &= f - 1, j++) {
                const int l = ctz32(f);
                li[k] |= (uint32_t)l << (8 * j);
                sv |= (uint32_t)(((l < 16 ? sp0 : sp1) >> (4 * (l & 15))) & 0xF) << (4 + 4 * j);
            }
            int id = -1;
            for (int q = 0; q < FAST_NSIG; q++) {                    /* ids in order of appearance: the common ones are low */
                const uint32_t old = atomicCAS(&sigs[q], 0u, sv);
                if (old == 0u || old == sv) { id = q; break; }
            }
            if (id < 0) ok = false; else sg[k] = (uint8_t)id;
        }
        if (ok) { cf.li0 = li[0]; cf.li1 = li[1]; cf.sig0 = sg[0]; cf.sig1 = sg[1]; cf.n0 = (uint8_t)n0; cf.n1 = (uint8_t)n1; cf.ok = 1; }
    }
    cls[s] = cf;
}

/* byte offsets of the direct-path tables of T pod types inside one buffer (global: fast_tables_kernel writes it,
 * the filter reads it through L1, the sweep copies it to shared memory): TB | SUB0 | SUB1 | GD | TyFast */
__host__ __device__ __forceinline__ size_t ftab_off_tb(int) { return 0; }
__host__ __device__ __forceinline__ size_t ftab_off_gd(int T) { return (size_t)T * 256; }
__host__ __device__ __forceinline__ size_t ftab_off_ty(int T) { return (size_t)T * 272; }
__host__ __device__ __forceinline__ size_t ftab_small_bytes(int T) { return (size_t)T * 288; }       /* TB | GD | TyFast: copied to shared memory */
__host__ __device__ __forceinline__ size_t ftab_off_sub0(int T) { return ftab_small_bytes(T); }
__host__ __device__ __forceinline__ size_t ftab_off_sub1(int T) { return ftab_small_bytes(T) + (size_t)T * FAST_NSIG * 64; }
__host__ __device__ __forceinline__ size_t ftab_bytes(int T) { return ftab_small_bytes(T) + (size_t)T * FAST_NSIG * 128; }

__device__ __noinline__ uint32_t nic_sub_solve(const double* cap, const PodType& t, int S, uint32_t mk, uint32_t inuse,
                                               unsigned long long sp0, unsigned long long sp1);

struct TablesArgs {
    const PodType* types;
    int n_types;
    const uint32_t* sigs;
    uint8_t* out;
    double cap[NHD_MAX_SPEED_CLASSES];
};

/* the direct-path tables of a batch's pod types (one CTA per type, 256 threads): see the comment above */
__global__ void fast_tables_kernel(const TablesArgs a)
{
    const int T = a.n_types, tt = blockIdx.x, i = threadIdx.x;
    if (tt >= T) return;
    const PodType& ty = a.types[tt];
    const bool direct = ty.valid_map && !ty.needs_gpu && !ty.pci && ty.G <= 2;
    {
        /* NIC stage per NUMA node (Matcher.py:242-268): per (type, NIC signature, NICs in use) and tuple p, whether
         * the groups p puts on NUMA 0 (SUB0) / NUMA 1 (SUB1) get NICs there, and which; blockIdx.y walks the signatures */
        const int e = blockIdx.y * 256 + i;                       /* (signature, NICs in use) */
        const int sg = e >> 4, iu = e & 15;
        const uint32_t sv = a.sigs[sg];
        uint32_t w0 = 0, w1 = 0;
        const int n_k = (int)(sv & 15);
        if ((sv >> 31) && direct && iu < (1 << n_k)) {
            const uint32_t mk = (1u << n_k) - 1;
            const unsigned long long sp = (sv >> 4) & 0xFFFFu;
            const int G = ty.G, gmask = (1 << G) - 1;
            for (int p = 0; p <= gmask; p++) {
                const int S1 = (int)(__brev((unsigned)p) >> (32 - G)), S0 = gmask & ~S1;
                const uint32_t r0 = nic_sub_solve(a.cap, ty, S0, mk, (uint32_t)iu, sp, 0ULL);
                const uint32_t r1 = nic_sub_solve(a.cap, ty, S1, mk, (uint32_t)iu, sp, 0ULL);
                w0 |= (((r0 >> 31) << 7) | (r0 & 3) | (((r0 >> 8) & 3) << 2)) << (8 * p);
                w1 |= (((r1 >> 31) << 7) | (r1 & 3) | (((r1 >> 8) & 3) << 2)) << (8 * p);
            }
        }
        reinterpret_cast<uint32_t*>(a.out + ftab_off_sub0(T))[tt * FAST_NSIG * 16 + e] = w0;
        reinterpret_cast<uint32_t*>(a.out + ftab_off_sub1(T))[tt * FAST_NSIG * 16 + e] = w1;
    }
    if (blockIdx.y != 0) return;
    {
        /* CPU stage per socket (Matcher.py:203-212 with K = 2): which tuples q = 2p + m fit c free cores on NUMA k */
        const int f = (i >> 7) & 1, k = (i >> 6) & 1, c = i & 63;
        const uint8_t* cl = f ? ty.cl_smt : ty.cl_nosmt;
        const int L = ty.G + 1;
        uint32_t m = 0;
        for (int q = 0; q < (1 << L) && L <= 3; q++) {
            int n = 0;
            for (int g = 0; g < L; g++) if (((q >> (L - 1 - g)) & 1) == k) n += cl[g];
            if (n <= c || (c == 63 && n <= 255)) m |= 1u << q;       /* the free count saturates at 63 in the index */
        }
        a.out[ftab_off_tb(T) + (size_t)tt * 256 + i] = (uint8_t)m;
    }
    if (i < 8) {
        /* cores the groups of tuple p take from each socket */
        const int f = (i >> 2) & 1, p = i & 3;
        const uint8_t* cl = f ? ty.cl_smt : ty.cl_nosmt;
        int n0 = 0, n1 = 0;
        for (int g = 0; g < ty.G && ty.G <= 2; g++) { if ((p >> (ty.G - 1 - g)) & 1) n1 += cl[g]; else n0 += cl[g]; }
        reinterpret_cast<uint16_t*>(a.out + ftab_off_gd(T))[tt * 8 + i] = (uint16_t)((n0 & 0xFF) | ((n1 & 0xFF) << 8));
    }
    if (i == 0) {
        TyFast f;
        f.G = ty.G; f.n_misc = ty.pod.n_misc; f.misc_smt = (ty.pod.flags & NHD_POD_MISC_SMT) ? 1 : 0; f.nic_groups = ty.nic_groups;
        f.direct = direct ? 1 : 0;
        f.pad_[0] = f.pad_[1] = f.pad_[2] = 0; f.hugepages_gb = ty.pod.hugepages_gb; f.pad2_ = 0;
        reinterpret_cast<TyFast*>(a.out + ftab_off_ty(T))[tt] = f;
    }
}

/* bit 7 of each byte of x -> bits 0..3 */
__device__ __forceinline__ uint32_t gather_b7(uint32_t x)
{
    return ((((x >> 7) & 0x01010101u) * 0x01020408u) >> 24) & 0xFu;
}

/* ------------------------------------------------------------------ TMA / mbarrier helpers */

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
/* 1-D bulk async copy global -> shared, completion counted on an mbarrier (SASS: UBLKCP) */
__device__ __forceinline__ void tma_load_1d(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

/* ------------------------------------------------------------------ snapshot predicate kernel */

struct FilterArgs {
    const uint8_t* nodes;        /* tiled node array, padded to SUPER_NODES */
    const PodType* types;
    int n_types;
    int n_nodes;
    int super_lo, super_hi;      /* super-tiles this launch covers (this rank's shard)        */
    int type_split;              /* CTAs per super-tile: the pod types are dealt over them     */
    int words;                   /* u64 words per bitmap row of the OUTPUT window              */
    int word_base;               /* first u64 word (node / 64) of the output window            */
    uint64_t* bitmaps;           /* [n_types + 2 + n_names][words]: F[0..T), NOGPU, BUSY, one per node-group name in use */
    uint64_t names_used;         /* node-group names some pod of the batch asks for (0: gate folded into the types) */
    uint4* dyn;                  /* [window nodes][2]: NodeDyn summaries; entry 0 = node 64 * word_base */
    const uint16_t* class_id;    /* hardware class of every node */
    const uint8_t* ftab;         /* direct-path tables (fast_tables_kernel) or null */
    const uint8_t* mapt;
    const ClsFast* cls;
    double now0;                 /* clock of the first pod, for the BUSY snapshot */
    double min_busy;
    double cap[NHD_MAX_SPEED_CLASSES];
};

/* The general predicate, out of line and on its own copy of the record: its tuple / search arrays live in local
 * memory, and inlined it would drag the caller's record there as well.  Only shapes outside the register-only form
 * come here (other than 2 NUMA nodes, more than two groups). */
__device__ __noinline__ bool node_feasible_general(const nhd_node_rec r, const PodType* t, const double* cap)
{
    return node_feasible(r, *t, cap);
}

__global__ void __launch_bounds__(FILTER_THREADS, 2)
filter_kernel(const FilterArgs a)
{
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* stage_buf = smem;                                          /* FILTER_STAGES x SUPER_BYTES */
    PodType* s_types = reinterpret_cast<PodType*>(smem + FILTER_STAGES * SUPER_BYTES);
    __shared__ __align__(8) uint64_t full_bar[FILTER_STAGES];
    __shared__ double s_cap[NHD_MAX_SPEED_CLASSES];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid < NHD_MAX_SPEED_CLASSES) s_cap[tid] = a.cap[tid];       /* ordered by the barrier below */
    /* CTA = (position in the walk over the super-tiles, type chunk): with few super-tiles per GPU (small clusters,
     * node-sharded ranks) the pod types are dealt over several CTAs so that the whole machine still works */
    const int TS = a.type_split, tch = (int)blockIdx.x % TS, cta = (int)blockIdx.x / TS, ncta = (int)gridDim.x / TS;
    const int n_my = (a.super_hi - a.super_lo - cta + ncta - 1) / ncta;
    if (n_my <= 0) return;

    if (tid == 0) {
        for (int s = 0; s < FILTER_STAGES; s++) mbar_init(&full_bar[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    auto issue = [&](int it) {                                          /* thread 0 only */
        int st = a.super_lo + cta + it * ncta;
        int s = it % FILTER_STAGES;
        mbar_expect_tx(&full_bar[s], SUPER_BYTES);
        tma_load_1d(stage_buf + s * SUPER_BYTES, a.nodes + (size_t)st * SUPER_BYTES, SUPER_BYTES, &full_bar[s]);
    };
    if (tid == 0)
        for (int it = 0; it < FILTER_STAGES && it < n_my; it++) issue(it);

    /* pod types: small tables are copied to shared memory while the first tile is in flight */
    const bool types_in_smem = a.n_types <= TYPES_SMEM_MAX;
    if (types_in_smem) {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(a.types);
        uint32_t* dst = reinterpret_cast<uint32_t*>(s_types);
        const int nw = a.n_types * (int)(sizeof(PodType) / 4);
        for (int i = tid; i < nw; i += FILTER_THREADS) dst[i] = src[i];
        __syncthreads();
    }
    const PodType* types = types_in_smem ? s_types : a.types;
    uint32_t* out32 = reinterpret_cast<uint32_t*>(a.bitmaps);
    const size_t words32 = (size_t)a.words * 2;

    for (int it = 0; it < n_my; it++) {
        const int s = it % FILTER_STAGES;
        const int st = a.super_lo + cta + it * ncta;
        mbar_wait(&full_bar[s], (it / FILTER_STAGES) & 1);

        RecU u;
        const uint8_t* tile = stage_buf + s * SUPER_BYTES + warp * TILE_BYTES;
#pragma unroll
        for (int c = 0; c < REC_CHUNKS; c++)
            u.q[c] = *reinterpret_cast<const uint4*>(tile + c * 512 + lane * 16);
        __syncthreads();                                                /* stage s fully consumed */
        if (tid == 0 && it + FILTER_STAGES < n_my) issue(it + FILTER_STAGES);

        const int node = st * SUPER_NODES + tid;
        const bool valid = node < a.n_nodes;

        /* per-node summary for the sweep */
        union { NodeDyn d; uint4 q[2]; } du;
        if (valid) { make_dyn(u.r, du.d); du.d.hw_class = a.class_id[node]; }
        else { du.q[0] = make_uint4(0, 0, 0, 0); du.q[1] = du.q[0]; }
        if (tch == 0) {
            const size_t dn = (size_t)node - (size_t)a.word_base * 64;
            a.dyn[dn * 2] = du.q[0];
            a.dyn[dn * 2 + 1] = du.q[1];
        }
        /* direct path (CPU-only NUMA-mode types with <= 2 groups on 2-NUMA nodes whose class the tables cover): the
         * node's part of the table indices, once for all types.  Same tables and the same answer as the sweep's
         * fast_eval: feasible <=> MAPT holds a mapping for (CPU mask, NIC mask) (Matcher.py:203-276, :349) */
        bool shape_ok = false;
        uint32_t d_i0 = 0, d_i1 = 0, d_c0 = 0, d_c1 = 0, d_smt = 0;
        if (valid && a.ftab && u.r.n_numa == 2 && du.d.hw_class != NHD_NO_CLASS) {
            const ClsFast cf = a.cls[du.d.hw_class];
            if (cf.ok) {
                shape_ok = true;
                uint32_t iu0 = 0, iu1 = 0;
                for (int j = 0; j < cf.n0; j++) iu0 |= ((u.r.nic_inuse >> ((cf.li0 >> (8 * j)) & 31)) & 1u) << j;
                for (int j = 0; j < cf.n1; j++) iu1 |= ((u.r.nic_inuse >> ((cf.li1 >> (8 * j)) & 31)) & 1u) << j;
                d_i0 = (uint32_t)cf.sig0 * 16 + iu0; d_i1 = (uint32_t)cf.sig1 * 16 + iu1;
                d_c0 = du.d.fc[0] < 63 ? du.d.fc[0] : 63; d_c1 = du.d.fc[1] < 63 ? du.d.fc[1] : 63;
                d_smt = rec_smt(u.r) ? 1 : 0;
            }
        }
        const int T_ = a.n_types;
        const uint8_t* f_tb = a.ftab;
        const uint32_t* f_sub0 = reinterpret_cast<const uint32_t*>(a.ftab + ftab_off_sub0(T_));
        const uint32_t* f_sub1 = reinterpret_cast<const uint32_t*>(a.ftab + ftab_off_sub1(T_));
        const TyFast* f_ty = reinterpret_cast<const TyFast*>(a.ftab + ftab_off_ty(T_));

        /* every other (type, node) pair of the common shape: the register-only predicate, its node part once */
        const bool k2 = valid && u.r.n_numa == 2;
        Pre2 pre;
        if (k2) make_pre2(u.r, du.d.fc[0], du.d.fc[1], pre);

        const size_t w32 = ((size_t)node >> 5) - (size_t)a.word_base * 2;
        for (int t = tch; t < a.n_types; t += TS) {
            bool f;
            if (shape_ok && f_ty[t].direct) {
                const uint32_t w0 = __ldg(&f_sub0[t * FAST_NSIG * 16 + d_i0]), w1 = __ldg(&f_sub1[t * FAST_NSIG * 16 + d_i1]);
                const uint32_t mC = gather_b7(w0 & w1);
                const uint32_t mB = __ldg(&f_tb[((t * 2 + d_smt) * 2 + 0) * 64 + d_c0]) & __ldg(&f_tb[((t * 2 + d_smt) * 2 + 1) * 64 + d_c1]);
                const uint32_t mi = f_ty[t].G == 2 ? ((mB << 4) | mC) : (4096 + (((mB & 15) << 2) | (mC & 3)));
                f = node_gates(u.r, types[t]) && (__ldg(&a.mapt[mi]) & 0x80) != 0;
            } else if (k2 && types[t].G >= 1 && types[t].G <= 2)
                f = node_feasible_k2(u.r, types[t], s_cap, pre);
            else
                f = valid && node_feasible_general(u.r, &types[t], s_cap);
            uint32_t bal = __ballot_sync(0xFFFFFFFFu, f);
            if (lane == 0) out32[(size_t)t * words32 + w32] = bal;
        }
        if (tch != 0) continue;
        uint32_t nog = __ballot_sync(0xFFFFFFFFu, valid && u.r.n_gpus == 0);
        uint32_t bsy = __ballot_sync(0xFFFFFFFFu, valid && node_busy(u.r, a.now0, a.min_busy));
        if (lane == 0) {
            out32[(size_t)a.n_types * words32 + w32] = nog;
            out32[(size_t)(a.n_types + 1) * words32 + w32] = bsy;
        }
        /* InitialNodeFilter per group name (NHDScheduler.py:241-243): nodes carrying name j */
        int r = 0;
        for (uint64_t g = a.names_used; g; g &= g - 1, r++) {
            const int jn = ctz64(g);
            const uint32_t hasg = __ballot_sync(0xFFFFFFFFu, valid && ((u.r.group_mask >> jn) & 1));
            if (lane == 0) out32[(size_t)(a.n_types + 2 + r) * words32 + w32] = hasg;
        }
    }
}

/*
 * Node-sharded ranks: after the one collective of the batch (an all-gather of every rank's slot: the NodeDyn
 * summaries and the bitmap columns of its nodes) the slots are laid back out as the arrays the sweep reads.
 * Slot q covers super-tiles [q*S, (q+1)*S): S*256 summaries, then rows x S*4 bitmap words.
 */
__global__ void unpack_slots_kernel(const uint4* __restrict__ xchg, int ws, int S, int n_super, int rows, int W,
                                    uint4* __restrict__ dyn, uint64_t* __restrict__ bitmaps)
{
    const size_t slot16 = (size_t)S * 2 * (SUPER_NODES + rows);           /* 16-byte units per slot */
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= slot16 * (size_t)ws) return;
    const int q = (int)(i / slot16);
    const size_t r = i % slot16;
    const int lo = q * S, hi = lo + S < n_super ? lo + S : n_super;
    if (lo >= hi) return;
    const size_t dyn16 = (size_t)S * SUPER_NODES * 2;
    if (r < dyn16) {
        if (r < (size_t)(hi - lo) * SUPER_NODES * 2) dyn[(size_t)lo * SUPER_NODES * 2 + r] = xchg[i];
    } else {
        const size_t b = r - dyn16;                                          /* 16 bytes = two words of one row */
        const int row = (int)(b / ((size_t)S * 2)), k2 = (int)(b % ((size_t)S * 2));
        if (k2 * 2 < (hi - lo) * 4) {
            const uint4 v = xchg[i];
            uint64_t* dst = bitmaps + (size_t)row * W + (size_t)lo * 4 + (size_t)k2 * 2;
            dst[0] = (uint64_t)v.x | ((uint64_t)v.y << 32);
            dst[1] = (uint64_t)v.z | ((uint64_t)v.w << 32);
        }
    }
}

/* ------------------------------------------------------------------ select + assign sweep */

#ifdef NHD_PROFILE
#define PROF_DECL long long prof_t0 = clock64(); long long prof_acc[16] = {0}; long long prof_cnt[16] = {0};
#define PROF_MARK(i) do { long long t_ = clock64(); prof_acc[i] += t_ - prof_t0; prof_cnt[i]++; prof_t0 = t_; } while (0)
#define PROF_COUNT(i) do { prof_cnt[i]++; } while (0)
#define PROF2_DECL long long p2_t0 = clock64();
#define PROF2(i) do { long long t_ = clock64(); if (cx.lane == 0) atomicAdd(&a.prof[16 + (i)], (unsigned long long)(t_ - p2_t0)); p2_t0 = t_; } while (0)
#define PROF_FLUSH(buf) do { if (lane == 0) for (int i_ = 0; i_ < 16; i_++) { (buf)[i_] = (unsigned long long)prof_acc[i_]; (buf)[32 + i_] = (unsigned long long)prof_cnt[i_]; } } while (0)
#define PROF_ADD(i, n) do { const unsigned long long n_ = (unsigned long long)(n); if (cx.lane == 0) atomicAdd(&a.prof[48 + (i)], n_); } while (0)
#define PROFL_DECL long long pl_t0 = clock64();
#define PROFL(i) do { long long t_ = clock64(); atomicAdd(&a.prof[16 + (i)], (unsigned long long)(t_ - pl_t0)); atomicAdd(&a.prof[48 + (i)], 1ULL); pl_t0 = clock64(); } while (0)
#else
#define PROF_ADD(i, n)
#define PROFL_DECL
#define PROFL(i)
#define PROF2_DECL
#define PROF2(i)
#define PROF_DECL
#define PROF_MARK(i)
#define PROF_COUNT(i)
#define PROF_FLUSH(buf)
#endif

#ifdef NHD_CHECKS
/* debugging aid: first directly committed decision the general path disagrees with -> prof[56..63] */
#define CHK_FAIL(code, x0, x1, x2) do { if (lane == 0 && atomicCAS(&a.prof[56], 0ULL, (unsigned long long)(code)) == 0ULL) { \
    a.prof[57] = (unsigned long long)(x0); a.prof[58] = (unsigned long long)(x1); a.prof[59] = (unsigned long long)(x2); a.prof[60] = (unsigned long long)wid; a.prof[61] = (unsigned long long)i; __threadfence_system(); } } while (0)
#define CHK_SANE(du_, node_, where_) do { const int k_ = ((du_).d.info >> 2) & 7; \
    if (k_ < 1 || k_ > 4 || (du_).d.n_nics > 32 || (du_).d.n_gpus > 16 || (node_) < 0 || (node_) >= a.n_nodes) CHK_FAIL(where_, node_, (du_).q[0].z, (du_).q[1].y); } while (0)
#else
#define CHK_FAIL(code, x0, x1, x2)
#define CHK_SANE(du_, node_, where_)
#endif

constexpr int SWEEP_THREADS = 256;
constexpr int SMEMO_SLOTS = 256;                  /* shared-memory front of the mapping memo (16 B)  */
constexpr int DMEMO_SLOTS = 128;                  /* decision memo (48 B entries), generic path only  */
constexpr int SPMEMO_SLOTS = 256;                 /* NIC sub-problem memo (16 B entries)             */

constexpr int DCACHE_SLOTS = 512;                 /* node-summary cache (32 B entries + tag)          */
constexpr int SWEEP_TYPES_SMEM_MAX = 64;

struct SweepArgs {
    uint8_t* nodes;
    const PodType* types;
    const int32_t* pod_type;
    const double* now;
    nhd_binding* out;
    int n_pods, n_types, n_nodes, words;
    int dual;                    /* 1: constant clock -> standing decisions per pod type (see sweep_kernel) */
    int sweep_flags;             /* bit 0: never sweep the two pod classes side by side; bits 8..: debug switches */
    int n_names;                 /* > 0: per-pod node-group masks, one bitmap per name after BUSY */
    uint64_t names_used;
    const uint64_t* pod_groups;  /* [n_pods] when n_names > 0 */
    uint64_t* bitmaps;           /* [n_types + 2][words] */
    uint4* dyn;                  /* NodeDyn summaries */
    int32_t* cursors;            /* global fallback: [n_types][2] */
    int32_t* busy_list;          /* nodes whose BUSY bit is set */
    int32_t* pend_pod;           /* [n_nodes] pod whose resolution is pending on the node */
    uint64_t* memo;              /* MEMO_SLOTS x 2 words (global, persists across batches) */
    const uint8_t* mapt;         /* MAPT_BYTES: GetNumaGroupIdx table of the direct path (mapt_kernel, once per handle) */
    const uint8_t* mapt2;        /* MAPT2_BYTES: the same with the GPU stage (mapt2_kernel); read by resolve_kernel */
    const uint32_t* sigs;        /* FAST_NSIG per-NUMA NIC signatures (cls_fast_kernel, at load / update time) */
    const uint8_t* ftab;         /* direct-path tables of the batch's pod types (fast_tables_kernel), null when T > FAST_MAX_TYPES */
    const struct ClsFast* cls_fast;   /* [CLASS_SLOTS] */
    unsigned long long* prof;    /* debug counters (NHD_PROFILE builds) */
    double min_busy;
    double cap[NHD_MAX_SPEED_CLASSES];
};

/* mapping memo: (K, G, stage-mask ballots) -> (gtuple index, misc NUMA), for K^(G+1) <= 32.
 * The three ballots are indexed by q = p*K + m (A and C use the m == 0 lanes). */
__device__ __forceinline__ uint64_t memo_mix(uint64_t x)
{
    x ^= x >> 33; x *= 0xff51afd7ed558ccdULL; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL; x ^= x >> 33;
    return x;
}

/* miss path of the mapping memo (lane 0): global LUT, else the CPython set emulation; out of line */
__device__ __noinline__ int choose_mapping_slow(uint4* smemo, int ss, uint64_t* gmemo, int K, int G,
                                                uint32_t balA, uint32_t balB, uint32_t balC, uint32_t tag)
{
    const uint64_t h = memo_mix(((uint64_t)balA << 32 | balB) ^ ((uint64_t)balC * 0x9E3779B97F4A7C15ULL) ^ tag);
    /* global memo: key = two words */
    const uint64_t k0 = (uint64_t)balA << 32 | balB, k1tag = ((uint64_t)tag << 32) | balC;
    int free_slot = -1, val = -2;
    for (int probe = 0; probe < 8; probe++) {
        const int s = (int)(((h >> 16) + probe) & (MEMO_SLOTS - 1));
        const ulonglong2 ge = __ldcg(reinterpret_cast<const ulonglong2*>(gmemo) + s);   /* one 16-byte access: two warps share this table */
        const uint64_t g0 = ge.x, g1 = ge.y;
        if (!(g1 >> 63)) { free_slot = s; break; }
        if (g0 == k0 && (g1 & 0xFFFF0000FFFFFFFFULL) == k1tag) { val = (int)((g1 >> 32) & 0xFFFF); break; }
    }
    if (val == -2) {
        TMask ma = tm_zero(), mb = tm_zero(), mc = tm_zero();
        mb.w[0] = balB;
        const int np = ipow(K, G);
        for (int p = 0; p < np; p++) {
            if ((balA >> (p * K)) & 1) tm_set(ma, p);
            if ((balC >> (p * K)) & 1) tm_set(mc, p);
        }
        int ps, ms;
        val = choose_mapping(K, G, ma, mb, mc, &ps, &ms) ? (ps | (ms << 8)) : 0xFFFF;
        if (free_slot >= 0)
            reinterpret_cast<ulonglong2*>(gmemo)[free_slot] = make_ulonglong2(k0, k1tag | ((uint64_t)val << 32));
    }
    smemo[ss] = make_uint4(balA, balB, balC, tag | (uint32_t)val);
    return val == 0xFFFF ? -1 : val;
}

/* lane-0 only.  Returns -1 infeasible, else ps | ms << 8.  The shared-memory hit is inline. */
__device__ __forceinline__ int choose_mapping_memo(uint4* smemo, int smemo_mask, uint64_t* gmemo, int K, int G,
                                                   uint32_t balA, uint32_t balB, uint32_t balC)
{
    const uint32_t tag = 0x80000000u | ((uint32_t)K << 24) | ((uint32_t)G << 16);
    uint32_t h32 = (balB * 0x9E3779B1u) ^ (balC * 0x85EBCA77u) ^ (balA * 0xC2B2AE3Du) ^ tag;
    h32 ^= h32 >> 15;
    const int ss = (int)(h32 & (uint32_t)smemo_mask);
    const uint4 e = smemo[ss];
    if (e.x == balA && e.y == balB && e.z == balC && (e.w & 0xFFFF0000u) == tag) {
        const int v = (int)(e.w & 0xFFFF);
        return v == 0xFFFF ? -1 : v;
    }
    return choose_mapping_slow(smemo, ss, gmemo, K, G, balA, balB, balC, tag);
}

/*
 * Decision memo entry (48 B).  Everything AttemptScheduling decides for (pod type, node) apart
 * from the core ids is a pure function of
 *     pod type, hardware class of the node, which GPUs and NICs are taken, and, per NUMA node,
 *     the largest per-socket demand any NUMA tuple of this type can make that still fits the
 *     free physical cores (the tuple predicates of Matcher.py:204-212 compare the free count
 *     with sums of sub-sets of the type's per-group demands and nothing else),
 * which is exactly the key.  Values are only ever produced by the full evaluation below.
 */
struct DEntry {
    unsigned long long a;        /* type(12) | class(12) | gpu_used(16) | effective fc 4 x 6 */
    uint32_t nic_inuse;
    uint8_t  state;              /* 0 empty, 1 no mapping, 2 placed, 3 assignment fails */
    uint8_t  ms, ncl, ng;
    uint32_t pn, idx, li;        /* per-group NUMA node / per-NUMA NIC index / NIC list index, one byte each */
    uint32_t claimed;            /* claimed NIC list indices in CPython set order */
    uint32_t gi;                 /* first four picked GPU indices */
    uint16_t gpu_used_new;
    uint8_t  fail_status;
    uint8_t  pad_;
    uint32_t pad2_[2];
};
static_assert(sizeof(DEntry) == 48, "DEntry is three 16-byte chunks");

struct PMap { uint32_t pn, idx, li, ms; };      /* a mapping, one byte per group */

__device__ __forceinline__ uint32_t pack_digits(int ps, int K, int G)
{
    uint8_t d[NHD_MAX_GROUPS] = {0, 0, 0, 0};
    tuple_digits(ps, K, G, d);
    return (uint32_t)d[0] | ((uint32_t)d[1] << 8) | ((uint32_t)d[2] << 16) | ((uint32_t)d[3] << 24);
}

/*
 * Full evaluation of (pod type, node) — memo miss path.  All 32 lanes enter with the same
 * arguments; for K^(G+1) <= 32 each lane owns one (G+1)-tuple and the stage masks are warp
 * ballots, otherwise lane 0 enumerates.  Returns feasibility and the mapping (uniform).
 */
__device__ __noinline__ bool evaluate_full(const SweepArgs& a, uint4* smemo, int smemo_mask, const nhd_node_rec& r, const NodeDyn& d,
                              const PodType& t, int lane, PMap& pm)
{
    const int K = r.n_numa, G = t.G;
    const bool smt = rec_smt(r);
    const int nq = ipow(K, G + 1);
    if (nq <= 32) {
        const uint64_t gsw = t.pci ? free_gpus_per_switch(r) : 0;
        int fg[NHD_MAX_NUMA], fc[NHD_MAX_NUMA];
        free_gpus(r, fg);
        for (int k = 0; k < NHD_MAX_NUMA; k++) fc[k] = d.fc[k];
        uint8_t dg[NHD_MAX_GROUPS + 1], idx[NHD_MAX_GROUPS] = {0, 0, 0, 0}, li[NHD_MAX_GROUPS] = {0, 0, 0, 0};
        bool okA = false, okB = false, okC = false;
        if (lane < nq) {
            tuple_digits(lane, K, G + 1, dg);
            const int mm = dg[G];
            okB = cpu_ok(t, dg, mm, K, fc, smt);
            if (mm == 0) {
                okA = gpu_ok(t, dg, K, fg);
                okC = nic_first_fit(r, t, dg, K, a.cap, gsw, idx, li);
            }
        }
        const uint32_t balA = __ballot_sync(0xFFFFFFFFu, okA);
        const uint32_t balB = __ballot_sync(0xFFFFFFFFu, okB);
        const uint32_t balC = __ballot_sync(0xFFFFFFFFu, okC);
        if (!(balA && balB && balC)) return false;
        int v = -1;
        if (lane == 0) v = choose_mapping_memo(smemo, smemo_mask, a.memo, K, G, balA, balB, balC);
        v = __shfl_sync(0xFFFFFFFFu, v, 0);
        if (v < 0) return false;
        const int ps = v & 0xFF;
        uint32_t pk = 0, pl = 0;
        for (int g = 0; g < NHD_MAX_GROUPS; g++) { pk |= (uint32_t)idx[g] << (8 * g); pl |= (uint32_t)li[g] << (8 * g); }
        pm.idx = __shfl_sync(0xFFFFFFFFu, pk, ps * K);
        pm.li = __shfl_sync(0xFFFFFFFFu, pl, ps * K);
        pm.pn = pack_digits(ps, K, G);
        pm.ms = (uint32_t)(v >> 8);
        return true;
    }
    /* large enumerations: scalar on lane 0 */
    uint32_t okl = 0, pk = 0, pl = 0;
    int ps = 0, ms = 0;
    if (lane == 0) {
        const uint64_t gsw = t.pci ? free_gpus_per_switch(r) : 0;
        TMask ma, mb, mc;
        if (stage_masks_fc(r, d.fc, t, a.cap, gsw, ma, mb, mc) && choose_mapping(K, G, ma, mb, mc, &ps, &ms)) {
            uint8_t dg[NHD_MAX_GROUPS], idx[NHD_MAX_GROUPS] = {0, 0, 0, 0}, li[NHD_MAX_GROUPS] = {0, 0, 0, 0};
            tuple_digits(ps, K, G, dg);
            nic_first_fit(r, t, dg, K, a.cap, gsw, idx, li);
            for (int g = 0; g < NHD_MAX_GROUPS; g++) { pk |= (uint32_t)idx[g] << (8 * g); pl |= (uint32_t)li[g] << (8 * g); }
            okl = 1;
        }
    }
    okl = __shfl_sync(0xFFFFFFFFu, okl, 0);
    if (!okl) return false;
    ps = __shfl_sync(0xFFFFFFFFu, ps, 0);
    pm.ms = (uint32_t)__shfl_sync(0xFFFFFFFFu, ms, 0);
    pm.idx = __shfl_sync(0xFFFFFFFFu, pk, 0);
    pm.li = __shfl_sync(0xFFFFFFFFu, pl, 0);
    pm.pn = pack_digits(ps, K, G);
    return true;
}

/* resource part of one decision: GPU picks (Node.py:707-726) and NIC claim order
 * (NHDScheduler.py:302), a pure function of (pod type, mapping, gpu_used, static GPU/NIC layout) */
struct Picks {
    unsigned long long gi_lo, gi_hi;     /* gpu_index[16] */
    uint32_t claimed, gpu_used_new;
    int ng, ncl, fail_status;            /* fail_status: 0 or NHD_ASSIGN_FAILED / NHD_REF_WOULD_CRASH */
};

__device__ __noinline__ void compute_picks(const nhd_node_rec& r, const PodType& t, const PMap& pm, uint32_t gpu_used, int n_gpus, Picks& pk)
{
    const int G = t.G;
    pk.gi_lo = pk.gi_hi = 0; pk.claimed = 0; pk.ng = pk.ncl = 0; pk.fail_status = 0;
    int n_rec = 0;
    uint8_t rec[NHD_MAX_GROUPS] = {0, 0, 0, 0};
    bool fail = false;
    for (int g = 0; g < G && !fail; g++) {
        const nhd_pod_group& pg = t.pod.groups[g];
        const int numa = (pm.pn >> (8 * g)) & 0xFF, lig = (pm.li >> (8 * g)) & 0xFF;
        if (pg.n_gpus) {
            const int nsw = nic_switch(r, lig);
            for (int jg = 0; jg < pg.n_gpus; jg++) {
                const uint32_t fr = ~gpu_used & ((1u << n_gpus) - 1);
                int dev = -1;
                for (uint32_t f = fr; f; f &= f - 1) {              /* GetFreePciGpuFromNic :648-655 */
                    const int gi = ctz32(f);
                    if (gpu_switch(r, gi) == nsw) { dev = gi; break; }
                }
                if (dev < 0) {
                    if (t.pci) { fail = true; break; }              /* :711-713 */
                    const uint32_t f = fr & r.gpu_numa_mask[numa];  /* GetNextGpuFree :495-500 */
                    if (f) dev = ctz32(f);
                }
                if (dev < 0) { fail = true; break; }
                gpu_used |= 1u << dev;
                if (pk.ng < 8) pk.gi_lo |= (unsigned long long)dev << (8 * pk.ng);
                else if (pk.ng < 16) pk.gi_hi |= (unsigned long long)dev << (8 * (pk.ng - 8));
                pk.ng++;
            }
            if (fail) break;
        }
        if (pg.flags & NHD_GRP_HAS_NIC_CORES) rec[n_rec++] = (uint8_t)lig;
    }
    if (fail) {                                                      /* Node.py:825-837 */
        pk.fail_status = n_rec ? NHD_REF_WOULD_CRASH : NHD_ASSIGN_FAILED;
        pk.gi_lo = pk.gi_hi = 0; pk.ng = 0;
        return;
    }
    pk.gpu_used_new = gpu_used;
    uint8_t outc[NHD_MAX_GROUPS] = {0, 0, 0, 0};
    pk.ncl = claimed_nic_order(rec, n_rec, outc);
    pk.claimed = (uint32_t)outc[0] | ((uint32_t)outc[1] << 8) | ((uint32_t)outc[2] << 16) | ((uint32_t)outc[3] << 24);
}

/* set / clear one bit of a 64-bit bitmap word with a native 32-bit atomic (works for shared and global) */
__device__ __forceinline__ void bit_set(uint64_t* words, int bit)
{
    atomicOr(reinterpret_cast<unsigned int*>(words) + (bit >> 5), 1u << (bit & 31));
}
__device__ __forceinline__ void bit_clear(uint64_t* words, int bit)
{
    atomicAnd(reinterpret_cast<unsigned int*>(words) + (bit >> 5), ~(1u << (bit & 31)));
}

/* bitmap word read: shared memory, or L2 (the sweep updates global bitmaps with atomics, which bypass L1) */
template <bool SMEM>
__device__ __forceinline__ uint64_t ldw(const uint64_t* p)
{
    if (SMEM) return *p;
    return __ldcg(reinterpret_cast<const unsigned long long*>(p));
}

#define NHD_PENDING      100          /* internal binding status: node chosen, mapping not resolved yet */
#define NHD_DYN_PENDING  0x20         /* NodeDyn.info: the node's first pod of this batch is still unresolved */

/* per-warp view of the sweep's shared-memory tables */
struct ClsNic;
struct SweepCtx {
    uint4* smemo;            /* mapping memo front      */
    uint4* dmemo;            /* decision memo           */
    uint4* dcache;           /* node-summary cache      */
    int32_t* dtag;
    const uint8_t* s_eff;    /* effective free-core tables [T][2][64] */
    const PodType* types;
    bool types_in_smem;
    int lane;
    int smemo_mask, dmemo_mask, dcache_mask, spmemo_mask, clsnic_mask;   /* slice sizes - 1 */
    const uint16_t* s_needb; /* [T][2][32] per-tuple socket demand for 2-NUMA nodes: need0 | need1 << 8 */
    struct ClsNic* clsnic;   /* CLSNIC_SLOTS x 48 B: static NIC layout per hardware class */
    uint4* spmemo;           /* SPMEMO_SLOTS x 16 B: first surviving NIC assignment of (type, groups S, NUMA k, NICs in use there) */
    const FastTables* ft;    /* direct-path tables (null when the batch has too many pod types) */
};

union DynU { NodeDyn d; uint4 q[2]; __device__ DynU() {} };

/*
 * Node summaries: HBM (later batches and commit_kernel read them) behind a direct-mapped shared-memory
 * cache per sweeping warp, written through: HBM is current for every node at all times, the cache only
 * shortens the chain.  One warp owns a cache (one CTA per pod class when the classes run side by side).
 */
__device__ __forceinline__ void load_dyn(const SweepArgs& a, const SweepCtx& cx, int node, DynU& du)
{
    const int cs = node & cx.dcache_mask;
    if (cx.dtag[cs] == node) { du.q[0] = cx.dcache[2 * cs]; du.q[1] = cx.dcache[2 * cs + 1]; }
    else { du.q[0] = __ldcg(&a.dyn[(size_t)node * 2]); du.q[1] = __ldcg(&a.dyn[(size_t)node * 2 + 1]); }   /* L2: the sweep also updates summaries with atomics */
}

__device__ __forceinline__ bool same_dyn(const DynU& x, const DynU& y)
{
    return x.q[0].x == y.q[0].x && x.q[0].y == y.q[0].y && x.q[0].z == y.q[0].z && x.q[0].w == y.q[0].w &&
           x.q[1].x == y.q[1].x && x.q[1].y == y.q[1].y && x.q[1].z == y.q[1].z && x.q[1].w == y.q[1].w;
}

/* write-through: HBM copy + the warp's cache slot (tag last) */
__device__ __forceinline__ void store_dyn(const SweepArgs& a, const SweepCtx& cx, int node, const DynU& du)
{
    const int cs = node & cx.dcache_mask;
    __syncwarp();                                        /* every lane has finished reading the cache */
    const uint4 half = cx.lane == 0 ? du.q[0] : du.q[1];      /* a select, not an index: keeps the summary in registers */
    if (cx.lane < 2) {
        a.dyn[(size_t)node * 2 + cx.lane] = half;
        cx.dcache[2 * cs + cx.lane] = half;
    }
    __syncwarp();
    if (cx.lane == 2) cx.dtag[cs] = node;
}

/* claimed NIC order, list({x[0] for x in nic_list}) (NHDScheduler.py:302), registers only:
 * the 8-slot CPython set table lives in one 64-bit word (slot byte = NIC index + 1) */
__device__ __forceinline__ uint32_t claimed_order_packed(uint32_t rec, int n_rec, int& ncl)
{
    if (n_rec <= 1) { ncl = n_rec; return n_rec ? (rec & 0xFF) : 0u; }
    unsigned long long slots = 0;
    for (int e = 0; e < n_rec; e++) {
        const uint32_t v = (rec >> (8 * e)) & 0xFF;
        uint32_t i = v & 7, perturb = v;
        for (;;) {
            const uint32_t sl = (uint32_t)(slots >> (8 * i)) & 0xFF;
            if (sl == 0) { slots |= (unsigned long long)(v + 1) << (8 * i); break; }
            if (sl == v + 1) break;
            perturb >>= 5;
            i = (i * 5 + 1 + perturb) & 7;
        }
    }
    uint32_t out = 0;
    ncl = 0;
    for (int i = 0; i < 8; i++) {
        const uint32_t sl = (uint32_t)(slots >> (8 * i)) & 0xFF;
        if (sl) { out |= (sl - 1) << (8 * ncl); ncl++; }
    }
    return out;
}

/*
 * NIC stage of Matcher.py:242-268 restricted to one NUMA node: the first surviving assignment of the groups
 * S (bit g = group g, taken in group order, first group most significant in the reference's product order) to
 * the NICs `mk` (list-index mask, ascending = NodeNic.idx order) of that NUMA node, with the reference's fp64
 * subtraction order.  Returns feasible << 31 | one byte per member of S: its NodeNic.idx.  Cold path (memoised).
 */
__device__ __noinline__ uint32_t nic_sub_solve(const double* cap, const PodType& t, int S, uint32_t mk, uint32_t inuse,
                                               unsigned long long sp0, unsigned long long sp1)
{
    bool feas = false;
    uint32_t r_idx = 0, r_li = 0;
    {
        /* members of S in group order, and their demands, in registers */
        const int n = popc32((uint32_t)S);
        int sr = S;
        const int g0 = sr ? ctz32((uint32_t)sr) : 0; sr &= sr - 1;
        const int g1 = sr ? ctz32((uint32_t)sr) : 0; sr &= sr - 1;
        const int g2 = sr ? ctz32((uint32_t)sr) : 0; sr &= sr - 1;
        const int g3 = sr ? ctz32((uint32_t)sr) : 0;
        const double rx[NHD_MAX_GROUPS] = {t.pod.groups[g0].rx_gbps, t.pod.groups[g1].rx_gbps, t.pod.groups[g2].rx_gbps, t.pod.groups[g3].rx_gbps};
        const double tx[NHD_MAX_GROUPS] = {t.pod.groups[g0].tx_gbps, t.pod.groups[g1].tx_gbps, t.pod.groups[g2].tx_gbps, t.pod.groups[g3].tx_gbps};
        auto capof = [&](int l) -> double {
            if ((inuse >> l) & 1) return 0.0;
            const int sc = (int)(((l < 16 ? sp0 : sp1) >> (4 * (l & 15))) & 0xF);
            return cap[sc];
        };
        if (n == 0) feas = true;
        else if (mk != 0) {
            for (uint32_t f0 = mk; f0 && !feas; f0 &= f0 - 1) {
                const int l0 = ctz32(f0);
                const double c0 = capof(l0);
                const double r0 = c0 - rx[0], t0 = c0 - tx[0];
                if (r0 < 0 || t0 < 0) continue;
                if (n == 1) { feas = true; r_li = l0; break; }
                for (uint32_t f1 = mk; f1 && !feas; f1 &= f1 - 1) {
                    const int l1 = ctz32(f1);
                    const double c1 = capof(l1);
                    const double r1 = (l1 == l0 ? r0 : c1) - rx[1], t1 = (l1 == l0 ? t0 : c1) - tx[1];
                    if (r1 < 0 || t1 < 0) continue;
                    if (n == 2) { feas = true; r_li = l0 | (l1 << 8); break; }
                    for (uint32_t f2 = mk; f2 && !feas; f2 &= f2 - 1) {
                        const int l2 = ctz32(f2);
                        const double c2 = capof(l2);
                        const double b2r = l2 == l1 ? r1 : (l2 == l0 ? r0 : c2), b2t = l2 == l1 ? t1 : (l2 == l0 ? t0 : c2);
                        const double r2 = b2r - rx[2], t2 = b2t - tx[2];
                        if (r2 < 0 || t2 < 0) continue;
                        if (n == 3) { feas = true; r_li = l0 | (l1 << 8) | (l2 << 16); break; }
                        for (uint32_t f3 = mk; f3; f3 &= f3 - 1) {
                            const int l3 = ctz32(f3);
                            const double c3 = capof(l3);
                            const double b3r = l3 == l2 ? r2 : (l3 == l1 ? r1 : (l3 == l0 ? r0 : c3));
                            const double b3t = l3 == l2 ? t2 : (l3 == l1 ? t1 : (l3 == l0 ? t0 : c3));
                            if (b3r - rx[3] < 0 || b3t - tx[3] < 0) continue;
                            feas = true; r_li = l0 | (l1 << 8) | (l2 << 16) | ((uint32_t)l3 << 24);
                            break;
                        }
                    }
                }
            }
            if (feas)
                for (int e = 0; e < n; e++) {
                    const int l = (r_li >> (8 * e)) & 0xFF;
                    r_idx |= (uint32_t)popc32(mk & ((1u << l) - 1)) << (8 * e);      /* NodeNic.idx = rank inside the NUMA node */
                }
        }
    }
    return r_idx | (feas ? 0x80000000u : 0u);
}

/* static NIC layout of one hardware class, cached in shared memory (32 B) */
struct ClsNic {
    uint32_t tag; uint32_t m0, m1;        /* NIC list-index masks of NUMA 0 / 1 */
    uint32_t nk;                          /* n_0 | n_1 << 8, bit 31: some NUMA node has more than 8 NICs */
    unsigned long long sp0, sp1;          /* speed-class nibbles by list index */
    uint32_t spk0, spk1;                  /* speed-class nibbles of NUMA 0 / 1 in NUMA-local order (<= 8 NICs) */
    uint32_t pad_[2];
};
static_assert(sizeof(ClsNic) == 48, "ClsNic is three 16-byte chunks");
constexpr int CLSNIC_SLOTS = 64;

/*
 * CPU-only pod, NUMA mode, on a 2-NUMA node (the reference's deployment shape) — the decision
 * factorises and is computed directly, without enumerating joint NIC choices:
 *   CPU stage   (Matcher.py:203-212)  lane q compares the type's precomputed per-socket demand of
 *               tuple q with the two free-core counts: one ballot;
 *   GPU stage   (Matcher.py:118-129)  no GPUs requested: every tuple passes;
 *   NIC stage   (Matcher.py:242-268)  NICs of different NUMA nodes do not interact (no PCI pruning in
 *               NUMA mode), so the first surviving entry for a tuple is the pair of first
 *               surviving sub-assignments of {groups on NUMA 0} and {groups on NUMA 1}.  Lane
 *               k*16 + S solves "groups S on the NICs of NUMA k" with the reference's own
 *               order (first group most significant, fp64 subtraction in group order); tuple
 *               lanes then read their two halves with shuffles;
 *   GetNumaGroupIdx (Matcher.py:423-452)  mapping memo on the three masks.
 * Same results as evaluate_full + compute_picks; returns 1 (not a candidate) or 2 (placed).
 */
__device__ __forceinline__ int resolve_cpu2(const SweepArgs& a, const SweepCtx& cx, int ti, const PodType& t, int node,
                            const DynU& du, PMap& pm, Picks& pk, bool& missed)
{
    PROF2_DECL
    const int lane = cx.lane, G = t.G, nq = 1 << (G + 1), gmask = (1 << G) - 1;
    const bool smt = (du.d.info & NHD_DYN_SMT) != 0;
    const uint32_t nb = cx.s_needb[(ti * 2 + (smt ? 1 : 0)) * 32 + lane];
    const bool okB = lane < nq && (nb & 0xFF) <= du.d.fc[0] && (nb >> 8) <= du.d.fc[1];
    const uint32_t balB = __ballot_sync(0xFFFFFFFFu, okB);
    if (!balB) return 1;
    const uint32_t balA = 0x55555555u & (nq >= 32 ? 0xFFFFFFFFu : ((1u << nq) - 1));

    /* static NIC layout of the node's hardware class */
    /* per-warp table: read by all lanes, refilled by lane 0 between two __syncwarp()s */
    ClsNic* ce = &cx.clsnic[du.d.hw_class & cx.clsnic_mask];
    uint32_t m0, m1, nk, spk0, spk1;
    unsigned long long sp0, sp1;
    __syncwarp();
    const uint32_t want = (uint32_t)du.d.hw_class + 1u;
    bool hit = ce->tag == want;
    m0 = ce->m0; m1 = ce->m1; nk = ce->nk; sp0 = ce->sp0; sp1 = ce->sp1; spk0 = ce->spk0; spk1 = ce->spk1;
    hit = __all_sync(0xFFFFFFFFu, hit);
    if (!hit) {
        missed = true;
        const uint4 c5 = *reinterpret_cast<const uint4*>(a.nodes + chunk_off(node, 5));
        const uint4 c7 = *reinterpret_cast<const uint4*>(a.nodes + chunk_off(node, 7));
        m0 = c5.x; m1 = c5.y;
        sp0 = (unsigned long long)c7.x | ((unsigned long long)c7.y << 32);
        sp1 = (unsigned long long)c7.z | ((unsigned long long)c7.w << 32);
        const int n0 = popc32(m0), n1 = popc32(m1);
        nk = (uint32_t)n0 | ((uint32_t)n1 << 8) | ((n0 > 8 || n1 > 8) ? 0x80000000u : 0u);
        spk0 = spk1 = 0;
        int j = 0;
        for (uint32_t f = m0; f && j < 8; f &= f - 1, j++) { const int l = ctz32(f); spk0 |= (uint32_t)(((l < 16 ? sp0 : sp1) >> (4 * (l & 15))) & 0xF) << (4 * j); }
        j = 0;
        for (uint32_t f = m1; f && j < 8; f &= f - 1, j++) { const int l = ctz32(f); spk1 |= (uint32_t)(((l < 16 ? sp0 : sp1) >> (4 * (l & 15))) & 0xF) << (4 * j); }
        __syncwarp();
        if (lane == 0) {
            ce->m0 = m0; ce->m1 = m1; ce->nk = nk; ce->sp0 = sp0; ce->sp1 = sp1; ce->spk0 = spk0; ce->spk1 = spk1;
            ce->tag = want;
        }
        __syncwarp();
    }

    PROF2(0);   /* B mask + class layout */
    /* ---- sub-problems: lane = k * 16 + S ---- */
    const int k = lane >> 4, S = lane & 15;
    const uint32_t mk = k ? m1 : m0;
    const uint32_t inuse = du.d.nic_inuse;
    bool feas = false, s_miss = false;
    uint32_t r_idx = 0, r_li = 0;                      /* one byte per member of S, in group order */
    uint4* se = cx.spmemo;
    uint4 s_new = make_uint4(0, 0, 0, 0);
    if (S <= gmask) {
      /* the sub-problem depends on (type, S) and on the NICs of this NUMA node only: their count,
       * speeds and which are taken, in NUMA-local order — memo keyed by exactly that */
      uint32_t inuse_k = 0;
      {
          int jl = 0;
          for (uint32_t f = mk; f; f &= f - 1, jl++) inuse_k |= ((inuse >> ctz32(f)) & 1u) << jl;
      }
      const bool wide = (nk >> 31) != 0;
      const uint32_t n_k = (k ? (nk >> 8) : nk) & 0xFF;
      const uint32_t skey = 0x80000000u | (uint32_t)ti | ((uint32_t)S << 12) | (n_k << 16) |
                            (wide ? (0x40000000u | ((uint32_t)k << 24)) : 0u);
      const uint32_t skey2 = wide ? (uint32_t)du.d.hw_class : (k ? spk1 : spk0);
      uint32_t sh = skey * 0x9E3779B1u ^ inuse_k * 0x85EBCA77u ^ skey2 * 0xC2B2AE3Du;
      sh ^= sh >> 15;
      se = &cx.spmemo[sh & cx.spmemo_mask];
      const uint4 sv = *se;
      if (sv.x == skey && sv.y == inuse_k && sv.z == skey2) {
        feas = (sv.w >> 31) != 0; r_idx = sv.w & 0x7FFFFFFFu;
      } else {
        const uint32_t rr = nic_sub_solve(a.cap, t, S, mk, inuse, sp0, sp1);
        feas = (rr >> 31) != 0; r_idx = rr & 0x7FFFFFFFu;
        s_new = make_uint4(skey, inuse_k, skey2, r_idx | (feas ? 0x80000000u : 0u));
        s_miss = true;
      }
    }
    {
        /* a miss is stored once every lane has read the table, one lane at a time (lanes may share a slot) */
        const uint32_t mm = __ballot_sync(0xFFFFFFFFu, s_miss);
        __syncwarp();
        for (uint32_t m = mm; m; m &= m - 1) {
            if (lane == ctz32(m)) *se = s_new;
            __syncwarp();
        }
    }
    PROF2(1);   /* per-NUMA sub-problems */
    /* ---- tuple lanes combine their two halves ---- */
    bool okC = lane < nq && !(lane & 1);
    {
        /* every lane takes part in the shuffles; only tuple lanes use the result */
        const int p = (lane >> 1) & gmask;
        const int s1 = (int)(__brev((unsigned)p) >> (32 - G));       /* groups on NUMA 1: digit g of the tuple is bit G-1-g of p */
        const int s0 = gmask & ~s1;
        const int f0 = __shfl_sync(0xFFFFFFFFu, (int)feas, s0);
        const int f1 = __shfl_sync(0xFFFFFFFFu, (int)feas, 16 + s1);
        okC = okC && f0 && f1;
    }
    const uint32_t balC = __ballot_sync(0xFFFFFFFFu, okC);
    if (!balC) return 1;
    PROF2(2);   /* combine */
    int v = -1;
    if (lane == 0) v = choose_mapping_memo(cx.smemo, cx.smemo_mask, a.memo, 2, G, balA, balB, balC);
    v = __shfl_sync(0xFFFFFFFFu, v, 0);
    PROF2(3);   /* mapping memo */
    if (v < 0) return 1;
    const int ps = v & 0xFF;
    pm.ms = (uint32_t)(v >> 8);
    const int s1 = (int)(__brev((unsigned)ps) >> (32 - G));
    pm.pn = ((uint32_t)s1 & 1u) | (((uint32_t)s1 & 2u) << 7) | (((uint32_t)s1 & 4u) << 14) | (((uint32_t)s1 & 8u) << 21);   /* one byte per group */
    const int s0 = gmask & ~s1;
    const uint32_t ix0 = __shfl_sync(0xFFFFFFFFu, r_idx, s0), ix1 = __shfl_sync(0xFFFFFFFFu, r_idx, 16 + s1);
    pm.idx = pm.li = 0;
    uint32_t rec = 0;
    int n_rec = 0, e0 = 0, e1 = 0;
    for (int g = 0; g < G; g++) {
        uint32_t l, x;
        if ((s1 >> g) & 1) { x = (ix1 >> (8 * e1)) & 0xFF; e1++; l = (uint32_t)nth_bit32(m1, (int)x); }
        else { x = (ix0 >> (8 * e0)) & 0xFF; e0++; l = (uint32_t)nth_bit32(m0, (int)x); }     /* NodeNic.idx -> index in Node.nics */
        pm.li |= l << (8 * g);
        pm.idx |= x << (8 * g);
        if ((t.nic_groups >> g) & 1) { rec |= l << (8 * n_rec); n_rec++; }
    }
    PROF2(4);   /* expand */
    pk.claimed = claimed_order_packed(rec, n_rec, pk.ncl);
    pk.gi_lo = pk.gi_hi = 0; pk.ng = 0; pk.fail_status = 0;
    pk.gpu_used_new = du.d.gpu_used;
    PROF2(5);   /* claim order */
    return 2;
}

/*
 * What would AttemptScheduling do with a pod of type ti on this node, given its summary?
 * Returns 1 (FindNode would not offer the node), 2 (placed) or 3 (SetPhysicalIdsFromMapping
 * fails) plus the mapping and the resource picks.  Decision memo first, full evaluation on a miss.
 */
__device__ __forceinline__ int direct_single(const SweepCtx& cx, int ti, const DynU& du, PMap& pm, Picks& pk);

__device__ __forceinline__ int resolve_decision(const SweepArgs& a, const SweepCtx& cx, int ti, const PodType& t, int node,
                                                const DynU& du, PMap& pm, Picks& pk, bool& missed)
{
    missed = false;
    if (summary_infeasible(t, du.d)) return 1;
    if (cx.ft) {
        /* CPU-only NUMA-mode type with <= 2 groups on a classed 2-NUMA node: the table-driven evaluation of the
         * standing decisions, for this one (type, node) — every lane computes the same */
        const int st = direct_single(cx, ti, du, pm, pk);
        if (st) return st;
    }
    const bool fast2 = cx.s_needb && t.total_gpus == 0 && !t.pci && ((du.d.info >> 2) & 7) == 2 && du.d.hw_class != NHD_NO_CLASS && ti < 4096;
    if (fast2) return resolve_cpu2(a, cx, ti, t, node, du, pm, pk, missed);    /* CPU-only pod on a 2-NUMA node: direct */
    const bool smt = (du.d.info & NHD_DYN_SMT) != 0;
    const int need = smt ? t.need_smt : t.need_nosmt;
    const bool memoable = cx.types_in_smem && du.d.hw_class != NHD_NO_CLASS && need <= 63 && t.total_gpus <= 4;
    unsigned long long key = (unsigned long long)ti | ((unsigned long long)du.d.hw_class << 12) |
                             ((unsigned long long)du.d.gpu_used << 24);
    if (memoable) {
        const uint8_t* eff = cx.s_eff + ti * 128 + (smt ? 64 : 0);
#pragma unroll
        for (int k = 0; k < NHD_MAX_NUMA; k++) {
            const int cc = du.d.fc[k] < 63 ? du.d.fc[k] : 63;
            key |= (unsigned long long)eff[cc] << (40 + 6 * k);
        }
    }
    const uint32_t hsh = (uint32_t)(memo_mix(key ^ ((unsigned long long)du.d.nic_inuse << 17)));
    uint4* de = &cx.dmemo[3 * (hsh & cx.dmemo_mask)];
    union { DEntry e; uint4 q[3]; } eu;
    eu.q[0] = de[0];
    if (memoable && eu.e.state != 0 && eu.e.a == key && eu.e.nic_inuse == du.d.nic_inuse) {
        const int state = eu.e.state;
        if (state >= 2) {
            eu.q[1] = de[1];
            eu.q[2] = de[2];
            pm.pn = eu.e.pn; pm.idx = eu.e.idx; pm.li = eu.e.li; pm.ms = eu.e.ms;
            pk.gi_lo = eu.e.gi; pk.gi_hi = 0; pk.claimed = eu.e.claimed; pk.gpu_used_new = eu.e.gpu_used_new;
            pk.ng = eu.e.ng; pk.ncl = eu.e.ncl; pk.fail_status = eu.e.fail_status;
        }
        return state;
    }
    missed = true;
    int state;
    {
    /* full evaluation on the node's static description + summary */
    RecU u;
#pragma unroll
    for (int cc = 2; cc < REC_CHUNKS; cc++)
        u.q[cc] = *reinterpret_cast<const uint4*>(a.nodes + chunk_off(node, cc));
    apply_dyn(u.r, du.d);
    state = 1;
    /* the out-of-line helpers get copies: taking the address of du / pm / pk would pin the hot
     * path's per-pod state in local memory */
    const NodeDyn dcopy = du.d;
    PMap pm2 = {0, 0, 0, 0};
    if (evaluate_full(a, cx.smemo, cx.smemo_mask, u.r, dcopy, t, cx.lane, pm2)) {
        Picks pk2;
        compute_picks(u.r, t, pm2, dcopy.gpu_used, dcopy.n_gpus, pk2);
        pk = pk2;
        state = pk2.fail_status ? 3 : 2;
    }
    pm = pm2;
    }
    __syncwarp();                                        /* every lane has read the entry */
    if (memoable && cx.lane == 0) {
        eu.e.a = key; eu.e.nic_inuse = du.d.nic_inuse;
        eu.e.state = (uint8_t)state; eu.e.ms = (uint8_t)pm.ms; eu.e.ncl = (uint8_t)pk.ncl; eu.e.ng = (uint8_t)pk.ng;
        eu.e.pn = pm.pn; eu.e.idx = pm.idx; eu.e.li = pm.li;
        eu.e.claimed = pk.claimed; eu.e.gi = (uint32_t)pk.gi_lo;
        eu.e.gpu_used_new = (uint16_t)pk.gpu_used_new; eu.e.fail_status = (uint8_t)pk.fail_status; eu.e.pad_ = 0;
        eu.e.pad2_[0] = eu.e.pad2_[1] = 0;
        de[0] = eu.q[0]; de[1] = eu.q[1]; de[2] = eu.q[2];
    }
    __syncwarp();
    return state;
}

/*
 * Apply a decision: everything of SetBusy + SetPhysicalIdsFromMapping + ClaimPodNICResources
 * (NHDScheduler.py:289-304, Node.py:663-841) except the core ids, on the summary; writes the
 * binding header (the core ids follow in assign_cores_kernel).  Returns true when placed.
 */
__device__ __forceinline__ bool apply_decision(const SweepCtx& cx, const PodType& t, int node, NodeDyn& d, const PMap& pm,
                                               const Picks& pk, double now, nhd_binding* bout, int chunks = 8)
{
    const int G = t.G;
    const bool smt_node = (d.info & NHD_DYN_SMT) != 0;
    const bool fail = pk.fail_status != 0;
    d.busy_time = now;                                              /* NHDScheduler.py:289 */
    d.info |= NHD_DYN_TOUCHED;
    uint32_t w0s, w2, w14 = 0;
    if (fail) {                                                      /* Node.py:825-837: cores/GPUs given back, busy stays */
        w0s = (uint32_t)pk.fail_status;
        w2 = (uint32_t)G;
    } else {
        /* per-socket core accounting: a group's two batches remove cl[g] cores from its socket
         * (Matcher.py:179-194 counts exactly what Node.py:502-519 will take); the misc batch on
         * an SMT node takes min(n, what is left) cores when it may not pair hyperthreads */
        const uint8_t* cl = smt_node ? t.cl_smt : t.cl_nosmt;
        uint32_t fcw = (uint32_t)d.fc[0] | ((uint32_t)d.fc[1] << 8) | ((uint32_t)d.fc[2] << 16) | ((uint32_t)d.fc[3] << 24);
        const uint32_t fc_before = fcw;
        w14 = (uint32_t)d.consumed[0] | ((uint32_t)d.consumed[1] << 8) | ((uint32_t)d.consumed[2] << 16) | ((uint32_t)d.consumed[3] << 24);
        for (int g = 0; g < G; g++) fcw -= (uint32_t)cl[g] << (8 * ((pm.pn >> (8 * g)) & 0xFF));
        {
            const int sh = 8 * (int)pm.ms;
            const int wd = batch_width(smt_node, (t.pod.flags & NHD_POD_MISC_SMT) != 0, t.pod.n_misc, (fcw >> sh) & 0xFF);
            fcw -= (uint32_t)wd << sh;
        }
        const uint32_t cons = w14 + (fc_before - fcw);               /* per byte, no borrows: each width <= what is free */
#pragma unroll
        for (int k = 0; k < NHD_MAX_NUMA; k++) { d.fc[k] = (uint8_t)(fcw >> (8 * k)); d.consumed[k] = (uint8_t)(cons >> (8 * k)); }
        d.gpu_used = (uint16_t)pk.gpu_used_new;
        if (t.pod.hugepages_gb > 0) d.free_hugepages_gb -= t.pod.hugepages_gb;      /* Node.py:794-796 */
        for (int e = 0; e < pk.ncl; e++) d.nic_inuse |= 1u << ((pk.claimed >> (8 * e)) & 0xFF);   /* Node.py:644-646 */
        w0s = NHD_PLACED;
        w2 = (uint32_t)G | ((uint32_t)pk.ng << 16) | ((uint32_t)pk.ncl << 24);
    }
    /* bytes: 12 gpu_numa[4] 16 cpu_numa[5] 21 nic_numa[4] 25 nic_idx[4] 29 nic_list_index[4] 33 claimed[4] 40 gpu_index[16] 56 cores */
    const uint32_t claimed = fail ? 0u : pk.claimed;
    const uint32_t w4 = G < 4 ? (pm.pn | (pm.ms << (8 * G))) : pm.pn;
    const uint32_t w5 = (G == 4 ? pm.ms : 0u) | (pm.pn << 8);
    const uint32_t w6 = (pm.pn >> 24) | (pm.idx << 8);
    const uint32_t w7 = (pm.idx >> 24) | (pm.li << 8);
    const uint32_t w8 = (pm.li >> 24) | (claimed << 8);
    const uint32_t w9 = claimed >> 24;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (cx.lane == 0) v = make_uint4(w0s, (uint32_t)node, w2, pm.pn);
    else if (cx.lane == 1) v = make_uint4(w4, w5, w6, w7);
    else if (cx.lane == 2) v = make_uint4(w8, w9, (uint32_t)pk.gi_lo, (uint32_t)(pk.gi_lo >> 32));
    else if (cx.lane == 3) v = make_uint4((uint32_t)pk.gi_hi, (uint32_t)(pk.gi_hi >> 32), w14, 0);
    if (cx.lane < chunks) reinterpret_cast<uint4*>(bout)[cx.lane] = v;      /* chunks 4..7 are zero until the core ids */
    return !fail;
}

/* the rare in-sweep resolution of a deferred pod (node revisited): kept out of line */
__device__ __noinline__ void resolve_pending(const SweepArgs& a, const SweepCtx& cx, int tj, const PodType& tjy, int node,
                                             DynU& du, nhd_binding* bout)
{
    PMap pmj = {0, 0, 0, 0};
    Picks pkj;
    pkj.fail_status = 0;
    bool mj;
    du.d.info &= ~NHD_DYN_PENDING;
    resolve_decision(a, cx, tj, tjy, node, du, pmj, pkj, mj);
    apply_decision(cx, tjy, node, du.d, pmj, pkj, du.d.busy_time, bout);
    store_dyn(a, cx, node, du);
    __syncwarp();
}

/*
 * ---------------------------------------------------------------- standing decisions (constant-clock batches)
 *
 * On a constant clock (the batch case) the sweep keeps, for every pod type, what the next pod of that type
 * will do — a pure function of (type, first-fit node, that node's summary):
 *   CPU-only types  the first-fit node of the GPU-less pass (first set bit of F[t] & NOGPU, Matcher.py:412-416),
 *                   the mapping and the node's summary after the pod (NHD_SLOT_FAST);
 *   GPU types       the first candidate that is not busy (Matcher.py:107-111); if no pod of this batch was bound
 *                   there its snapshot bit is exact and the pod only stamps the node (NHD_SLOT_DEFER).
 * A pod commits its type's slot in a handful of instructions; the slots made for the node it changed are then
 * worked out again, ONE LANE PER TYPE, all types side by side.  So that this is short, everything a decision
 * needs is tabulated when the sweep starts (all 256 threads, a few microseconds):
 *   TB    [type][smt][numa][free cores]   -> which (G+1)-tuples pass the CPU stage on that socket (Matcher.py:203-212)
 *   SUB0/1[type][NIC signature][in use]   -> per G-tuple: does the NIC stage (Matcher.py:242-268) survive on NUMA 0 / 1
 *                                            for the groups the tuple puts there, and which NodeNic.idx they get
 *                                            (nic_sub_solve: the reference's order, fp64 subtraction order)
 *   MAPT  [CPU mask][NIC mask]            -> GetNumaGroupIdx (Matcher.py:423-452), i.e. CPython set order; a pure
 *                                            function, filled once per handle (mapt_kernel)
 *   GD    [type][smt][tuple]              -> cores the groups take from each socket
 *   CLS   [hardware class]                -> NIC list indices per NUMA node and the two NIC signatures
 * and a decision is five table reads and some arithmetic.  The direct path covers CPU-only NUMA-mode types with
 * at most two groups on 2-NUMA nodes with a hardware class and at most four NICs per NUMA node (the reference's
 * deployment shape).  Anything else — spills onto GPU nodes, GPU pods on nodes already bound to, other node or
 * type shapes — is NHD_SLOT_SLOW: the pod takes the ordinary path below.  One warp does all of this in pod
 * order: no inter-warp hand-off exists.  The binding of a directly decided pod is written out in packed form
 * (NHD_PENDING_FAST) and formatted by resolve_kernel, off the sequential chain.
 */
/* what a lane knows about the node it evaluates besides the summary: the NICs in use in NodeNic.idx order
 * (NUMA 0 in bits 0-3, NUMA 1 in bits 4-7) and the class entry (li0, li1, sig0 | sig1 << 8 | n0 << 16 | n1 << 24) */
struct NodeAux { uint32_t iu, li0, li1, sig; };

/*
 * One lane, one pod type, no branches: what AttemptScheduling does with a pod of type `tl` on a node with
 * summary du (CPU-only type and node shape covered by the tables: the caller checks TyFast.direct / ClsFast.ok).
 * Returns true when the pod is placed; then dec / da / iu_after describe the mapping, the summary after the pod
 * (SetBusy + the bookkeeping of SetPhysicalIdsFromMapping, Node.py:663-841, + ClaimPodNICResources) and the NICs
 * in use afterwards.
 */
template <bool SUB_SMEM>
__device__ __forceinline__ bool fast_eval(const FastTables& ft, int tl, const TyFast& ty, const DynU& du, const NodeAux& ax,
                                          double now, uint32_t& dec, DynU& da, uint32_t& iu_after)
{
    const int smt = (du.d.info >> 1) & 1;                                     /* NHD_DYN_SMT */
    /* the standing decisions read the rows in shared memory (fast_node_aux admits only the first FAST_NSIG_SMEM
     * signatures there); the general path reads any signature's row from global memory */
    const uint32_t w0 = SUB_SMEM ? ft.sub0s[(tl * FAST_NSIG_SMEM + (ax.sig & 0xFF)) * 16 + (ax.iu & 15)]
                                 : __ldg(&ft.sub0[(tl * FAST_NSIG + (ax.sig & 0xFF)) * 16 + (ax.iu & 15)]);
    const uint32_t w1 = SUB_SMEM ? ft.sub1s[(tl * FAST_NSIG_SMEM + ((ax.sig >> 8) & 0xFF)) * 16 + ((ax.iu >> 4) & 15)]
                                 : __ldg(&ft.sub1[(tl * FAST_NSIG + ((ax.sig >> 8) & 0xFF)) * 16 + ((ax.iu >> 4) & 15)]);
    const uint32_t mC = gather_b7(w0 & w1);                                   /* Matcher.py:242-276 */
    const uint32_t fc0 = du.q[0].x & 0xFF, fc1 = (du.q[0].x >> 8) & 0xFF;
    const uint32_t mB = ft.tb[((tl * 2 + smt) * 2 + 0) * 64 + (fc0 < 63 ? fc0 : 63)] &
                        ft.tb[((tl * 2 + smt) * 2 + 1) * 64 + (fc1 < 63 ? fc1 : 63)];      /* Matcher.py:203-212 */
    const uint32_t mi = ty.G == 2 ? ((mB << 4) | mC) : (4096 + (((mB & 15) << 2) | (mC & 3)));
    const uint32_t mv = ft.mapt[mi];                                          /* Matcher.py:349, :423-452 */
    const bool feas = (mv & 0x80) != 0 && ty.hugepages_gb <= du.d.free_hugepages_gb;      /* Matcher.py:78 */
    const uint32_t ps = mv & 3, ms = (mv >> 2) & 1;
    const uint32_t gd = ft.gd[(tl * 2 + smt) * 4 + ps];
    uint32_t f0 = fc0 - (gd & 0xFF), f1 = fc1 - (gd >> 8);
    {
        const uint32_t avail = ms ? f1 : f0, n = ty.n_misc;
        const uint32_t wd = !smt ? n : (ty.misc_smt ? (n + 1) >> 1 : (n < avail ? n : avail));     /* batch_width */
        f0 -= ms ? 0u : wd;
        f1 -= ms ? wd : 0u;
    }
    const uint32_t e0 = (w0 >> (8 * ps)) & 0xFF, e1 = (w1 >> (8 * ps)) & 0xFF;
    /* NICs the groups claim (Node.py:742-755, :644-646); G <= 2: group 0 is the high digit of the tuple */
    uint32_t claim = 0, ciu = 0;
    {
        const uint32_t numa0 = ty.G == 2 ? (ps >> 1) & 1 : ps & 1;
        const uint32_t x0 = (numa0 ? e1 : e0) & 3;
        const uint32_t l0 = ((numa0 ? ax.li1 : ax.li0) >> (8 * x0)) & 31;
        const uint32_t t0 = ty.nic_groups & 1u;
        claim |= t0 << l0; ciu |= t0 << (x0 + 4 * numa0);
        const uint32_t numa1 = ps & 1;
        const uint32_t sh1 = numa1 == numa0 ? 2u : 0u;                        /* second member of that NUMA node's set, or first */
        const uint32_t x1 = ((numa1 ? e1 : e0) >> sh1) & 3;
        const uint32_t l1 = ((numa1 ? ax.li1 : ax.li0) >> (8 * x1)) & 31;
        const uint32_t t1 = ty.G == 2 ? (ty.nic_groups >> 1) & 1u : 0u;
        claim |= t1 << l1; ciu |= t1 << (x1 + 4 * numa1);
    }
    da.q[0] = du.q[0]; da.q[1] = du.q[1];
    const uint32_t fcw = (du.q[0].x & 0xFFFF0000u) | f0 | (f1 << 8);
    da.q[0].x = fcw;
    da.q[0].y = du.q[0].y + (du.q[0].x - fcw);              /* per byte, no borrows: each width <= what is free */
    da.q[0].z = du.q[0].z | ((uint32_t)NHD_DYN_TOUCHED << 16);
    da.q[0].w = du.q[0].w | claim;
    da.q[1].x = du.q[1].x - (uint32_t)(ty.hugepages_gb > 0 ? ty.hugepages_gb : 0);       /* Node.py:794-796 */
    da.d.busy_time = now;                                     /* NHDScheduler.py:289 */
    iu_after = ax.iu | ciu;
    dec = ps | (ms << 2) | (e0 << 8) | (e1 << 16);
    return feas;
}

/* summary of a node for the direct path: the cache, else HBM — through L1 while no pod of the batch has been
 * bound to the node (its summary is the snapshot's, immutable), from L2 otherwise */
__device__ __forceinline__ void fast_load_dyn(const SweepArgs& a, const SweepCtx& cx, const uint64_t* touched, int node, DynU& du)
{
    const int cs = node & cx.dcache_mask;
    if (cx.dtag[cs] == node) { du.q[0] = cx.dcache[2 * cs]; du.q[1] = cx.dcache[2 * cs + 1]; }
    else if ((touched[node >> 6] >> (node & 63)) & 1) { du.q[0] = __ldcg(&a.dyn[(size_t)node * 2]); du.q[1] = __ldcg(&a.dyn[(size_t)node * 2 + 1]); }
    else { du.q[0] = a.dyn[(size_t)node * 2]; du.q[1] = a.dyn[(size_t)node * 2 + 1]; }
}

/* class entry and compact in-use bits of a node with summary du; false when the direct path does not cover it */
__device__ __forceinline__ bool fast_node_aux(const FastTables& ft, const DynU& du, NodeAux& ax, bool smem_rows = true)
{
    ax.iu = ax.li0 = ax.li1 = ax.sig = 0;
    if (((du.d.info >> 2) & 7) != 2 || du.d.hw_class == NHD_NO_CLASS) return false;
    const ClsFast cf = ft.cls[du.d.hw_class];
    /* the sweep keeps the table rows of the first few NIC signatures in shared memory (a generic or global load on
     * this chain costs 3-5 % of the whole sweep, measured); rarer signatures take the general path */
    if (!cf.ok || (smem_rows && (cf.sig0 >= FAST_NSIG_SMEM || cf.sig1 >= FAST_NSIG_SMEM))) return false;
    const uint32_t inuse = du.d.nic_inuse;
    uint32_t iu = 0;
    for (int j = 0; j < cf.n0; j++) iu |= ((inuse >> ((cf.li0 >> (8 * j)) & 31)) & 1u) << j;
    for (int j = 0; j < cf.n1; j++) iu |= ((inuse >> ((cf.li1 >> (8 * j)) & 31)) & 1u) << (4 + j);
    ax.iu = iu; ax.li0 = cf.li0; ax.li1 = cf.li1;
    ax.sig = (uint32_t)cf.sig0 | ((uint32_t)cf.sig1 << 8) | ((uint32_t)cf.n0 << 16) | ((uint32_t)cf.n1 << 24);
    return true;
}

/* resolve_decision's direct case: 0 = not covered by the tables, 1 = FindNode would not offer the node, 2 = placed
 * (mapping and picks filled in like resolve_cpu2 does) */
__device__ __forceinline__ int direct_single(const SweepCtx& cx, int ti, const DynU& du, PMap& pm, Picks& pk)
{
    const FastTables& ft = *cx.ft;
    const TyFast ty = ft.ty[ti];
    if (!ty.direct) return 0;
    NodeAux ax;
    if (!fast_node_aux(ft, du, ax, false)) return 0;
    uint32_t dec = 0, iu2 = 0;
    DynU da;
    if (!fast_eval<false>(ft, ti, ty, du, ax, 0.0, dec, da, iu2)) return 1;
    const int G = ty.G, ps = dec & 3;
    const uint32_t e0 = (dec >> 8) & 0xFF, e1 = (dec >> 16) & 0xFF;
    uint32_t pn = 0, idx = 0, li = 0, rec = 0;
    int n_rec = 0, k0 = 0, k1 = 0;
    for (int g = 0; g < G; g++) {
        const int numa = (ps >> (G - 1 - g)) & 1;
        const uint32_t x = numa ? (e1 >> (2 * k1++)) & 3 : (e0 >> (2 * k0++)) & 3;
        const uint32_t l = ((numa ? ax.li1 : ax.li0) >> (8 * x)) & 31;             /* NodeNic.idx -> index in Node.nics */
        pn |= (uint32_t)numa << (8 * g); idx |= x << (8 * g); li |= l << (8 * g);
        if ((ty.nic_groups >> g) & 1) { rec |= l << (8 * n_rec); n_rec++; }
    }
    pm.pn = pn; pm.idx = idx; pm.li = li; pm.ms = (dec >> 2) & 1;
    pk.claimed = claimed_order_packed(rec, n_rec, pk.ncl);                          /* NHDScheduler.py:302 */
    pk.gi_lo = pk.gi_hi = 0; pk.ng = 0; pk.fail_status = 0;
    pk.gpu_used_new = du.d.gpu_used;
    return 2;
}

/* per-lane standing decision (lane t = pod type t), kept in registers */
struct LaneSlot {
    int node, kind;          /* NHD_SLOT_* */
    uint32_t dec, w14;       /* FAST: packed mapping; NodeDyn.consumed before the pod */
    DynU after;              /* FAST: summary once the pod is placed */
    NodeAux ax;              /* FAST: class entry of the node, NICs in use once the pod is placed */
    int c;                   /* CPU-only types: word of F[t] & NOGPU the lane is at, and what is left of it */
    uint64_t w;
};

/*
 * Bring the lanes' standing decisions up to date after a pod (lane t = pod type t; all 32 lanes call).
 *   eval_first   a directly decided pod was just committed at node0 (summary st0, aux ax0): EVERY lane with a
 *                directly evaluable CPU-only type evaluates its type there, so that the bits of F at nodes pods have
 *                been bound to stay exact; lanes whose decision was for node0 take the result as their new decision.
 *                A lane whose type no longer fits clears the bit (resources only shrink inside a batch) and, if node0
 *                was its candidate, moves on to its next one;
 *   rescan_cpu / rescan_gpu   lanes that must look their candidate up again (after the ordinary path).
 * Every pass of the loop evaluates all lanes that need it side by side; lanes only part ways to scan and load.
 */
template <bool SMEM_BITMAPS>
__device__ __forceinline__ void lanes_refresh(const SweepArgs& a, const SweepCtx& cx, const FastTables& ft, const TyFast& ty, int tl,
                                              bool l_direct, bool l_cpu, bool l_gpu, LaneSlot& sl, uint64_t* BM, const uint64_t* NOGPU,
                                              const uint64_t* BUSY, const uint64_t* touched, int W, int32_t* cursors, double now,
                                              bool eval_first, int node0, const DynU& st0, const NodeAux& ax0,
                                              uint32_t rescan_cpu, uint32_t rescan_gpu)
{
    const int lane = cx.lane;
    uint64_t* F = BM + (size_t)tl * W;
    bool need = eval_first && l_direct;
    bool pointing = sl.node == node0;
    bool dead = !eval_first && l_cpu && ((rescan_cpu >> lane) & 1);
    int cur_node = node0;
    DynU cur;
    cur.q[0] = st0.q[0]; cur.q[1] = st0.q[1];
    NodeAux cax = ax0;
    __syncwarp();
    if (dead && sl.c >= 0 && sl.c < W)                       /* the ordinary path may have cleared bits of this word */
        sl.w &= ldw<SMEM_BITMAPS>(&F[sl.c]);
    for (;;) {
        if (__any_sync(0xFFFFFFFFu, need)) {
            PROF_ADD(0, 1);                                  /* evaluation passes */
            PROF_ADD(1, __popc(__ballot_sync(0xFFFFFFFFu, need)));      /* lanes evaluating */
            uint32_t dec = 0, iu2 = 0;
            DynU da;
            const bool feas = fast_eval<true>(ft, tl, ty, cur, cax, now, dec, da, iu2);
            if (need) {
                if (feas) {
                    if (pointing) {
                        sl.node = cur_node; sl.kind = NHD_SLOT_FAST; sl.dec = dec; sl.w14 = cur.q[0].y;
                        sl.after.q[0] = da.q[0]; sl.after.q[1] = da.q[1];
                        sl.ax = cax; sl.ax.iu = iu2;
                    }
                } else {
                    bit_clear(F, cur_node);
                    if (sl.c == (cur_node >> 6)) sl.w &= ~(1ULL << (cur_node & 63));
                    dead = pointing;
                }
            }
            need = false;
        }
        if (!__any_sync(0xFFFFFFFFu, dead)) break;
        PROF_ADD(2, 1);                                      /* passes with lanes moving on */
        PROF_ADD(3, __popc(__ballot_sync(0xFFFFFFFFu, dead)));          /* lanes moving on */
        if (dead) {
            /* next candidate of the GPU-less pass (Matcher.py:412-416) */
            if (sl.c < W)
                while (sl.w == 0) {
                    sl.c++;
                    if (sl.c >= W) break;
                    sl.w = ldw<SMEM_BITMAPS>(&F[sl.c]) & ldw<SMEM_BITMAPS>(&NOGPU[sl.c]);
                }
            if (sl.c >= W) { sl.node = -1; sl.kind = NHD_SLOT_SLOW; }        /* the pod will spill: ordinary path */
            else {
                cur_node = sl.c * 64 + ctz64(sl.w);
                fast_load_dyn(a, cx, touched, cur_node, cur);
                if (l_direct && fast_node_aux(ft, cur, cax)) { need = true; pointing = true; }
                else { sl.node = cur_node; sl.kind = NHD_SLOT_SLOW; }         /* a shape the tables do not cover */
            }
            dead = false;
        }
    }
    if (l_gpu && ((rescan_gpu >> lane) & 1)) {
        /* first candidate that is not busy (Matcher.py:107-111) */
        int c = cursors[tl * 3 + 2];
        const int c_in = c;
        uint64_t w = 0;
        while (c < W) {
            w = ldw<SMEM_BITMAPS>(&F[c]) & ~ldw<SMEM_BITMAPS>(&BUSY[c]);
            if (w) break;
            c++;
        }
        if (c != c_in) cursors[tl * 3 + 2] = c;
        if (c >= W) { sl.node = -1; sl.kind = NHD_SLOT_NONE; }            /* final: busy bits are only set on a constant clock */
        else {
            const int node = c * 64 + ctz64(w);
            sl.node = node;
            /* no pod of this batch was bound there: the snapshot bit is exact; else the ordinary path */
            sl.kind = ((touched[c] >> (node & 63)) & 1) ? NHD_SLOT_SLOW : NHD_SLOT_DEFER;
        }
    }
    __syncwarp();
}

/*
 * One pod on the general path (see sweep_kernel): first fit over the bitmaps, live re-validation on the node's summary,
 * assignment, eager invalidation.  Kept out of line so that the short loop of the standing decisions is compiled on
 * its own (registers, scheduling).  Returns the node whose summary / BUSY / touched state the pod changed, or -1.
 */
struct OrdState {
    uint64_t* BM; uint64_t* NOGPU; uint64_t* BUSY; const uint64_t* GB; uint64_t* s_touched;
    int32_t* cursors; const PodType* types;
    int W, T;
    bool multi, eager, cclock, fast;
    int all_need, all_big, all_hp, all_gpus;
    int n_busy;                       /* entries of the busy list */
    double cur_now, busy_oldest;      /* clock the BUSY bitmap stands at; oldest stamp on the busy list */
};

template <bool SMEM_BITMAPS>
__device__ __noinline__ int ordinary_pod(const SweepArgs& a, const SweepCtx& cx, OrdState& os, int i, int ti, double now,
                                         unsigned long long gm)
{
    const int lane = cx.lane, W = os.W, T = os.T;
    uint64_t* const BM = os.BM;
    uint64_t* const NOGPU = os.NOGPU;
    uint64_t* const BUSY = os.BUSY;
    const uint64_t* const GB = os.GB;
    uint64_t* const s_touched = os.s_touched;
    int32_t* const cursors = os.cursors;
    const PodType* const types = os.types;
    const bool multi = os.multi, eager = os.eager, cclock = os.cclock, fast = os.fast;
    const int all_need = os.all_need, all_big = os.all_big, all_hp = os.all_hp, all_gpus = os.all_gpus;
    int& n_busy = os.n_busy;
    double& cur_now = os.cur_now;
    double& busy_oldest = os.busy_oldest;
    const PodType& t = types[ti];
    nhd_binding* bout = &a.out[i];
    uint64_t* F = BM + (size_t)ti * W;
    int commit_node = -1;
    const int wid = 0;                /* (check builds name the sweeping warp) */
    (void)wid;
    PROF_DECL
    do {

        /* ---- busy window bookkeeping when the clock moved (Node.py:847-850) ---- */
        if (now > cur_now && now - busy_oldest < a.min_busy) {
            /* forwards, and not even the oldest stamp on the list has left the window: nothing changes */
            cur_now = now;
        } else if (now != cur_now) {
            double oldest = 1e300;
            if (now < cur_now) {
                /* clock went backwards: rebuild from the summaries */
                n_busy = 0;
                for (int n0 = 0; n0 < W * 64; n0 += 32) {
                    int n = n0 + lane;
                    bool b = false;
                    if (n < a.n_nodes) {
                        double bt = __ldcg(&reinterpret_cast<const NodeDyn*>(a.dyn)[n].busy_time);
                        b = (now - bt) < a.min_busy;
                        if (b && bt < oldest) oldest = bt;
                    }
                    uint32_t bal = __ballot_sync(0xFFFFFFFFu, b);
                    if (lane == 0) reinterpret_cast<uint32_t*>(BUSY)[n0 >> 5] = bal;
                    if (b) a.busy_list[n_busy + popc32(bal & ((1u << lane) - 1))] = n;
                    n_busy += popc32(bal);
                }
            } else {
                int kept = 0;
                for (int e0 = 0; e0 < n_busy; e0 += 32) {
                    int e = e0 + lane;
                    int n = -1;
                    bool b = false;
                    if (e < n_busy) {
                        n = a.busy_list[e];
                        double bt = __ldcg(&reinterpret_cast<const NodeDyn*>(a.dyn)[n].busy_time);
                        b = (now - bt) < a.min_busy;
                        if (b && bt < oldest) oldest = bt;
                        if (!b) atomicAnd(reinterpret_cast<unsigned long long*>(&BUSY[n >> 6]), ~(1ULL << (n & 63)));
                    }
                    uint32_t bal = __ballot_sync(0xFFFFFFFFu, b);
                    __syncwarp();
                    if (b) a.busy_list[kept + popc32(bal & ((1u << lane) - 1))] = n;   /* kept <= e0 */
                    __syncwarp();
                    kept += popc32(bal);
                }
                n_busy = kept;
            }
            for (int tt = lane; tt < T; tt += 32) cursors[tt * 3 + 2] = 0;   /* busy bits may have cleared */
            /* the oldest stamp still inside the window (stamps added from here on are newer) */
            for (int d = 16; d >= 1; d >>= 1) {
                const double o = __shfl_sync(0xFFFFFFFFu, oldest, lane ^ d);
                oldest = o < oldest ? o : oldest;
            }
            busy_oldest = oldest;
            __syncwarp();
            cur_now = now;
        }

        if (!t.valid_map) {
            if (lane < 8) reinterpret_cast<uint4*>(bout)[lane] = make_uint4(lane == 0 ? NHD_BAD_MAP_TYPE : 0, lane == 0 ? 0xFFFFFFFFu : 0, lane == 0 ? t.G : 0, 0);
            break;
        }

        /* ---- first fit ---- */
        int chosen = -1;
        bool deferred = false;
        DynU du;
        PMap pm = {0, 0, 0, 0};
        Picks pk;
        pk.fail_status = 0;
        const bool skip_busy = t.needs_gpu != 0;                         /* Matcher.py:107-111 */
        /* nodes whose groups intersect the pod's (NHDScheduler.py:241); all ones when the gate is in F */
        auto elig = [&](int w) -> uint64_t {
            if (!multi) return ~0ULL;
            uint64_t e = 0;
            for (unsigned long long g = gm; g; g &= g - 1)
                e |= ldw<SMEM_BITMAPS>(&GB[(size_t)popc64(a.names_used & ((1ULL << ctz64(g)) - 1)) * W + w]);
            return e;
        };
        for (int pass = t.needs_gpu ? 1 : 0; pass < 2 && chosen < 0; pass++) {
            /* (1) the cursor: first word with any candidate of this pass */
            int c = __shfl_sync(0xFFFFFFFFu, cursors[ti * 3 + pass], 0);     /* one read for all lanes */
            const int c_in = c;
            uint64_t raw = 0;
            while (c < W) {
                raw = ldw<SMEM_BITMAPS>(&F[c]) & (pass == 0 ? ldw<SMEM_BITMAPS>(&NOGPU[c]) : ~0ULL);
                if (raw) break;
                int found = W;
                for (int base = c + 1; base < W; base += 32) {
                    const int w = base + lane;
                    const uint64_t r = (w < W) ? (ldw<SMEM_BITMAPS>(&F[w]) & (pass == 0 ? ldw<SMEM_BITMAPS>(&NOGPU[w]) : ~0ULL)) : 0;
                    const uint32_t nz = __ballot_sync(0xFFFFFFFFu, r != 0);
                    if (nz) { found = base + ctz32(nz); break; }
                }
                c = found;
            }
            if (c != c_in) {
                __syncwarp();
                if (lane == 0) cursors[ti * 3 + pass] = c;
                __syncwarp();
            }
            if (c >= W) continue;
            /* (2) candidates from there on, skipping busy nodes for GPU pods */
            int cb = c;
            if (skip_busy && !multi) { const int c2 = cursors[ti * 3 + 2]; cb = c2 > c ? c2 : c; }
            bool first = true;
            while (cb < W) {
                /* first look: the cursor word was just read */
                uint64_t word = (first && cb == c) ? raw : (ldw<SMEM_BITMAPS>(&F[cb]) & (pass == 0 ? ldw<SMEM_BITMAPS>(&NOGPU[cb]) : ~0ULL));
                first = false;
                if (multi) word &= elig(cb);
                if (skip_busy) word &= ~ldw<SMEM_BITMAPS>(&BUSY[cb]);
                if (!word) {
                    int found = W;
                    for (int base = cb + 1; base < W; base += 32) {
                        const int w = base + lane;
                        uint64_t r = (w < W) ? (ldw<SMEM_BITMAPS>(&F[w]) & (pass == 0 ? ldw<SMEM_BITMAPS>(&NOGPU[w]) : ~0ULL) & elig(w)) : 0;
                        if (skip_busy && w < W) r &= ~ldw<SMEM_BITMAPS>(&BUSY[w]);
                        const uint32_t nz = __ballot_sync(0xFFFFFFFFu, r != 0);
                        if (nz) { found = base + ctz32(nz); break; }
                    }
                    cb = found;
                    if (skip_busy && !multi) {
                        __syncwarp();
                        if (lane == 0) cursors[ti * 3 + 2] = cb;
                        __syncwarp();
                    }
                    continue;
                }
                const int node = cb * 64 + ctz64(word);
                const uint64_t nbit = 1ULL << (node & 63);
                PROF_MARK(1);      /* bitmap scan */

                if (skip_busy && !(s_touched[cb] & nbit)) {
                    /* no pod of this batch was bound here: the snapshot bit is exact (and the node is not
                     * busy), so the pod is placed; what it takes is resolved later */
                    chosen = node;
                    deferred = true;
                    break;
                }
                load_dyn(a, cx, node, du);
                CHK_SANE(du, node, 6);
                if (du.d.info & NHD_DYN_PENDING) {
                    /* the pod that took this node first is still unresolved: do it now, in order */
                    const int pj = a.pend_pod[node];
                    const int tj = a.pod_type[pj];
                    DynU dtmp;
                    dtmp.q[0] = du.q[0]; dtmp.q[1] = du.q[1];
                    resolve_pending(a, cx, tj, types[tj], node, dtmp, &a.out[pj]);
                    du.q[0] = dtmp.q[0]; du.q[1] = dtmp.q[1];
                    PROF_COUNT(12);
                }
                /* active / maintenance / node group are static inside a batch and already part of F */
                bool missed;
                const int state = resolve_decision(a, cx, ti, t, node, du, pm, pk, missed);
                if (missed) { PROF_MARK(3); } else { PROF_MARK(2); }      /* summary + decision: memo miss / hit */
                if (state >= 2) { chosen = node; break; }
                PROF_COUNT(8);     /* stale candidate */
                /* resources only shrink inside a batch: the node stays infeasible for this type */
                __syncwarp();                            /* every lane has read the word */
                if (lane == 0) bit_clear(F, node);
                __syncwarp();
            }
        }
        if (chosen < 0) {
            if (lane < 8) reinterpret_cast<uint4*>(bout)[lane] = make_uint4(lane == 0 ? NHD_NO_CANDIDATE : 0, lane == 0 ? 0xFFFFFFFFu : 0, lane == 0 ? t.G : 0, 0);
            break;
        }
        PROF_MARK(4);      /* loop exit */
        commit_node = chosen;

        bool placed = false;
        if (deferred) {
            /* stamp the node (NHDScheduler.py:289) and leave a note for resolve_kernel / a later visitor */
            __syncwarp();                                /* every lane has read the touched word */
            if (lane == 0) {
                NodeDyn* gd = reinterpret_cast<NodeDyn*>(a.dyn) + chosen;
                gd->busy_time = now;
                atomicOr(reinterpret_cast<unsigned int*>(&gd->gpu_used), (unsigned int)(NHD_DYN_TOUCHED | NHD_DYN_PENDING) << 16);
                a.pend_pod[chosen] = i;
                reinterpret_cast<uint2*>(bout)[0] = make_uint2(NHD_PENDING, (uint32_t)chosen);
                bit_set(s_touched, chosen);
            }
        } else {
            placed = apply_decision(cx, t, chosen, du.d, pm, pk, now, bout);
            store_dyn(a, cx, chosen, du);
            /* the touched / BUSY bitmaps are only ever consulted for GPU pods, which cannot fit a GPU-less node */
            if (lane == 0 && (du.d.n_gpus || fast)) bit_set(s_touched, chosen);
        }
        PROF_MARK(5);      /* assignment */
        if (a.min_busy > 0.0 && (deferred || du.d.n_gpus)) {             /* now - busy_time == 0 < MIN_BUSY_SECS */
            const uint64_t bit = 1ULL << (chosen & 63);
            if (!(ldw<SMEM_BITMAPS>(&BUSY[chosen >> 6]) & bit)) {
                __syncwarp();
                if (lane == 0) {
                    bit_set(BUSY, chosen);
                    if (!cclock) a.busy_list[n_busy] = chosen;
                }
                n_busy++;
                if (now < busy_oldest) busy_oldest = now;
            }
        }
        /* eager invalidation: pod types that can no longer fit here lose their bit now, so later
         * pods of those types never stop at this node (exact: summary_infeasible is a necessary condition) */
        bool roomy = false;
        if (eager && placed) {
            const NodeDyn& nd = du.d;
            const int sum = nd.fc[0] + nd.fc[1] + nd.fc[2] + nd.fc[3];
            int mx = nd.fc[0] > nd.fc[1] ? nd.fc[0] : nd.fc[1];
            const int mx2 = nd.fc[2] > nd.fc[3] ? nd.fc[2] : nd.fc[3];
            mx = mx > mx2 ? mx : mx2;
            const uint32_t alln = nd.n_nics >= 32 ? 0xFFFFFFFFu : ((1u << nd.n_nics) - 1);
            roomy = sum >= all_need && mx >= all_big && nd.free_hugepages_gb >= all_hp && (nd.nic_inuse & alln) != alln &&
                    (nd.n_gpus == 0 || popc32(~(uint32_t)nd.gpu_used & ((1u << nd.n_gpus) - 1)) >= all_gpus);
        }
        if (eager && placed && !roomy) {
            for (int tb = 0; tb < T; tb += 32) {
                const int tt = tb + lane;
                if (tt < T && summary_infeasible(types[tt], du.d))
                    bit_clear(BM + (size_t)tt * W, chosen);
            }
        }
    } while (0);
    __syncwarp();
    return commit_node;
}

/*
 * Decision sweep.  One CTA — or two, one per pod class, when the classes provably cannot meet (see the
 * certificate below); in each, warp 0 walks its pods in order (all lanes execute the scalar parts
 * redundantly, so there is no intra-warp hand-off), the other warps only help to stage tables
 * into shared memory.  Per pod on the general path (ordinary_pod):
 *   first fit   cursor word of the type's feasibility bitmap (minus busy nodes; GPU-less nodes
 *               first for CPU-only pods, Matcher.py:412-416), 32-wide ballot search when empty;
 *   untouched?  the snapshot bit of a node no pod of this batch was bound to is exact, so a GPU
 *               pod just takes the node (busy stamp, BUSY bit) and its mapping is worked out
 *               later, in parallel, by resolve_kernel — or right here if the node is revisited;
 *   validate    otherwise the node's 32-byte summary: exact cheap rejects, the decision memo,
 *               (miss) the full tuple evaluation + GPU picks + NIC claim order;
 *   assign      hugepages, busy stamp, per-socket core accounting, binding header, summary
 *               write-back (Node.py:663-841 minus the core ids);
 *   invalidate  every pod type that can no longer fit on the node loses its bit right away.
 * On a constant clock the standing decisions above short-cut all of this for the common cases.
 */
template <bool SMEM_BITMAPS>
__global__ void __launch_bounds__(SWEEP_THREADS, 1)
sweep_kernel(const SweepArgs a)
{
    extern __shared__ __align__(1024) uint8_t smem[];
    const int tid = threadIdx.x, lane = tid & 31;
    const int W = a.words, T = a.n_types;
    const int wid = tid >> 5;
    const int dbg = a.sweep_flags >> 8;       /* debug switch: 1 = no standing decisions (ordinary path for every pod) */
    SweepCtx cx;
    cx.lane = lane;
    cx.ft = nullptr;
    cx.smemo_mask = SMEMO_SLOTS - 1;
    cx.dmemo_mask = DMEMO_SLOTS - 1;
    cx.spmemo_mask = SPMEMO_SLOTS - 1;
    cx.clsnic_mask = CLSNIC_SLOTS - 1;
    cx.dcache_mask = DCACHE_SLOTS - 1;
    cx.smemo = reinterpret_cast<uint4*>(smem);                                 /* SMEMO_SLOTS x 16 B */
    cx.dmemo = reinterpret_cast<uint4*>(smem + SMEMO_SLOTS * 16);              /* DMEMO_SLOTS x 48 B */
    cx.dcache = reinterpret_cast<uint4*>(smem + SMEMO_SLOTS * 16 + DMEMO_SLOTS * 48);   /* DCACHE_SLOTS x 32 B */
    int32_t* dtag_all = reinterpret_cast<int32_t*>(smem + SMEMO_SLOTS * 16 + DMEMO_SLOTS * 48 + DCACHE_SLOTS * 32);
    cx.dtag = dtag_all;
    ClsNic* clsnic_all = reinterpret_cast<ClsNic*>(dtag_all + DCACHE_SLOTS + 4);     /* CLSNIC_SLOTS x 48 B */
    uint4* spmemo_all = reinterpret_cast<uint4*>(clsnic_all + CLSNIC_SLOTS);         /* SPMEMO_SLOTS x 16 B */
    cx.clsnic = clsnic_all;
    cx.spmemo = spmemo_all;
    uint8_t* p0 = reinterpret_cast<uint8_t*>(spmemo_all + SPMEMO_SLOTS);
    PodType* s_types = reinterpret_cast<PodType*>(p0);
    cx.types_in_smem = T <= SWEEP_TYPES_SMEM_MAX;
    uint8_t* p1 = p0 + (cx.types_in_smem ? ((T * sizeof(PodType) + 15) & ~(size_t)15) : 0);
    uint8_t* s_eff = p1;                                                        /* [T][2][64] effective-fc tables */
    cx.s_eff = s_eff;
    uint16_t* s_needb = reinterpret_cast<uint16_t*>(p1 + (cx.types_in_smem ? (size_t)T * 128 : 0));   /* [T][2][32] */
    cx.s_needb = cx.types_in_smem ? s_needb : nullptr;
    uint8_t* p2 = reinterpret_cast<uint8_t*>(s_needb) + (cx.types_in_smem ? (size_t)T * 128 : 0);
    int32_t* s_cursors = reinterpret_cast<int32_t*>(p2);                        /* [T][3] */
    uint8_t* p3 = p2 + (((size_t)T * 3 * 4 + 15) & ~(size_t)15);
    /* standing decisions and their tables (constant clock, one lane per type) */
    const bool fast_cap = cx.types_in_smem && T <= FAST_MAX_TYPES;
    uint8_t* s_tb = p3;                                                         /* [T][2][2][64] */
    uint16_t* s_gd = reinterpret_cast<uint16_t*>(s_tb + (fast_cap ? (size_t)T * 256 : 0));               /* [T][2][4] */
    TyFast* s_ty = reinterpret_cast<TyFast*>(s_gd + (fast_cap ? (size_t)T * 8 : 0));                       /* [T] */
    uint32_t* s_sub0s = reinterpret_cast<uint32_t*>(s_ty + (fast_cap ? T : 0));                            /* [T][FAST_NSIG_SMEM][16] */
    uint32_t* s_sub1s = s_sub0s + (fast_cap ? (size_t)T * FAST_NSIG_SMEM * 16 : 0);
    uint8_t* s_mapt = reinterpret_cast<uint8_t*>(s_sub1s + (fast_cap ? (size_t)T * FAST_NSIG_SMEM * 16 : 0));   /* MAPT_BYTES (+ pad) */
    int* s_cnt = reinterpret_cast<int*>(s_mapt + (fast_cap ? ((MAPT_BYTES + 15) & ~15) : 0));              /* [T + 2] candidate counts, CPU-only pods, flag */
    uint64_t* s_touched = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(s_cnt) + (fast_cap ? (((size_t)(T + 2) * 4 + 15) & ~(size_t)15) : 0));   /* [W] */
    uint64_t* s_bitmaps = s_touched + W;

    if (fast_cap && tid < T + 2) s_cnt[tid] = 0;
    __syncthreads();
    for (int i = tid; i < SMEMO_SLOTS + DMEMO_SLOTS * 3; i += SWEEP_THREADS)
        reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
    for (int i = tid; i < CLSNIC_SLOTS * 3 + SPMEMO_SLOTS; i += SWEEP_THREADS) reinterpret_cast<uint4*>(clsnic_all)[i] = make_uint4(0, 0, 0, 0);
    for (int i = tid; i < DCACHE_SLOTS; i += SWEEP_THREADS) dtag_all[i] = -1;
    for (int i = tid; i < W; i += SWEEP_THREADS) s_touched[i] = 0;
    const bool have_tables = fast_cap && a.ftab != nullptr && !(dbg & 4);
    const bool fast = have_tables && a.dual != 0 && a.n_names == 0 && !(dbg & 1);
    if (have_tables) {
        for (int i = tid; i < (MAPT_BYTES + 15) / 16; i += SWEEP_THREADS)
            reinterpret_cast<uint4*>(s_mapt)[i] = reinterpret_cast<const uint4*>(a.mapt)[i];
        /* the direct-path tables of this batch's pod types (fast_tables_kernel): one contiguous copy; the
         * shared-memory areas s_tb | s_gd | s_ty are laid out like the head of the buffer; the NIC-stage tables
         * (SUB0 / SUB1: one row per NIC signature, up to FAST_NSIG of them) stay in global memory, read through L1 */
        for (int i = tid; i < (int)(ftab_small_bytes(T) / 16); i += SWEEP_THREADS)
            reinterpret_cast<uint4*>(s_tb)[i] = reinterpret_cast<const uint4*>(a.ftab)[i];
        for (int i = tid; i < T * FAST_NSIG_SMEM * 16; i += SWEEP_THREADS) {        /* rows of the first signatures */
            const int tt = i / (FAST_NSIG_SMEM * 16), r = i % (FAST_NSIG_SMEM * 16);
            s_sub0s[i] = reinterpret_cast<const uint32_t*>(a.ftab + ftab_off_sub0(T))[tt * FAST_NSIG * 16 + r];
            s_sub1s[i] = reinterpret_cast<const uint32_t*>(a.ftab + ftab_off_sub1(T))[tt * FAST_NSIG * 16 + r];
        }
    }
    if (fast) {
        /* "no CPU-only pod can spill" certificate: a CPU-only pod touches one node, and a node no pod of the batch
         * was bound to keeps its exact snapshot bit; a type with more GPU-less candidates than there are CPU-only
         * pods therefore never runs out of them (or it has no candidate anywhere).  Then CPU-only pods only ever
         * touch GPU-less nodes, GPU pods only GPU nodes, and the two classes can be swept side by side. */
        {
            const uint64_t* gb = a.bitmaps;                                  /* HBM copy: the shared-memory one is still being staged */
            for (int tt = 0; tt < T; tt++) {
                const PodType& ty = a.types[tt];
                if (ty.needs_gpu || !ty.valid_map) continue;
                int c0 = 0, c1 = 0;
                for (int w = tid; w < W; w += SWEEP_THREADS) {
                    const uint64_t f = gb[(size_t)tt * W + w];
                    c0 += popc64(f & gb[(size_t)T * W + w]);
                    c1 += f != 0;
                }
                if (c0) atomicAdd(&s_cnt[tt], c0);
                if (c1) atomicOr(&s_cnt[T + 1], 1 << (tt & 31));              /* the type has candidates at all */
            }
            int nc = 0;
            for (int i = tid; i < a.n_pods; i += SWEEP_THREADS) nc += a.types[a.pod_type[i]].needs_gpu ? 0 : 1;
            if (nc) atomicAdd(&s_cnt[T], nc);
        }
    }
    if (cx.types_in_smem) {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(a.types);
        uint32_t* dst = reinterpret_cast<uint32_t*>(s_types);
        for (int i = tid; i < T * (int)(sizeof(PodType) / 4); i += SWEEP_THREADS) dst[i] = src[i];
        /* effective free-core count: the largest sum of a sub-set of the type's per-group demands that
         * does not exceed c — all the tuple predicates can ever learn about a socket with c free cores */
        for (int i = tid; i < T * 128; i += SWEEP_THREADS) {
            const int tt = i >> 7, f = (i >> 6) & 1, c = i & 63;
            const PodType& ty = a.types[tt];
            const uint8_t* cl = f ? ty.cl_smt : ty.cl_nosmt;
            const int n = ty.G + 1;
            int best = 0;
            for (int sub = 0; sub < (1 << n); sub++) {
                int sum = 0;
                for (int b = 0; b < n; b++) if ((sub >> b) & 1) sum += cl[b];
                if (sum <= c && sum > best) best = sum;
            }
            s_eff[i] = (uint8_t)best;
        }
        /* per-tuple socket demand on 2-NUMA nodes (Matcher.py:203-212 with K = 2) */
        for (int i = tid; i < T * 64; i += SWEEP_THREADS) {
            const int tt = i >> 6, f = (i >> 5) & 1, q = i & 31;
            const PodType& ty = a.types[tt];
            const uint8_t* cl = f ? ty.cl_smt : ty.cl_nosmt;
            const int L = ty.G + 1;
            int n0 = 0, n1 = 0;
            if (q < (1 << L)) {
                for (int g = 0; g < L; g++) { if ((q >> (L - 1 - g)) & 1) n1 += cl[g]; else n0 += cl[g]; }
            } else { n0 = n1 = 255; }
            s_needb[i] = (uint16_t)((n0 > 255 ? 255 : n0) | ((n1 > 255 ? 255 : n1) << 8));
        }
    }
    if (SMEM_BITMAPS) {
        const uint4* src = reinterpret_cast<const uint4*>(a.bitmaps);
        uint4* dst = reinterpret_cast<uint4*>(s_bitmaps);
        const int n16 = (T + 2 + a.n_names) * W / 2;
        for (int i = tid; i < n16; i += SWEEP_THREADS) dst[i] = src[i];
    }
    /* cursors[t*3 + 0/1]: first word that may hold a candidate (pass 0 / 1); [t*3 + 2]: first
     * word that may hold a NON-BUSY candidate (valid while the clock stands still) */
    int32_t* cursors = s_cursors;
    for (int i = tid; i < T * 3; i += SWEEP_THREADS) cursors[i] = 0;
    __syncthreads();
    /* side-by-side mode: CTA 0 sweeps the CPU-only pods, CTA 1 the GPU pods (see the certificate above; both CTAs
     * compute it from the same inputs); with a busy window every GPU pod of the batch lands on a node no pod was
     * bound to, so CTA 1 only scans and stamps */
    bool split = false;
    if (fast && a.min_busy > 0.0 && !(dbg & 2) && !(a.sweep_flags & 1)) {
        split = true;
        for (int tt = 0; tt < T; tt++) {
            const PodType& ty = a.types[tt];
            if (ty.needs_gpu || !ty.valid_map) continue;
            if (!(s_cnt[tt] > s_cnt[T] || !((s_cnt[T + 1] >> (tt & 31)) & 1))) split = false;
        }
    }
    /* the sweep proper is one warp; side by side: warp 0 of CTA 0 takes the CPU-only pods, warp 0 of CTA 1 (its own
     * SM, its own copy of the bitmaps) the GPU pods — the two classes share nothing they both write */
    if (wid >= 1 || (blockIdx.x == 1 && !split)) return;
    if (blockIdx.x == 1) {
        uint64_t* const BMg = SMEM_BITMAPS ? s_bitmaps : a.bitmaps;
        uint64_t* const BUSYg = BMg + (size_t)(T + 1) * W;
        int32_t* const curs = s_cursors;
        const PodType* tys = cx.types_in_smem ? s_types : a.types;
        for (int i0 = 0; i0 < a.n_pods; i0 += 32) {
            const int my_ti = (i0 + lane < a.n_pods) ? a.pod_type[i0 + lane] : 0;
            const double my_now = (i0 + lane < a.n_pods) ? a.now[i0 + lane] : 0.0;
            uint32_t todo = __ballot_sync(0xFFFFFFFFu, i0 + lane < a.n_pods && tys[my_ti].needs_gpu && tys[my_ti].valid_map);
            for (; todo; todo &= todo - 1) {
                const int j = ctz32(todo), i = i0 + j;
                const int ti = __shfl_sync(0xFFFFFFFFu, my_ti, j);
                const double now = __shfl_sync(0xFFFFFFFFu, my_now, j);
                const uint64_t* F = BMg + (size_t)ti * W;
                /* first candidate that is not busy (Matcher.py:107-111); every lane walks the same words */
                int c = curs[ti * 3 + 2];
                uint64_t w = 0;
                while (c < W) {
                    w = ldw<SMEM_BITMAPS>(&F[c]) & ~ldw<SMEM_BITMAPS>(&BUSYg[c]);
                    if (w) break;
                    c++;
                }
                __syncwarp();
                if (c >= W) {
                    if (lane < 8) reinterpret_cast<uint4*>(&a.out[i])[lane] = make_uint4(lane == 0 ? NHD_NO_CANDIDATE : 0, lane == 0 ? 0xFFFFFFFFu : 0, lane == 0 ? tys[ti].G : 0, 0);
                    if (lane == 8) curs[ti * 3 + 2] = c;
                    __syncwarp();
                    continue;
                }
                const int node = c * 64 + ctz64(w);
                /* stamp the node (NHDScheduler.py:289), note the pod for resolve_kernel, take the node out of this
                 * window's candidates (now - busy_time == 0 < MIN_BUSY_SECS): one store per lane */
                NodeDyn* gd = reinterpret_cast<NodeDyn*>(a.dyn) + node;
                if (lane == 0) gd->busy_time = now;
                else if (lane == 1) atomicOr(reinterpret_cast<unsigned int*>(&gd->gpu_used), (unsigned int)(NHD_DYN_TOUCHED | NHD_DYN_PENDING) << 16);
                else if (lane == 2) a.pend_pod[node] = i;
                else if (lane == 3) reinterpret_cast<uint2*>(&a.out[i])[0] = make_uint2(NHD_PENDING, (uint32_t)node);
                else if (lane == 4) bit_set(BUSYg, node);
                else if (lane == 5) bit_set(s_touched, node);
                else if (lane == 6) curs[ti * 3 + 2] = c;
                __syncwarp();
            }
        }
        return;
    }

    uint64_t* const BM = SMEM_BITMAPS ? s_bitmaps : a.bitmaps;
    uint64_t* const NOGPU = BM + (size_t)T * W;
    uint64_t* const BUSY = BM + (size_t)(T + 1) * W;
    const uint64_t* const GB = BM + (size_t)(T + 2) * W;
    const bool multi = a.n_names > 0;
    const PodType* types = cx.types_in_smem ? s_types : a.types;
    cx.types = types;
    const bool eager = T <= 64;
    /* the most demanding type decides whether a placement can have made the node unfit for anybody */
    int all_need = 0, all_big = 0, all_hp = 0, all_gpus = 0;
    for (int tt = 0; tt < T && eager; tt++) {
        const PodType& ty = types[tt];
        const int nd = ty.need_smt > ty.need_nosmt ? ty.need_smt : ty.need_nosmt;
        const int bg = ty.max_smt > ty.max_nosmt ? ty.max_smt : ty.max_nosmt;
        all_need = nd > all_need ? nd : all_need;
        all_big = bg > all_big ? bg : all_big;
        all_hp = ty.pod.hugepages_gb > all_hp ? ty.pod.hugepages_gb : all_hp;
        all_gpus = ty.total_gpus > all_gpus ? ty.total_gpus : all_gpus;
    }

    /* standing decisions: constant clock, the node-group gate folded into the types, one lane per type */
    const bool cclock = a.dual != 0;
    uint32_t cpu_mask = 0, gpu_mask = 0;
    unsigned long long gpu_pods_mask = 0;                   /* (side by side) types whose pods CTA 1 sweeps */
    FastTables ft;
    ft.tb = s_tb; ft.mapt = s_mapt; ft.gd = s_gd; ft.ty = s_ty; ft.cls = a.cls_fast;
    ft.sub0s = s_sub0s; ft.sub1s = s_sub1s;
    ft.sub0 = a.ftab ? reinterpret_cast<const uint32_t*>(a.ftab + ftab_off_sub0(T)) : nullptr;
    ft.sub1 = a.ftab ? reinterpret_cast<const uint32_t*>(a.ftab + ftab_off_sub1(T)) : nullptr;
    /* the general path (out of line) gets its own copy: taking the address of `ft` would move the hot loop's table
     * pointers from registers to local memory (measured: 9 % of the sweep) */
    FastTables ft_general = ft;
    SweepCtx cx_general = cx;        /* likewise the per-warp view: ordinary_pod takes it by reference */
#ifdef NHD_CHECKS
    cx_general.ft = nullptr;         /* check builds re-derive the standing decisions with the independent warp-wide evaluation */
    (void)ft_general;
#else
    cx_general.ft = have_tables ? &ft_general : nullptr;
#endif
    DynU st_none;
    st_none.q[0] = make_uint4(0, 0, 0, 0); st_none.q[1] = st_none.q[0];
    NodeAux ax_none = {0, 0, 0, 0};
    /* lane t = pod type t: its type record and its standing decision live in registers */
    const int tl = lane < T ? lane : 0;
    TyFast myty;
    myty.G = 1; myty.n_misc = 0; myty.misc_smt = 0; myty.nic_groups = 0; myty.direct = 0; myty.hugepages_gb = 0;
    bool l_cpu = false, l_gpu = false, l_direct = false;
    LaneSlot sl;
    sl.node = -1; sl.kind = NHD_SLOT_SLOW; sl.dec = sl.w14 = 0; sl.after.q[0] = st_none.q[0]; sl.after.q[1] = st_none.q[0];
    sl.ax = ax_none; sl.c = -1; sl.w = 0;
    const double now0 = a.n_pods > 0 ? a.now[0] : 0.0;
    if (fast) {
        for (int tt = 0; tt < T; tt++) {
            const PodType& ty = types[tt];
            if (!ty.valid_map) continue;
            if (ty.needs_gpu) gpu_mask |= 1u << tt; else cpu_mask |= 1u << tt;
        }
        gpu_pods_mask = gpu_mask;
        if (split) gpu_mask = 0;                            /* CTA 1 sweeps the GPU pods */
        if (lane < T) myty = s_ty[lane];
        l_cpu = (cpu_mask >> lane) & 1; l_gpu = (gpu_mask >> lane) & 1;
        l_direct = l_cpu && myty.direct;
        lanes_refresh<SMEM_BITMAPS>(a, cx, ft, myty, tl, l_direct, l_cpu, l_gpu, sl, BM, NOGPU, BUSY, s_touched, W, cursors, now0,
                                    false, -1, st_none, ax_none, cpu_mask, gpu_mask);
    }

    /* busy list from the BUSY snapshot (filter_kernel evaluated it for now[0]) */
    int n_busy = 0;
    for (int w0 = 0; w0 < W && !cclock; w0 += 32) {      /* (a constant clock needs no list) */
        uint64_t word = (w0 + lane < W) ? ldw<SMEM_BITMAPS>(&BUSY[w0 + lane]) : 0;
        int cnt = popc64(word);
        int pre = cnt;                                   /* inclusive scan over lanes */
        for (int d = 1; d < 32; d <<= 1) {
            int v = __shfl_up_sync(0xFFFFFFFFu, pre, d);
            if (lane >= d) pre += v;
        }
        int pos = n_busy + pre - cnt;
        while (word) {
            a.busy_list[pos++] = (w0 + lane) * 64 + ctz64(word);
            word &= word - 1;
        }
        n_busy += __shfl_sync(0xFFFFFFFFu, pre, 31);
    }
    __syncwarp();
    OrdState os;
    os.BM = BM; os.NOGPU = NOGPU; os.BUSY = BUSY; os.GB = GB; os.s_touched = s_touched; os.cursors = cursors; os.types = types;
    os.W = W; os.T = T; os.multi = multi; os.eager = eager; os.cclock = cclock; os.fast = fast;
    os.all_need = all_need; os.all_big = all_big; os.all_hp = all_hp; os.all_gpus = all_gpus;
    os.n_busy = n_busy;
    os.cur_now = a.n_pods > 0 ? a.now[0] : 0.0;
    os.busy_oldest = -1e300;              /* oldest stamp on the busy list; unknown for the snapshot's list: first clock step scans */
    PROF_DECL

    for (int i0 = 0; i0 < a.n_pods; i0 += 32) {
      /* the next 32 pods' types and clocks in one coalesced read */
      const int my_ti = (i0 + lane < a.n_pods) ? a.pod_type[i0 + lane] : 0;
      const double my_now = (i0 + lane < a.n_pods) ? a.now[i0 + lane] : 0.0;
      const unsigned long long my_gm = (multi && i0 + lane < a.n_pods) ? a.pod_groups[i0 + lane] : 0ULL;
      /* this CTA's pods of the chunk: all of them, or (side by side) all but the GPU pods CTA 1 sweeps */
      const bool in_chunk = i0 + lane < a.n_pods;
      uint32_t todo = __ballot_sync(0xFFFFFFFFu, in_chunk && !(split && ((gpu_pods_mask >> my_ti) & 1)));
      for (; todo; todo &= todo - 1) {
        const int j = ctz32(todo);
        const int i = i0 + j;
        const int ti = __shfl_sync(0xFFFFFFFFu, my_ti, j);
        const double now = cclock ? now0 : __shfl_sync(0xFFFFFFFFu, my_now, j);
        const unsigned long long gm = multi ? (__shfl_sync(0xFFFFFFFFu, my_gm, j) & a.names_used) : 0ULL;
        const PodType& t = types[ti];
        nhd_binding* bout = &a.out[i];
        uint64_t* F = BM + (size_t)ti * W;

        /* ---- standing decision of the pod's type (held by lane ti) ---- */
        bool handled = false, fast_commit = false;
        int commit_node = -1;                  /* node this pod changed (summary, BUSY / touched bits) */
        DynU da;
        da.q[0] = make_uint4(0, 0, 0, 0); da.q[1] = da.q[0];
        NodeAux dax = ax_none;
        if (fast) {
            const int kind = __shfl_sync(0xFFFFFFFFu, sl.kind, ti), node = __shfl_sync(0xFFFFFFFFu, sl.node, ti);
            if (kind == NHD_SLOT_FAST) {
                const uint32_t dec = __shfl_sync(0xFFFFFFFFu, sl.dec, ti), w14 = __shfl_sync(0xFFFFFFFFu, sl.w14, ti);
                da.q[0].x = __shfl_sync(0xFFFFFFFFu, sl.after.q[0].x, ti); da.q[0].y = __shfl_sync(0xFFFFFFFFu, sl.after.q[0].y, ti);
                da.q[0].z = __shfl_sync(0xFFFFFFFFu, sl.after.q[0].z, ti); da.q[0].w = __shfl_sync(0xFFFFFFFFu, sl.after.q[0].w, ti);
                da.q[1].x = __shfl_sync(0xFFFFFFFFu, sl.after.q[1].x, ti); da.q[1].y = __shfl_sync(0xFFFFFFFFu, sl.after.q[1].y, ti);
                da.q[1].z = __shfl_sync(0xFFFFFFFFu, sl.after.q[1].z, ti); da.q[1].w = __shfl_sync(0xFFFFFFFFu, sl.after.q[1].w, ti);
                dax.iu = __shfl_sync(0xFFFFFFFFu, sl.ax.iu, ti); dax.li0 = __shfl_sync(0xFFFFFFFFu, sl.ax.li0, ti);
                dax.li1 = __shfl_sync(0xFFFFFFFFu, sl.ax.li1, ti); dax.sig = __shfl_sync(0xFFFFFFFFu, sl.ax.sig, ti);
#ifdef NHD_CHECKS
                {
                    DynU dx; load_dyn(a, cx, node, dx);
                    CHK_SANE(dx, node, 2);
                    if (dx.q[0].y != w14) CHK_FAIL(3, node, dx.q[0].y, w14);
                    PMap pmx = {0, 0, 0, 0}; Picks pkx; pkx.fail_status = 0; bool msx;
                    const int stx = resolve_decision(a, cx, ti, t, node, dx, pmx, pkx, msx);
                    if (stx < 2) CHK_FAIL(4, node, stx, 0);
                    else {
                        nhd_binding* scratch = &a.out[a.n_pods];      /* spare record behind the batch */
                        apply_decision(cx, t, node, dx.d, pmx, pkx, now, scratch);
                        __syncwarp();
                        if (!same_dyn(dx, da)) CHK_FAIL(5, node, dx.q[0].x, da.q[0].x);
                        /* the packed mapping: tuple, misc NUMA, NodeNic.idx per group */
                        const int ps = dec & 3, G = t.G;
                        uint32_t pn = 0, ix = 0; int k0 = 0, k1 = 0;
                        for (int g = 0; g < G; g++) {
                            const int numa = (ps >> (G - 1 - g)) & 1;
                            const uint32_t x = numa ? (((dec >> 16) & 0xFF) >> (2 * k1++)) & 3 : (((dec >> 8) & 0xFF) >> (2 * k0++)) & 3;
                            pn |= (uint32_t)numa << (8 * g); ix |= x << (8 * g);
                        }
                        if (pn != pmx.pn || ix != pmx.idx || ((dec >> 2) & 1) != pmx.ms) CHK_FAIL(8, node, dec, pmx.pn);
                    }
                    /* and it is the first fit of the GPU-less pass */
                    for (int w = lane; w < (node >> 6); w += 32)
                        if (ldw<SMEM_BITMAPS>(&F[w]) & ldw<SMEM_BITMAPS>(&NOGPU[w])) CHK_FAIL(6, node, w, 0);
                    if ((ldw<SMEM_BITMAPS>(&F[node >> 6]) & ldw<SMEM_BITMAPS>(&NOGPU[node >> 6])) & ((1ULL << (node & 63)) - 1)) CHK_FAIL(7, node, 0, 0);
                    if (!((ldw<SMEM_BITMAPS>(&F[node >> 6]) >> (node & 63)) & 1)) CHK_FAIL(9, node, 0, 0);
                }
#endif
                /* commit: summary (cache + HBM, written through), touched bit, packed binding */
                const int cs = node & cx.dcache_mask;
                __syncwarp();
                if (lane < 2) {
                    const uint4 half = lane == 0 ? da.q[0] : da.q[1];
                    cx.dcache[2 * cs + lane] = half;
                    a.dyn[(size_t)node * 2 + lane] = half;
                } else if (lane == 2) { cx.dtag[cs] = node; bit_set(s_touched, node); }
                else if (lane == 3) *reinterpret_cast<uint4*>(bout) = make_uint4(NHD_PENDING_FAST, (uint32_t)node, dec, w14);
                commit_node = node;
                handled = true; fast_commit = true;
                PROF_COUNT(13);
            } else if (kind == NHD_SLOT_DEFER) {
                /* stamp the node (NHDScheduler.py:289) and leave a note for resolve_kernel / a later visitor */
                const bool was_busy = ((ldw<SMEM_BITMAPS>(&BUSY[node >> 6]) >> (node & 63)) & 1) != 0;
                __syncwarp();
                if (lane == 0) {
                    NodeDyn* gd = reinterpret_cast<NodeDyn*>(a.dyn) + node;
                    gd->busy_time = now;
                    atomicOr(reinterpret_cast<unsigned int*>(&gd->gpu_used), (unsigned int)(NHD_DYN_TOUCHED | NHD_DYN_PENDING) << 16);
                    a.pend_pod[node] = i;
                    reinterpret_cast<uint2*>(bout)[0] = make_uint2(NHD_PENDING, (uint32_t)node);
                } else if (lane == 1) bit_set(s_touched, node);
                else if (lane == 2 && a.min_busy > 0.0 && !was_busy) bit_set(BUSY, node);      /* now - busy_time == 0 < MIN_BUSY_SECS */
                commit_node = node;
                handled = true;
                PROF_COUNT(12);
            } else if (kind == NHD_SLOT_NONE) {
                if (lane < 8) reinterpret_cast<uint4*>(bout)[lane] = make_uint4(lane == 0 ? NHD_NO_CANDIDATE : 0, lane == 0 ? 0xFFFFFFFFu : 0, lane == 0 ? t.G : 0, 0);
                handled = true;
            }
        }
        PROF_MARK(0);      /* pod header / standing decision */
        if (!handled) commit_node = ordinary_pod<SMEM_BITMAPS>(a, cx_general, os, i, ti, now, gm);
        __syncwarp();
        if (fast) {
            if (fast_commit) {
                lanes_refresh<SMEM_BITMAPS>(a, cx, ft, myty, tl, l_direct, l_cpu, l_gpu, sl, BM, NOGPU, BUSY, s_touched, W, cursors, now,
                                            true, commit_node, da, dax, 0u, 0u);
            } else {
                /* every standing decision made for the node this pod changed is out of date; after the ordinary path
                 * the pod's own type as well (it may have given up the node its slot names) */
                uint32_t st = handled ? 0u : (1u << ti);
                if (commit_node >= 0) st |= __ballot_sync(0xFFFFFFFFu, sl.node == commit_node);
                if (st & (cpu_mask | gpu_mask))
                    lanes_refresh<SMEM_BITMAPS>(a, cx, ft, myty, tl, l_direct, l_cpu, l_gpu, sl, BM, NOGPU, BUSY, s_touched, W, cursors, now,
                                                false, -1, st_none, ax_none, st & cpu_mask, st & gpu_mask);
            }
        }
        PROF_MARK(6);      /* write-back + refresh */
      }
    }
    PROF_FLUSH(a.prof);
}

/*
 * Pods the sweep bound to a node without working out the mapping (first pod on an untouched
 * node): one thread per pod, all independent — the node's summary is still the snapshot's,
 * apart from the busy stamp.  Same arithmetic as the sweep's miss path, scalar.
 */
__global__ void resolve_kernel(const SweepArgs a)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n_pods) return;
    const int status = a.out[i].status;
    if (status == NHD_PENDING_FAST) {
        /* decided directly by the sweep: format the binding header from the packed mapping (the node's summary is
         * final already); same words as apply_decision writes */
        const uint4 hd = *reinterpret_cast<const uint4*>(&a.out[i]);
        const int node = (int)hd.y;
        const PodType& t = a.types[a.pod_type[i]];
        const int G = t.G, ps = hd.z & 3;
        const uint32_t ms = (hd.z >> 2) & 1, e0 = (hd.z >> 8) & 0xFF, e1 = (hd.z >> 16) & 0xFF;
        const uint4 c5 = *reinterpret_cast<const uint4*>(a.nodes + chunk_off(node, 5));
        uint32_t pn = 0, idx = 0, li = 0, rec = 0;
        int n_rec = 0, k0 = 0, k1 = 0;
        for (int g = 0; g < G; g++) {
            const int numa = (ps >> (G - 1 - g)) & 1;
            const uint32_t x = numa ? (e1 >> (2 * k1++)) & 3 : (e0 >> (2 * k0++)) & 3;
            const uint32_t l = (uint32_t)nth_bit32(numa ? c5.y : c5.x, (int)x);        /* NodeNic.idx -> index in Node.nics */
            pn |= (uint32_t)numa << (8 * g); idx |= x << (8 * g); li |= l << (8 * g);
            if ((t.nic_groups >> g) & 1) { rec |= l << (8 * n_rec); n_rec++; }
        }
        int ncl = 0;
        const uint32_t claimed = claimed_order_packed(rec, n_rec, ncl);                 /* NHDScheduler.py:302 */
        const uint32_t w2 = (uint32_t)G | ((uint32_t)ncl << 24);
        const uint32_t w4 = G < 4 ? (pn | (ms << (8 * G))) : pn;
        const uint32_t w5 = (G == 4 ? ms : 0u) | (pn << 8);
        const uint32_t w6 = (pn >> 24) | (idx << 8);
        const uint32_t w7 = (idx >> 24) | (li << 8);
        const uint32_t w8 = (li >> 24) | (claimed << 8);
        const uint32_t w9 = claimed >> 24;
        uint4* o = reinterpret_cast<uint4*>(&a.out[i]);
        o[0] = make_uint4(NHD_PLACED, (uint32_t)node, w2, pn);
        o[1] = make_uint4(w4, w5, w6, w7);
        o[2] = make_uint4(w8, w9, 0, 0);
        o[3] = make_uint4(0, 0, hd.w, 0);
        for (int c = 4; c < 8; c++) o[c] = make_uint4(0, 0, 0, 0);
        return;
    }
    if (status != NHD_PENDING) return;
    const int node = a.out[i].node;
    const PodType& t = a.types[a.pod_type[i]];
    RecU u;
#pragma unroll
    for (int c = 2; c < REC_CHUNKS; c++)
        u.q[c] = *reinterpret_cast<const uint4*>(a.nodes + chunk_off(node, c));
    DynU du;
    du.q[0] = a.dyn[(size_t)node * 2];
    du.q[1] = a.dyn[(size_t)node * 2 + 1];
    du.d.info &= ~NHD_DYN_PENDING;
    apply_dyn(u.r, du.d);
    union { nhd_binding b; uint4 q[8]; } bu;
    for (int c = 0; c < 8; c++) bu.q[c] = make_uint4(0, 0, 0, 0);
    bu.b.node = node;
    const uint64_t gsw = t.pci ? free_gpus_per_switch(u.r) : 0;
    Mapping m;
    bool mapped = false;
    if (u.r.n_numa == 2 && t.G >= 1 && t.G <= 2 && a.mapt2) {
        /* the common shape: stage masks without arrays, GetNumaGroupIdx from the table, then the first NIC entry of
         * the chosen tuple — the same values as the general branch below */
        Pre2 pre;
        make_pre2(u.r, du.d.fc[0], du.d.fc[1], pre);
        uint32_t mA, mB, mC;
        if (stage_masks_k2(u.r, t, a.cap, pre, mA, mB, mC)) {
            const uint32_t e = __ldg(&a.mapt2[t.G == 2 ? ((mA << 12) | (mB << 4) | mC) : (65536u + ((mA << 6) | (mB << 2) | mC))]);
            if (e & 0x80) {
                const int p0 = t.G == 2 ? (int)((e >> 1) & 1) : (int)(e & 1), p1 = (int)(e & 1);
                uint32_t idx = 0, li = 0;
                nic_first_fit2(u.r, t, p0, p1, a.cap, gsw, &idx, &li);
                m.gpu_numa[0] = (uint8_t)p0; m.gpu_numa[1] = (uint8_t)(t.G == 2 ? p1 : 0); m.gpu_numa[2] = m.gpu_numa[3] = 0;
                m.misc_numa = (uint8_t)((e >> 2) & 1);
                m.nic_idx[0] = (uint8_t)(idx & 0xFF); m.nic_idx[1] = (uint8_t)((idx >> 8) & 0xFF); m.nic_idx[2] = m.nic_idx[3] = 0;
                m.nic_li[0] = (uint8_t)(li & 0xFF); m.nic_li[1] = (uint8_t)((li >> 8) & 0xFF); m.nic_li[2] = m.nic_li[3] = 0;
                mapped = true;
            }
        }
    } else {
        TMask ma, mb, mc;
        int ps = 0, ms = 0;
        if (stage_masks_fc(u.r, du.d.fc, t, a.cap, gsw, ma, mb, mc) && choose_mapping(u.r.n_numa, t.G, ma, mb, mc, &ps, &ms)) {
            tuple_digits(ps, u.r.n_numa, t.G, m.gpu_numa);
            m.misc_numa = (uint8_t)ms;
            nic_first_fit(u.r, t, m.gpu_numa, u.r.n_numa, a.cap, gsw, m.nic_idx, m.nic_li);
            mapped = true;
        }
    }
    if (mapped) {
        assign_resources(u.r, du.d, t, m, du.d.busy_time, &bu.b);
    } else {
        bu.b.status = NHD_NO_CANDIDATE;        /* cannot happen: the snapshot bit said feasible */
        bu.b.node = -1;
    }
    a.dyn[(size_t)node * 2] = du.q[0];
    a.dyn[(size_t)node * 2 + 1] = du.q[1];
    for (int c = 0; c < 8; c++) reinterpret_cast<uint4*>(&a.out[i])[c] = bu.q[c];
}

/* ------------------------------------------------------------------ core ids + commit */

struct FinishArgs {
    uint8_t* nodes;
    const PodType* types;
    const int32_t* pod_type;
    nhd_binding* out;
    const uint4* dyn;
    int n_pods;
};

/* stage A: the logical core ids of every placed pod, all pods in parallel, from the records as
 * they were at the start of the batch (the sweep never writes them) and the prefix offsets. */
__global__ void assign_cores_kernel(const FinishArgs a)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n_pods) return;
    union { nhd_binding b; uint4 q[8]; } bu;
    for (int c = 0; c < 8; c++) bu.q[c] = reinterpret_cast<const uint4*>(&a.out[i])[c];
    if (bu.b.status != NHD_PLACED) return;
    RecU u;
    load_rec(a.nodes, bu.b.node, u);
    assign_cores_from_snapshot(u.r, a.types[a.pod_type[i]], &bu.b);
    for (int c = 0; c < 8; c++) reinterpret_cast<uint4*>(&a.out[i])[c] = bu.q[c];
}

/* commit: fold the batch into the records (core masks by atomic OR, the rest from the summaries) */
__global__ void commit_kernel(const FinishArgs a)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n_pods) return;
    const nhd_binding* b = &a.out[i];
    const int node = b->node;
    if (node < 0) return;
    if (b->status == NHD_PLACED) {
        unsigned long long m[4] = {0, 0, 0, 0};
        for (int k = 0; k < b->n_cores; k++) m[b->cores[k] >> 6] |= 1ULL << (b->cores[k] & 63);
        for (int w = 0; w < 4; w++)
            if (m[w]) atomicOr(reinterpret_cast<unsigned long long*>(a.nodes + chunk_off(node, w >> 1) + (w & 1) * 8), m[w]);
    }
    /* every pod bound to this node writes the node's final summary: identical values */
    const NodeDyn d = reinterpret_cast<const NodeDyn*>(a.dyn)[node];
    uint8_t* c2 = a.nodes + chunk_off(node, 2);
    *reinterpret_cast<uint16_t*>(c2 + 0) = d.gpu_used;
    *reinterpret_cast<uint32_t*>(c2 + 4) = d.nic_inuse;
    *reinterpret_cast<int32_t*>(c2 + 8) = d.free_hugepages_gb;
    *reinterpret_cast<double*>(a.nodes + chunk_off(node, 3)) = d.busy_time;
}

/* ------------------------------------------------------------------ explanation (nhd_explain) */

constexpr int EXPLAIN_THREADS = 256;
constexpr int EXPLAIN_NONE = 0x7FFFFFFF;          /* first-fit slot before any feasible node is seen */

struct ExplainArgs {
    const uint8_t* nodes;        /* tiled node array (read only) */
    const PodType* types;        /* [n_types] explain types: descriptor with the pod's own group mask */
    const double* now;           /* [n_types] clock of each explain type */
    int n_types;
    int n_nodes;
    int32_t* counts;             /* [n_types][NHD_WHY_COUNT], zeroed by the caller */
    int32_t* first;              /* [n_types][2]: first feasible node, first feasible node without GPUs (EXPLAIN_NONE) */
    uint8_t* reasons;            /* [n_types][n_nodes] or null */
    double min_busy;
    double cap[NHD_MAX_SPEED_CLASSES];
};

/* One thread per (node, explain type): blockIdx.y = type, 32 consecutive nodes per warp, so each 16-byte chunk of
 * the tiled records is one 512-byte coalesced read per warp.  Counts are summed per warp (one ballot per reason,
 * one atomicAdd per warp and non-zero reason); first fit takes the lowest lane of a ballot, one atomicMin per warp.
 * The node records are only read, and no buffer of the solve is touched. */
__global__ void __launch_bounds__(EXPLAIN_THREADS)
explain_kernel(const ExplainArgs a)
{
    const int t = blockIdx.y;
    const int node = blockIdx.x * EXPLAIN_THREADS + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const bool valid = node < a.n_nodes;
    int why = -1;
    bool nogpu = false;
    if (valid) {
        RecU u;
        load_rec(a.nodes, node, u);
        why = node_reason(u.r, a.types[t], a.cap, a.now[t], a.min_busy);
        nogpu = u.r.n_gpus == 0;
        if (a.reasons) a.reasons[(size_t)t * a.n_nodes + node] = (uint8_t)why;
    }
    const int base = node - lane;
#pragma unroll
    for (int w = 0; w < NHD_WHY_COUNT; w++) {
        const uint32_t bal = __ballot_sync(0xFFFFFFFFu, why == w);
        if (lane == 0 && bal) atomicAdd(&a.counts[t * NHD_WHY_COUNT + w], popc32(bal));
        if (w == NHD_WHY_FEASIBLE) {
            const uint32_t ng = __ballot_sync(0xFFFFFFFFu, why == w && nogpu);
            if (lane == 0 && bal) atomicMin(&a.first[t * 2 + 0], base + ctz32(bal));
            if (lane == 0 && ng) atomicMin(&a.first[t * 2 + 1], base + ctz32(ng));
        }
    }
}

} // namespace nhd
