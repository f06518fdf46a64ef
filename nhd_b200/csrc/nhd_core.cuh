/*
 * nhd_core.cuh — per-(pod type, node) placement arithmetic of the B200 solver.
 *
 * Everything here is scalar, branch-light bitmask code over the packed
 * nhd_node_rec (include/nhd_b200.h).  The CUDA kernels (nhd_kernels.cu) call
 * these functions from the snapshot predicate kernel (one thread per node) and
 * from the sequential select+assign sweep.  The functions are
 * __host__ __device__ only so that tests/emu can compile the very same logic
 * with g++ and diff it against the oracle without a GPU; the shipped library
 * never runs them on the host.
 *
 * What each block replaces in the reference (file:line under /root/reference):
 *   free_cores / free_gpus / nic tables   nhd/Node.py:250-296, 456-462
 *   gpu_ok / cpu_ok / nic_first_fit       nhd/Matcher.py:95-276 (+ PCI pruning :295-335)
 *   choose_mapping (+ the set emulator)   nhd/Matcher.py:337-389, 423-452
 *   cpu_batch                             nhd/Node.py:502-519
 *   assign_pod                            nhd/Node.py:663-841, nhd/NHDScheduler.py:289,302-304
 */
#pragma once

#include <stdint.h>
#include "../../include/nhd_b200.h"

#if defined(__CUDACC__)
#define NHD_HD __host__ __device__ __forceinline__
#define NHD_HDN __host__ __device__ __noinline__
#else
#define NHD_HD inline
#define NHD_HDN inline
#endif

namespace nhd {

/* ---------------------------------------------------------------- bit helpers */
NHD_HD int popc32(uint32_t x)
{
#ifdef __CUDA_ARCH__
    return __popc(x);
#else
    return __builtin_popcount(x);
#endif
}
NHD_HD int popc64(uint64_t x)
{
#ifdef __CUDA_ARCH__
    return __popcll(x);
#else
    return __builtin_popcountll(x);
#endif
}
NHD_HD int ctz32(uint32_t x)      /* x != 0 */
{
#ifdef __CUDA_ARCH__
    return __ffs((int)x) - 1;
#else
    return __builtin_ctz(x);
#endif
}
NHD_HD int ctz64(uint64_t x)      /* x != 0 */
{
#ifdef __CUDA_ARCH__
    return __ffsll((long long)x) - 1;
#else
    return __builtin_ctzll(x);
#endif
}
/* index of the n-th (0-based) set bit of x, -1 if fewer */
NHD_HD int nth_bit32(uint32_t x, int n)
{
    for (; n > 0 && x; n--) x &= x - 1;          /* n is tiny (a per-NUMA NIC index) */
    return x ? ctz32(x) : -1;
}

/* 256-bit core mask (logical core c = bit c) */
struct M256 { uint64_t w[4]; };

NHD_HD M256 m_zero() { M256 r; r.w[0] = r.w[1] = r.w[2] = r.w[3] = 0; return r; }
NHD_HD M256 m_and(const M256& a, const M256& b) { M256 r; for (int i = 0; i < 4; i++) r.w[i] = a.w[i] & b.w[i]; return r; }
NHD_HD M256 m_or(const M256& a, const M256& b) { M256 r; for (int i = 0; i < 4; i++) r.w[i] = a.w[i] | b.w[i]; return r; }
NHD_HD M256 m_andnot(const M256& a, const M256& b) { M256 r; for (int i = 0; i < 4; i++) r.w[i] = a.w[i] & ~b.w[i]; return r; }
NHD_HD int  m_popc(const M256& a) { return popc64(a.w[0]) + popc64(a.w[1]) + popc64(a.w[2]) + popc64(a.w[3]); }
NHD_HD bool m_test(const M256& a, int c) { return (a.w[c >> 6] >> (c & 63)) & 1; }
NHD_HD void m_set(M256& a, int c) { a.w[c >> 6] |= 1ULL << (c & 63); }
NHD_HD void m_clr(M256& a, int c) { a.w[c >> 6] &= ~(1ULL << (c & 63)); }
/* bits [lo, hi) */
NHD_HD M256 m_range(int lo, int hi)
{
    M256 r;
    for (int i = 0; i < 4; i++) {
        int a = lo - 64 * i, b = hi - 64 * i;
        a = a < 0 ? 0 : a;
        b = b > 64 ? 64 : b;
        uint64_t m = 0;
        if (b > a) m = (b - a == 64) ? ~0ULL : (((1ULL << (b - a)) - 1) << a);
        r.w[i] = m;
    }
    return r;
}
NHD_HD M256 m_shr(const M256& a, int s)   /* 0 <= s < 256 */
{
    M256 r;
    int ws = s >> 6, bs = s & 63;
    for (int i = 0; i < 4; i++) {
        uint64_t lo = (i + ws < 4) ? a.w[i + ws] : 0;
        uint64_t hi = (i + ws + 1 < 4) ? a.w[i + ws + 1] : 0;
        r.w[i] = bs ? ((lo >> bs) | (hi << (64 - bs))) : lo;
    }
    return r;
}
NHD_HD M256 m_shl(const M256& a, int s)   /* 0 <= s < 256 */
{
    M256 r;
    int ws = s >> 6, bs = s & 63;
    for (int i = 3; i >= 0; i--) {
        uint64_t hi = (i - ws >= 0) ? a.w[i - ws] : 0;
        uint64_t lo = (i - ws - 1 >= 0) ? a.w[i - ws - 1] : 0;
        r.w[i] = bs ? ((hi << bs) | (lo >> (64 - bs))) : hi;
    }
    return r;
}

/* ---------------------------------------------------------------- pod type */

/* Device-side pod type: the wire descriptor plus the request vectors of
 * CfgTopology.GetTotal{Gpus,Cpus,NICs}Requested (CfgTopology.py:199-232) and the
 * per-group physical-core demand of Matcher.py:179-201, all precomputed once per
 * distinct descriptor by the host. */
struct PodType {
    nhd_pod pod;
    uint8_t G;
    uint8_t needs_gpu;                 /* sum(req_gpus) > 0 (Matcher.py:107) == any group has GPUs (:406-410) */
    uint8_t pci;                       /* map_type == PCI */
    uint8_t valid_map;                 /* map_type in {NUMA, PCI} (Matcher.py:45) */
    uint8_t tot[NHD_MAX_GROUPS];       /* len(proc_cores) + sum(len(gpu.cpu_cores)) */
    uint8_t cl_smt[NHD_MAX_GROUPS + 1];    /* physical cores needed on an SMT node, [G] = misc */
    uint8_t cl_nosmt[NHD_MAX_GROUPS + 1];  /* ... on a non-SMT node */
    uint8_t total_gpus;
    uint8_t need_smt;                  /* sum of cl_smt (saturated at 255): no tuple ever asks a socket for more */
    uint8_t need_nosmt;
    uint8_t max_smt;                   /* largest single entry of cl_smt: some socket must offer that much */
    uint8_t max_nosmt;
    uint8_t has_bw;                    /* some group asks for NIC bandwidth (rx or tx > 0) */
    uint8_t nic_groups;                /* bit g: group g has RX/TX cores, i.e. claims its NIC (Node.py:742-755) */
    uint8_t pad2_[7];
};

NHD_HD void make_pod_type(const nhd_pod& p, PodType& t)
{
    t.pod = p;
    t.G = p.n_groups;
    t.pci = p.map_type == NHD_MAP_PCI;
    t.valid_map = (p.map_type == NHD_MAP_NUMA || p.map_type == NHD_MAP_PCI);
    int gpus = 0;
    for (int g = 0; g < NHD_MAX_GROUPS + 1; g++) t.cl_smt[g] = t.cl_nosmt[g] = 0;
    for (int g = 0; g < NHD_MAX_GROUPS; g++) t.tot[g] = 0;
    for (int g = 0; g < p.n_groups && g < NHD_MAX_GROUPS; g++) {
        const nhd_pod_group& pg = p.groups[g];
        int tot = pg.n_proc;
        for (int j = 0; j < pg.n_gpus && j < NHD_MAX_GROUP_GPUS; j++) tot += pg.gpu_feeders[j];
        gpus += pg.n_gpus;
        t.tot[g] = (uint8_t)tot;
        int a = (pg.flags & NHD_GRP_PROC_SMT) ? (tot + 1) / 2 : tot;                    /* Matcher.py:182-185 */
        int b = (pg.flags & NHD_GRP_HELPER_SMT) ? (pg.n_helpers + 1) / 2 : pg.n_helpers; /* :187-190 */
        t.cl_smt[g] = (uint8_t)(a + b);
        t.cl_nosmt[g] = (uint8_t)(tot + pg.n_helpers);                                    /* :194 */
    }
    /* Matcher.py:197-201: on SMT nodes the misc cores are always halved (the SMT flag
     * tested there is an Enum member, hence always true). */
    if (p.n_groups <= NHD_MAX_GROUPS) {
        t.cl_smt[p.n_groups] = (uint8_t)((p.n_misc + 1) / 2);
        t.cl_nosmt[p.n_groups] = p.n_misc;
    }
    t.total_gpus = (uint8_t)gpus;
    t.needs_gpu = gpus > 0;
    int ns = 0, nn = 0;
    for (int g = 0; g <= NHD_MAX_GROUPS; g++) { ns += t.cl_smt[g]; nn += t.cl_nosmt[g]; }
    t.need_smt = (uint8_t)(ns > 255 ? 255 : ns);
    t.need_nosmt = (uint8_t)(nn > 255 ? 255 : nn);
    int ms = 0, mn = 0, bw = 0;
    for (int g = 0; g <= NHD_MAX_GROUPS; g++) { ms = t.cl_smt[g] > ms ? t.cl_smt[g] : ms; mn = t.cl_nosmt[g] > mn ? t.cl_nosmt[g] : mn; }
    for (int g = 0; g < p.n_groups && g < NHD_MAX_GROUPS; g++)
        if (p.groups[g].rx_gbps > 0.0 || p.groups[g].tx_gbps > 0.0) bw = 1;
    t.max_smt = (uint8_t)ms; t.max_nosmt = (uint8_t)mn; t.has_bw = (uint8_t)bw;
    t.nic_groups = 0;
    for (int g = 0; g < p.n_groups && g < NHD_MAX_GROUPS; g++)
        if (p.groups[g].flags & NHD_GRP_HAS_NIC_CORES) t.nic_groups |= (uint8_t)(1u << g);
    for (int i = 0; i < 7; i++) t.pad2_[i] = 0;
}

/* ---------------------------------------------------------------- record validation */

/* Limits of the packed layout and internal consistency of one nhd_node_rec (include/nhd_b200.h).
 * 0 = ok, -1 = malformed, -2 = valid for the reference but outside the packed limits. */
NHD_HD int validate_node_rec(const nhd_node_rec& r)
{
    const int K = r.n_numa;
    if (K < 1 || K > NHD_MAX_NUMA) return -2;
    const int phys = r.phys_cores;
    const bool smt = (r.flags & NHD_NODE_SMT) != 0;
    if (phys < 1 || phys % K != 0) return -2;
    if ((smt ? 2 * phys : phys) > NHD_MAX_LCORES) return -2;
    if (r.n_gpus > NHD_MAX_GPUS || r.n_nics > NHD_MAX_NICS) return -2;
    uint32_t gseen = 0, nseen = 0;
    for (int k = 0; k < NHD_MAX_NUMA; k++) {
        if (k >= K && (r.gpu_numa_mask[k] || r.nic_numa_mask[k])) return -1;
        if ((gseen & r.gpu_numa_mask[k]) || (nseen & r.nic_numa_mask[k])) return -1;
        gseen |= r.gpu_numa_mask[k];
        nseen |= r.nic_numa_mask[k];
    }
    const uint32_t gall = r.n_gpus ? ((1u << r.n_gpus) - 1) : 0;
    const uint32_t nall = r.n_nics >= 32 ? 0xFFFFFFFFu : ((1u << r.n_nics) - 1);
    if (gseen != gall || nseen != nall) return -1;
    if ((r.gpu_used & ~gall) || (r.nic_inuse & ~nall)) return -1;
    const double bt = r.busy_time;
    if (!(bt == bt) || bt > 1.7e308 || bt < -1.7e308) return -1;       /* NaN / infinity */
    return 0;
}

/* ---------------------------------------------------------------- node queries */

NHD_HD M256 rec_used(const nhd_node_rec& r) { M256 m; for (int i = 0; i < 4; i++) m.w[i] = r.used[i]; return m; }
NHD_HD bool rec_smt(const nhd_node_rec& r) { return (r.flags & NHD_NODE_SMT) != 0; }

/* physical cores c < phys whose hyperthreads are all unused (Node.py:257-262) */
NHD_HD M256 eligible_phys(const nhd_node_rec& r)
{
    M256 u = rec_used(r);
    M256 e = m_andnot(m_range(0, r.phys_cores), u);
    if (rec_smt(r)) e = m_andnot(e, m_shr(u, r.phys_cores));
    return e;
}

/* Node.GetFreeCpuCores (Node.py:250-264) */
NHD_HD void free_cores(const nhd_node_rec& r, int* fc)
{
    M256 e = eligible_phys(r);
    int per = r.phys_cores / r.n_numa;
    for (int k = 0; k < r.n_numa; k++) fc[k] = m_popc(m_and(e, m_range(k * per, (k + 1) * per)));
}

/* Node.GetFreeNumaGPUs (Node.py:456-462) */
NHD_HD void free_gpus(const nhd_node_rec& r, int* fg)
{
    uint32_t fr = ~(uint32_t)r.gpu_used & ((1u << r.n_gpus) - 1);
    for (int k = 0; k < r.n_numa; k++) fg[k] = popc32(fr & r.gpu_numa_mask[k]);
}

NHD_HD int gpu_switch(const nhd_node_rec& r, int i) { return (int)((r.gpu_sw >> (4 * i)) & 0xF); }
NHD_HD int nic_switch(const nhd_node_rec& r, int i) { return (int)((r.nic_sw[i >> 4] >> (4 * (i & 15))) & 0xF); }
NHD_HD int nic_speed_class(const nhd_node_rec& r, int i) { return (int)((r.nic_speed[i >> 4] >> (4 * (i & 15))) & 0xF); }

/* Node.GetFreeGPUPCICount (Node.py:266-273): free GPUs per local switch id, packed 4 bits each
 * (a node has at most 16 GPUs, but a count of 16 would not fit: saturate at 15, which is
 * still >= NHD_MAX_GROUPS, the largest value it is ever compared with). */
NHD_HD uint64_t free_gpus_per_switch(const nhd_node_rec& r)
{
    uint64_t cnt = 0;
    uint32_t fr = ~(uint32_t)r.gpu_used & ((1u << r.n_gpus) - 1);
    while (fr) {
        int i = ctz32(fr);
        fr &= fr - 1;
        int s = gpu_switch(r, i);
        if (((cnt >> (4 * s)) & 0xF) < 15) cnt += 1ULL << (4 * s);
    }
    return cnt;
}

/* Node.GetFreeNumaNicResources (Node.py:283-296), sharing disabled: a NIC offers
 * speed * NIC_BW_AVAIL_PERCENT in each direction, or nothing once a pod uses it. */
NHD_HD double nic_free_bw(const nhd_node_rec& r, int li, const double* cap)
{
    return ((r.nic_inuse >> li) & 1) ? 0.0 : cap[nic_speed_class(r, li)];
}

/* Node.IsBusy (Node.py:847-850) */
NHD_HD bool node_busy(const nhd_node_rec& r, double now, double min_busy)
{
    return (now - r.busy_time) < min_busy;
}

/* Pod-independent gates: InitialNodeFilter (NHDScheduler.py:241-243) and
 * FilterPodResources (Matcher.py:73,78). */
NHD_HD bool node_gates(const nhd_node_rec& r, const PodType& t)
{
    if (!(r.flags & NHD_NODE_ACTIVE)) return false;
    if ((r.group_mask & t.pod.group_mask) == 0) return false;
    if (r.flags & NHD_NODE_MAINTENANCE) return false;
    if (t.pod.hugepages_gb > r.free_hugepages_gb) return false;
    return true;
}

/* ---------------------------------------------------------------- NUMA tuples */

/* tuple #idx of itertools.product(range(K), repeat=L): first element most significant */
NHD_HD void tuple_digits(int idx, int K, int L, uint8_t* p)
{
    if (K == 2) { for (int i = L - 1; i >= 0; i--) { p[i] = (uint8_t)(idx & 1); idx >>= 1; } }
    else if (K == 4) { for (int i = L - 1; i >= 0; i--) { p[i] = (uint8_t)(idx & 3); idx >>= 2; } }
    else if (K == 1) { for (int i = 0; i < L; i++) p[i] = 0; }
    else { for (int i = L - 1; i >= 0; i--) { p[i] = (uint8_t)(idx % K); idx /= K; } }
}
NHD_HD int ipow(int K, int L) { int r = 1; for (int i = 0; i < L; i++) r *= K; return r; }

/* GPU stage predicate for one tuple (Matcher.py:121-129) */
NHD_HD bool gpu_ok(const PodType& t, const uint8_t* p, int K, const int* fg)
{
    int ttl[NHD_MAX_NUMA] = {0, 0, 0, 0};
    for (int g = 0; g < t.G; g++) ttl[p[g]] += t.pod.groups[g].n_gpus;
    for (int k = 0; k < K; k++) if (ttl[k] > fg[k]) return false;
    return true;
}

/* CPU stage predicate for one (G+1)-tuple (Matcher.py:204-212); m = NUMA node of the misc cores */
NHD_HD bool cpu_ok(const PodType& t, const uint8_t* p, int m, int K, const int* fc, bool smt)
{
    const uint8_t* cl = smt ? t.cl_smt : t.cl_nosmt;
    int ttl[NHD_MAX_NUMA] = {0, 0, 0, 0};
    for (int g = 0; g < t.G; g++) ttl[p[g]] += cl[g];
    ttl[m] += cl[t.G];
    for (int k = 0; k < K; k++) if (ttl[k] > fc[k]) return false;
    return true;
}

/*
 * NIC stage for one NUMA tuple p: the FIRST entry of filts['nic'] whose NUMA part is p,
 * after the PCI-switch pruning when map_type == PCI.
 *
 * The reference enumerates, for this p, every joint choice of per-NUMA NIC indices
 * (NUMA 0's combination most significant, inside a NUMA node the first group most
 * significant; Matcher.py:245-258), keeps the choices where no NIC goes negative after
 * subtracting the groups' (rx, tx) in group order (:261-268), and in PCI mode drops
 * choices that put more groups on a PCIe switch than it has free GPUs (:312-322).
 * Both constraints only tighten as groups are added (speeds are >= 0), so a
 * depth-first search in that same significance order with pruning returns exactly the
 * first surviving entry.  Returns false when no entry survives.
 */
NHD_HD bool nic_first_fit(const nhd_node_rec& r, const PodType& t, const uint8_t* p, int K,
                          const double* cap, uint64_t gsw, uint8_t* out_idx, uint8_t* out_li)
{
    const int G = t.G;
    int ord[NHD_MAX_GROUPS];
    int n = 0;
    for (int k = 0; k < K; k++)
        for (int g = 0; g < G; g++)
            if (p[g] == k) {
                if (r.nic_numa_mask[k] == 0) return false;      /* product(range(0), ...) is empty (:247) */
                ord[n++] = g;
            }
    int choice[NHD_MAX_GROUPS], li[NHD_MAX_GROUPS];
    double rrx[NHD_MAX_GROUPS], rtx[NHD_MAX_GROUPS];
    int d = 0;
    choice[0] = 0;
    for (;;) {
        const int g = ord[d];
        const uint32_t nm = r.nic_numa_mask[p[g]];
        const int l = nth_bit32(nm, choice[d]);
        if (l < 0) {                                           /* exhausted this level: backtrack */
            if (d == 0) return false;
            d--;
            choice[d]++;
            continue;
        }
        double rx = nic_free_bw(r, l, cap), tx = rx;
        for (int e = d - 1; e >= 0; e--)
            if (li[e] == l) { rx = rrx[e]; tx = rtx[e]; break; }
        rx -= t.pod.groups[g].rx_gbps;                          /* fp64, group order (:262-263) */
        tx -= t.pod.groups[g].tx_gbps;
        bool ok = !(rx < 0) && !(tx < 0);
        if (ok && t.pci) {
            const int s = nic_switch(r, l);
            int cnt = 1;
            for (int e = 0; e < d; e++) cnt += (nic_switch(r, li[e]) == s);
            ok = cnt <= (int)((gsw >> (4 * s)) & 0xF);
        }
        if (!ok) { choice[d]++; continue; }
        li[d] = l; rrx[d] = rx; rtx[d] = tx;
        if (d == G - 1) break;
        d++;
        choice[d] = 0;
    }
    for (int e = 0; e < G; e++) {
        out_idx[ord[e]] = (uint8_t)choice[e];
        out_li[ord[e]] = (uint8_t)li[e];
    }
    return true;
}

/*
 * Snapshot predicate: would node r be in filts[1] after IntersectResources for pod
 * type t, ignoring the time-dependent busy window?  True iff some NUMA tuple p passes
 * the GPU stage, has a CPU tuple (p, m) and a surviving NIC entry — i.e. the three-way
 * set intersection of Matcher.py:349 is non-empty.
 */
NHD_HD bool node_feasible(const nhd_node_rec& r, const PodType& t, const double* cap)
{
    if (!t.valid_map) return false;
    if (!node_gates(r, t)) return false;
    const int K = r.n_numa, G = t.G;
    int fg[NHD_MAX_NUMA], fc[NHD_MAX_NUMA];
    free_gpus(r, fg);
    free_cores(r, fc);
    /* cheap necessary conditions before enumerating tuples */
    {
        int sg = 0, sc = 0, need = 0;
        const uint8_t* cl = rec_smt(r) ? t.cl_smt : t.cl_nosmt;
        for (int k = 0; k < K; k++) { sg += fg[k]; sc += fc[k]; }
        for (int g = 0; g <= G; g++) need += cl[g];
        if (t.total_gpus > sg || need > sc) return false;
    }
    const uint64_t gsw = t.pci ? free_gpus_per_switch(r) : 0;
    const bool smt = rec_smt(r);
    const int np = ipow(K, G);
    uint8_t p[NHD_MAX_GROUPS], idx[NHD_MAX_GROUPS], li[NHD_MAX_GROUPS];
    for (int pi = 0; pi < np; pi++) {
        tuple_digits(pi, K, G, p);
        if (!gpu_ok(t, p, K, fg)) continue;
        bool c = false;
        for (int m = 0; m < K && !c; m++) c = cpu_ok(t, p, m, K, fc, smt);
        if (!c) continue;
        if (nic_first_fit(r, t, p, K, cap, gsw, idx, li)) return true;
    }
    return false;
}

/*
 * Why FindNode drops node r for pod type t at clock now: the FIRST stage of the reference path that removes it
 * (NHD_WHY_*, include/nhd_b200.h), NHD_WHY_FEASIBLE if none does.  The group test comes before the active test
 * here, as in InitialNodeFilter (NHDScheduler.py:241-245), unlike node_gates.  The stages are the predicates
 * node_feasible is built from: the GPU stage is non-empty iff some G-tuple passes gpu_ok, the CPU stage iff some
 * (G+1)-tuple passes cpu_ok (Matcher.py:203-216: every tuple, not only those of the GPU stage), the NIC stage iff
 * some G-tuple has a surviving entry without the PCIe pruning, the intersection (Matcher.py:349) iff one tuple
 * passes all three, and the PCI-mode node survives iff that still holds with the pruning (:295-335).
 */
NHD_HD int node_reason(const nhd_node_rec& r, const PodType& t, const double* cap, double now, double min_busy)
{
    if ((r.group_mask & t.pod.group_mask) == 0) return NHD_WHY_NOT_IN_GROUP;
    if (!(r.flags & NHD_NODE_ACTIVE)) return NHD_WHY_INACTIVE;
    if (r.flags & NHD_NODE_MAINTENANCE) return NHD_WHY_MAINTENANCE;
    if (t.pod.hugepages_gb > r.free_hugepages_gb) return NHD_WHY_HUGEPAGES;
    if (!t.valid_map) return NHD_WHY_MAP_TYPE;
    if (t.needs_gpu && node_busy(r, now, min_busy)) return NHD_WHY_BUSY;
    const int K = r.n_numa, G = t.G;
    int fg[NHD_MAX_NUMA], fc[NHD_MAX_NUMA];
    free_gpus(r, fg);
    free_cores(r, fc);
    const bool smt = rec_smt(r);
    /* 15 free GPUs on every switch: more than the <= NHD_MAX_GROUPS groups that can share one, so the PCI test of
     * nic_first_fit always passes — the NIC stage as Matcher.FilterNumaTopology leaves it */
    const uint64_t no_pruning = ~0ULL;
    const uint64_t gsw = t.pci ? free_gpus_per_switch(r) : no_pruning;
    bool any_gpu = false, any_cpu = false, any_nic = false, isect = false, isect_pruned = false;
    const int np = ipow(K, G);
    uint8_t p[NHD_MAX_GROUPS], idx[NHD_MAX_GROUPS], li[NHD_MAX_GROUPS];
    for (int pi = 0; pi < np && !isect_pruned; pi++) {
        tuple_digits(pi, K, G, p);
        const bool g = gpu_ok(t, p, K, fg);
        bool c = false;
        for (int m = 0; m < K && !c; m++) c = cpu_ok(t, p, m, K, fc, smt);
        any_gpu |= g;
        any_cpu |= c;
        if (any_nic && !(g && c)) continue;           /* nothing left to learn from this tuple's NICs */
        const bool n = nic_first_fit(r, t, p, K, cap, no_pruning, idx, li);
        any_nic |= n;
        if (!(g && c && n)) continue;
        isect = true;
        isect_pruned = !t.pci || nic_first_fit(r, t, p, K, cap, gsw, idx, li);
    }
    if (!any_gpu) return NHD_WHY_GPU;
    if (!any_cpu) return NHD_WHY_CPU;
    if (!any_nic) return NHD_WHY_NIC;
    if (!isect) return NHD_WHY_NUMA;
    if (!isect_pruned) return NHD_WHY_PCIE;
    return NHD_WHY_FEASIBLE;
}

/*
 * The same predicate for the common shape — a 2-NUMA node and a pod of one or two groups — written so that
 * nothing is indexed dynamically: the record, the per-NUMA counts and the search state all stay in registers
 * (node_feasible keeps its tuples, demand sums and NIC search stack in arrays, which the GPU puts in local
 * memory).  Only EXISTENCE of a surviving entry matters here, so the order of enumeration is free; what must
 * not change is the arithmetic of each test: fp64 subtraction in group order on a shared NIC
 * (Matcher.py:261-268), the per-switch count of the PCI pruning (:312-322).  The part that does not depend on
 * the pod type is computed once per node (Pre2).
 */
struct Pre2 {
    int fc0, fc1;                /* Node.GetFreeCpuCores */
    int fg0, fg1;                /* Node.GetFreeNumaGPUs */
    uint64_t gsw;                /* Node.GetFreeGPUPCICount, 4 bits per local switch id */
    bool smt;
};

NHD_HD void make_pre2(const nhd_node_rec& r, int fc0, int fc1, Pre2& q)
{
    const uint32_t fr = ~(uint32_t)r.gpu_used & ((1u << r.n_gpus) - 1);
    q.fc0 = fc0; q.fc1 = fc1;
    q.fg0 = popc32(fr & r.gpu_numa_mask[0]);
    q.fg1 = popc32(fr & r.gpu_numa_mask[1]);
    q.gsw = fr ? free_gpus_per_switch(r) : 0;
    q.smt = rec_smt(r);
}

NHD_HD int nic_switch2(const nhd_node_rec& r, int l)
{
    return (int)(((l < 16 ? r.nic_sw[0] : r.nic_sw[1]) >> (4 * (l & 15))) & 0xF);
}
NHD_HD double nic_free_bw2(const nhd_node_rec& r, int l, const double* cap)
{
    const int sc = (int)(((l < 16 ? r.nic_speed[0] : r.nic_speed[1]) >> (4 * (l & 15))) & 0xF);
    return ((r.nic_inuse >> l) & 1) ? 0.0 : cap[sc];
}

/* NIC stage of one NUMA tuple (p0, p1), G <= 2: does filts['nic'] keep an entry with this NUMA part? */
NHD_HD bool nic_any_fit2(const nhd_node_rec& r, const PodType& t, int p0, int p1, const double* cap, uint64_t gsw)
{
    const uint32_t nm0 = p0 ? r.nic_numa_mask[1] : r.nic_numa_mask[0];
    const double rx0 = t.pod.groups[0].rx_gbps, tx0 = t.pod.groups[0].tx_gbps;
    if (t.G == 1) {
        for (uint32_t m = nm0; m; m &= m - 1) {
            const int l = ctz32(m);
            const double c = nic_free_bw2(r, l, cap);
            if ((c - rx0 < 0) || (c - tx0 < 0)) continue;
            if (t.pci && ((gsw >> (4 * nic_switch2(r, l))) & 0xF) < 1) continue;
            return true;
        }
        return false;
    }
    const uint32_t nm1 = p1 ? r.nic_numa_mask[1] : r.nic_numa_mask[0];
    const double rx1 = t.pod.groups[1].rx_gbps, tx1 = t.pod.groups[1].tx_gbps;
    if (nm1 == 0) return false;
    for (uint32_t m = nm0; m; m &= m - 1) {
        const int l0 = ctz32(m);
        const double c0 = nic_free_bw2(r, l0, cap);
        const double r0 = c0 - rx0, q0 = c0 - tx0;
        if ((r0 < 0) || (q0 < 0)) continue;
        const int s0 = nic_switch2(r, l0);
        const int f0 = (int)((gsw >> (4 * s0)) & 0xF);
        if (t.pci && f0 < 1) continue;
        for (uint32_t n = nm1; n; n &= n - 1) {
            const int l1 = ctz32(n);
            double r1, q1;
            if (l1 == l0) { r1 = r0 - rx1; q1 = q0 - tx1; }        /* what group 0 left of the NIC (:261-268) */
            else { const double c1 = nic_free_bw2(r, l1, cap); r1 = c1 - rx1; q1 = c1 - tx1; }
            if ((r1 < 0) || (q1 < 0)) continue;
            if (t.pci) {
                const int s1 = nic_switch2(r, l1);
                if (s1 == s0 ? f0 < 2 : ((gsw >> (4 * s1)) & 0xF) < 1) continue;
            }
            return true;
        }
    }
    return false;
}

/* node_feasible for r.n_numa == 2 and t.G <= 2 (the caller checks both) */
NHD_HD bool node_feasible_k2(const nhd_node_rec& r, const PodType& t, const double* cap, const Pre2& q)
{
    if (!t.valid_map) return false;
    if (!node_gates(r, t)) return false;
    const uint8_t* cl = q.smt ? t.cl_smt : t.cl_nosmt;
    const bool two = t.G > 1;
    const int c0 = cl[0], c1 = two ? cl[1] : 0, cm = two ? cl[2] : cl[1];
    const int g0 = t.pod.groups[0].n_gpus, g1 = two ? t.pod.groups[1].n_gpus : 0;
    if (g0 + g1 > q.fg0 + q.fg1 || c0 + c1 + cm > q.fc0 + q.fc1) return false;
    const int np = two ? 4 : 2;
    for (int pi = 0; pi < np; pi++) {
        const int p0 = two ? (pi >> 1) : pi, p1 = pi & 1;           /* first element most significant */
        const int a1 = (p0 ? g0 : 0) + ((two && p1) ? g1 : 0), a0 = g0 + g1 - a1;
        if (a0 > q.fg0 || a1 > q.fg1) continue;                    /* Matcher.py:121-129 */
        const int b1 = (p0 ? c0 : 0) + ((two && p1) ? c1 : 0), b0 = c0 + c1 - b1;
        if (!((b0 + cm <= q.fc0 && b1 <= q.fc1) || (b0 <= q.fc0 && b1 + cm <= q.fc1))) continue;   /* :204-212 */
        if (nic_any_fit2(r, t, p0, p1, cap, q.gsw)) return true;
    }
    return false;
}

/*
 * The three stage masks of stage_masks_fc in the same register-only form (r.n_numa == 2, t.G <= 2): bit p of mA /
 * mC = NUMA tuple p passes the GPU stage / keeps a NIC entry, bit 2p + m of mB = CPU tuple (p, m) passes.  With the
 * GetNumaGroupIdx table over (mA, mB, mC) (mapt2_kernel) this is everything the mapping of a pod needs on such a node.
 */
NHD_HD bool stage_masks_k2(const nhd_node_rec& r, const PodType& t, const double* cap, const Pre2& q,
                           uint32_t& mA, uint32_t& mB, uint32_t& mC)
{
    const uint8_t* cl = q.smt ? t.cl_smt : t.cl_nosmt;
    const bool two = t.G > 1;
    const int c0 = cl[0], c1 = two ? cl[1] : 0, cm = two ? cl[2] : cl[1];
    const int g0 = t.pod.groups[0].n_gpus, g1 = two ? t.pod.groups[1].n_gpus : 0;
    const int np = two ? 4 : 2;
    mA = mB = mC = 0;
    for (int pi = 0; pi < np; pi++) {
        const int p0 = two ? (pi >> 1) : pi, p1 = pi & 1;
        const int a1 = (p0 ? g0 : 0) + ((two && p1) ? g1 : 0), a0 = g0 + g1 - a1;
        if (a0 <= q.fg0 && a1 <= q.fg1) mA |= 1u << pi;
        const int b1 = (p0 ? c0 : 0) + ((two && p1) ? c1 : 0), b0 = c0 + c1 - b1;
        if (b0 + cm <= q.fc0 && b1 <= q.fc1) mB |= 1u << (2 * pi);
        if (b0 <= q.fc0 && b1 + cm <= q.fc1) mB |= 2u << (2 * pi);
        if (nic_any_fit2(r, t, p0, p1, cap, t.pci ? q.gsw : 0)) mC |= 1u << pi;
    }
    return mA != 0 && mB != 0 && mC != 0;
}

/*
 * nic_first_fit for the NUMA tuple (p0, p1), same shapes: the FIRST surviving entry in the reference's order — NUMA 0's
 * groups vary slowest, inside a NUMA node the first group (Matcher.py:245-258).  Packed result: per group g the
 * per-NUMA NodeNic.idx in bits 8g.. of *idx and the index in Node.nics in bits 8g.. of *li.
 */
NHD_HD bool nic_first_fit2(const nhd_node_rec& r, const PodType& t, int p0, int p1, const double* cap, uint64_t gsw,
                           uint32_t* idx, uint32_t* li)
{
    const bool two = t.G > 1;
    /* level order: a group on NUMA 0 before a group on NUMA 1, else group order */
    const int ga = (two && p0 > p1) ? 1 : 0, gb = 1 - ga;
    const uint32_t nma = (ga ? p1 : p0) ? r.nic_numa_mask[1] : r.nic_numa_mask[0];
    const double rxa = t.pod.groups[ga].rx_gbps, txa = t.pod.groups[ga].tx_gbps;
    for (uint32_t m = nma; m; m &= m - 1) {
        const int la = ctz32(m);
        const double ca = nic_free_bw2(r, la, cap);
        const double ra = ca - rxa, qa = ca - txa;
        if ((ra < 0) || (qa < 0)) continue;
        const int sa = nic_switch2(r, la);
        const int fa = (int)((gsw >> (4 * sa)) & 0xF);
        if (t.pci && fa < 1) continue;
        const uint32_t ia = (uint32_t)popc32(nma & ((1u << la) - 1));
        if (!two) { *idx = ia; *li = (uint32_t)la; return true; }
        const uint32_t nmb = (gb ? p1 : p0) ? r.nic_numa_mask[1] : r.nic_numa_mask[0];
        const double rxb = t.pod.groups[gb].rx_gbps, txb = t.pod.groups[gb].tx_gbps;
        for (uint32_t n = nmb; n; n &= n - 1) {
            const int lb = ctz32(n);
            double rb, qb;
            if (lb == la) { rb = ra - rxb; qb = qa - txb; }
            else { const double cb = nic_free_bw2(r, lb, cap); rb = cb - rxb; qb = cb - txb; }
            if ((rb < 0) || (qb < 0)) continue;
            if (t.pci) {
                const int sb = nic_switch2(r, lb);
                if (sb == sa ? fa < 2 : ((gsw >> (4 * sb)) & 0xF) < 1) continue;
            }
            const uint32_t ib = (uint32_t)popc32(nmb & ((1u << lb) - 1));
            *idx = (ia << (8 * ga)) | (ib << (8 * gb));
            *li = ((uint32_t)la << (8 * ga)) | ((uint32_t)lb << (8 * gb));
            return true;
        }
    }
    return false;
}

/* ---------------------------------------------------------------- CPython set emulation */

/*
 * The order in which the reference walks its candidate tuples is the iteration order of
 * CPython sets of int tuples (Matcher.py:129,141,212,220,349,365).  This is the
 * product's own model of that table (Objects/setobject.c, CPython 3.8-3.12: 8 initial
 * slots, LINEAR_PROBES 9, perturb shift 5, resize at fill*5 >= mask*3 to the smallest
 * power of two > 4*used, re-insertion in old slot order) and of the tuple hash
 * (Objects/tupleobject.c).  Keys are tuple indices of product(range(K), repeat=L).
 */
NHD_HD uint64_t py_tuple_hash(int idx, int K, int L)
{
    const uint64_t P1 = 11400714785074694791ULL, P2 = 14029467366897019727ULL, P5 = 2870177450012600261ULL;
    uint8_t d[8];
    tuple_digits(idx, K, L, d);
    uint64_t acc = P5;
    for (int i = 0; i < L; i++) {
        acc += (uint64_t)d[i] * P2;           /* hash(small int) == the int */
        acc = (acc << 31) | (acc >> 33);
        acc *= P1;
    }
    acc += (uint64_t)L ^ (P5 ^ 3527539ULL);
    return acc == ~0ULL ? 1546275796ULL : acc;
}

template <int SLOTS>
struct PySet {
    uint16_t slot[SLOTS];      /* tuple index + 1, 0 = empty */
    int mask, fill, K, L;

    NHD_HD void init(int K_, int L_)
    {
        K = K_; L = L_; mask = 7; fill = 0;
        for (int i = 0; i < 8; i++) slot[i] = 0;
    }
    NHD_HD void insert_clean(uint16_t* tab, int msk, int idx) const
    {
        uint64_t h = py_tuple_hash(idx, K, L), perturb = h;
        uint64_t i = h & (uint64_t)msk;
        for (;;) {
            if (!tab[i]) { tab[i] = (uint16_t)(idx + 1); return; }
            if (i + 9 <= (uint64_t)msk) {
                for (int j = 1; j <= 9; j++)
                    if (!tab[i + j]) { tab[i + j] = (uint16_t)(idx + 1); return; }
            }
            perturb >>= 5;
            i = (i * 5 + 1 + perturb) & (uint64_t)msk;
        }
    }
    NHD_HD bool has(int idx) const
    {
        uint64_t h = py_tuple_hash(idx, K, L), perturb = h;
        uint64_t i = h & (uint64_t)mask;
        for (;;) {
            int probes = (i + 9 <= (uint64_t)mask) ? 9 : 0;
            for (int j = 0; j <= probes; j++) {
                if (!slot[i + j]) return false;
                if (slot[i + j] == idx + 1) return true;
            }
            perturb >>= 5;
            i = (i * 5 + 1 + perturb) & (uint64_t)mask;
        }
    }
    NHD_HD void add(int idx)
    {
        uint64_t h = py_tuple_hash(idx, K, L), perturb = h;
        uint64_t i = h & (uint64_t)mask;
        for (;;) {
            int probes = (i + 9 <= (uint64_t)mask) ? 9 : 0;
            for (int j = 0; j <= probes; j++) {
                if (!slot[i + j]) { i += j; goto found_unused; }
                if (slot[i + j] == idx + 1) return;
            }
            perturb >>= 5;
            i = (i * 5 + 1 + perturb) & (uint64_t)mask;
        }
found_unused:
        slot[i] = (uint16_t)(idx + 1);
        fill++;
        if (fill * 5 < mask * 3) return;
        /* resize: smallest power of two > 4 * used, old entries re-inserted in slot order */
        int newsize = 8;
        while (newsize <= fill * 4) newsize <<= 1;
        uint16_t old[SLOTS / 4 > 8 ? SLOTS / 4 : 8];    /* the old table is at most a quarter of SLOTS */
        int oldmask = mask;
        for (int k = 0; k <= oldmask; k++) old[k] = slot[k];
        for (int k = 0; k < newsize; k++) slot[k] = 0;
        mask = newsize - 1;
        for (int k = 0; k <= oldmask; k++)
            if (old[k]) insert_clean(slot, mask, old[k] - 1);
    }
    /* list(s): indices in slot order */
    NHD_HD int list(uint8_t* out) const
    {
        int n = 0;
        for (int i = 0; i <= mask; i++) if (slot[i]) out[n++] = (uint8_t)(slot[i] - 1);
        return n;
    }
};

/* a & b with CPython's rule: walk the smaller operand (the right one on ties) in slot
 * order, keep members of the other (setobject.c set_intersection) */
template <int SA, int SB, int SO>
NHD_HD void pyset_and(const PySet<SA>& a, const PySet<SB>& b, PySet<SO>& out)
{
    out.init(a.K, a.L);
    if (b.fill > a.fill) {
        for (int i = 0; i <= a.mask; i++) if (a.slot[i] && b.has(a.slot[i] - 1)) out.add(a.slot[i] - 1);
    } else {
        for (int i = 0; i <= b.mask; i++) if (b.slot[i] && a.has(b.slot[i] - 1)) out.add(b.slot[i] - 1);
    }
}

/* 256-bit tuple-feasibility mask, bit = tuple index */
struct TMask { uint64_t w[4]; };
NHD_HD bool tm_test(const TMask& m, int i) { return (m.w[i >> 6] >> (i & 63)) & 1; }
NHD_HD void tm_set(TMask& m, int i) { m.w[i >> 6] |= 1ULL << (i & 63); }
NHD_HD TMask tm_zero() { TMask m; m.w[0] = m.w[1] = m.w[2] = m.w[3] = 0; return m; }

/*
 * GetNumaGroupIdx on top of IntersectResources for ONE node, given which tuples passed
 * each stage: maskA over product(range(K), repeat=G) (GPU stage), maskB over
 * repeat=G+1 (CPU stage), maskC over repeat=G (NUMA tuples that keep at least one NIC
 * entry).  Reproduces, including CPython set order:
 *   A_list = list(set of A tuples added in product order)          Matcher.py:113-141
 *   B_list likewise                                                :175-220
 *   intersect = list(set(A_list) & set(prefixes of B_list) & set(C numa parts))   :344-349
 *   gpu list = intersect when something was removed, else A_list   :365-368
 *   gtuple   = first element with the largest max-min group count  :428-439
 *   ctuple   = first B_list entry whose prefix is gtuple           :442-444
 * Returns false when the intersection is empty; else *p_star = index of gtuple,
 * *m_star = last element of ctuple.
 */
NHD_HDN bool choose_mapping(int K, int G, const TMask& maskA, const TMask& maskB, const TMask& maskC,
                            int* p_star, int* m_star)
{
    const int np = ipow(K, G), nq = np * K;
    PySet<128> sa;  sa.init(K, G);
    for (int i = 0; i < np; i++) if (tm_test(maskA, i)) sa.add(i);
    if (sa.fill == 0) return false;
    PySet<512> sb;  sb.init(K, G + 1);
    for (int i = 0; i < nq; i++) if (tm_test(maskB, i)) sb.add(i);
    if (sb.fill == 0) return false;
    uint8_t a_list[64], b_list[256];
    const int na = sa.list(a_list), nb = sb.list(b_list);

    PySet<128> sg, sc, sn, t1, isect;
    sg.init(K, G);
    for (int i = 0; i < na; i++) sg.add(a_list[i]);
    sc.init(K, G);
    for (int i = 0; i < nb; i++) sc.add(b_list[i] / K);          /* x[:-1] */
    sn.init(K, G);
    for (int i = 0; i < np; i++) if (tm_test(maskC, i)) sn.add(i); /* first appearance = product order */
    pyset_and(sg, sc, t1);
    pyset_and(t1, sn, isect);
    if (isect.fill == 0) return false;

    uint8_t i_list[64];
    const int ni = isect.list(i_list);
    const uint8_t* gl = a_list;
    int ngl = na;
    if (ni != na) { gl = i_list; ngl = ni; }                       /* intersect is a subset of A */

    int best = -1, bestv = -1;
    for (int x = 0; x < ngl; x++) {
        uint8_t d[NHD_MAX_GROUPS];
        tuple_digits(gl[x], K, G, d);
        int mx = 0, mn = 1 << 20;
        for (int y = 0; y < K; y++) {
            int c = 0;
            for (int g = 0; g < G; g++) c += (d[g] == y);
            mx = c > mx ? c : mx;
            mn = c < mn ? c : mn;
        }
        if (mx - mn > bestv) { bestv = mx - mn; best = x; }        /* strict '>' keeps the first */
    }
    *p_star = gl[best];
    for (int i = 0; i < nb; i++)
        if (b_list[i] / K == *p_star) { *m_star = b_list[i] % K; return true; }
    return false;   /* unreachable: p_star is in set(prefixes of B) */
}

/* list({x[0] for x in nic_list}) for up to NHD_MAX_GROUPS small ints (NHDScheduler.py:302):
 * an 8-slot table, hash(i) == i, no resize below five distinct keys. */
NHD_HD int claimed_nic_order(const uint8_t* li, int n, uint8_t* out)
{
    int slot[8];
    for (int i = 0; i < 8; i++) slot[i] = -1;
    for (int e = 0; e < n; e++) {
        uint64_t h = li[e], perturb = h, i = h & 7;
        for (;;) {
            if (slot[i] < 0) { slot[i] = li[e]; break; }
            if (slot[i] == li[e]) break;
            perturb >>= 5;
            i = (i * 5 + 1 + perturb) & 7;
        }
    }
    int m = 0;
    for (int i = 0; i < 8; i++) if (slot[i] >= 0) out[m++] = (uint8_t)slot[i];
    return m;
}

/* ---------------------------------------------------------------- evaluation of one node */

/*
 * Full evaluation of (pod type, node) on the node's CURRENT state: decides feasibility
 * and, when feasible, the mapping GetNumaGroupIdx would return.
 */
struct Mapping {
    uint8_t gpu_numa[NHD_MAX_GROUPS];
    uint8_t misc_numa;
    uint8_t nic_idx[NHD_MAX_GROUPS];
    uint8_t nic_li[NHD_MAX_GROUPS];
};

/* Stage masks of one node on its current state: which NUMA tuples pass the GPU stage (a),
 * the CPU stage (b, over G+1 tuples) and keep a NIC entry (c).  False when a stage is empty. */
NHD_HD bool stage_masks(const nhd_node_rec& r, const PodType& t, const double* cap, uint64_t gsw,
                        TMask& ma, TMask& mb, TMask& mc)
{
    const int K = r.n_numa, G = t.G;
    int fg[NHD_MAX_NUMA], fc[NHD_MAX_NUMA];
    free_gpus(r, fg);
    free_cores(r, fc);
    const bool smt = rec_smt(r);
    const int np = ipow(K, G);
    ma = tm_zero(); mb = tm_zero(); mc = tm_zero();
    uint8_t p[NHD_MAX_GROUPS], idx[NHD_MAX_GROUPS], li[NHD_MAX_GROUPS];
    bool anyA = false, anyB = false, anyC = false;
    for (int pi = 0; pi < np; pi++) {
        tuple_digits(pi, K, G, p);
        if (gpu_ok(t, p, K, fg)) { tm_set(ma, pi); anyA = true; }
        for (int m = 0; m < K; m++)
            if (cpu_ok(t, p, m, K, fc, smt)) { tm_set(mb, pi * K + m); anyB = true; }
        if (nic_first_fit(r, t, p, K, cap, gsw, idx, li)) { tm_set(mc, pi); anyC = true; }
    }
    return anyA && anyB && anyC;
}

NHD_HDN bool evaluate_mapping(const nhd_node_rec& r, const PodType& t, const double* cap, Mapping* out)
{
    const int K = r.n_numa, G = t.G;
    const uint64_t gsw = t.pci ? free_gpus_per_switch(r) : 0;
    TMask ma, mb, mc;
    if (!stage_masks(r, t, cap, gsw, ma, mb, mc)) return false;
    int ps, ms;
    if (!choose_mapping(K, G, ma, mb, mc, &ps, &ms)) return false;
    tuple_digits(ps, K, G, out->gpu_numa);
    out->misc_numa = (uint8_t)ms;
    nic_first_fit(r, t, out->gpu_numa, K, cap, gsw, out->nic_idx, out->nic_li);
    return true;
}

/* ---------------------------------------------------------------- physical assignment */

/*
 * Node.GetFreeCpuBatch (Node.py:502-519): walk ALL logical ids in ascending order, take
 * ids on socket `numa` that are unused and (on SMT nodes) whose sibling is unused —
 * judged against the state at call time, nothing is marked during the walk.  An SMT
 * request takes [core, sibling] while at least two are still needed.
 * Returns the number of ids written to out (== num on success).
 */
NHD_HD int cpu_batch(const nhd_node_rec& r, int numa, int num, bool smt_req, uint8_t* out)
{
    const int phys = r.phys_cores, per = phys / r.n_numa;
    const bool smt = rec_smt(r);
    M256 e = m_and(eligible_phys(r), m_range(numa * per, (numa + 1) * per));
    if (smt) e = m_or(e, m_shl(e, phys));      /* both hyperthreads of a free core are eligible ids */
    int n = 0;
    for (int w = 0; w < 4 && num > 0; w++) {
        uint64_t bits = e.w[w];
        while (bits && num > 0) {
            int c = 64 * w + ctz64(bits);
            bits &= bits - 1;
            if (smt && smt_req && num >= 2) {
                out[n++] = (uint8_t)c;
                out[n++] = (uint8_t)(c < phys ? c + phys : c - phys);
                num -= 2;
            } else {
                out[n++] = (uint8_t)c;
                num -= 1;
            }
        }
    }
    return n;
}

NHD_HD void mark_used(nhd_node_rec& r, int c) { r.used[c >> 6] |= 1ULL << (c & 63); }

/*
 * Node.SetPhysicalIdsFromMapping (Node.py:663-841) + SetBusy (NHDScheduler.py:289) +
 * ClaimPodNICResources (NHDScheduler.py:302-304) on the packed record.  r is updated in
 * place; on failure every core/GPU taken so far is given back (Node.py:825-830) but the
 * busy stamp stays.  b->status, node-independent fields and the physical ids are filled.
 */
NHD_HDN void assign_pod(nhd_node_rec& r, const PodType& t, const Mapping& m, double now, nhd_binding* b)
{
    const nhd_node_rec saved = r;
    const int G = t.G;
    r.busy_time = now;                                             /* NHDScheduler.py:289 */
    int nc = 0, ng = 0, n_nic_rec = 0;
    uint8_t nic_rec[NHD_MAX_GROUPS];
    uint8_t batch[NHD_MAX_POD_CORES + 2];
    bool hp_taken = false;
    bool fail = false;

    for (int g = 0; g < G; g++) {
        b->gpu_numa[g] = m.gpu_numa[g];
        b->cpu_numa[g] = m.gpu_numa[g];
        b->nic_numa[g] = m.gpu_numa[g];
        b->nic_idx[g] = m.nic_idx[g];
        b->nic_list_index[g] = m.nic_li[g];
    }
    b->cpu_numa[G] = m.misc_numa;
    b->n_groups = (uint8_t)G;

    for (int g = 0; g < G && !fail; g++) {
        const nhd_pod_group& pg = t.pod.groups[g];
        const int numa = m.gpu_numa[g];
        const int req = t.tot[g];
        if (cpu_batch(r, numa, req, (pg.flags & NHD_GRP_PROC_SMT) != 0, batch) != req) { fail = true; break; }   /* :685 */
        int ci = 0;
        const int nsw = nic_switch(r, m.nic_li[g]);
        for (int j = 0; j < pg.n_gpus; j++) {                       /* :707-732 */
            uint32_t fr = ~(uint32_t)r.gpu_used & ((1u << r.n_gpus) - 1);
            int dev = -1;
            for (uint32_t f = fr; f; f &= f - 1) {                  /* GetFreePciGpuFromNic :648-655 */
                int i = ctz32(f);
                if (gpu_switch(r, i) == nsw) { dev = i; break; }
            }
            if (dev < 0) {
                if (t.pci) { fail = true; break; }                  /* :711-713 */
                uint32_t f = fr & r.gpu_numa_mask[numa];            /* GetNextGpuFree :495-500 */
                if (f) dev = ctz32(f);
            }
            if (dev < 0) { fail = true; break; }                    /* :718-720 */
            r.gpu_used |= (uint16_t)(1u << dev);
            if (ng < NHD_MAX_POD_GPUS) b->gpu_index[ng] = (uint8_t)dev;
            ng++;
            for (int k = 0; k < pg.gpu_feeders[j]; k++) {
                mark_used(r, batch[ci]);
                if (nc < NHD_MAX_POD_CORES) b->cores[nc] = batch[ci];
                nc++; ci++;
            }
        }
        if (fail) break;
        for (int k = 0; k < pg.n_proc; k++) {                       /* :735-739 */
            mark_used(r, batch[ci]);
            if (nc < NHD_MAX_POD_CORES) b->cores[nc] = batch[ci];
            nc++; ci++;
        }
        if (pg.flags & NHD_GRP_HAS_NIC_CORES) nic_rec[n_nic_rec++] = m.nic_li[g];   /* :742-755 */
        const int nh = pg.n_helpers;                                /* :773-788 */
        if (cpu_batch(r, numa, nh, (pg.flags & NHD_GRP_HELPER_SMT) != 0, batch) != nh) { fail = true; break; }
        for (int k = 0; k < nh; k++) {
            mark_used(r, batch[k]);
            if (nc < NHD_MAX_POD_CORES) b->cores[nc] = batch[k];
            nc++;
        }
    }
    if (!fail) {
        if (t.pod.hugepages_gb > 0) { r.free_hugepages_gb -= t.pod.hugepages_gb; hp_taken = true; }   /* :794-796 */
        const int nm = t.pod.n_misc;                                                  /* :799-811 */
        if (cpu_batch(r, m.misc_numa, nm, (t.pod.flags & NHD_POD_MISC_SMT) != 0, batch) != nm) fail = true;
        else
            for (int k = 0; k < nm; k++) {
                mark_used(r, batch[k]);
                if (nc < NHD_MAX_POD_CORES) b->cores[nc] = batch[k];
                nc++;
            }
    }
    if (fail) {                                                      /* :825-837 */
        const double bt = r.busy_time;
        r = saved;
        r.busy_time = bt;
        if (hp_taken) r.free_hugepages_gb -= t.pod.hugepages_gb;   /* the unwind never restores hugepages */
        b->n_cores = b->n_gpus = b->n_claimed = 0;
        for (int i = 0; i < NHD_MAX_POD_CORES; i++) b->cores[i] = 0;
        for (int i = 0; i < NHD_MAX_POD_GPUS; i++) b->gpu_index[i] = 0;
        b->status = n_nic_rec ? NHD_REF_WOULD_CRASH : NHD_ASSIGN_FAILED;
        return;
    }
    b->n_cores = (uint8_t)nc;
    b->n_gpus = (uint8_t)ng;
    const int ncl = claimed_nic_order(nic_rec, n_nic_rec, b->claimed_nics);          /* NHDScheduler.py:302 */
    b->n_claimed = (uint8_t)ncl;
    for (int i = 0; i < ncl; i++) r.nic_inuse |= 1u << b->claimed_nics[i];          /* Node.py:644-646 */
    b->status = NHD_PLACED;
}


/* ================================================================================== */
/* Two-stage placement: decisions on a per-node summary, core ids deferred             */
/* ================================================================================== */

/*
 * NodeDyn — the mutable summary of one node the sequential sweep works on (32 bytes).
 *
 * Every decision of the reference path depends on the 256-bit core mask only through
 * Node.GetFreeCpuCores (Node.py:250-264), i.e. the number of fully free physical cores per
 * NUMA node.  Node.GetFreeCpuBatch (Node.py:502-519) always hands out the LOWEST eligible
 * ids of a socket, so whatever a batch of pods took from a socket is a prefix of the
 * snapshot's eligible-core list; `consumed[k]` is the length of that prefix.  The sweep
 * therefore tracks counts only, and the actual core ids are reconstructed afterwards, for
 * all pods in parallel, from the snapshot mask and the pod's prefix offsets
 * (assign_cores_from_snapshot).
 */
struct NodeDyn {
    uint8_t  fc[NHD_MAX_NUMA];        /* free physical cores per NUMA node (current)              */
    uint8_t  consumed[NHD_MAX_NUMA];  /* eligible cores consumed since the snapshot, per NUMA node */
    uint16_t gpu_used;
    uint16_t info;                    /* bit0 touched by this batch, bit1 SMT node, bits 2-4 n_numa */
    uint32_t nic_inuse;
    int32_t  free_hugepages_gb;
    uint16_t hw_class;                /* id of the node's static hardware description, 0xFFFF = none */
    uint8_t  n_gpus;
    uint8_t  n_nics;
    double   busy_time;
};
#define NHD_DYN_TOUCHED 1
#define NHD_DYN_SMT     2
#define NHD_NO_CLASS    0xFFFF
static_assert(sizeof(NodeDyn) == 32, "NodeDyn must be two 16-byte chunks");

NHD_HD void make_dyn(const nhd_node_rec& r, NodeDyn& d)
{
    int fc[NHD_MAX_NUMA] = {0, 0, 0, 0};
    free_cores(r, fc);
    for (int k = 0; k < NHD_MAX_NUMA; k++) { d.fc[k] = (uint8_t)fc[k]; d.consumed[k] = 0; }
    d.gpu_used = r.gpu_used;
    d.info = (uint16_t)((rec_smt(r) ? NHD_DYN_SMT : 0) | (r.n_numa << 2));
    d.nic_inuse = r.nic_inuse;
    d.free_hugepages_gb = r.free_hugepages_gb;
    d.hw_class = NHD_NO_CLASS;
    d.n_gpus = r.n_gpus;
    d.n_nics = r.n_nics;
    d.busy_time = r.busy_time;
}

/* overlay the summary on a record that holds the static fields */
NHD_HD void apply_dyn(nhd_node_rec& r, const NodeDyn& d)
{
    r.gpu_used = d.gpu_used;
    r.nic_inuse = d.nic_inuse;
    r.free_hugepages_gb = d.free_hugepages_gb;
    r.busy_time = d.busy_time;
}

/*
 * Cheap NECESSARY conditions for (pod type, node summary) to be feasible; true means the node
 * cannot be in filts[1] (so skipping it is exact).  Covers the ways a node typically fills up:
 * hugepages (Matcher.py:78), total / largest-chunk core demand (:203-212), free GPUs (:118-129)
 * and every NIC already owned by a pod (Node.py:292) while the pod wants bandwidth.
 */
NHD_HD bool summary_infeasible(const PodType& t, const NodeDyn& d)
{
    if (t.pod.hugepages_gb > d.free_hugepages_gb) return true;
    const bool smt = (d.info & NHD_DYN_SMT) != 0;
    const int need = smt ? t.need_smt : t.need_nosmt, big = smt ? t.max_smt : t.max_nosmt;
    const int sum = d.fc[0] + d.fc[1] + d.fc[2] + d.fc[3];
    int mx = d.fc[0] > d.fc[1] ? d.fc[0] : d.fc[1];
    const int mx2 = d.fc[2] > d.fc[3] ? d.fc[2] : d.fc[3];
    mx = mx > mx2 ? mx : mx2;
    if (sum < need || mx < big) return true;
    if (t.total_gpus) {
        const uint32_t fr = ~(uint32_t)d.gpu_used & ((1u << d.n_gpus) - 1);
        if (popc32(fr) < t.total_gpus) return true;
    }
    if (t.has_bw) {
        const uint32_t all = d.n_nics >= 32 ? 0xFFFFFFFFu : ((1u << d.n_nics) - 1);
        if ((d.nic_inuse & all) == all) return true;
    }
    return false;
}

/* stage_masks with the free-core counts taken from the summary */
NHD_HD bool stage_masks_fc(const nhd_node_rec& r, const uint8_t* fc8, const PodType& t, const double* cap,
                           uint64_t gsw, TMask& ma, TMask& mb, TMask& mc)
{
    const int K = r.n_numa, G = t.G;
    int fg[NHD_MAX_NUMA], fc[NHD_MAX_NUMA];
    free_gpus(r, fg);
    for (int k = 0; k < NHD_MAX_NUMA; k++) fc[k] = fc8[k];
    const bool smt = rec_smt(r);
    const int np = ipow(K, G);
    ma = tm_zero(); mb = tm_zero(); mc = tm_zero();
    uint8_t p[NHD_MAX_GROUPS], idx[NHD_MAX_GROUPS], li[NHD_MAX_GROUPS];
    bool anyA = false, anyB = false, anyC = false;
    for (int pi = 0; pi < np; pi++) {
        tuple_digits(pi, K, G, p);
        if (gpu_ok(t, p, K, fg)) { tm_set(ma, pi); anyA = true; }
        for (int m = 0; m < K; m++)
            if (cpu_ok(t, p, m, K, fc, smt)) { tm_set(mb, pi * K + m); anyB = true; }
        if (nic_first_fit(r, t, p, K, cap, gsw, idx, li)) { tm_set(mc, pi); anyC = true; }
    }
    return anyA && anyB && anyC;
}

/* physical cores a GetFreeCpuBatch(num, smt) call removes from a socket's eligible list,
 * given `avail` eligible cores there (Node.py:502-519): SMT pairs take one core per two ids;
 * a non-SMT request on an SMT node takes one core per id and, once the first-half ids run
 * out, continues with the siblings of the cores it just took. */
NHD_HD int batch_width(bool smt_node, bool smt_req, int num, int avail)
{
    if (!smt_node) return num;
    if (smt_req) return (num + 1) / 2;
    return num < avail ? num : avail;
}

/*
 * Everything of SetPhysicalIdsFromMapping except the core ids (Node.py:663-841), on the
 * summary: GPU picks, NIC claim order, hugepages, busy stamp, and the per-socket core
 * accounting.  r holds the node's static fields with the summary overlaid (apply_dyn).
 * b->cores[0..3] temporarily carries the pod's prefix offsets for assign_cores_from_snapshot.
 */
NHD_HD void assign_resources(const nhd_node_rec& r, NodeDyn& d, const PodType& t, const Mapping& m, double now,
                             nhd_binding* b)
{
    const int G = t.G;
    const bool smt_node = (d.info & NHD_DYN_SMT) != 0;
    d.busy_time = now;                                             /* NHDScheduler.py:289 */
    d.info |= NHD_DYN_TOUCHED;
    b->n_groups = (uint8_t)G;
    for (int g = 0; g < G; g++) {
        b->gpu_numa[g] = m.gpu_numa[g];
        b->cpu_numa[g] = m.gpu_numa[g];
        b->nic_numa[g] = m.gpu_numa[g];
        b->nic_idx[g] = m.nic_idx[g];
        b->nic_list_index[g] = m.nic_li[g];
    }
    b->cpu_numa[G] = m.misc_numa;

    uint16_t gpu_used = d.gpu_used;
    int ng = 0, n_nic_rec = 0;
    uint8_t nic_rec[NHD_MAX_GROUPS];
    bool fail = false;
    for (int g = 0; g < G && !fail; g++) {
        const nhd_pod_group& pg = t.pod.groups[g];
        const int numa = m.gpu_numa[g];
        const int nsw = pg.n_gpus ? nic_switch(r, m.nic_li[g]) : 0;
        for (int j = 0; j < pg.n_gpus; j++) {                       /* Node.py:707-726 */
            uint32_t fr = ~(uint32_t)gpu_used & ((1u << r.n_gpus) - 1);
            int dev = -1;
            for (uint32_t f = fr; f; f &= f - 1) {
                int i = ctz32(f);
                if (gpu_switch(r, i) == nsw) { dev = i; break; }
            }
            if (dev < 0) {
                if (t.pci) { fail = true; break; }
                uint32_t f = fr & r.gpu_numa_mask[numa];
                if (f) dev = ctz32(f);
            }
            if (dev < 0) { fail = true; break; }
            gpu_used |= (uint16_t)(1u << dev);
            if (ng < NHD_MAX_POD_GPUS) b->gpu_index[ng] = (uint8_t)dev;
            ng++;
        }
        if (fail) break;
        if (pg.flags & NHD_GRP_HAS_NIC_CORES) nic_rec[n_nic_rec++] = m.nic_li[g];
    }
    if (fail) {                                                      /* Node.py:825-837 */
        b->n_cores = b->n_gpus = b->n_claimed = 0;
        for (int i = 0; i < NHD_MAX_POD_GPUS; i++) b->gpu_index[i] = 0;
        b->status = n_nic_rec ? NHD_REF_WOULD_CRASH : NHD_ASSIGN_FAILED;
        return;
    }
    /* core accounting in call order: per group the proc batch then the helper batch, then misc */
    uint8_t fc[NHD_MAX_NUMA];
    for (int k = 0; k < NHD_MAX_NUMA; k++) { fc[k] = d.fc[k]; b->cores[k] = d.consumed[k]; }
    for (int g = 0; g < G; g++) {
        const nhd_pod_group& pg = t.pod.groups[g];
        const int k = m.gpu_numa[g];
        int w = batch_width(smt_node, (pg.flags & NHD_GRP_PROC_SMT) != 0, t.tot[g], fc[k]);
        fc[k] = (uint8_t)(fc[k] - w);
        w = batch_width(smt_node, (pg.flags & NHD_GRP_HELPER_SMT) != 0, pg.n_helpers, fc[k]);
        fc[k] = (uint8_t)(fc[k] - w);
    }
    {
        const int k = m.misc_numa;
        int w = batch_width(smt_node, (t.pod.flags & NHD_POD_MISC_SMT) != 0, t.pod.n_misc, fc[k]);
        fc[k] = (uint8_t)(fc[k] - w);
    }
    for (int k = 0; k < NHD_MAX_NUMA; k++) {
        d.consumed[k] = (uint8_t)(d.consumed[k] + (d.fc[k] - fc[k]));
        d.fc[k] = fc[k];
    }
    d.gpu_used = gpu_used;
    if (t.pod.hugepages_gb > 0) d.free_hugepages_gb -= t.pod.hugepages_gb;
    b->n_gpus = (uint8_t)ng;
    const int ncl = claimed_nic_order(nic_rec, n_nic_rec, b->claimed_nics);
    b->n_claimed = (uint8_t)ncl;
    for (int i = 0; i < ncl; i++) d.nic_inuse |= 1u << b->claimed_nics[i];
    b->status = NHD_PLACED;
}

/*
 * The core ids of one placed pod, from the node's SNAPSHOT record (state at the start of the
 * batch) and the pod's prefix offsets (b->cores[0..3] as left by assign_resources): the first
 * offsets[k] eligible cores of socket k went to earlier pods of the batch.  Fills b->cores /
 * b->n_cores and returns the logical ids taken as a mask.
 */
NHD_HDN M256 assign_cores_from_snapshot(const nhd_node_rec& snap, const PodType& t, nhd_binding* b)
{
    nhd_node_rec r = snap;
    const int per = r.phys_cores / r.n_numa;
    int offs[NHD_MAX_NUMA];
    for (int k = 0; k < NHD_MAX_NUMA; k++) { offs[k] = b->cores[k]; b->cores[k] = 0; }
    for (int k = 0; k < r.n_numa; k++) {
        int off = offs[k];
        M256 e = m_and(eligible_phys(r), m_range(k * per, (k + 1) * per));
        for (int w = 0; w < 4 && off > 0; w++) {
            uint64_t bits = e.w[w];
            while (bits && off > 0) {
                mark_used(r, 64 * w + ctz64(bits));                /* a used first-half id retires the whole core */
                bits &= bits - 1;
                off--;
            }
        }
    }
    const M256 before = rec_used(r);
    uint8_t batch[NHD_MAX_POD_CORES + 2];
    int nc = 0;
    const int G = t.G;
    for (int g = 0; g < G; g++) {
        const nhd_pod_group& pg = t.pod.groups[g];
        const int numa = b->gpu_numa[g];
        int n = cpu_batch(r, numa, t.tot[g], (pg.flags & NHD_GRP_PROC_SMT) != 0, batch);
        for (int k = 0; k < n; k++) { mark_used(r, batch[k]); if (nc < NHD_MAX_POD_CORES) b->cores[nc] = batch[k]; nc++; }
        n = cpu_batch(r, numa, pg.n_helpers, (pg.flags & NHD_GRP_HELPER_SMT) != 0, batch);
        for (int k = 0; k < n; k++) { mark_used(r, batch[k]); if (nc < NHD_MAX_POD_CORES) b->cores[nc] = batch[k]; nc++; }
    }
    {
        int n = cpu_batch(r, b->cpu_numa[G], t.pod.n_misc, (t.pod.flags & NHD_POD_MISC_SMT) != 0, batch);
        for (int k = 0; k < n; k++) { mark_used(r, batch[k]); if (nc < NHD_MAX_POD_CORES) b->cores[nc] = batch[k]; nc++; }
    }
    b->n_cores = (uint8_t)nc;
    return m_andnot(rec_used(r), before);
}

} // namespace nhd
