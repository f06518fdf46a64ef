"""Why FindNode drops a node, restated in Python from the reference's statements on packed records.

TEST INFRASTRUCTURE: the explanation oracle.  It follows the reference path statement by statement —
InitialNodeFilter (nhd/NHDScheduler.py:239-245), FilterPodResources (nhd/Matcher.py:65-84), the map-type test
(:45-47), FilterNumaTopology (:86-280), the PCI pruning and the intersection of IntersectResources (:283-353) and
SelectNode (:393-421) — over the values the Node getters return for a packed record (Node.py:225-296,456-462,
847-850), without sharing code with the CUDA core (nhd_b200/csrc/nhd_core.cuh).  It is itself pinned to the
unmodified reference by tests/golden/explain/cases.json (tests/golden/make_explain_golden.py).
"""
import itertools
import math
from collections import defaultdict

import numpy as np

from nhd_b200 import wire


def _bits(x):
    return [i for i in range(64) if (int(x) >> i) & 1]


def node_view(r, speed_table, nic_bw_avail_percent=0.9):
    """What the Node getters return for record r: free GPUs / physical cores per NUMA node, per-NUMA NIC
    (rx, tx) free bandwidth and switch, free GPUs per switch."""
    K, phys = int(r['n_numa']), int(r['phys_cores'])
    smt = bool(int(r['flags']) & wire.NODE_SMT)
    used = [int(w) for w in r['used']]

    def is_used(c):
        return (used[c >> 6] >> (c & 63)) & 1

    per = phys // K
    free_cpu = [0] * K                                   # GetFreeCpuCores (Node.py:250-264)
    for c in range(phys):
        if not is_used(c) and not (smt and is_used(c + phys)):
            free_cpu[c // per] += 1
    n_gpus = int(r['n_gpus'])
    gpu_numa = [next(k for k in range(K) if (int(r['gpu_numa_mask'][k]) >> g) & 1) for g in range(n_gpus)]
    gpu_free = [not ((int(r['gpu_used']) >> g) & 1) for g in range(n_gpus)]
    free_gpu = [sum(1 for g in range(n_gpus) if gpu_free[g] and gpu_numa[g] == k) for k in range(K)]   # GetFreeNumaGPUs
    gsw = defaultdict(lambda: 0)                         # GetFreeGPUPCICount (Node.py:266-273)
    for g in range(n_gpus):
        if gpu_free[g]:
            gsw[(int(r['gpu_sw']) >> (4 * g)) & 0xF] += 1
    nic_free, nic_sw = [[] for _ in range(K)], [[] for _ in range(K)]
    for j in range(int(r['n_nics'])):                    # GetFreeNumaNicResources / GetNumaNICPCIResources (:275-296)
        k = next(k for k in range(K) if (int(r['nic_numa_mask'][k]) >> j) & 1)
        sc = (int(r['nic_speed'][j >> 4]) >> (4 * (j & 15))) & 0xF
        bw = 0 if (int(r['nic_inuse']) >> j) & 1 else float(speed_table[sc]) * nic_bw_avail_percent
        nic_free[k].append([bw, bw])
        nic_sw[k].append((int(r['nic_sw'][j >> 4]) >> (4 * (j & 15))) & 0xF)
    return {'K': K, 'smt': smt, 'free_cpu': free_cpu, 'free_gpu': free_gpu, 'gsw': gsw,
            'nic_free': nic_free, 'nic_sw': nic_sw}


def pod_view(p):
    """CfgTopology.GetTotal{Gpus,Cpus,NICs}Requested (CfgTopology.py:199-232) of a packed pod."""
    G = int(p['n_groups'])
    gs = [p['groups'][g] for g in range(G)]
    req_gpus = [int(g['n_gpus']) for g in gs]
    proc = []
    for g in gs:
        tot = int(g['n_proc']) + sum(int(x) for x in g['gpu_feeders'][:int(g['n_gpus'])])
        proc.append(((tot, bool(int(g['flags']) & wire.GRP_PROC_SMT)),
                     (int(g['n_helpers']), bool(int(g['flags']) & wire.GRP_HELPER_SMT))))
    req_nics = [(float(g['rx_gbps']), float(g['tx_gbps'])) for g in gs]
    return {'G': G, 'req_gpus': req_gpus, 'proc': proc, 'misc': int(p['n_misc']), 'req_nics': req_nics,
            'map_type': int(p['map_type']), 'hugepages': int(p['hugepages_gb']), 'group_mask': int(p['group_mask'])}


def _nic_fits(v, pv, p, prune):
    """Is there one entry of nic_cands for NUMA tuple p (Matcher.py:242-268) that survives, with ``prune``, the PCI
    switch test (:312-322)?  The reference enumerates every joint NIC choice and subtracts the groups' (rx, tx) in
    group order; a choice survives if nothing went negative.  Bandwidth only ever decreases, so a search in group
    order that stops at the first negative value finds a survivor iff the enumeration has one."""
    G = pv['G']
    if any(len(v['nic_free'][p[g]]) == 0 for g in range(G)):
        return False                                    # product(range(0), ...) is empty (:247)

    def rec(g, ttl, chosen):
        if g == G:
            if not prune:
                return True
            cnt = defaultdict(lambda: 0)
            for (k, i) in chosen:
                cnt[v['nic_sw'][k][i]] += 1
            return all(v['gsw'][s] >= n for s, n in cnt.items())
        k = p[g]
        for i in range(len(v['nic_free'][k])):
            t = [row[:] for row in ttl[k]]
            t[i][0] -= pv['req_nics'][g][0]
            t[i][1] -= pv['req_nics'][g][1]
            if t[i][0] < 0 or t[i][1] < 0:
                continue
            ttl2 = list(ttl)
            ttl2[k] = t
            if rec(g + 1, ttl2, chosen + [(k, i)]):
                return True
        return False

    return rec(0, [[row[:] for row in x] for x in v['nic_free']], [])


def explain_node(r, p, speed_table, now, nic_bw_avail_percent=0.9, min_busy_secs=30.0):
    """wire.WHY_* code of node record r for packed pod p at clock now."""
    pv = pod_view(p)
    flags = int(r['flags'])
    if not (int(r['group_mask']) & pv['group_mask']):                      # NHDScheduler.py:241
        return wire.WHY_NOT_IN_GROUP
    if not flags & wire.NODE_ACTIVE:                                        # :242
        return wire.WHY_INACTIVE
    if flags & wire.NODE_MAINTENANCE:                                       # Matcher.py:73
        return wire.WHY_MAINTENANCE
    if pv['hugepages'] > int(r['free_hugepages_gb']):                       # :78
        return wire.WHY_HUGEPAGES
    if pv['map_type'] not in (wire.MAP_NUMA, wire.MAP_PCI):                 # :45
        return wire.WHY_MAP_TYPE
    if sum(pv['req_gpus']) > 0 and (now - float(r['busy_time'])) < min_busy_secs:   # :107-108, Node.py:847-850
        return wire.WHY_BUSY
    v = node_view(r, speed_table, nic_bw_avail_percent)
    K, G = v['K'], pv['G']
    gpu_t = set()                                                           # :117-129
    for q in itertools.product(range(K), repeat=G):
        ttl = [0] * K
        for i, n in enumerate(q):
            ttl[n] += pv['req_gpus'][i]
        if all(ttl[x] <= v['free_gpu'][x] for x in range(K)):
            gpu_t.add(q)
    if not gpu_t:
        return wire.WHY_GPU
    clist = []                                                              # :179-201
    for t in pv['proc']:
        if v['smt']:
            clist.append((int(math.ceil(t[0][0] / 2.0)) if t[0][1] else t[0][0]) +
                         (int(math.ceil(t[1][0] / 2.0)) if t[1][1] else t[1][0]))
        else:
            clist.append(t[0][0] + t[1][0])
    clist.append(int(math.ceil(pv['misc'] / 2.0)) if v['smt'] else pv['misc'])   # the SMT test there is always true
    cpu_t = set()                                                           # :203-212
    for q in itertools.product(range(K), repeat=G + 1):
        ttl = [0] * K
        for i, n in enumerate(q):
            ttl[n] += clist[i]
        if all(ttl[x] <= v['free_cpu'][x] for x in range(K)):
            cpu_t.add(q[:-1])
    if not cpu_t:
        return wire.WHY_CPU
    nic_t = {q for q in itertools.product(range(K), repeat=G) if _nic_fits(v, pv, q, False)}
    if not nic_t:
        return wire.WHY_NIC
    isect = gpu_t & cpu_t & nic_t                                           # :349
    if not isect:
        return wire.WHY_NUMA
    if pv['map_type'] == wire.MAP_PCI and not any(_nic_fits(v, pv, q, True) for q in isect):
        return wire.WHY_PCIE
    return wire.WHY_FEASIBLE


def explain(recs, p, speed_table, now, nic_bw_avail_percent=0.9, min_busy_secs=30.0):
    """(codes[node] uint8, first_fit): every node's reason and the node FindNode returns (SelectNode,
    Matcher.py:400-421: a pod without GPUs takes the first feasible node without GPUs if there is one), or -1."""
    codes = np.array([explain_node(r, p, speed_table, now, nic_bw_avail_percent, min_busy_secs) for r in recs],
                     dtype=np.uint8)
    feas = np.flatnonzero(codes == wire.WHY_FEASIBLE)
    if len(feas) == 0:
        return codes, -1
    if sum(pod_view(p)['req_gpus']) == 0:
        for n in feas:
            if int(recs[n]['n_gpus']) == 0:
                return codes, int(n)
    return codes, int(feas[0])


def counts_of(codes):
    return np.bincount(np.asarray(codes, dtype=np.int64), minlength=wire.WHY_COUNT).astype(np.int32)
