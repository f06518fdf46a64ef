/*
 * nhd_b200.h — C-ABI of the B200-native NHD placement solver.
 *
 * This is the drop-in boundary for the one hot path of Viasat/nhd: the node
 * filter -> NUMA/PCIe intersection -> node select -> physical assignment loop.
 * The reference has no FFI; its seam is the Python method surface
 *     Matcher.FindNode(nl, top)                      nhd/Matcher.py:27-63
 *     Node.SetPhysicalIdsFromMapping(mapping, top)   nhd/Node.py:663-841
 *     Node.ClaimPodNICResources(nidx)                nhd/Node.py:644-646
 * driven once per pending pod by NHDScheduler.AttemptScheduling
 * (nhd/NHDScheduler.py:277-304) after NHDScheduler.InitialNodeFilter
 * (nhd/NHDScheduler.py:235-247).  One call of nhd_solve_batch() replaces that
 * whole per-pod sequence for a batch of pods, with the reference's strict
 * sequential semantics (pod i sees the cluster after pods 0..i-1).
 *
 * Conventions: plain C, caller owns every buffer, all functions return an
 * int32 status (0 = NHD_OK, negative = error), no exceptions cross the
 * boundary, a handle is not re-entrant (the reference has a single scheduler
 * thread, nhd/NHDScheduler.py:43).  Every pointer is a HOST pointer unless the
 * name ends in _dev.
 */
#ifndef NHD_B200_H
#define NHD_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- limits of the packed layout (checked by nhd_validate_*) -------------- */
#define NHD_MAX_NUMA           4    /* Node.numa_nodes (== sockets, Node.py:336)      */
#define NHD_MAX_GROUPS         4    /* len(CfgTopology.proc_groups)                   */
#define NHD_MAX_TUPLES         256  /* numa^(groups+1) must not exceed this; numa = the largest NUMA count among the
                                        nodes the filter could accept (active, not in maintenance) at staging time */
#define NHD_MAX_GPUS           16   /* len(Node.gpus)                                 */
#define NHD_MAX_NICS           32   /* len(Node.nics) (schedulable NICs / VFs)        */
#define NHD_MAX_LCORES         256  /* len(Node.cores) (logical cores)                */
#define NHD_MAX_SWITCHES       16   /* distinct PCIe switch ids on one node           */
#define NHD_MAX_SPEED_CLASSES  16   /* distinct NIC link speeds in the cluster        */
#define NHD_MAX_GROUP_GPUS     8    /* len(ProcGroup.group_gpus)                      */
#define NHD_MAX_POD_GPUS       16   /* GPUs requested by one pod                      */
#define NHD_MAX_POD_CORES      72   /* cores requested by one pod                     */
#define NHD_MAX_GROUP_NAMES    64   /* distinct node-group names in the cluster       */

/* ---- return codes ---------------------------------------------------------- */
#define NHD_OK                  0
#define NHD_ERR_INVALID        -1   /* bad argument / malformed record                */
#define NHD_ERR_UNSUPPORTED    -2   /* valid for the reference, outside packed limits */
#define NHD_ERR_CUDA           -3   /* CUDA runtime failure (see nhd_last_error)      */
#define NHD_ERR_NCCL           -4   /* NCCL failure / NCCL not loadable               */
#define NHD_ERR_STATE          -5   /* call order (e.g. solve before load)            */
#define NHD_ERR_LABELS         -6   /* Node.ParseLabels would return False (node ignored) */

/* ---- per-pod outcome (nhd_binding.status) ---------------------------------- */
#define NHD_PLACED              0   /* FindNode found a node and assignment succeeded (NHDScheduler.py:291-304) */
#define NHD_NO_CANDIDATE        1   /* FindNode returned (None,)   (Matcher.py:52,60)                           */
#define NHD_ASSIGN_FAILED       2   /* SetPhysicalIdsFromMapping raised IndexError, clean unwind (Node.py:825-837) */
#define NHD_REF_WOULD_CRASH     3   /* unwind hit the buggy NIC rollback (Node.py:831-835); state as IndexError  */
#define NHD_BAD_MAP_TYPE        4   /* map_type not NUMA/PCI -> (None,) (Matcher.py:45-47)                       */

/* CfgTopology.TopologyMapType values (CfgTopology.py:41-45) */
#define NHD_MAP_INVALID         0
#define NHD_MAP_NUMA            1
#define NHD_MAP_PCI             2
#define NHD_MAP_NONE            3

/* nhd_node_rec.flags */
#define NHD_NODE_SMT            0x01  /* Node.smt_enabled   (Node.py:335) */
#define NHD_NODE_ACTIVE         0x02  /* Node.active        (NHDScheduler.py:242) */
#define NHD_NODE_MAINTENANCE    0x04  /* Node.maintenance   (Matcher.py:73) */

/* nhd_pod_group.flags */
#define NHD_GRP_PROC_SMT        0x01  /* ProcGroup.proc_smt   == SMT_ENABLED */
#define NHD_GRP_HELPER_SMT      0x02  /* ProcGroup.helper_smt == SMT_ENABLED */
#define NHD_GRP_HAS_NIC_CORES   0x04  /* any proc core with nic_dir RX or TX (Node.py:742) */

/* nhd_pod.flags */
#define NHD_POD_MISC_SMT        0x01  /* CfgTopology.misc_cores_smt == SMT_ENABLED */

/*
 * nhd_node_rec — the complete decision-relevant state of one Node
 * (nhd/Node.py:100-131), 128 bytes.  Everything the reference reads on the hot
 * path is here; names, MACs, GPU device ids and the NIC speed_used/pods_used
 * counters stay with the caller (they never influence a decision while
 * ENABLE_SHARING is False, Node.py:20,292).
 *
 *  logical core c (Node.cores[c]):  socket(c) = (c % phys_cores) / (phys_cores / n_numa)
 *                                   sibling(c) = c +- phys_cores when SMT      (Node.py:343-350)
 *  gpus[i] / nics[i] are in Node.gpus / Node.nics list order (label order, Node.py:388-432).
 *  A NIC's per-NUMA index NodeNic.idx (Node.py:413-418) is its rank among the
 *  set bits of nic_numa_mask[numa].
 *  Switch ids are node-local 4-bit aliases of NodeGpu/NodeNic.pciesw (only
 *  equality is ever tested: Matcher.py:316-320, Node.py:651).
 */
typedef struct nhd_node_rec {
    uint64_t used[4];            /* bit c = Node.cores[c].used (reserved cores included)      */
    uint16_t gpu_used;           /* bit i = Node.gpus[i].used                                  */
    uint8_t  n_gpus;             /* len(Node.gpus)                                             */
    uint8_t  n_nics;             /* len(Node.nics)                                             */
    uint32_t nic_inuse;          /* bit i = Node.nics[i].pods_used > 0                         */
    int32_t  free_hugepages_gb;  /* Node.mem.free_hugepages_gb                                 */
    uint8_t  n_numa;             /* Node.numa_nodes                                            */
    uint8_t  flags;              /* NHD_NODE_*                                                 */
    uint16_t phys_cores;         /* label nfd-extras-cpu.num_cores (physical cores, Node.py:334) */
    double   busy_time;          /* Node.busy_time (monotonic seconds, Node.py:115,845)        */
    uint64_t group_mask;         /* bit j = cluster group name j in Node.groups                */
    uint16_t gpu_numa_mask[NHD_MAX_NUMA];  /* bit i = (Node.gpus[i].numa_node == k)            */
    uint64_t gpu_sw;             /* nibble i = local switch id of Node.gpus[i]                 */
    uint32_t nic_numa_mask[NHD_MAX_NUMA];  /* bit i = (Node.nics[i].numa_node == k)            */
    uint64_t nic_sw[2];          /* nibble i = local switch id of Node.nics[i]                 */
    uint64_t nic_speed[2];       /* nibble i = speed class of Node.nics[i] (nhd_params.speed_gbps) */
} nhd_node_rec;

/* One ProcGroup of a pod request (CfgTopology.py:82-110), 32 bytes. */
typedef struct nhd_pod_group {
    uint8_t n_gpus;              /* len(group_gpus)                                            */
    uint8_t n_proc;              /* len(proc_cores)                                            */
    uint8_t n_helpers;           /* len(misc_cores) of the group ("helper" cores)              */
    uint8_t flags;               /* NHD_GRP_*                                                  */
    uint8_t gpu_feeders[NHD_MAX_GROUP_GPUS]; /* len(group_gpus[j].cpu_cores)                   */
    uint8_t pad_[4];
    double  rx_gbps;             /* sum of nic_speed over RX proc cores, core order (CfgTopology.py:219-232) */
    double  tx_gbps;             /* same for TX                                                */
} nhd_pod_group;

/* One pending pod: CfgTopology (CfgTopology.py:126-143) + its node-group list
 * (NHDScheduler.py:238, K8SMgr.py:160-163), 144 bytes. */
typedef struct nhd_pod {
    uint8_t  n_groups;           /* len(proc_groups), 1..NHD_MAX_GROUPS                        */
    uint8_t  map_type;           /* NHD_MAP_*                                                  */
    uint8_t  n_misc;             /* len(CfgTopology.misc_cores)                                */
    uint8_t  flags;              /* NHD_POD_*                                                  */
    int32_t  hugepages_gb;       /* CfgTopology.hugepages_gb                                   */
    uint64_t group_mask;         /* bit j = cluster group name j requested by the pod          */
    nhd_pod_group groups[NHD_MAX_GROUPS];
} nhd_pod;

/*
 * nhd_binding — everything AttemptScheduling learns for one pod, 128 bytes:
 * the node, the mapping dict FindNode returns (Matcher.py:452), every value
 * SetPhysicalIdsFromMapping writes into the CfgTopology (Node.py:724-811) and
 * the NIC list handed to ClaimPodNICResources (NHDScheduler.py:302-304).
 */
typedef struct nhd_binding {
    int32_t status;              /* NHD_PLACED ...                                             */
    int32_t node;                /* node index in load order, -1 when none                     */
    uint8_t n_groups;
    uint8_t n_cores;             /* entries used in cores[]                                    */
    uint8_t n_gpus;              /* entries used in gpu_index[]                                */
    uint8_t n_claimed;           /* entries used in claimed_nics[]                             */
    uint8_t gpu_numa[NHD_MAX_GROUPS];      /* mapping['gpu']                                   */
    uint8_t cpu_numa[NHD_MAX_GROUPS + 1];  /* mapping['cpu'] (last used entry = misc cores)    */
    uint8_t nic_numa[NHD_MAX_GROUPS];      /* mapping['nic'][g][0]                             */
    uint8_t nic_idx[NHD_MAX_GROUPS];       /* mapping['nic'][g][1] (per-NUMA NodeNic.idx)      */
    uint8_t nic_list_index[NHD_MAX_GROUPS];/* index of that NIC in Node.nics                   */
    uint8_t claimed_nics[NHD_MAX_GROUPS];  /* list({x[0] for x in nic_list}), CPython set order */
    uint8_t pad_[3];
    uint8_t gpu_index[NHD_MAX_POD_GPUS];   /* index in Node.gpus per requested GPU, group-major */
    /* logical core ids in canonical order: per group [feeder cores of gpu 0..][proc cores]
     * [helper cores]; then the top-level misc cores (Node.py:728-811). */
    uint8_t cores[NHD_MAX_POD_CORES];
} nhd_binding;

/* Solver parameters: the module constants of nhd/Node.py:18-20,107. */
typedef struct nhd_params {
    double   nic_bw_avail_percent;   /* NIC_BW_AVAIL_PERCENT (0.9)                             */
    double   min_busy_secs;          /* Node.MIN_BUSY_SECS (30.0)                              */
    int32_t  enable_sharing;         /* ENABLE_SHARING; only 0 is supported                    */
    int32_t  n_speed_classes;
    double   speed_gbps[NHD_MAX_SPEED_CLASSES]; /* NodeNic.speed (= label Mb/s / 1e3) per class */
    int32_t  device;                 /* CUDA device ordinal                                    */
    int32_t  rank;                   /* node-shard rank, 0 when single GPU                     */
    int32_t  world_size;             /* number of GPUs sharing the node set                    */
    int32_t  reserved_;              /* 0.  Test hook: low byte 1 = the general one-warp sweep only, 2 = never sweep the two pod
                                      * classes side by side; bit 8 = no standing decisions, bit 9 = same as 2, bit 10 = no direct-path tables;
                                      * all settings produce identical bindings (tests/test_gpu_parity.py)      */
    uint8_t  nccl_unique_id[128];    /* from nhd_nccl_unique_id() on rank 0; unused if world_size==1 */
} nhd_params;

/* per-call device timings of the last nhd_solve_batch (CUDA events, ms) */
typedef struct nhd_timing {
    float filter_ms;             /* snapshot predicate kernel                                  */
    float exchange_ms;           /* NCCL all-gather + slot unpack (0 when world_size == 1)     */
    float sweep_ms;              /* select + assign sweep kernel                               */
    float total_ms;              /* first launch to last kernel end                            */
    int32_t n_types;             /* distinct pod descriptors in the batch                      */
    int32_t n_launches;          /* kernels launched by the call                               */
} nhd_timing;

typedef struct nhd_handle nhd_handle;

void    nhd_default_params(nhd_params* p);
int32_t nhd_nccl_unique_id(uint8_t out[128]);
/* (nodes x distinct pod types of a batch) from which world_size > 1 handles split the snapshot filter over the ranks
 * and exchange the results with one all-gather; smaller batches are filtered whole by every rank with no collective
 * (the reference has no counterpart: it is one process, NHDScheduler.py:43).  NHD_SHARD_MIN_PAIRS in the environment
 * — the same on every rank — overrides the default (2^21) for handles created afterwards. */
int64_t nhd_shard_min_pairs(void);
int32_t nhd_create(const nhd_params* p, nhd_handle** out);
int32_t nhd_destroy(nhd_handle* h);
const char* nhd_last_error(const nhd_handle* h);

/* Page-locked host buffers: records / pods / bindings placed here move to and from the device
 * without a staging copy (anything else is staged internally). */
int32_t nhd_alloc_pinned(uint64_t bytes, void** out);
int32_t nhd_free_pinned(void* p);

/* Host-side validation of wire records against the limits above (nhd_load_nodes runs the same
 * check on the device). */
int32_t nhd_validate_node(const nhd_node_rec* rec);
int32_t nhd_validate_pod(const nhd_pod* pod);

/* Full upload (start-up, ResetResources; NHDScheduler.py:74-105,146-159). */
int32_t nhd_load_nodes(nhd_handle* h, int32_t n_nodes, const nhd_node_rec* recs);
/* Claim / release / cordon / maintenance / group deltas between batches
 * (NHDScheduler.py:107-205,533-570): overwrite records idx[0..n). */
int32_t nhd_update_nodes(nhd_handle* h, int32_t n, const int32_t* idx, const nhd_node_rec* recs);
/* Download the current records [first, first+n). */
int32_t nhd_read_nodes(nhd_handle* h, int32_t first, int32_t n, nhd_node_rec* out);

/* Snapshot / restore of the device mirror (device-to-device; used by benchmarks
 * to replay a batch from the same cluster state). */
int32_t nhd_snapshot(nhd_handle* h);
int32_t nhd_restore(nhd_handle* h);

/*
 * Solve a batch with sequential semantics.  now[i] is the value
 * time.monotonic() would return while pod i is scheduled (Node.py:845,848).
 * Host buffers in, host buffers out; the device mirror is updated in place.
 */
int32_t nhd_solve_batch(nhd_handle* h, int32_t n_pods, const nhd_pod* pods,
                        const double* now, nhd_binding* out);

/*
 * The three phases of nhd_solve_batch, separately callable so that a caller (or a
 * benchmark) can keep a batch resident in HBM:
 *   nhd_stage_batch    validate, de-duplicate descriptors into pod types, host -> device
 *   nhd_solve_staged   launch the kernels on the staged batch (asynchronous)
 *   nhd_fetch_bindings wait, device -> host
 * nhd_sync only waits (bindings stay on the device).
 */
int32_t nhd_stage_batch(nhd_handle* h, int32_t n_pods, const nhd_pod* pods, const double* now);
int32_t nhd_solve_staged(nhd_handle* h);
int32_t nhd_fetch_bindings(nhd_handle* h, nhd_binding* out);
int32_t nhd_sync(nhd_handle* h);

/* Debug / tests: run only the snapshot predicate kernel on the staged batch, so that
 * nhd_read_filter returns the bitmaps before the sweep edits them. */
int32_t nhd_run_filter_only(nhd_handle* h);

int32_t nhd_last_timing(const nhd_handle* h, nhd_timing* out);

/* Per-pod-type feasibility bitmaps of the last solve's snapshot filter
 * (debug / tests): words[t * words_per_type + w], bit b of word w = node 64*w+b. */
int32_t nhd_read_filter(nhd_handle* h, int32_t* n_types, int32_t* words_per_type,
                        uint64_t* words, int64_t capacity_words, int32_t* pod_type, int32_t n_pods);

/* Debug: 64 words of per-phase cycle accumulators / counters of the last sweep; only non-zero
 * in libraries built with -DNHD_PROFILE. */
int32_t nhd_debug_counters(nhd_handle* h, uint64_t* out64);

/* ---- node ingest (host side, no GPU): NFD label dictionary -> nhd_node_rec --------------------
 * Replaces Node.ParseLabels (nhd/Node.py:468-487: InitGroups :312, InitMaintenance :324, InitCores :328,
 * InitNics :378, InitGpus :428, InitMisc :440) + Node.SetHugepages (:489-493) for a node the scheduler has
 * just discovered (nhd/NHDScheduler.py:122-140), and the packing of the resulting Node object.
 * An nhd_ingest holds the two cluster-wide dictionaries the records refer to: node-group names -> bits of
 * group_mask, NIC link speeds -> speed classes (= nhd_params.speed_gbps).  What the placement loop does not
 * need (interface names, MACs, the gateway string) stays with the caller, addressed by label position. */
typedef struct nhd_ingest nhd_ingest;

typedef struct nhd_node_aux {
    int32_t data_vlan;                     /* DATA_PLANE_VLAN                (Node.py:441-446)   */
    int32_t res_hugepages_gb;              /* RES_HUGEPAGES_GB, 0 if absent  (Node.py:451-453)   */
    int32_t n_reserved_cores;              /* len(Node.reserved_cores)       (Node.py:368-371)   */
    int32_t gw_label;                      /* index of the DATA_DEFAULT_GW label                  */
    int32_t gpu_device_id[NHD_MAX_GPUS];   /* Node.gpus[i].device_id, -1 beyond n_gpus            */
    int32_t nic_label[NHD_MAX_NICS];       /* index of the label Node.nics[i] came from, -1 beyond n_nics */
} nhd_node_aux;

int32_t nhd_ingest_create(nhd_ingest** out);
int32_t nhd_ingest_destroy(nhd_ingest* g);
/* keys / values: the node's labels in dictionary order (NIC / GPU list order follows label order).
 * NHD_ERR_LABELS: the reference's ParseLabels returns False; NHD_ERR_INVALID: it would raise;
 * NHD_ERR_UNSUPPORTED: beyond NHD_MAX_*.  aux may be NULL. */
int32_t nhd_ingest_node(nhd_ingest* g, int32_t n_labels, const char* const* keys, const char* const* values,
                        int32_t active, int32_t hugepages_alloc_gb, int32_t hugepages_free_gb,
                        nhd_node_rec* rec, nhd_node_aux* aux);
/* '.'-joined group names (the NHD_GROUP label / pod group annotation) -> group_mask bits */
int32_t nhd_ingest_group_mask(nhd_ingest* g, const char* dotted_names, int32_t create, uint64_t* mask);
/* speed classes seen so far, for nhd_params.speed_gbps */
int32_t nhd_ingest_speed_table(const nhd_ingest* g, double out[NHD_MAX_SPEED_CLASSES], int32_t* n_classes);

/* ---- node statistics from packed records (host side) ------------------------------------------
 * What NHDScheduler.GetBasicNodeStats (nhd/NHDScheduler.py:355-378) reads off a Node, for records that came
 * back from the device mirror (nhd_read_nodes): the counters the packed state carries.  totalhuge_gb,
 * totalpods and the per-NIC used speeds are not part of the placement state and stay with the caller. */
typedef struct nhd_node_stats {
    int32_t freegpu;                       /* Node.GetFreeGpuCount()      (Node.py:235-237) */
    int32_t totalgpu;                      /* Node.GetTotalGPUs()         (Node.py:239-241) */
    int32_t freecpu;                       /* Node.GetFreeCpuCoreCount(): logical cores, with SMT only those whose
                                            * sibling is free too         (Node.py:225-233) */
    int32_t totalcpu;                      /* Node.GetTotalCPUs() = len(Node.cores)         (Node.py:243-245) */
    int32_t freehuge_gb;                   /* Node.GetFreeHugepages()     (Node.py:171-173) */
    int32_t active;                        /* Node.GetNodeActive()        (Node.py:163-165) */
    int32_t maintenance;
    int32_t nics_in_use;                   /* NICs with pods_used > 0 */
    int32_t free_cores_numa[NHD_MAX_NUMA]; /* Node.GetFreeCpuCores(): free physical cores per NUMA node (Node.py:250-264) */
    int32_t free_gpus_numa[NHD_MAX_NUMA];  /* Node.GetFreeNumaGPUs()      (Node.py:456-462) */
} nhd_node_stats;
int32_t nhd_node_stats_from_records(int32_t n, const nhd_node_rec* recs, nhd_node_stats* out);

/* ---- explanation: why FindNode drops a node for a pod ------------------------------------------
 * The reference logs, node by node, the first stage of its path that removes a node (Matcher.py INFO
 * records); nhd_explain computes that stage for every (pod, loaded node) pair on the device.  A node
 * gets exactly one code: the first of the list below that applies, judged on the current records at
 * the pod's clock now[i]. */
#define NHD_WHY_FEASIBLE        0   /* in filts[1] when SelectNode runs                (Matcher.py:393-421) */
#define NHD_WHY_NOT_IN_GROUP    1   /* no node group in common with the pod            (NHDScheduler.py:241) */
#define NHD_WHY_INACTIVE        2   /* in the group but not active                     (NHDScheduler.py:242-245) */
#define NHD_WHY_MAINTENANCE     3   /* node in maintenance                             (Matcher.py:73-75) */
#define NHD_WHY_HUGEPAGES       4   /* too few free 1 GB hugepages                     (Matcher.py:78-79) */
#define NHD_WHY_MAP_TYPE        5   /* pod map type neither NUMA nor PCI               (Matcher.py:45-47) */
#define NHD_WHY_BUSY            6   /* GPU pod, last deployment within MIN_BUSY_SECS   (Matcher.py:107-111) */
#define NHD_WHY_GPU             7   /* GPU stage empty                                 (Matcher.py:132-134) */
#define NHD_WHY_CPU             8   /* CPU stage over (G+1)-tuples empty               (Matcher.py:214-216) */
#define NHD_WHY_NIC             9   /* NIC stage empty without the PCIe pruning        (Matcher.py:270-272) */
#define NHD_WHY_PCIE           10   /* intersection non-empty only without the PCIe-switch pruning (Matcher.py:295-335,349-353) */
#define NHD_WHY_NUMA           11   /* GPU / CPU / NIC NUMA tuples do not intersect    (Matcher.py:349-353) */
#define NHD_WHY_COUNT          12

/* Read-only: the records, the snapshot, a staged batch, the last bindings, nhd_read_filter and
 * nhd_last_timing are left as they were; returns after a synchronise.  Pods are validated as
 * nhd_stage_batch validates them.  On a world_size > 1 handle the call is local to the rank (every
 * rank holds every record) and runs no collective.
 *   counts     [n_pods][NHD_WHY_COUNT]: nodes per reason; each row sums to the loaded node count
 *   first_fit  [n_pods] or NULL: the node FindNode would return now (load order), -1 if none
 *   reasons    [n_pods][n_nodes] or NULL: the reason code of every node */
int32_t nhd_explain(nhd_handle* h, int32_t n_pods, const nhd_pod* pods, const double* now,
                    int32_t* counts, int32_t* first_fit, uint8_t* reasons);

#ifdef __cplusplus
}
#endif
#endif /* NHD_B200_H */
