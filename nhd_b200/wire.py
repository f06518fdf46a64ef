"""numpy dtypes that mirror the C-ABI wire structs of ``include/nhd_b200.h`` byte for byte."""
import numpy as np

MAX_NUMA = 4
MAX_GROUPS = 4
MAX_TUPLES = 256
MAX_GPUS = 16
MAX_NICS = 32
MAX_LCORES = 256
MAX_SWITCHES = 16
MAX_SPEED_CLASSES = 16
MAX_GROUP_GPUS = 8
MAX_POD_GPUS = 16
MAX_POD_CORES = 72
MAX_GROUP_NAMES = 64

# error codes (include/nhd_b200.h)
OK, ERR_INVALID, ERR_UNSUPPORTED, ERR_CUDA, ERR_NCCL, ERR_STATE, ERR_LABELS = 0, -1, -2, -3, -4, -5, -6

# nhd_binding.status
PLACED, NO_CANDIDATE, ASSIGN_FAILED, REF_WOULD_CRASH, BAD_MAP_TYPE = 0, 1, 2, 3, 4
STATUS_NAMES = {PLACED: 'placed', NO_CANDIDATE: 'none', ASSIGN_FAILED: 'assign_failed',
                REF_WOULD_CRASH: 'ref_would_crash', BAD_MAP_TYPE: 'bad_map_type'}

# nhd_explain reason codes (NHD_WHY_*): the first stage of the reference path that drops a node for a pod
(WHY_FEASIBLE, WHY_NOT_IN_GROUP, WHY_INACTIVE, WHY_MAINTENANCE, WHY_HUGEPAGES, WHY_MAP_TYPE, WHY_BUSY, WHY_GPU, WHY_CPU,
 WHY_NIC, WHY_PCIE, WHY_NUMA) = range(12)
WHY_COUNT = 12
WHY_NAMES = ('FEASIBLE', 'NOT_IN_GROUP', 'INACTIVE', 'MAINTENANCE', 'HUGEPAGES', 'MAP_TYPE', 'BUSY', 'GPU', 'CPU',
             'NIC', 'PCIE', 'NUMA')
# short text per code, in the style of kube-scheduler's "0/N nodes are available: 3 <text>, ..."
WHY_TEXT = ('feasible', "not in the pod's node groups", 'inactive', 'in maintenance', 'too few free hugepages',
            'unsupported topology map type', 'busy after a recent GPU deployment', 'too few free GPUs per NUMA node',
            'too few free CPU cores', 'too little free NIC bandwidth', 'no NIC on a PCIe switch with a free GPU',
            'GPUs, CPU cores and NICs on different NUMA nodes')

MAP_INVALID, MAP_NUMA, MAP_PCI, MAP_NONE = 0, 1, 2, 3
NODE_SMT, NODE_ACTIVE, NODE_MAINTENANCE = 1, 2, 4
GRP_PROC_SMT, GRP_HELPER_SMT, GRP_HAS_NIC_CORES = 1, 2, 4
POD_MISC_SMT = 1

NODE_DTYPE = np.dtype([
    ('used', '<u8', (4,)),
    ('gpu_used', '<u2'), ('n_gpus', 'u1'), ('n_nics', 'u1'),
    ('nic_inuse', '<u4'), ('free_hugepages_gb', '<i4'),
    ('n_numa', 'u1'), ('flags', 'u1'), ('phys_cores', '<u2'),
    ('busy_time', '<f8'), ('group_mask', '<u8'),
    ('gpu_numa_mask', '<u2', (MAX_NUMA,)), ('gpu_sw', '<u8'),
    ('nic_numa_mask', '<u4', (MAX_NUMA,)),
    ('nic_sw', '<u8', (2,)), ('nic_speed', '<u8', (2,)),
], align=False)
assert NODE_DTYPE.itemsize == 128

POD_GROUP_DTYPE = np.dtype([
    ('n_gpus', 'u1'), ('n_proc', 'u1'), ('n_helpers', 'u1'), ('flags', 'u1'),
    ('gpu_feeders', 'u1', (MAX_GROUP_GPUS,)), ('pad_', 'u1', (4,)),
    ('rx_gbps', '<f8'), ('tx_gbps', '<f8'),
], align=False)
assert POD_GROUP_DTYPE.itemsize == 32

POD_DTYPE = np.dtype([
    ('n_groups', 'u1'), ('map_type', 'u1'), ('n_misc', 'u1'), ('flags', 'u1'),
    ('hugepages_gb', '<i4'), ('group_mask', '<u8'),
    ('groups', POD_GROUP_DTYPE, (MAX_GROUPS,)),
], align=False)
assert POD_DTYPE.itemsize == 144

BINDING_DTYPE = np.dtype([
    ('status', '<i4'), ('node', '<i4'),
    ('n_groups', 'u1'), ('n_cores', 'u1'), ('n_gpus', 'u1'), ('n_claimed', 'u1'),
    ('gpu_numa', 'u1', (MAX_GROUPS,)), ('cpu_numa', 'u1', (MAX_GROUPS + 1,)),
    ('nic_numa', 'u1', (MAX_GROUPS,)), ('nic_idx', 'u1', (MAX_GROUPS,)),
    ('nic_list_index', 'u1', (MAX_GROUPS,)), ('claimed_nics', 'u1', (MAX_GROUPS,)),
    ('pad_', 'u1', (3,)),
    ('gpu_index', 'u1', (MAX_POD_GPUS,)),
    ('cores', 'u1', (MAX_POD_CORES,)),
], align=False)
assert BINDING_DTYPE.itemsize == 128

# nhd_node_aux: what nhd_ingest_node reads from the labels besides the packed record
NODE_AUX_DTYPE = np.dtype([
    ('data_vlan', '<i4'), ('res_hugepages_gb', '<i4'), ('n_reserved_cores', '<i4'), ('gw_label', '<i4'),
    ('gpu_device_id', '<i4', (MAX_GPUS,)), ('nic_label', '<i4', (MAX_NICS,)),
])
assert NODE_AUX_DTYPE.itemsize == 16 + 4 * MAX_GPUS + 4 * MAX_NICS

# nhd_node_stats: GetBasicNodeStats counters of one packed record
NODE_STATS_DTYPE = np.dtype([
    ('freegpu', '<i4'), ('totalgpu', '<i4'), ('freecpu', '<i4'), ('totalcpu', '<i4'), ('freehuge_gb', '<i4'),
    ('active', '<i4'), ('maintenance', '<i4'), ('nics_in_use', '<i4'),
    ('free_cores_numa', '<i4', (MAX_NUMA,)), ('free_gpus_numa', '<i4', (MAX_NUMA,)),
])
assert NODE_STATS_DTYPE.itemsize == 64
