"""ctypes loader of the C-ABI library (nhd_b200/libnhd_b200.so, include/nhd_b200.h).

The library is the product: if it is missing or cannot be loaded this module raises —
there is no Python or CPU implementation of the solver to fall back to."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, os.environ.get('NHD_B200_LIB', 'libnhd_b200.so'))

# every symbol include/nhd_b200.h declares
EXPORTS = ('nhd_default_params', 'nhd_nccl_unique_id', 'nhd_shard_min_pairs', 'nhd_create', 'nhd_destroy', 'nhd_last_error',
           'nhd_validate_node', 'nhd_validate_pod', 'nhd_load_nodes', 'nhd_update_nodes', 'nhd_read_nodes',
           'nhd_snapshot', 'nhd_restore', 'nhd_solve_batch', 'nhd_stage_batch', 'nhd_solve_staged',
           'nhd_fetch_bindings', 'nhd_sync', 'nhd_run_filter_only', 'nhd_last_timing', 'nhd_read_filter',
           'nhd_debug_counters', 'nhd_alloc_pinned', 'nhd_free_pinned',
           'nhd_ingest_create', 'nhd_ingest_destroy', 'nhd_ingest_node', 'nhd_ingest_group_mask',
           'nhd_ingest_speed_table', 'nhd_node_stats_from_records', 'nhd_explain')


class Params(ctypes.Structure):
    _fields_ = [('nic_bw_avail_percent', ctypes.c_double), ('min_busy_secs', ctypes.c_double),
                ('enable_sharing', ctypes.c_int32), ('n_speed_classes', ctypes.c_int32),
                ('speed_gbps', ctypes.c_double * 16),
                ('device', ctypes.c_int32), ('rank', ctypes.c_int32), ('world_size', ctypes.c_int32),
                ('reserved_', ctypes.c_int32), ('nccl_unique_id', ctypes.c_uint8 * 128)]


class Timing(ctypes.Structure):
    _fields_ = [('filter_ms', ctypes.c_float), ('exchange_ms', ctypes.c_float), ('sweep_ms', ctypes.c_float),
                ('total_ms', ctypes.c_float), ('n_types', ctypes.c_int32), ('n_launches', ctypes.c_int32)]


_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f'{LIB_PATH} is missing: build it with `python -m nhd_b200.build` '
                           '(nvcc, sm_100a). The B200 solver has no CPU fallback.')
    L = ctypes.CDLL(LIB_PATH)
    if hasattr(L, 'nhd_emulated_device') and os.environ.get('NHD_B200_ALLOW_EMULATED') != '1':
        # tests build the library's sources on a CPU emulation of CUDA to exercise the kernels' logic without a
        # GPU; that build is never a way to *run* the solver
        raise RuntimeError(f'{LIB_PATH} is a CPU-emulated test build, not the CUDA library; refusing to load it '
                           '(set NHD_B200_ALLOW_EMULATED=1 only in tests). The B200 solver has no CPU fallback.')
    vp, i32, i64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64
    sig = {
        'nhd_default_params': (None, [ctypes.POINTER(Params)]),
        'nhd_nccl_unique_id': (i32, [vp]),
        'nhd_shard_min_pairs': (i64, []),
        'nhd_create': (i32, [ctypes.POINTER(Params), ctypes.POINTER(vp)]),
        'nhd_destroy': (i32, [vp]),
        'nhd_last_error': (ctypes.c_char_p, [vp]),
        'nhd_validate_node': (i32, [vp]),
        'nhd_validate_pod': (i32, [vp]),
        'nhd_load_nodes': (i32, [vp, i32, vp]),
        'nhd_update_nodes': (i32, [vp, i32, vp, vp]),
        'nhd_read_nodes': (i32, [vp, i32, i32, vp]),
        'nhd_snapshot': (i32, [vp]),
        'nhd_restore': (i32, [vp]),
        'nhd_solve_batch': (i32, [vp, i32, vp, vp, vp]),
        'nhd_stage_batch': (i32, [vp, i32, vp, vp]),
        'nhd_solve_staged': (i32, [vp]),
        'nhd_fetch_bindings': (i32, [vp, vp]),
        'nhd_sync': (i32, [vp]),
        'nhd_run_filter_only': (i32, [vp]),
        'nhd_last_timing': (i32, [vp, ctypes.POINTER(Timing)]),
        'nhd_read_filter': (i32, [vp, ctypes.POINTER(i32), ctypes.POINTER(i32), vp, i64, vp, i32]),
        'nhd_debug_counters': (i32, [vp, vp]),
        'nhd_alloc_pinned': (i32, [ctypes.c_uint64, ctypes.POINTER(vp)]),
        'nhd_free_pinned': (i32, [vp]),
        'nhd_ingest_create': (i32, [ctypes.POINTER(vp)]),
        'nhd_ingest_destroy': (i32, [vp]),
        'nhd_ingest_node': (i32, [vp, i32, ctypes.POINTER(ctypes.c_char_p), ctypes.POINTER(ctypes.c_char_p), i32, i32, i32, vp, vp]),
        'nhd_ingest_group_mask': (i32, [vp, ctypes.c_char_p, i32, ctypes.POINTER(ctypes.c_uint64)]),
        'nhd_ingest_speed_table': (i32, [vp, vp, ctypes.POINTER(i32)]),
        'nhd_node_stats_from_records': (i32, [i32, vp, vp]),
        'nhd_explain': (i32, [vp, i32, vp, vp, vp, vp, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L
