"""``Solver`` — thin object wrapper over the C-ABI handle (include/nhd_b200.h).

Works on packed numpy records (``nhd_b200.wire``); the object-level drop-in lives in
``nhd_b200.Matcher``.  All compute happens in the CUDA library."""
import ctypes

import os

import numpy as np

from nhd_b200 import _lib, wire

ERR_NAMES = {-1: 'NHD_ERR_INVALID', -2: 'NHD_ERR_UNSUPPORTED', -3: 'NHD_ERR_CUDA', -4: 'NHD_ERR_NCCL',
             -5: 'NHD_ERR_STATE'}


class SolverError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f'{ERR_NAMES.get(code, code)}: {msg}')
        self.code = code


def nccl_unique_id() -> bytes:
    buf = (ctypes.c_uint8 * 128)()
    rc = _lib.load().nhd_nccl_unique_id(buf)
    if rc != 0:
        raise SolverError(rc, 'nhd_nccl_unique_id')
    return bytes(buf)


def shard_min_pairs() -> int:
    """(nodes x distinct pod types) from which a world_size > 1 handle created now would node-shard its filter
    (``nhd_shard_min_pairs``; ``NHD_SHARD_MIN_PAIRS`` in the environment of every rank overrides the default)."""
    return int(_lib.load().nhd_shard_min_pairs())


def pinned_array(n, dtype):
    """numpy array of n records in page-locked host memory (nhd_alloc_pinned): such buffers go to
    and from the device without a staging copy.  Keep the returned array alive while in use."""
    L = _lib.load()
    dtype = np.dtype(dtype)
    nbytes = max(1, n * dtype.itemsize)
    ptr = ctypes.c_void_p()
    rc = L.nhd_alloc_pinned(nbytes, ctypes.byref(ptr))
    if rc != 0:
        raise SolverError(rc, 'nhd_alloc_pinned')
    buf = (ctypes.c_char * nbytes).from_address(ptr.value)
    arr = np.frombuffer(buf, dtype=dtype, count=n)
    _PINNED[id(arr)] = (ptr, buf)
    return arr


_PINNED = {}


class Solver:
    def __init__(self, speed_table, nic_bw_avail_percent=0.9, min_busy_secs=30.0, device=0,
                 rank=0, world_size=1, nccl_id: bytes = None, single_warp: bool = False, cpu_warps: int = 0,
                 sweep_debug: int = 0):
        self._L = _lib.load()
        p = _lib.Params()
        self._L.nhd_default_params(ctypes.byref(p))
        p.nic_bw_avail_percent = nic_bw_avail_percent
        p.min_busy_secs = min_busy_secs
        speeds = [float(x) for x in speed_table]
        nz = max([i + 1 for i, s in enumerate(speeds) if s != 0.0], default=0)
        p.n_speed_classes = nz
        for i, s in enumerate(speeds[:16]):
            p.speed_gbps[i] = s
        p.device, p.rank, p.world_size = device, rank, world_size
        # test knobs (all settings produce identical bindings): single_warp = the general one-warp sweep only;
        # cpu_warps = 1: never sweep the two pod classes side by side; sweep_debug bit 0: no standing decisions,
        # bit 1: same as cpu_warps = 1, bit 2: no direct-path tables in the sweep (warp-wide evaluation everywhere)
        p.reserved_ = (1 if single_warp else (cpu_warps + 1 if cpu_warps else 0)) | \
            ((int(sweep_debug) | int(os.environ.get('NHD_SWEEP_DEBUG', '0'))) << 8)
        if world_size > 1:
            if not nccl_id or len(nccl_id) != 128:
                raise ValueError('world_size > 1 needs the 128-byte NCCL unique id of rank 0')
            ctypes.memmove(p.nccl_unique_id, nccl_id, 128)
        self._h = ctypes.c_void_p()
        rc = self._L.nhd_create(ctypes.byref(p), ctypes.byref(self._h))
        if rc != 0:
            msg = self._L.nhd_last_error(self._h).decode() if self._h else 'no usable CUDA device (no CPU fallback)'
            if self._h:
                self._L.nhd_destroy(self._h)
                self._h = None
            raise SolverError(rc, msg)
        self.n_nodes = 0
        self.n_pods = 0

    def close(self):
        if getattr(self, '_h', None):
            self._L.nhd_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise SolverError(rc, self._L.nhd_last_error(self._h).decode())

    # ---- cluster mirror -------------------------------------------------------------
    def load_nodes(self, recs):
        recs = np.ascontiguousarray(recs, dtype=wire.NODE_DTYPE)
        self._ck(self._L.nhd_load_nodes(self._h, len(recs), recs.ctypes.data))
        self.n_nodes = len(recs)

    def update_nodes(self, idx, recs):
        idx = np.ascontiguousarray(idx, dtype='<i4')
        recs = np.ascontiguousarray(recs, dtype=wire.NODE_DTYPE)
        assert len(idx) == len(recs)
        self._ck(self._L.nhd_update_nodes(self._h, len(idx), idx.ctypes.data, recs.ctypes.data))

    def read_nodes(self, first=0, n=None):
        n = self.n_nodes - first if n is None else n
        out = np.zeros(n, dtype=wire.NODE_DTYPE)
        self._ck(self._L.nhd_read_nodes(self._h, first, n, out.ctypes.data))
        return out

    def snapshot(self):
        self._ck(self._L.nhd_snapshot(self._h))

    def restore(self):
        self._ck(self._L.nhd_restore(self._h))

    # ---- batches --------------------------------------------------------------------
    def solve_batch(self, pods, now, out=None):
        pods = np.ascontiguousarray(pods, dtype=wire.POD_DTYPE)
        now = np.ascontiguousarray(now, dtype='<f8')
        assert len(pods) == len(now)
        if out is None:
            out = np.zeros(len(pods), dtype=wire.BINDING_DTYPE)
        self._ck(self._L.nhd_solve_batch(self._h, len(pods), pods.ctypes.data, now.ctypes.data, out.ctypes.data))
        self.n_pods = len(pods)
        return out

    def stage_batch(self, pods, now):
        pods = np.ascontiguousarray(pods, dtype=wire.POD_DTYPE)
        now = np.ascontiguousarray(now, dtype='<f8')
        assert len(pods) == len(now)
        self._ck(self._L.nhd_stage_batch(self._h, len(pods), pods.ctypes.data, now.ctypes.data))
        self.n_pods = len(pods)

    def solve_staged(self):
        self._ck(self._L.nhd_solve_staged(self._h))

    def sync(self):
        self._ck(self._L.nhd_sync(self._h))

    def fetch_bindings(self, out=None):
        if out is None:
            out = np.zeros(self.n_pods, dtype=wire.BINDING_DTYPE)
        self._ck(self._L.nhd_fetch_bindings(self._h, out.ctypes.data))
        return out

    def timing(self):
        t = _lib.Timing()
        self._ck(self._L.nhd_last_timing(self._h, ctypes.byref(t)))
        return {k: getattr(t, k) for k, _ in t._fields_}

    def debug_counters(self):
        out = np.zeros(64, dtype='<u8')
        self._ck(self._L.nhd_debug_counters(self._h, out.ctypes.data))
        return out

    def explain(self, pods, now, detail=False):
        """Why each node is dropped for each pod, on the current records (``nhd_explain``; changes nothing).
        Returns (counts[pod, WHY_COUNT] nodes per ``wire.WHY_*`` reason, first_fit[pod] the node FindNode would
        pick now or -1, reasons[pod, node] uint8 codes when ``detail`` else None)."""
        pods = np.ascontiguousarray(pods, dtype=wire.POD_DTYPE)
        now = np.ascontiguousarray(np.broadcast_to(np.asarray(now, dtype='<f8'), (len(pods),)))
        counts = np.zeros((len(pods), wire.WHY_COUNT), dtype='<i4')
        first = np.zeros(len(pods), dtype='<i4')
        reasons = np.zeros((len(pods), self.n_nodes), dtype=np.uint8) if detail else None
        self._ck(self._L.nhd_explain(self._h, len(pods), pods.ctypes.data, now.ctypes.data, counts.ctypes.data,
                                     first.ctypes.data, reasons.ctypes.data if detail else None))
        return counts, first, reasons

    def filter_bitmaps(self):
        """Runs only the snapshot predicate kernel on the staged batch; returns
        (feas[type, node] bool, nogpu[node], busy[node], pod_type[pod])."""
        self._ck(self._L.nhd_run_filter_only(self._h))
        nt, wpt = ctypes.c_int32(), ctypes.c_int32()
        self._ck(self._L.nhd_read_filter(self._h, ctypes.byref(nt), ctypes.byref(wpt), None, 0, None, 0))
        words = np.zeros((nt.value + 2) * wpt.value, dtype='<u8')
        pt = np.zeros(self.n_pods, dtype='<i4')
        self._ck(self._L.nhd_read_filter(self._h, ctypes.byref(nt), ctypes.byref(wpt), words.ctypes.data,
                                         len(words), pt.ctypes.data, len(pt)))
        bits = np.unpackbits(words.view(np.uint8), bitorder='little').reshape(nt.value + 2, wpt.value * 64)
        bits = bits[:, :self.n_nodes].astype(bool)
        return bits[:nt.value], bits[nt.value], bits[nt.value + 1], pt
