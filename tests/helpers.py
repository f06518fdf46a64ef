"""Shared test helpers: run a packed scenario through the oracle / the host-emulated core."""
import ctypes
import hashlib
import json
import os

import numpy as np

from nhd_b200 import wire

FROZEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'frozen')


def digest(x):
    """Short fingerprint of bytes, of an array's bytes or of a JSON value (dict key order ignored, as by ==).  The
    frozen reference outcomes (golden/frozen, golden/make_frozen_golden.py) keep large values in this form."""
    if isinstance(x, bytes):
        raw = x
    elif isinstance(x, np.ndarray):
        raw = np.ascontiguousarray(x).tobytes()
    else:
        raw = json.dumps(x, sort_keys=True, separators=(',', ':')).encode()
    return hashlib.sha256(raw).hexdigest()[:16]


def frozen(name):
    """What the unmodified reference computed for a test module's cases (golden/make_frozen_golden.py)."""
    with open(os.path.join(FROZEN, name + '.json')) as f:
        return json.load(f)


def emu_solve(emu, recs, speed_table, pods, now, bw=0.9, min_busy=30.0, two_stage=False):
    recs = np.ascontiguousarray(recs, dtype=wire.NODE_DTYPE).copy()
    pods = np.ascontiguousarray(pods, dtype=wire.POD_DTYPE)
    now = np.ascontiguousarray(now, dtype='<f8')
    speed = np.ascontiguousarray(speed_table, dtype='<f8')
    out = np.zeros(len(pods), dtype=wire.BINDING_DTYPE)
    fn = emu.nhd_emu_solve2 if two_stage else emu.nhd_emu_solve
    fn.argtypes = [ctypes.c_double, ctypes.c_double, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p,
                   ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    rc = fn(bw, min_busy, speed.ctypes.data, len(recs), recs.ctypes.data, len(pods),
                           pods.ctypes.data, now.ctypes.data, out.ctypes.data)
    assert rc == 0, f'emu error {rc}'
    return out, recs


def emu_feasible(emu, recs, speed_table, pod, bw=0.9, k2=False):
    """node_feasible per node; k2=True: the register-only 2-NUMA form (2 = form does not apply to that node / pod)."""
    recs = np.ascontiguousarray(recs, dtype=wire.NODE_DTYPE)
    pod = np.ascontiguousarray(pod, dtype=wire.POD_DTYPE).reshape(1)
    speed = np.ascontiguousarray(speed_table, dtype='<f8')
    out = np.zeros(len(recs), dtype=np.uint8)
    fn = emu.nhd_emu_feasible_k2 if k2 else emu.nhd_emu_feasible
    fn.argtypes = [ctypes.c_double, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    fn(bw, speed.ctypes.data, len(recs), recs.ctypes.data, pod.ctypes.data, out.ctypes.data)
    return out


def binding_bytes_equal(a, b):
    """Bindings compared on every meaningful byte (pad excluded)."""
    names = [n for n in a.dtype.names if n != 'pad_']
    return all(np.array_equal(a[n], b[n]) for n in names)


def first_binding_diff(a, b):
    for i in range(len(a)):
        for n in a.dtype.names:
            if n != 'pad_' and not np.array_equal(a[i][n], b[i][n]):
                return f'pod {i} field {n}: {a[i][n]} != {b[i][n]}'
    return None


class OracleSolver:
    """Stand-in with ``nhd_b200.solver.Solver``'s interface whose batches are computed by the C oracle.
    TEST INFRASTRUCTURE: lets the host-side scheduler logic (``nhd_b200.NHDScheduler``) run in the
    ``-m "not gpu"`` suite, where no CUDA device exists; the GPU tests run the same scenarios through
    the real ``Solver``.  Never used by the product."""

    def __init__(self, speed_table, nic_bw_avail_percent=0.9, min_busy_secs=30.0, device=0):
        from oracle import binding
        self._oracle = binding
        self._speed = np.ascontiguousarray(speed_table, dtype='<f8').copy()
        self._bw, self._min_busy = nic_bw_avail_percent, min_busy_secs
        self._recs = np.zeros(0, dtype=wire.NODE_DTYPE)
        self.closed = False

    def load_nodes(self, recs):
        self._recs = np.ascontiguousarray(recs, dtype=wire.NODE_DTYPE).copy()

    def update_nodes(self, idx, recs):
        for i, r in zip(np.asarray(idx), np.ascontiguousarray(recs, dtype=wire.NODE_DTYPE)):
            self._recs[int(i)] = r

    def read_nodes(self, first=0, n=None):
        return self._recs[first:(None if n is None else first + n)].copy()

    def solve_batch(self, pods, now):
        out, final = self._oracle.solve(self._recs, self._speed, pods, now, self._bw, self._min_busy)
        self._recs = final
        return out

    def snapshot(self):
        self._snap = self._recs.copy()

    def restore(self):
        self._recs = self._snap.copy()

    def close(self):
        self.closed = True
