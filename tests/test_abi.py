"""CPU-only checks of the drop-in boundary: the C-ABI library loads, exports every function the
header declares, agrees with the numpy wire dtypes on struct sizes, validates records on the host,
and refuses to run without a GPU instead of falling back to a CPU path."""
import ctypes
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

import workload
from nhd_b200 import _lib, wire

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, 'include', 'nhd_b200.h')


@pytest.fixture(scope='module')
def lib():
    from nhd_b200 import build
    build.build()
    return _lib.load()


def test_every_declared_symbol_is_exported(lib):
    text = open(HEADER).read()
    declared = set(re.findall(r'^\s*(?:int32_t|int64_t|void|const char\*)\s+(nhd_\w+)\s*\(', text, flags=re.M))
    assert len(declared) >= 18
    assert declared == set(_lib.EXPORTS)
    for name in declared:
        assert hasattr(lib, name), name


def test_struct_sizes_match_header():
    src = '#include <stdio.h>\n#include "nhd_b200.h"\nint main(){printf("%zu %zu %zu %zu %zu %zu\\n",' \
          'sizeof(nhd_node_rec),sizeof(nhd_pod_group),sizeof(nhd_pod),sizeof(nhd_binding),sizeof(nhd_params),' \
          'sizeof(nhd_timing));return 0;}\n'
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, 't.c')
        open(c, 'w').write(src)
        exe = os.path.join(d, 't')
        subprocess.run(['gcc', '-I', os.path.join(ROOT, 'include'), '-o', exe, c], check=True)
        sizes = [int(x) for x in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()]
    assert sizes[:4] == [wire.NODE_DTYPE.itemsize, wire.POD_GROUP_DTYPE.itemsize, wire.POD_DTYPE.itemsize,
                         wire.BINDING_DTYPE.itemsize] == [128, 32, 144, 128]
    assert sizes[4] == ctypes.sizeof(_lib.Params) and sizes[5] == ctypes.sizeof(_lib.Timing)


def test_host_validation(lib):
    recs, _, pods, _ = workload.make_workload(3, n_nodes=64, n_pods=32)
    for i in range(len(recs)):
        assert lib.nhd_validate_node(recs[i:i + 1].ctypes.data) == 0
    for i in range(len(pods)):
        assert lib.nhd_validate_pod(pods[i:i + 1].ctypes.data) == 0
    bad = recs[:1].copy()
    bad['n_numa'] = 5
    assert lib.nhd_validate_node(bad.ctypes.data) == -2          # NHD_ERR_UNSUPPORTED
    bad = recs[:1].copy()
    bad['phys_cores'] = 33                                       # not divisible by sockets
    assert lib.nhd_validate_node(bad.ctypes.data) == -2
    bad = recs[:1].copy()
    bad['gpu_used'] = 0xFFFF
    bad['n_gpus'] = 0
    bad['gpu_numa_mask'] = 0
    assert lib.nhd_validate_node(bad.ctypes.data) == -1          # NHD_ERR_INVALID
    badp = pods[:1].copy()
    badp['n_groups'] = 0                                         # crashes the reference (Matcher.py:346)
    assert lib.nhd_validate_pod(badp.ctypes.data) == -1
    badp = pods[:1].copy()
    badp['n_groups'] = 5
    assert lib.nhd_validate_pod(badp.ctypes.data) == -2
    badp = pods[:1].copy()
    badp['groups'][0][0]['rx_gbps'] = -1.0
    assert lib.nhd_validate_pod(badp.ctypes.data) == -1


def test_no_cpu_fallback(lib):
    """Without a CUDA device nhd_create fails loudly (NHD_ERR_CUDA); with one it succeeds."""
    p = _lib.Params()
    lib.nhd_default_params(ctypes.byref(p))
    assert p.nic_bw_avail_percent == 0.9 and p.min_busy_secs == 30.0 and p.world_size == 1
    h = ctypes.c_void_p()
    rc = lib.nhd_create(ctypes.byref(p), ctypes.byref(h))
    assert rc in (0, -3)
    if rc == 0:
        lib.nhd_destroy(h)
    else:
        assert not h
        from nhd_b200.solver import Solver, SolverError
        with pytest.raises(SolverError):
            Solver([100.0])
    p.enable_sharing = 1                                         # only the shipped default (Node.py:20) is supported
    assert lib.nhd_create(ctypes.byref(p), ctypes.byref(h)) == -2


def test_product_does_not_import_oracle():
    """The oracle is test infrastructure: nothing under nhd_b200/ may import, include or link it."""
    pkg = os.path.join(ROOT, 'nhd_b200')
    pat = re.compile(r'(import\s+oracle|from\s+oracle|#include\s+"[^"]*oracle|libnhd_oracle|oracle/|'
                     r'^\s*import\s+tests\b|^\s*from\s+tests\b|cuda_emu)', re.M)
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.h', '.cpp')):
                text = open(os.path.join(dirpath, f)).read()
                assert not pat.search(text), os.path.join(dirpath, f)


def test_emulated_test_build_is_refused_by_the_loader():
    """A CPU-emulated build of the library (tests/emu) must never stand in for the CUDA library by accident."""
    import subprocess
    import sys
    sys.path.insert(0, os.path.join(ROOT, 'tests', 'emu'))
    try:
        import build_emu_cuda
    finally:
        sys.path.pop(0)
    emu = build_emu_cuda.build()
    code = ('from nhd_b200 import _lib\n'
            'try:\n    _lib.load(); print("LOADED")\n'
            'except RuntimeError as e:\n    print("REFUSED" if "CPU-emulated" in str(e) else "OTHER")\n')
    env = dict(os.environ, NHD_B200_LIB=emu)
    env.pop('NHD_B200_ALLOW_EMULATED', None)
    out = subprocess.run([sys.executable, '-c', code], cwd=ROOT, env=env, capture_output=True, text=True).stdout
    assert out.strip() == 'REFUSED'


def test_shard_threshold_default_and_environment(lib, monkeypatch):
    """nhd_shard_min_pairs: 2^21 unless NHD_SHARD_MIN_PAIRS holds a non-negative integer (anything else is ignored)."""
    monkeypatch.delenv('NHD_SHARD_MIN_PAIRS', raising=False)
    assert lib.nhd_shard_min_pairs() == 1 << 21
    for text, want in (('1', 1), ('0', 0), ('123456789012', 123456789012), ('abc', 1 << 21), ('-5', 1 << 21), ('', 1 << 21),
                       ('12x', 1 << 21)):
        monkeypatch.setenv('NHD_SHARD_MIN_PAIRS', text)
        assert lib.nhd_shard_min_pairs() == want, text
