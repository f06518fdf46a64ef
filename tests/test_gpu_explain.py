"""nhd_explain on the device (explain_kernel): the reference's per-node reasons through the C-ABI, Solver.explain and
Matcher.Explain.  Also runs on the CPU-emulated device (tests/test_emulated_device.py), where the full-size case
runs on a node prefix."""
import ctypes
import os

import numpy as np
import pytest

import workload
from nhd_b200 import wire
from tests import explain_model, ref_compare, scenarios
from tests.test_explain import _emu_reason, golden_probes, reason_lib  # noqa: F401  (reason_lib: fixture)

pytestmark = pytest.mark.gpu

EMULATED = os.environ.get('NHD_B200_ALLOW_EMULATED') == '1'


def _solver(speed, min_busy=30.0):
    from nhd_b200.solver import Solver
    return Solver(speed, min_busy_secs=min_busy)


def test_golden_probes_through_the_library(oracle_lib):
    solvers = {}
    n = 0
    try:
        for recs, speed, pod, now, mb, codes, first in golden_probes(oracle_lib):
            key = (tuple(np.asarray(speed).tolist()), mb)
            if key not in solvers:
                solvers[key] = _solver(speed, mb)
            s = solvers[key]
            s.load_nodes(recs)
            counts, ff, reasons = s.explain(pod.reshape(1), [now], detail=True)
            assert reasons[0].tolist() == codes, (n, reasons[0].tolist(), codes)
            assert int(ff[0]) == first and counts[0].tolist() == explain_model.counts_of(codes).tolist(), n
            n += 1
    finally:
        for s in solvers.values():
            s.close()
    assert n >= 300


def test_random_scenarios_against_the_oracle_with_detail(oracle_lib):
    """Whole pending sets in one call (several explain types, repeated descriptors, two clocks) on partially filled
    clusters of every flavour."""
    for seed in range(8):
        flavor = ('mixed', 'wild', 'vf', 'big')[seed % 4]
        scn = scenarios.random_scenario(64000 + seed, n_nodes=40 if not EMULATED else 24, n_pods=48, flavor=flavor)
        recs, pods, now, layout = ref_compare.pack_scenario(scn)
        speed = layout.speed_table()
        _, filled = oracle_lib.solve(recs, speed, pods[:24], now[:24])
        q = np.concatenate([pods[24:], pods[24:28]])
        t = np.concatenate([now[24:], now[24:28] + 31.0])
        s = _solver(speed)
        try:
            s.load_nodes(filled)
            counts, ff, reasons = s.explain(q, t, detail=True)
        finally:
            s.close()
        for i in range(len(q)):
            want, wff = explain_model.explain(filled, q[i], speed, float(t[i]))
            assert np.array_equal(reasons[i], want), (seed, i, reasons[i], want)
            assert int(ff[i]) == wff and np.array_equal(counts[i], explain_model.counts_of(want)), (seed, i)
            assert int(counts[i].sum()) == len(filled)


def test_first_fit_is_the_node_a_one_pod_solve_binds(oracle_lib):
    for seed in range(6):
        scn = scenarios.random_scenario(65000 + seed, n_nodes=32, n_pods=40, flavor=('mixed', 'wild')[seed % 2])
        recs, pods, now, layout = ref_compare.pack_scenario(scn)
        pods[3]['map_type'] = wire.MAP_NONE
        s = _solver(layout.speed_table())
        try:
            s.load_nodes(recs)
            s.solve_batch(pods[:20], now[:20])
            for i in range(20, 40):
                _, ff, _ = s.explain(pods[i:i + 1], now[i:i + 1])
                s.snapshot()
                b = s.solve_batch(pods[i:i + 1], now[i:i + 1])[0]
                s.restore()
                assert int(ff[0]) == int(b['node']), (seed, i)
                assert (int(ff[0]) < 0) == (int(b['status']) in (wire.NO_CANDIDATE, wire.BAD_MAP_TYPE))
            _, ff, _ = s.explain(pods[3:4], now[3:4])
            assert int(ff[0]) == -1
        finally:
            s.close()


def test_explain_is_read_only(oracle_lib):
    from nhd_b200 import _lib
    scn = scenarios.random_scenario(66000, n_nodes=48, n_pods=60, flavor='mixed')
    recs, pods, now, layout = ref_compare.pack_scenario(scn)
    s = _solver(layout.speed_table())
    try:
        s.load_nodes(recs)
        s.snapshot()                                         # snapshot = initial records
        s.stage_batch(pods[:30], now[:30])
        feas0, nog0, busy0, pt0 = s.filter_bitmaps()          # filter of the staged batch
        t0 = s.timing()
        rec0 = s.read_nodes()
        s.explain(pods, now, detail=True)
        s.explain(pods[30:], now[30:] + 100.0)
        assert s.read_nodes().tobytes() == rec0.tobytes()
        nt, wpt = ctypes.c_int32(), ctypes.c_int32()
        s._ck(s._L.nhd_read_filter(s._h, ctypes.byref(nt), ctypes.byref(wpt), None, 0, None, 0))
        words = np.zeros((nt.value + 2) * wpt.value, dtype='<u8')
        pt = np.zeros(30, dtype='<i4')
        s._ck(s._L.nhd_read_filter(s._h, ctypes.byref(nt), ctypes.byref(wpt), words.ctypes.data, len(words),
                                   pt.ctypes.data, len(pt)))
        bits = np.unpackbits(words.view(np.uint8), bitorder='little').reshape(nt.value + 2, -1)[:, :len(recs)]
        assert np.array_equal(bits[:nt.value].astype(bool), feas0) and np.array_equal(pt, pt0)
        assert s.timing() == t0
        # a batch staged before the call and solved after it binds as if the call had not happened
        s.restore()
        s.stage_batch(pods[:30], now[:30])
        s.explain(pods[30:], now[30:], detail=True)
        s.solve_staged()
        got = s.fetch_bindings()
        s.restore()
        s.explain(pods, now)
        after_restore = s.read_nodes()
        want = s.solve_batch(pods[:30], now[:30])
        assert got.tobytes() == want.tobytes()
        assert after_restore.tobytes() == recs.tobytes()       # the snapshot survived the calls
        assert t0['n_types'] == s.timing()['n_types']
        assert _lib.load() is s._L
    finally:
        s.close()


def test_error_codes_are_those_of_stage_batch():
    recs, speed, pods, now = workload.make_workload(1)
    s = _solver(speed)
    L = s._L
    counts = np.zeros((len(pods), wire.WHY_COUNT), dtype='<i4')

    def both(p, t):
        p = np.ascontiguousarray(p, dtype=wire.POD_DTYPE)
        t = np.ascontiguousarray(t, dtype='<f8')
        a = L.nhd_explain(s._h, len(p), p.ctypes.data, t.ctypes.data, counts.ctypes.data, None, None)
        b = L.nhd_stage_batch(s._h, len(p), p.ctypes.data, t.ctypes.data)
        return a, b

    try:
        assert both(pods, now) == (wire.ERR_STATE, wire.ERR_STATE)              # before a load
        s.load_nodes(recs)
        assert both(pods, now) == (wire.OK, wire.OK)
        bad = pods.copy()
        bad[1]['n_groups'] = 0
        assert both(bad, now) == (wire.ERR_INVALID, wire.ERR_INVALID)
        t = now.copy()
        t[2] = np.nan
        assert both(pods, t) == (wire.ERR_INVALID, wire.ERR_INVALID)
        big = pods.copy()
        big[0]['n_groups'] = 5
        assert both(big, now) == (wire.ERR_UNSUPPORTED, wire.ERR_UNSUPPORTED)
        # 4-NUMA nodes: a pod of 4 groups would need 4^5 tuples
        grp4 = scenarios.make_pod([scenarios.make_group() for _ in range(4)])
        scn = {'nodes': [scenarios.make_node('q0', sockets=4, phys_cores=32)], 'pods': [grp4] * 3, 'now': [1000.0] * 3}
        four, grp, _, _ = ref_compare.pack_scenario(scn)
        s.load_nodes(four)
        grp[0]['n_groups'] = grp[1]['n_groups'] = 1
        assert both(grp, [1000.0] * 3) == (wire.ERR_UNSUPPORTED, wire.ERR_UNSUPPORTED)
        assert 'pod 2' in L.nhd_last_error(s._h).decode()
    finally:
        s.close()


def test_matcher_explain_agrees_with_find_node():
    import nhd_b200.CfgTopology as cfg_mod
    import nhd_b200.Node as node_mod
    from nhd_b200.Matcher import Matcher
    scn = scenarios.random_scenario(67000, n_nodes=16, n_pods=30, flavor='mixed', min_busy_secs=30.0)
    nodes = scenarios.build_nodes(scn, node_mod)
    m = Matcher()
    agree = found = 0
    for pod, now in zip(scn['pods'], scn['now']):
        top = scenarios.build_top(pod, cfg_mod)
        nl = {n: v for n, v in nodes.items() if set(v.groups) & set(pod['groups']) and v.active}
        name, why = m.Explain(nl, top, now=now)
        assert set(why) == set(nl) and set(why.values()) <= set(wire.WHY_NAMES)
        assert (name is None) == ('FEASIBLE' not in why.values())
        res = m.FindNode(nl, scenarios.build_top(pod, cfg_mod), now=now)
        assert name == res[0]
        agree += 1
        found += name is not None
        if name is not None:                                 # follow the placement, as the scheduler would
            m.FindNodesBatch(nodes, [top], [pod['groups']], now=now)
    assert agree == 30 and found > 0


def test_baseline_config4_against_the_oracle(oracle_lib, reason_lib):
    """BASELINE config 4 (65 536 nodes, 16 pod types) on the state after one solved batch: every node's reason
    against the host build of node_reason (pinned to the explanation oracle), FEASIBLE against the C oracle's
    candidates, first fit against the oracle's one-pod solve.  A node prefix on the emulated device."""
    n_nodes = 1024 if EMULATED else None
    recs, speed, pods, now = workload.make_workload(4, n_nodes=n_nodes, n_pods=256 if EMULATED else None)
    types = workload.make_pod_types(4)
    s = _solver(speed)
    try:
        s.load_nodes(recs)
        s.solve_batch(pods, now)
        state = s.read_nodes()
        t = float(now[-1])
        counts, ff, reasons = s.explain(types, np.full(len(types), t), detail=True)
    finally:
        s.close()
    for i, p in enumerate(types):
        want = _emu_reason(reason_lib, state, speed, p, t, 30.0)
        assert np.array_equal(reasons[i], want), i
        assert np.array_equal(counts[i], explain_model.counts_of(want))
        cand = oracle_lib.candidates(state, speed, p, t).astype(bool)
        busy = (t - state['busy_time']) < 30.0
        if not int(p['groups']['n_gpus'][:int(p['n_groups'])].sum()):
            busy[:] = False                                   # the busy window only concerns GPU pods
        assert np.array_equal(want == wire.WHY_FEASIBLE, cand & ~busy), i
        b, _ = oracle_lib.solve(state, speed, p.reshape(1), [t])
        assert int(ff[i]) == int(b[0]['node']), i
    sample = np.random.default_rng(4).choice(len(state), 64, replace=False)
    for i in range(0, len(types), 4):                         # the Python oracle itself on a node sample
        want, _ = explain_model.explain(state[sample], types[i], speed, t)
        assert np.array_equal(reasons[i][sample], want), i
