"""CPU-only: the explanation of unschedulable pods (nhd_explain, Matcher.Explain, NHDScheduler(explain_failures=True)).

The explanation oracle (tests/explain_model.py) is pinned to the unmodified reference's own log records
(golden/explain/cases.json, every probe and every node); the product's node_reason (nhd_core.cuh compiled with g++)
is pinned to that oracle; the scheduler's summaries are checked on scripted sessions with the C oracle behind the
Solver interface."""
import ctypes
import json
import os
import re

import numpy as np
import pytest

from nhd_b200 import packing, wire
from tests import explain_model, fake_k8s, helpers, ref_compare, scenarios, sched_harness
from tests.conftest import has_reference

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, 'tests', 'golden', 'explain', 'cases.json')


def _pack_probe(pod, layout):
    import nhd_b200.CfgTopology as cfg_mod
    out = np.zeros(1, dtype=wire.POD_DTYPE)
    packing.pack_pod(scenarios.build_top(pod, cfg_mod), pod['groups'], layout, out=out[0])
    return out[0]


def _state_at(oracle_lib, scn, pos):
    """Packed records of scn's nodes after its first pos pods (the C oracle replays them)."""
    recs, pods, now, layout = ref_compare.pack_scenario(scn)
    mb = float(scn.get('min_busy_secs', 30.0))
    if pos:
        _, recs = oracle_lib.solve(recs, layout.speed_table(), pods[:pos], now[:pos], min_busy_secs=mb)
    return recs, layout


def golden_probes(oracle_lib):
    """(records, speed table, packed pod, now, min_busy, codes, first) of every frozen probe."""
    with open(GOLDEN) as f:
        doc = json.load(f)
    for st in doc['streams']:
        scn = st['scenario']
        states = {}
        for pr in st['probes']:
            if pr['pos'] not in states:
                states[pr['pos']] = _state_at(oracle_lib, scn, pr['pos'])
            recs, layout = states[pr['pos']]
            pod = _pack_probe(pr['pod'], layout)
            yield (recs, layout.speed_table(), pod, float(pr['now']), float(scn.get('min_busy_secs', 30.0)),
                   pr['codes'], pr['first'])


def test_oracle_explains_every_golden_probe_as_the_reference_logged_it(oracle_lib):
    n, seen = 0, set()
    for recs, speed, pod, now, mb, codes, first in golden_probes(oracle_lib):
        got, ff = explain_model.explain(recs, pod, speed, now, min_busy_secs=mb)
        assert got.tolist() == codes, (n, got.tolist(), codes)
        assert ff == first, (n, ff, first)
        seen.update(codes)
        n += 1
    assert n >= 300 and seen == set(range(wire.WHY_COUNT))


@pytest.fixture(scope='session')
def reason_lib(tmp_path_factory):
    """g++ build of node_reason (tests/emu/nhd_emu_reason.cpp on nhd_core.cuh), in a temporary directory."""
    import subprocess
    so = str(tmp_path_factory.mktemp('emu_reason') / '_emu_reason.so')
    subprocess.run(['g++', '-O2', '-std=c++17', '-x', 'c++', '-fPIC', '-shared', '-ffp-contract=off', '-o', so,
                    os.path.join(ROOT, 'tests', 'emu', 'nhd_emu_reason.cpp')], check=True)
    L = ctypes.CDLL(so)
    L.nhd_emu_reason.argtypes = [ctypes.c_double, ctypes.c_double, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p,
                                 ctypes.c_void_p, ctypes.c_double, ctypes.c_void_p]
    return L


def _emu_reason(lib, recs, speed, pod, now, min_busy):
    recs = np.ascontiguousarray(recs, dtype=wire.NODE_DTYPE)
    pod = np.ascontiguousarray(pod, dtype=wire.POD_DTYPE).reshape(1)
    sp = np.ascontiguousarray(speed, dtype='<f8')
    out = np.zeros(len(recs), dtype=np.uint8)
    assert lib.nhd_emu_reason(0.9, min_busy, sp.ctypes.data, len(recs), recs.ctypes.data, pod.ctypes.data, now,
                              out.ctypes.data) == 0
    return out


def test_core_node_reason_matches_the_oracle(oracle_lib, reason_lib):
    """node_reason (what explain_kernel evaluates per thread) == the oracle, node by node, on partially filled
    clusters of every flavour, NUMA and PCI pods, busy windows open and closed; and on the golden probes."""
    pairs, codes_seen, maps = 0, set(), set()
    for seed in range(48):
        flavor = ('mixed', 'wild', 'vf', 'big')[seed % 4]
        scn = scenarios.random_scenario(61000 + seed, n_nodes=12, n_pods=32, flavor=flavor)
        recs, pods, now, layout = ref_compare.pack_scenario(scn)
        speed = layout.speed_table()
        _, filled = oracle_lib.solve(recs, speed, pods[:16], now[:16])
        for i in range(16, 32):
            for t in (float(now[i]), float(now[i]) + 25.0):
                want, _ = explain_model.explain(filled, pods[i], speed, t)
                got = _emu_reason(reason_lib, filled, speed, pods[i], t, 30.0)
                assert np.array_equal(got, want), (seed, i, got, want)
                pairs += len(filled)
                codes_seen.update(want.tolist())
                maps.add(int(pods[i]['map_type']))
    for recs, speed, pod, now, mb, codes, _ in golden_probes(oracle_lib):
        assert _emu_reason(reason_lib, recs, speed, pod, now, mb).tolist() == codes
        pairs += len(recs)
    assert pairs >= 2000 and maps == {wire.MAP_NUMA, wire.MAP_PCI}
    assert {wire.WHY_GPU, wire.WHY_CPU, wire.WHY_NIC, wire.WHY_BUSY, wire.WHY_NUMA} <= codes_seen


@pytest.mark.reference
@pytest.mark.skipif(not has_reference(), reason='needs the unmodified reference')
def test_oracle_against_the_live_reference(oracle_lib):
    """Fresh seeds (not frozen) through the generator's own probe on the reference's objects."""
    import contextlib
    import io
    import sys
    sys.path.insert(0, os.path.join(ROOT, 'tests', 'golden'))
    try:
        import make_explain_golden as G
    finally:
        sys.path.pop(0)
    from oracle import ref_loader
    ref = ref_loader.load()
    matcher = ref.matcher.Matcher()
    n = 0
    for seed, flavor in enumerate(('mixed', 'wild', 'vf', 'big')):
        scn = scenarios.random_scenario(73000 + seed, 8, 16, flavor)
        ref.node.Node.MIN_BUSY_SECS = float(scn['min_busy_secs'])
        try:
            nodes = scenarios.build_nodes(scn, ref.node)
            for i, (pod, now) in enumerate(zip(scn['pods'], scn['now'])):
                if i % 4 == 0:
                    codes, first = G.probe(ref, matcher, nodes, pod, now)
                    recs, layout = _state_at(oracle_lib, scn, i)
                    got, ff = explain_model.explain(recs, _pack_probe(pod, layout), layout.speed_table(), now,
                                                    min_busy_secs=scn['min_busy_secs'])
                    assert got.tolist() == codes and ff == first, (seed, i, got.tolist(), codes, ff, first)
                    n += 1
                ref.clock.t = float(now)
                with contextlib.redirect_stdout(io.StringIO()):
                    ref_loader.attempt_scheduling(ref, matcher, nodes, scenarios.build_top(pod, ref.cfg), pod['groups'], now)
        finally:
            ref.node.Node.MIN_BUSY_SECS = 30.0
    assert n >= 12


def test_why_codes_match_the_header():
    with open(os.path.join(ROOT, 'include', 'nhd_b200.h')) as f:
        text = f.read()
    defs = {m.group(1): int(m.group(2)) for m in re.finditer(r'#define NHD_WHY_(\w+)\s+(\d+)', text)}
    assert defs.pop('COUNT') == wire.WHY_COUNT == len(wire.WHY_NAMES) == len(wire.WHY_TEXT)
    assert defs == {name: i for i, name in enumerate(wire.WHY_NAMES)}
    assert all(getattr(wire, 'WHY_' + name) == i for i, name in enumerate(wire.WHY_NAMES))


def test_unschedulable_message():
    from nhd_b200.NHDScheduler import OUTSIDE_LIMITS, unschedulable_message
    assert unschedulable_message({'CPU': 12, 'NOT_IN_GROUP': 3}, 15) == \
        "0/15 nodes are available: 3 not in the pod's node groups, 12 too few free CPU cores."
    assert unschedulable_message({'GPU': 2, OUTSIDE_LIMITS: 1, 'BUSY': 4}, 7) == \
        "0/7 nodes are available: 4 busy after a recent GPU deployment, 2 too few free GPUs per NUMA node, " \
        "1 outside the solver's limits."
    msg = unschedulable_message({'FEASIBLE': 2, 'BUSY': 1}, 3)
    assert msg.startswith('2/3 nodes are available now (busy windows expired since the attempt): ') and \
        msg.endswith('1 busy after a recent GPU deployment.')
    assert unschedulable_message({}, 0) == '0/0 nodes are available.'


class ExplainingOracleSolver(helpers.OracleSolver):
    """The C oracle behind the Solver interface, with the explanation oracle as ``explain``."""

    def explain(self, pods, now, detail=False):
        pods = np.ascontiguousarray(pods, dtype=wire.POD_DTYPE)
        now = np.broadcast_to(np.asarray(now, dtype='<f8'), (len(pods),))
        counts = np.zeros((len(pods), wire.WHY_COUNT), dtype=np.int32)
        first = np.zeros(len(pods), dtype=np.int32)
        reasons = np.zeros((len(pods), len(self._recs)), dtype=np.uint8)
        for i, p in enumerate(pods):
            reasons[i], first[i] = explain_model.explain(self._recs, p, self._speed, float(now[i]), self._bw, self._min_busy)
            counts[i] = explain_model.counts_of(reasons[i])
        return counts, first, (reasons if detail else None)


def _session(script, explain, checks=None):
    """sched_harness.run_mirror with explain_failures; ``checks`` collects (counts the scheduler emitted, counts the
    oracle gives for the host's node objects packed afresh after the pass)."""
    import nhd_b200.CfgTopology as cfg_mod
    import nhd_b200.Node as node_mod
    from nhd_b200.NHDScheduler import NHDScheduler
    node_mod.Node.MIN_BUSY_SECS = float(script['min_busy_secs'])
    clock = sched_harness.Clock(script['clock0'])
    k8s = fake_k8s.FakeK8s(script['nodes'], codec=script.get('codec', 'json'))
    sink = sched_harness.RpcSink()
    for st in script['init']:
        sched_harness.apply_k8s_op(k8s, clock, st)

    def parser(cfgtype, cfgstr):
        return fake_k8s.JsonCfgParser(cfgstr, cfg_mod)

    def make():
        s = NHDScheduler(k8s, parser, solver_factory=ExplainingOracleSolver, clock=clock, explain_failures=explain)
        if checks is not None:
            orig = s._explain_unplaced

            def wrapped(entries, s=s, orig=orig):
                orig(entries)
                recs = packing.pack_nodes([s.nodes[n] for n in s.nodes], s.cluster.layout)
                for e in entries:
                    pod = np.array(e.rec, dtype=wire.POD_DTYPE)
                    pod['group_mask'] = s.cluster.layout.groups_mask(e.groups, create=False)
                    codes, _ = explain_model.explain(recs, pod, s.cluster.layout.speed_table(), clock(),
                                                     min_busy_secs=node_mod.Node.MIN_BUSY_SECS)
                    want = {wire.WHY_NAMES[w]: int(c) for w, c in enumerate(explain_model.counts_of(codes)) if c}
                    checks.append((dict(s.failure_reasons[(e.key[0], e.key[1])]), want))
            s._explain_unplaced = wrapped
        s.Startup()
        return s

    s = None
    try:
        s = make()
        for st in script['steps']:
            op = st['op']
            if op in sched_harness.K8S_OPS:
                sched_harness.apply_k8s_op(k8s, clock, st)
            elif op == 'watch':
                s.HandleWatchItem({k: v for k, v in st.items() if k != 'op'})
            elif op == 'rpc':
                s.ParseRPCReq(st['msg'], sink)
            elif op == 'idle':
                s.CheckPendingPods()
            elif op == 'restart':
                s.close()
                s = make()
        doc = sched_harness.state_document(s, k8s, sink)
        return doc, {k: list(v) for k, v in k8s.events.items()}, dict(s.failure_reasons), s
    finally:
        node_mod.Node.MIN_BUSY_SECS = 30.0
        if s is not None:
            s.close()


def test_scheduler_explains_unschedulable_pods_without_changing_anything_else(oracle_lib):
    explained = 0
    for seed in range(10):
        script = sched_harness.random_script(88000 + seed, flavor=('mixed', 'wild')[seed % 2], n_nodes=6, n_steps=30)
        doc0, ev0, fr0, _ = _session(script, False)
        checks = []
        doc1, ev1, fr1, s1 = _session(script, True, checks)
        assert fr0 == {}
        unsched = {k: [e for e in v if e[0] == 'Unschedulable'] for k, v in ev1.items()}
        stripped = {k: [e for e in v if e[0] != 'Unschedulable'] for k, v in ev1.items()}
        assert stripped == ev0, seed
        doc1['k8s']['events'] = {k: [e for e in v if e[0] != 'Unschedulable'] for k, v in doc1['k8s']['events'].items()}
        assert json.dumps(doc1, sort_keys=True, default=str) == json.dumps(doc0, sort_keys=True, default=str), seed
        for got, want in checks:
            assert got == want, (seed, got, want)
        for (ns, pod), reasons in fr1.items():
            assert unsched.get((ns, pod)), (ns, pod)
            assert sum(reasons.values()) == len(s1.nodes)
            assert s1.pod_state.get((ns, pod), {}).get('state') != 'scheduled'
        for evs in unsched.values():
            for e in evs:
                assert e[1] == 'EVENT_TYPE_WARNING' and re.match(r'^\d+/\d+ nodes are available', e[2]), e
        explained += len(checks)
    assert explained >= 10
