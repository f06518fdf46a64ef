"""Generates tests/golden/explain/cases.json from the UNMODIFIED reference (build container only).

    python tests/golden/make_explain_golden.py

The reference tells an operator why a pod is pending only through its INFO log: Matcher.FindNode logs, node by node,
the stage that drops the node (nhd/Matcher.py:74,79,109,133,215,271,353), after InitialNodeFilter left out the nodes
outside the pod's node groups or inactive (nhd/NHDScheduler.py:241-245).  This script replays seeded scenario
streams of every flavour through the reference's own loop (as make_golden.py does) and, at several points, probes
the next pod and a few fixed pods with FindNode while a handler captures the Matcher logger's records.  Each record
names one node and one stage; that stage is the node's reason code (wire.WHY_*).  A node dropped at the
intersection is PCIE when the same probe with the NUMA map type keeps it, NUMA otherwise (FindNode changes no
node: the second probe sees the same state).

Stored per probe: the scenario (once per stream), the probe position (pods already scheduled), the pod, its clock,
the per-node codes and the node FindNode returned.  tests/test_explain.py compares the explanation oracle
(tests/explain_model.py) with every probe and every node, without the reference.
"""
import contextlib
import io
import json
import logging
import os
import re
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

import numpy as np                                   # noqa: E402

from nhd_b200 import wire                            # noqa: E402
from tests import scenarios as S                     # noqa: E402

OUT = os.path.join(HERE, 'explain', 'cases.json')

# Matcher log messages -> reason code (the node name is the first group)
_PATTERNS = [
    (re.compile(r'^Node (\S+) in maintenance\. Removing node'), wire.WHY_MAINTENANCE),                  # :74
    (re.compile(r'^Node (\S+) only has .* Removing node'), wire.WHY_HUGEPAGES),                         # :79
    (re.compile(r'^Dropping node (\S+) from candidate list beacause last deploy'), wire.WHY_BUSY),     # :109
    (re.compile(r'^Dropping node (\S+) from candidate list since not enough free GPUs'), wire.WHY_GPU),   # :133
    (re.compile(r'^Dropping node (\S+) from candidate list since not enough free CPU cores'), wire.WHY_CPU),   # :215
    (re.compile(r'^Dropping node (\S+) from candidate list since not enough free NIC'), wire.WHY_NIC),  # :271
    (re.compile(r'^Node (\S+) has no valid intersection candidates'), wire.WHY_NUMA),                   # :353
]


class _Capture(logging.Handler):
    def __init__(self):
        super().__init__(logging.DEBUG)
        self.msgs = []

    def emit(self, record):
        self.msgs.append(record.getMessage())


def _find_node_logged(matcher, nl, top):
    """FindNode(nl, top) with the Matcher logger's records captured (ref_loader disables logging: re-enabled
    around the call).  Returns (result, messages)."""
    cap = _Capture()
    lg = matcher.logger
    old_level, old_handlers = lg.level, lg.handlers
    lg.handlers = [cap]                               # (the reference's own handler writes to the terminal)
    lg.setLevel(logging.INFO)
    logging.disable(logging.NOTSET)
    try:
        with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
            res = matcher.FindNode(nl, top)
    finally:
        logging.disable(logging.CRITICAL)
        lg.handlers = old_handlers
        lg.setLevel(old_level)
    return res, cap.msgs


def _stage_codes(msgs, names):
    codes, map_type_error = {}, False
    for m in msgs:
        if m.startswith('Invalid mapping type'):                                                         # :46
            map_type_error = True
        for pat, code in _PATTERNS:
            x = pat.match(m)
            if x and x.group(1) in names:
                assert x.group(1) not in codes, (m, codes)
                codes[x.group(1)] = code
    return codes, map_type_error


def probe(ref, matcher, nodes, pod, now):
    """Per-node reason codes (node order) and the FindNode result index for one pod on the current objects."""
    ref.clock.t = float(now)
    names = list(nodes)
    codes = {}
    nl = {}
    for n, v in nodes.items():                        # InitialNodeFilter, NHDScheduler.py:239-245
        if len(set(v.groups) & set(pod['groups'])) == 0:
            codes[n] = wire.WHY_NOT_IN_GROUP
        elif not v.active:
            codes[n] = wire.WHY_INACTIVE
        else:
            nl[n] = v
    top = S.build_top(pod, ref.cfg)
    res, msgs = _find_node_logged(matcher, nl, top)
    staged, map_type_error = _stage_codes(msgs, set(nl))
    if pod['map_type'] == 'PCI' and any(c == wire.WHY_NUMA for c in staged.values()):
        numa_pod = dict(pod, map_type='NUMA')
        nl2 = dict(nl)                                # FindNode changes no node (it only edits its own filts)
        _, msgs2 = _find_node_logged(matcher, nl2, S.build_top(numa_pod, ref.cfg))
        staged2, _ = _stage_codes(msgs2, set(nl2))
        for n, c in staged.items():
            if c == wire.WHY_NUMA and n not in staged2:
                staged[n] = wire.WHY_PCIE
    for n in nl:
        if n in staged:
            codes[n] = staged[n]
        elif map_type_error:
            codes[n] = wire.WHY_MAP_TYPE
        else:
            codes[n] = wire.WHY_FEASIBLE
    first = names.index(res[0]) if res[0] is not None else -1
    return [int(codes[n]) for n in names], first


FIXED_PODS = [
    S.make_pod([S.make_group([(10, 10)], 2)], misc=1),                                   # small CPU pod
    S.make_pod([S.make_group([(10, 10)], 1, [1], 1)], misc=1),                           # one GPU
    S.make_pod([S.make_group([(20, 10)], 2, [1]), S.make_group([(20, 10)], 1, [1])], misc=2, map_type='PCI'),
    S.make_pod([S.make_group([(10, 10)], 1)], misc=1, map_type='NONE'),                  # neither NUMA nor PCI
    S.make_pod([S.make_group([(10, 10)], 4, [], 2)], misc=1, hugepages=12, groups=('g1',)),
]


def hand_built():
    """Shapes random streams rarely produce: NUMA (GPUs free only on NUMA 0, cores only on NUMA 1), PCIE (the
    only NIC with bandwidth sits on a switch without a free GPU) and an inactive node in the pod's group."""
    out = []
    gpus = [(0, 0, 0x10), (1, 0, 0x10)]
    nics = [('eth0', 100000, 0, 0x10), ('eth1', 100000, 1, 0x20)]
    # NUMA 0 has no isolated cores left (reserved_per_socket = whole socket), NUMA 1 has all of them
    numa_node = S.make_node('numa0', 2, 16, False, 0, gpus, nics, isolcpus='8-15', hp_alloc=64)
    ok_node = S.make_node('ok0', 2, 16, False, 1, gpus + [(2, 1, 0x20)], nics, hp_alloc=64)
    pci_node = S.make_node('pci0', 2, 16, False, 1, [(0, 0, 0x10), (1, 1, 0x30)],
                           [('eth0', 100000, 0, 0x20), ('eth1', 100000, 1, 0x30)], hp_alloc=64)
    pods = [S.make_pod([S.make_group([(10, 10)], 2, [1])], misc=0),
            S.make_pod([S.make_group([(10, 10)], 2, [1])], misc=0, map_type='PCI'),
            S.make_pod([S.make_group([(10, 10)], 1, [1])], misc=0, map_type='PCI'),
            S.make_pod([S.make_group([(50, 10)], 1, [1]), S.make_group([(50, 10)], 1, [1])], misc=0, map_type='PCI')]
    off_node = S.make_node('off0', 2, 16, False, 1, gpus, nics, hp_alloc=64, active=False)
    out.append({'nodes': [numa_node, ok_node, pci_node, off_node], 'pods': pods, 'now': [1000.0] * len(pods),
                'min_busy_secs': 0.0})
    return out


def main():
    from oracle import ref_loader
    ref = ref_loader.load()
    matcher = ref.matcher.Matcher()
    streams = []
    seeds = [('mixed', 8, 30), ('wild', 8, 30), ('vf', 6, 24), ('big', 6, 30), ('mixed', 12, 40), ('wild', 10, 36),
             ('vf', 8, 30), ('big', 8, 30)]
    for i, (flavor, n_nodes, n_pods) in enumerate(seeds):
        streams.append(S.random_scenario(52000 + i, n_nodes, n_pods, flavor, max_groups=3))
    streams += hand_built()
    doc = {'generator': 'tests/golden/make_explain_golden.py',
           'reference': 'Viasat/nhd v0.3.39, CPython ' + sys.version.split()[0], 'streams': []}
    seen = set()
    n_probes = 0
    for si, scn in enumerate(streams):
        ref.node.Node.MIN_BUSY_SECS = float(scn.get('min_busy_secs', 30.0))
        nodes = S.build_nodes(scn, ref.node)
        probes = []
        every = max(1, len(scn['pods']) // 6)
        for i, (pod, now) in enumerate(zip(scn['pods'], scn['now'])):
            if i % every == 0 or i == len(scn['pods']) - 1:
                for p, t in [(pod, now)] + [(fp, now) for fp in FIXED_PODS] + [(FIXED_PODS[1], now + 40.0)]:
                    codes, first = probe(ref, matcher, nodes, p, t)
                    probes.append({'pos': i, 'pod': p, 'now': t, 'codes': codes, 'first': first})
                    seen.update(codes)
            ref.clock.t = float(now)
            top = S.build_top(pod, ref.cfg)
            with contextlib.redirect_stdout(io.StringIO()):
                ref_loader.attempt_scheduling(ref, matcher, nodes, top, pod['groups'], now)
        ref.node.Node.MIN_BUSY_SECS = 30.0
        n_probes += len(probes)
        doc['streams'].append({'scenario': scn, 'probes': probes})
    missing = [wire.WHY_NAMES[c] for c in range(wire.WHY_COUNT) if c not in seen]
    assert not missing, f'reason codes never produced: {missing}'
    assert n_probes >= 300, n_probes
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    with open(OUT, 'w') as f:
        json.dump(doc, f, separators=(',', ':'))
    hist = np.bincount([c for s in doc['streams'] for p in s['probes'] for c in p['codes']], minlength=wire.WHY_COUNT)
    print(f'{len(streams)} streams, {n_probes} probes; per code: ' +
          ', '.join(f'{wire.WHY_NAMES[c]} {int(hist[c])}' for c in range(wire.WHY_COUNT)))


if __name__ == '__main__':
    main()
