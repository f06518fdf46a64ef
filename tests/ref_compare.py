"""Helpers that run one scenario through (a) the unmodified reference, (b) the C oracle,
(c) the CUDA solver, and compare the outcomes field by field.  Test infrastructure."""
import contextlib
import copy
import io

import numpy as np

from nhd_b200 import packing, wire
from tests import helpers, scenarios

_REF_STATUS = {'none': (wire.NO_CANDIDATE, wire.BAD_MAP_TYPE), 'placed': (wire.PLACED,),
               'assign_failed': (wire.ASSIGN_FAILED, wire.REF_WOULD_CRASH), 'crash': (wire.REF_WOULD_CRASH,)}


def run_reference(scn):
    """Schedules scn['pods'] one by one with the UNMODIFIED reference (build container only).
    Returns (outcomes, initial_records, final_records, layout, node_names)."""
    from oracle import ref_loader
    ref = ref_loader.load()
    ref.node.Node.MIN_BUSY_SECS = float(scn.get('min_busy_secs', 30.0))
    nodes = scenarios.build_nodes(scn, ref.node)
    names = list(nodes.keys())
    layout = packing.ClusterLayout()
    initial = packing.pack_nodes([nodes[n] for n in names], layout)
    matcher = ref.matcher.Matcher()
    outcomes = []
    for pod, now in zip(scn['pods'], scn['now']):
        top = scenarios.build_top(pod, ref.cfg)
        with contextlib.redirect_stdout(io.StringIO()):     # stray print at Matcher.py:329
            r = ref_loader.attempt_scheduling(ref, matcher, nodes, top, pod['groups'], now)
        o = {'status': r['status']}
        if r['status'] != 'none':
            node = nodes[r['node']]
            o['node'] = names.index(r['node'])
            m = r['mapping']
            o['mapping'] = {'gpu': list(m['gpu']), 'cpu': list(m['cpu']), 'nic': [list(x) for x in m['nic']]}
        if r['status'] == 'placed':
            res = scenarios.extract_result(top)
            o.update(res)
            o['nidx'] = list(r['nidx'])
            o['gpu_index'] = [next(i for i, g in enumerate(node.gpus) if g.device_id == d) for d in res['gpus']]
        outcomes.append(o)
    final = packing.pack_nodes([nodes[n] for n in names], layout)
    ref.node.Node.MIN_BUSY_SECS = 30.0
    run_reference.last_final_state = {n: scenarios.node_state(nodes[n]) for n in names}
    return outcomes, initial, final, layout, names


def pack_scenario(scn, node_mod=None, cfg_mod=None):
    """Scenario -> (records, pods, now, layout) using this repo's mirror classes by default."""
    if node_mod is None:
        import nhd_b200.Node as node_mod
    if cfg_mod is None:
        import nhd_b200.CfgTopology as cfg_mod
    nodes = scenarios.build_nodes(scn, node_mod)
    layout = packing.ClusterLayout()
    recs = packing.pack_nodes(list(nodes.values()), layout)
    pods = np.zeros(len(scn['pods']), dtype=wire.POD_DTYPE)
    for i, pod in enumerate(scn['pods']):
        top = scenarios.build_top(pod, cfg_mod)
        packing.pack_pod(top, pod['groups'], layout, out=pods[i])
    now = np.asarray(scn['now'], dtype='<f8')
    return recs, pods, now, layout


def binding_dict(b):
    """nhd_binding record -> plain dict of the meaningful fields."""
    G = int(b['n_groups'])
    d = {'status': int(b['status']), 'node': int(b['node'])}
    if d['node'] >= 0:
        d['mapping'] = {'gpu': [int(x) for x in b['gpu_numa'][:G]],
                        'cpu': [int(x) for x in b['cpu_numa'][:G + 1]],
                        'nic': [[int(b['nic_numa'][g]), int(b['nic_idx'][g])] for g in range(G)]}
    if d['status'] == wire.PLACED:
        d['cores'] = [int(x) for x in b['cores'][:int(b['n_cores'])]]
        d['gpu_index'] = [int(x) for x in b['gpu_index'][:int(b['n_gpus'])]]
        d['nidx'] = [int(x) for x in b['claimed_nics'][:int(b['n_claimed'])]]
        d['nic_list_index'] = [int(x) for x in b['nic_list_index'][:G]]
    return d


def diff_outcome(ref_o, b):
    """Returns a list of mismatch descriptions between a reference outcome and a binding."""
    bd = binding_dict(b)
    errs = []
    if bd['status'] not in _REF_STATUS[ref_o['status']]:
        errs.append(f"status ref={ref_o['status']} got={wire.STATUS_NAMES.get(bd['status'])}")
        return errs
    if ref_o['status'] == 'none':
        return errs
    if ref_o['node'] != bd['node']:
        errs.append(f"node ref={ref_o['node']} got={bd['node']}")
    if ref_o['mapping'] != bd.get('mapping'):
        errs.append(f"mapping ref={ref_o['mapping']} got={bd.get('mapping')}")
    if ref_o['status'] == 'placed':
        for k in ('cores', 'gpu_index', 'nidx'):
            if ref_o[k] != bd[k]:
                errs.append(f"{k} ref={ref_o[k]} got={bd[k]}")
    return errs


def compared_fields(status, d):
    """The fields diff_outcome compares for a reference outcome of this status, taken from d (a reference
    outcome or a binding_dict)."""
    if status == 'none':
        return None
    keys = ('node', 'mapping') + (('cores', 'gpu_index', 'nidx') if status == 'placed' else ())
    return {k: d.get(k) for k in keys}


def freeze_outcomes(outs):
    """A stream of reference outcomes as [one letter per pod for its status (n)one / (p)laced / (a)ssign_failed /
    (c)rash, digest of the fields diff_outcome compares, pod after pod]."""
    return [''.join(o['status'][0] for o in outs),
            helpers.digest([compared_fields(o['status'], o) for o in outs])]


def diff_frozen_outcomes(frozen, bindings):
    """diff_outcome over a stream kept by freeze_outcomes."""
    letters, want = frozen
    status_of = {s[0]: s for s in _REF_STATUS}
    if len(letters) != len(bindings):
        return [f'{len(bindings)} bindings for {len(letters)} reference outcomes']
    errs, got = [], []
    for i, (c, b) in enumerate(zip(letters, bindings)):
        bd = binding_dict(b)
        if bd['status'] not in _REF_STATUS[status_of[c]]:
            errs.append(f"pod {i}: status ref={status_of[c]} got={wire.STATUS_NAMES.get(bd['status'])}")
        got.append(compared_fields(status_of[c], bd))
    if not errs and helpers.digest(got) != want:
        errs.append(f'nodes / mappings / cores / GPUs / NICs are not what the reference chose: {got}')
    return errs


def records_equal(a, b):
    return a.tobytes() == b.tobytes()


def diff_records(a, b):
    out = []
    for i in range(len(a)):
        if a[i].tobytes() != b[i].tobytes():
            for name in a.dtype.names:
                if np.any(a[i][name] != b[i][name]):
                    out.append(f'node {i} field {name}: {a[i][name]} != {b[i][name]}')
    return out
