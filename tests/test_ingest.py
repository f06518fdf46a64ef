"""Node ingest (SURVEY 8f row 3): the library's label parser (`nhd_ingest_node`, csrc/nhd_ingest.cpp) must give
the records `packing.pack_node` makes of a Node that went through the reference's `Node.ParseLabels` +
`SetHugepages` (nhd/Node.py:468-493), byte for byte, and fail where and how the reference fails."""
import json
import os
import random

import numpy as np
import pytest

from nhd_b200 import Node as mirror_node
from nhd_b200 import packing, wire
from nhd_b200.ingest import LabelError, LabelIngest
from tests import helpers, scenarios

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'ingest', 'cases.json')


def _native(ing, case):
    """-> ('ok', rec, aux) | ('false'|'raises'|'unsupported', None, None)"""
    try:
        rec, aux = ing.node(case['labels'], case['active'], case['hp_alloc'], case['hp_free'], name=case['name'])
    except LabelError as e:
        kind = {wire.ERR_LABELS: 'false', wire.ERR_INVALID: 'raises', wire.ERR_UNSUPPORTED: 'unsupported'}[e.code]
        return kind, None, None
    return 'ok', rec, aux


def _object_path(node_mod, case, layout):
    """the same through Node objects (reference's or the mirror's) and pack_node"""
    n = node_mod.Node(case['name'], case['active'])
    try:
        ok = n.ParseLabels(case['labels'])
    except Exception:                                            # noqa: BLE001
        return 'raises', None, None
    if not ok:
        return 'false', None, None
    n.SetHugepages(case['hp_alloc'], case['hp_free'])
    try:
        rec = packing.pack_node(n, layout)
    except packing.UnsupportedError:
        return 'unsupported', None, None
    return 'ok', rec, n


def aux_of(n):
    """What the side outputs of the native ingest must say about a parsed Node object."""
    return {'data_vlan': n.data_vlan, 'res_hugepages_gb': n.mem.res_hugepages_gb,
            'n_reserved_cores': len(n.reserved_cores), 'gpu_device_id': [g.device_id for g in n.gpus],
            'nic_ifname': [x.ifname for x in n.nics]}


def native_aux(case, rec, aux):
    """aux_of for the side outputs of the native ingest of an accepted case."""
    n_gpus, n_nics = int(rec['n_gpus']), int(rec['n_nics'])
    assert (aux['gpu_device_id'][n_gpus:] == -1).all()
    keys = list(case['labels'].keys())
    assert keys[int(aux['gw_label'])] == 'DATA_DEFAULT_GW'
    return {'data_vlan': int(aux['data_vlan']), 'res_hugepages_gb': int(aux['res_hugepages_gb']),
            'n_reserved_cores': int(aux['n_reserved_cores']), 'gpu_device_id': aux['gpu_device_id'][:n_gpus].tolist(),
            'nic_ifname': [keys[i].split('.')[4] for i in aux['nic_label'][:n_nics]]}


def test_golden_cases_from_the_reference():
    """Frozen outcomes of the unmodified reference (tests/golden/make_ingest_golden.py), one cluster dictionary
    across all cases: group bits and speed classes must come out in the same order too."""
    g = json.load(open(GOLDEN))
    ing = LabelIngest()
    seen = {'ok': 0, 'false': 0, 'raises': 0, 'unsupported': 0}
    for case in g['cases']:
        exp = case['expect']
        want = exp['parse'] if exp['parse'] != 'ok' else ('unsupported' if exp['record'] == 'unsupported' else 'ok')
        kind, rec, aux = _native(ing, case)
        assert kind == want, (case['name'], kind, want)
        seen[kind] += 1
        if kind == 'ok':
            assert rec.tobytes().hex() == exp['record'], case['name']
            assert int(aux['data_vlan']) == exp['data_vlan']
            assert int(aux['res_hugepages_gb']) == exp['res_hugepages_gb']
            assert int(aux['n_reserved_cores']) == exp['n_reserved_cores']
            assert aux['gpu_device_id'][:int(rec['n_gpus'])].tolist() == exp['gpu_device_id']
            keys = list(case['labels'].keys())
            assert [keys[i].split('.')[4] for i in aux['nic_label'][:int(rec['n_nics'])]] == exp['nic_ifname']
    assert min(seen.values()) >= 10, seen
    assert ing.speed_table().tolist() == g['speed_table']
    for name, bit in g['group_bits'].items():
        assert ing.group_mask([name]) == 1 << bit
    ing.close()


@pytest.mark.parametrize('flavor', ['mixed', 'wild', 'vf', 'big'])
def test_native_ingest_matches_mirror_objects(flavor):
    ing, layout = LabelIngest(), packing.ClusterLayout()
    n_ok = 0
    for seed in range(12):
        scn = scenarios.random_scenario(33000 + seed * 7 + len(flavor), n_nodes=9, n_pods=1, flavor=flavor)
        for nd in scn['nodes']:
            case = {'name': nd['name'], 'labels': nd['labels'], 'active': nd.get('active', True),
                    'hp_alloc': nd['hp_alloc'], 'hp_free': nd['hp_free']}
            kind, rec, aux = _native(ing, case)
            okind, orec, n = _object_path(mirror_node, case, layout)
            assert kind == okind, (seed, nd['name'])
            if kind == 'ok':
                assert rec.tobytes() == orec.tobytes(), (seed, nd['name'])
                assert native_aux(case, rec, aux) == aux_of(n), (seed, nd['name'])
                n_ok += 1
    assert n_ok > 80
    assert ing.speed_table().tolist() == layout.speed_table().tolist()
    assert all(ing.group_mask([g]) == 1 << b for g, b in layout.group_bits.items())


def test_batch_ingest_feeds_the_record_validator():
    """nodes(): rejected nodes are skipped like BuildInitialNodeList does, the rest pass nhd_validate_node."""
    from nhd_b200 import _lib
    L = _lib.load()
    scn = scenarios.random_scenario(4242, n_nodes=20, n_pods=1, flavor='mixed')
    items = [(nd['labels'], nd.get('active', True), nd['hp_alloc'], nd['hp_free']) for nd in scn['nodes']]
    broken = dict(items[3][0])
    del broken['DATA_PLANE_VLAN']
    items[3] = (broken,) + items[3][1:]
    ing = LabelIngest()
    recs, kept = ing.nodes(items, skip_rejected=True)
    assert kept == [i for i in range(20) if i != 3] and len(recs) == 19
    for i in range(len(recs)):
        assert L.nhd_validate_node(recs[i:i + 1].ctypes.data) == 0
    with pytest.raises(LabelError):
        ing.nodes(items, strict=True)


def test_batch_ingest_brings_a_cluster_up_like_build_initial_node_list():
    """nodes(): the flow of NHDScheduler.BuildInitialNodeList (NHDScheduler.py:83-100) — a node whose labels are
    refused, whose parsing raises, or whose allocatable hugepages are 0 stays in the list, deactivated, and every
    node keeps its index (= the scheduler's preference order)."""
    scn = scenarios.random_scenario(4243, n_nodes=12, n_pods=1, flavor='mixed')
    items = [(nd['labels'], True, max(1, nd['hp_alloc']), nd['hp_free']) for nd in scn['nodes']]
    refused = dict(items[2][0]); del refused['DATA_PLANE_VLAN']                    # ParseLabels returns False
    items[2] = (refused,) + items[2][1:]
    raising = dict(items[5][0]); raising['DATA_PLANE_VLAN'] = 'not-a-number'        # int() raises inside ParseLabels
    items[5] = (raising,) + items[5][1:]
    items[7] = (items[7][0], True, 0, items[7][3])                                   # alloc == 0
    ing = LabelIngest()
    recs, kept = ing.nodes(items)
    assert len(recs) == 12 and kept == [i for i in range(12) if i not in (2, 5, 7)]
    active = (recs['flags'] & wire.NODE_ACTIVE) != 0
    assert active.tolist() == [i not in (2, 5, 7) for i in range(12)]
    # the untouched nodes are byte-identical to one-by-one ingest in the same order of dictionary growth
    ing2 = LabelIngest()
    for i, it in enumerate(items):
        if i in (2, 5):
            with pytest.raises(LabelError):
                ing2.node(*it)
            continue
        r, _ = ing2.node(*it)
        if i == 7:
            r = r.copy(); r['flags'] &= ~np.uint8(wire.NODE_ACTIVE)
        assert recs[i].tobytes() == r.tobytes(), i


def fuzzed_cases():
    from tests.golden import make_ingest_golden as mk
    return mk.mutations(random.Random(5), 400)


def test_fuzzed_labels_against_the_live_reference():
    """Seeded damage to valid label dictionaries: the native parser must do what the unmodified reference did
    (frozen by tests/golden/make_frozen_golden.py) — accept / return False / raise / beyond-limits — and give
    accepted records whose bytes hash as the reference's did, with the same side outputs."""
    frozen = helpers.frozen('ingest')
    ing = LabelIngest()
    kinds = {}
    for case, want in zip(fuzzed_cases(), frozen['fuzzed'], strict=True):
        kind, rec, aux = _native(ing, case)
        assert kind == want[0], (case['name'], kind, want[0], case['labels'])
        kinds[kind] = kinds.get(kind, 0) + 1
        if kind == 'ok':              # digests of the record and of aux_of the reference's Node
            assert helpers.digest(rec.tobytes()) == want[1], case['name']
            assert helpers.digest(native_aux(case, rec, aux)) == want[2], case['name']
    assert kinds.get('ok', 0) > 100 and kinds.get('raises', 0) > 10 and kinds.get('false', 0) > 5, kinds
    assert ing.speed_table().tolist() == frozen['fuzzed_speed_table']


# ---- node statistics off packed records (SURVEY 8f row 4, the part the packed state carries) -------------
def _stats_of_objects(nodes):
    rows = []
    for n in nodes:
        rows.append({'freegpu': n.GetFreeGpuCount(), 'totalgpu': n.GetTotalGPUs(), 'freecpu': n.GetFreeCpuCoreCount(),
                     'totalcpu': n.GetTotalCPUs(), 'freehuge_gb': n.GetFreeHugepages(), 'active': int(bool(n.GetNodeActive())),
                     # the per-NUMA counts are hot-path functions (a8 / a9): the reference has them, the mirror
                     # leaves them to the device
                     'free_cores_numa': list(n.GetFreeCpuCores()) if hasattr(n, 'GetFreeCpuCores') else None,
                     'free_gpus_numa': list(n.GetFreeNumaGPUs()) if hasattr(n, 'GetFreeNumaGPUs') else None,
                     'nics_in_use': sum(1 for x in n.nics if x.pods_used > 0)})
    return rows


def _check_stats(recs, rows):
    from nhd_b200.ingest import node_stats
    st = node_stats(recs)
    assert len(st) == len(rows)
    for s, r, rec in zip(st, rows, recs):
        for k in ('freegpu', 'totalgpu', 'freecpu', 'totalcpu', 'freehuge_gb', 'active', 'nics_in_use'):
            assert int(s[k]) == r[k], (k, int(s[k]), r[k])
        if r['free_cores_numa'] is not None:
            K = len(r['free_cores_numa'])
            assert s['free_cores_numa'][:K].tolist() == r['free_cores_numa'] and (s['free_cores_numa'][K:] == 0).all()
            assert s['free_gpus_numa'][:K].tolist() == r['free_gpus_numa']
        else:
            smt = int(rec['flags']) & wire.NODE_SMT
            assert int(s['free_cores_numa'].sum()) * (2 if smt else 1) == r['freecpu']
            assert int(s['free_gpus_numa'].sum()) == r['freegpu']


@pytest.mark.parametrize('flavor', ['mixed', 'wild', 'vf', 'big'])
def test_node_stats_match_mirror_getters_after_scheduling(oracle_lib, flavor):
    """Schedule a scenario with the oracle, write the bindings into the mirror objects, then the counters of the
    packed final records must be what the objects' getters report."""
    from nhd_b200 import CfgTopology as mirror_cfg
    from tests import ref_compare
    for seed in range(6):
        scn = scenarios.random_scenario(44000 + seed * 5 + len(flavor), n_nodes=8, n_pods=30, flavor=flavor)
        recs, pods, now, layout = ref_compare.pack_scenario(scn)
        bindings, final = oracle_lib.solve(recs, layout.speed_table(), pods, now)
        nodes = scenarios.build_nodes(scn, mirror_node)
        order = list(nodes.values())
        for pod, b, t in zip(scn['pods'], bindings, now):
            if int(b['node']) < 0:
                continue
            node = order[int(b['node'])]
            node.busy_time = float(t)
            if int(b['status']) == wire.PLACED:
                top = scenarios.build_top(pod, mirror_cfg)
                packing.apply_binding(node, top, b)
                node.ClaimPodNICResources([int(x) for x in b['claimed_nics'][:int(b['n_claimed'])]])
        assert packing.pack_nodes(order, layout).tobytes() == final.tobytes()
        _check_stats(final, _stats_of_objects(order))


def stats_scenarios():
    for seed, flavor in enumerate(['mixed', 'wild', 'vf', 'big', 'mixed', 'big']):
        yield seed, scenarios.random_scenario(45000 + seed, n_nodes=8, n_pods=30, flavor=flavor)


def test_node_stats_match_reference_getters_after_scheduling(oracle_lib):
    """Same against the unmodified reference: its own scheduler loop left Node objects behind whose getters
    (what GetBasicNodeStats calls, nhd/NHDScheduler.py:355-378) must agree with the packed records' counters.
    The records and the getters' answers are frozen (tests/golden/make_frozen_golden.py); the oracle must reach
    the same records from the scenario."""
    from tests import ref_compare
    frozen = helpers.frozen('ingest')['stats']
    for (seed, scn), want in zip(stats_scenarios(), frozen, strict=True):
        recs = np.frombuffer(bytes.fromhex(want['records']), dtype=wire.NODE_DTYPE)
        start, pods, now, layout = ref_compare.pack_scenario(scn)
        _, final = oracle_lib.solve(start, layout.speed_table(), pods, now)
        assert final.tobytes() == recs.tobytes(), seed
        _check_stats(recs, want['rows'])


@pytest.mark.parametrize('config,wild', [(4, False), (5, False), (4, True)])
def test_bench_clusters_are_what_the_ingest_makes_of_nfd_labels(config, wild):
    """SURVEY 8d: the synthetic clusters of workload.py (bench.py, the full-size parity tests) are packed records
    written with numpy for speed; every one of them is exactly what the native label ingest produces from the NFD
    label dictionary of that node (tests/pyref.node_def_from_record writes the labels), plus the occupancy the
    record carries (cores / GPUs / NICs in use, hugepages) — i.e. a state the reference reaches from those labels."""
    import workload
    from tests import pyref
    recs, speed = workload.make_cluster(config, n_nodes=600, wild=wild)
    ing = LabelIngest()
    for s in speed:                                   # same speed classes in the same order as the workload's table
        if s:
            pass
    got = np.zeros(len(recs), dtype=wire.NODE_DTYPE)
    for i, r in enumerate(recs):
        nd = pyref.node_def_from_record(i, r, speed, group_names=[f'g{b}' for b in range(64)] if config == 5 else None)
        rec, _ = ing.node(nd['labels'], nd['active'], nd['hp_alloc'], nd['hp_free'], name=nd['name'])
        got[i] = rec
    # static description: everything but the occupancy words
    for f in ('n_numa', 'phys_cores', 'n_gpus', 'n_nics', 'gpu_numa_mask', 'nic_numa_mask'):
        assert np.array_equal(got[f], recs[f]), f

    def switch_classes(r):
        # switch ids are node-local aliases (only equality is ever tested, Matcher.py:316-320, Node.py:651): compare the
        # partition of the GPUs and NICs into switches, numbered by first use
        ids = [(int(r['gpu_sw']) >> (4 * g)) & 0xF for g in range(int(r['n_gpus']))] + \
              [(int(r['nic_sw'][j >> 4]) >> (4 * (j & 15))) & 0xF for j in range(int(r['n_nics']))]
        first = {}
        return [first.setdefault(x, len(first)) for x in ids]
    for i in range(len(recs)):
        assert switch_classes(got[i]) == switch_classes(recs[i]), i
    assert np.array_equal(got['flags'] & (wire.NODE_SMT | wire.NODE_ACTIVE), recs['flags'] & (wire.NODE_SMT | wire.NODE_ACTIVE))
    # speed classes: the ingest numbers them in order of first appearance, the workload by its table
    tbl = ing.speed_table()
    for i in range(len(recs)):
        for j in range(int(recs[i]['n_nics'])):
            a = (int(got[i]['nic_speed'][j >> 4]) >> (4 * (j & 15))) & 0xF
            b = (int(recs[i]['nic_speed'][j >> 4]) >> (4 * (j & 15))) & 0xF
            assert tbl[a] == speed[b], (i, j)
    # occupancy only ever adds to what the labels give: reserved cores stay reserved, free hugepages as given
    assert np.array_equal(got['used'] & recs['used'], got['used'])
    assert np.array_equal(got['free_hugepages_gb'], recs['free_hugepages_gb'])
    assert (got['gpu_used'] == 0).all() and (got['nic_inuse'] == 0).all()
