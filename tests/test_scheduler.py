"""SURVEY 8f row 1 — the scheduler loop around the hot path (``nhd_b200.NHDScheduler``): the pending
set goes to the solver as one batch, and everything Kubernetes, ``pod_state`` and the ``Node``
objects end up with must be what the UNMODIFIED reference ``nhd.NHDScheduler.run()`` leaves behind
when it schedules the same pods one ``AttemptScheduling`` at a time.

* random scripted sessions — pods appearing, Kubernetes writes failing at every step the reference
  unwinds from, delete / create events, cordon, maintenance, group changes, restarts, RPCs — against
  fingerprints of the reference's end states (``tests/golden/frozen/scheduler.json``, made by
  ``tests/golden/make_frozen_golden.py``);
* frozen: ``tests/golden/sched/*.json`` (made by ``tests/golden/make_sched_golden.py`` from the
  reference), replayed here on CPU and, ``-m gpu``, through the CUDA solver on the B200 box.

On CPU the solver behind ``DeviceCluster`` is ``tests.helpers.OracleSolver`` (the C oracle behind the
``Solver`` interface, test infrastructure): these tests pin the *host* logic — batching, cutting a
batch after an unwind, delta uploads; the placement arithmetic is pinned elsewhere.
"""
import glob
import json
import os

import pytest

from tests import helpers, sched_harness as H

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), 'golden', 'sched', '*.json')))
IDS = [os.path.basename(p)[:-5] for p in GOLDEN]


def _load(path):
    with open(path) as f:
        return json.load(f)


def test_golden_present():
    assert len(GOLDEN) >= 16


@pytest.mark.parametrize('path', GOLDEN, ids=IDS)
def test_scheduler_reproduces_reference_sessions(oracle_lib, path):
    doc = _load(path)
    stats = {}
    got = H.run_mirror(doc['script'], solver_factory=helpers.OracleSolver, stats=stats)
    want = H.drop_speed_residue(doc['expected'], stats['assign_failed_nodes'])
    got = H.drop_speed_residue(got, stats['assign_failed_nodes'])
    assert H.first_difference(want, got) is None
    assert got == want
    assert stats['batches'] > 0 and stats['pods'] >= stats['batches']
    if 'assign_failures' in path:                        # failed assignments rewind the device inside the batch
        assert stats['rewinds'] > 0 and stats['assign_failed_nodes']


@pytest.mark.gpu
@pytest.mark.parametrize('path', GOLDEN, ids=IDS)
def test_scheduler_cuda_reproduces_reference_sessions(path):
    """The same sessions with the CUDA solver behind the scheduler (the product configuration)."""
    doc = _load(path)
    stats = {}
    got = H.run_mirror(doc['script'], stats=stats)
    want = H.drop_speed_residue(doc['expected'], stats['assign_failed_nodes'])
    got = H.drop_speed_residue(got, stats['assign_failed_nodes'])
    assert H.first_difference(want, got) is None
    assert got == want


def flavor_scripts(flavor):
    for seed in range(100, 112):
        yield seed, H.random_script(seed, flavor, codec='triad' if seed % 2 else 'json')


@pytest.mark.parametrize('flavor', ['mixed', 'vf', 'big', 'wild'])
def test_scheduler_matches_live_reference(oracle_lib, flavor):
    """Scripted sessions against the fingerprints (``sched_harness.fingerprint``) of the state documents the
    reference's ``run()`` ended in, frozen by ``tests/golden/make_frozen_golden.py``."""
    frozen = helpers.frozen('scheduler')[flavor]
    checked = binds = 0
    for (seed, script), want in zip(flavor_scripts(flavor), frozen, strict=True):
        stats = {}
        got = H.run_mirror(script, solver_factory=helpers.OracleSolver, stats=stats)
        names = stats['assign_failed_nodes']
        want = dict(want, residue={n: d for n, d in want['residue'].items() if n not in names})
        assert H.first_difference(want, H.fingerprint(got, names)) is None, (seed, flavor)
        checked += 1
        binds += len(got['k8s']['binds'])
    assert checked == 12 and binds > 100


def test_thread_function_equals_direct_driving(oracle_lib):
    """``NHDScheduler.run()`` (queue polling, idle counting, start-up flush) fed by the fake queues that drive
    the reference's ``run()`` ends where driving the handlers directly ends."""
    for seed, flavor, codec in ((3, 'mixed', 'json'), (4, 'wild', 'triad'), (5, 'vf', 'json')):
        script = H.random_script(seed, flavor, codec=codec)
        a = H.run_mirror(script, solver_factory=helpers.OracleSolver)
        b = H.run_mirror_loop(script, solver_factory=helpers.OracleSolver)
        assert H.first_difference(a, b) is None, (seed, flavor)


def test_pending_set_is_one_batch_and_unwinds_cut_it(oracle_lib):
    """No failing write: the whole pending set is ONE solver call.  A write that fails before the
    config annotation exists makes ``ReleasePodResources`` reset the cluster (``NHDScheduler.py:178-181``);
    the batch is cut there and the rest solved again — and only then."""
    from tests.golden.make_sched_golden import unwind_script
    script = unwind_script()
    clean = json.loads(json.dumps(script))
    for st in clean['init']:
        st['fail'] = []
    clean['steps'] = []
    stats = {}
    doc = H.run_mirror(clean, solver_factory=helpers.OracleSolver, stats=stats)
    assert stats['batches'] == 1 and stats['pods'] == len(clean['init']) and stats['full_loads'] == 1
    assert len(doc['k8s']['binds']) > 8

    script['steps'] = []
    stats = {}
    H.run_mirror(script, solver_factory=helpers.OracleSolver, stats=stats)
    # cuts: nad, gpumap, annotate (each resets); bind leaks and podobj / cfg never reach the solver
    assert stats['batches'] == 4, stats
    assert stats['pods'] > 12


def test_delta_uploads_only_touch_changed_nodes(oracle_lib):
    """Between batches only the nodes the host changed are re-sent (``nhd_update_nodes``)."""
    from nhd_b200.NHDScheduler import NHDScheduler
    import nhd_b200.CfgTopology as cfg_mod
    from tests import fake_k8s, scenarios
    nodes = [scenarios.make_node(f'n{i}', 2, 16, True, 1, nics=[('eth0', 100000, 0, 0x10), ('eth1', 100000, 1, 0x20)])
             for i in range(12)]
    k8s = fake_k8s.FakeK8s(nodes)
    clock = H.Clock(1000.0)
    s = NHDScheduler(k8s, lambda t, c: fake_k8s.JsonCfgParser(c, cfg_mod), solver_factory=helpers.OracleSolver,
                     clock=clock)
    pod = scenarios.make_pod([scenarios.make_group(pairs=((10, 10),), workers=1)], misc=1, hugepages=1)
    for i in range(5):
        k8s.add_pod('a', f'p{i}', pod, uid=f'u{i}')
    s.Startup()
    assert (s.cluster.full_loads, s.cluster.delta_nodes, s.cluster.batches) == (1, 0, 1)
    assert len(k8s.binds) == 5
    s.HandleWatchItem({'type': 'NHD_WATCH_TYPE_NODE_CORDON', 'node': 'n0'})
    s.HandleWatchItem({'type': 'NHD_WATCH_TYPE_NODE_CORDON', 'node': 'n0'})           # no change, no upload
    s.HandleWatchItem({'type': 'NHD_WATCH_TYPE_TRIAD_POD_DELETE', 'pod': {'ns': 'a', 'name': 'p1', 'uid': 'u1'}})
    k8s.add_pod('a', 'late', pod, uid='u9')
    s.CheckPendingPods()
    assert s.cluster.full_loads == 1 and s.cluster.batches == 2
    assert 1 <= s.cluster.delta_nodes <= 2          # n0 (cordon) and the node p1 ran on (may be n0)
    # the device copy equals the objects
    from nhd_b200 import packing
    want = packing.pack_nodes(list(s.nodes.values()), s.cluster.layout)
    assert s.cluster.read_records().tobytes() == want.tobytes()
    row = {r['name']: r for r in s.GetBasicNodeStats()}
    assert row['n0']['active'] is False
    s.close()


def test_scheduler_has_no_cpu_placement_path():
    """Without a CUDA device the default solver factory must raise, not fall back."""
    from nhd_b200 import _lib
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip('a GPU is present')
    except ImportError:
        pass
    from nhd_b200.NHDScheduler import NHDScheduler
    from nhd_b200.solver import SolverError
    import nhd_b200.CfgTopology as cfg_mod
    from tests import fake_k8s, scenarios
    _lib.load()
    k8s = fake_k8s.FakeK8s([scenarios.make_node('n0', nics=[('eth0', 100000, 0, 0x10), ('eth1', 100000, 1, 0x20)])])
    k8s.add_pod('a', 'p', scenarios.make_pod([scenarios.make_group()]))
    s = NHDScheduler(k8s, lambda t, c: fake_k8s.JsonCfgParser(c, cfg_mod))
    with pytest.raises(SolverError):
        s.Startup()


def test_requests_and_nodes_beyond_the_packed_limits_fail_loudly_not_fatally(oracle_lib):
    """A pod asking for more than the packed layout can describe gets a FailedScheduling event and is listed; an
    active node beyond the limits is kept out of placement and listed; everything else is scheduled as usual."""
    from nhd_b200.NHDScheduler import NHDScheduler
    import nhd_b200.CfgTopology as cfg_mod
    from tests import fake_k8s, scenarios
    nics = [('eth0', 100000, 0, 0x10), ('eth1', 100000, 1, 0x20)]
    nodes = [scenarios.make_node('huge', 2, 192, True, 2, nics=nics),          # 384 logical cores > NHD_MAX_LCORES
             scenarios.make_node('n1', 2, 32, True, 2, nics=nics), scenarios.make_node('n2', 2, 32, True, 2, nics=nics)]
    k8s = fake_k8s.FakeK8s(nodes)
    ok_pod = scenarios.make_pod([scenarios.make_group(pairs=((10, 10),), workers=2)], misc=1)
    k8s.add_pod('a', 'fits', ok_pod, uid='u1')
    k8s.add_pod('a', 'monster', scenarios.make_pod([scenarios.make_group(workers=80)]), uid='u2')   # > 72 cores per pod
    k8s.add_pod('a', 'fits2', ok_pod, uid='u3')
    s = NHDScheduler(k8s, lambda t, c: fake_k8s.JsonCfgParser(c, cfg_mod), solver_factory=helpers.OracleSolver,
                     clock=H.Clock(1000.0))
    s.Startup()
    assert [b[1] for b in k8s.binds] == ['fits', 'fits2'] and all(b[2] in ('n1', 'n2') for b in k8s.binds)
    assert 'huge' in s.cluster.unsupported_nodes and s.nodes['huge'].active
    assert [p[1] for p in s.unsupported_pods] == ['monster'] and s.failed_schedule_count == 1
    assert k8s.events[('a', 'monster')][-1][0] == 'FailedScheduling'
    assert s.pod_state[('a', 'monster')]['state'].name == 'POD_STATUS_FAILED'
    assert s.cluster.batches == 1
    s.close()


@pytest.mark.gpu
def test_cluster_dependent_limit_fails_one_pod_not_the_batch():
    """4 processing groups on a cluster with a 4-NUMA node exceed the solver's tuple enumeration (4^5 > 256,
    include/nhd_b200.h): the library refuses the batch naming the pod; the scheduler fails that pod and schedules
    the others."""
    from nhd_b200.NHDScheduler import NHDScheduler
    import nhd_b200.CfgTopology as cfg_mod
    from tests import fake_k8s, scenarios
    nics4 = [(f'eth{k}', 100000, k, 0x10 * (k + 1)) for k in range(4)]
    nodes = [scenarios.make_node('quad', 4, 64, True, 1, nics=nics4),
             scenarios.make_node('n1', 2, 32, True, 2, nics=nics4[:2]), scenarios.make_node('n2', 2, 32, True, 2, nics=nics4[:2])]
    k8s = fake_k8s.FakeK8s(nodes)
    small = scenarios.make_pod([scenarios.make_group(pairs=((10, 10),), workers=1)], misc=1)
    four = scenarios.make_pod([scenarios.make_group(pairs=((5, 5),), workers=1) for _ in range(4)], misc=1)
    for i, pod in enumerate([small, four, small, four, small]):
        k8s.add_pod('a', f'p{i}', pod, uid=f'u{i}')
    s = NHDScheduler(k8s, lambda t, c: fake_k8s.JsonCfgParser(c, cfg_mod), clock=H.Clock(1000.0))
    try:
        s.Startup()
        assert [b[1] for b in k8s.binds] == ['p0', 'p2', 'p4']
        assert [p[1] for p in s.unsupported_pods] == ['p1', 'p3'] and s.failed_schedule_count == 2
        assert 'tuple' in s.unsupported_pods[0][2]
    finally:
        s.close()
