"""Scripted scheduler sessions (SURVEY 8f row 1).  TEST INFRASTRUCTURE.

A *script* is plain JSON-able data: a cluster (``tests.scenarios`` nodes), the Kubernetes
operations that happen around the scheduler (pods appearing, phases changing, writes that will
fail), the controller's watch-queue items, gRPC requests, idle periods, clock steps and
scheduler restarts.  ``run_reference`` plays it to the UNMODIFIED ``nhd.NHDScheduler.run()``
(build container only; the thread function is called directly and fed through fake queues),
``run_mirror`` plays it to ``nhd_b200.NHDScheduler``; both return the same state document
(what Kubernetes saw, ``pod_state``, every node's resources, RPC answers) for comparison.
"""
import json
from queue import Empty

import numpy as np

from tests import fake_k8s, scenarios

K8S_OPS = ('add_pod', 'delete_pod', 'set_phase', 'clock')
FAIL_STEPS = ('podobj', 'cfg', 'nad', 'gpumap', 'annotate', 'bind')


# ----------------------------------------------------------------------------------------------
# script generation
# ----------------------------------------------------------------------------------------------
def random_script(seed, flavor='mixed', n_nodes=10, n_steps=28, fail_rate=0.15, codec='json'):
    rng = np.random.default_rng(seed)
    nodes = [scenarios.random_node(rng, f'n{i}', flavor) for i in range(n_nodes)]
    if rng.random() < 0.4:                                # a node whose labels ParseLabels refuses
        bad = scenarios.random_node(rng, 'nbad', flavor)
        del bad['labels']['DATA_PLANE_VLAN']
        nodes.insert(int(rng.integers(0, len(nodes) + 1)), bad)
    if rng.random() < 0.3:                                # alloc == 0 deactivates the node (NHDScheduler.py:94)
        nodes[int(rng.integers(0, len(nodes)))]['hp_alloc'] = 0
    counter = [0]
    known = []

    def new_pod():
        counter[0] += 1
        ns = 'solo' if counter[0] == 3 else ('ns' + str(int(rng.integers(0, 2))))
        name = 'solo' if counter[0] == 3 else f'pod{counter[0]}'
        fail = [str(rng.choice(FAIL_STEPS))] if rng.random() < fail_rate else []
        known.append((ns, name))
        return {'op': 'add_pod', 'ns': ns, 'name': name, 'uid': f'u{counter[0]}', 'fail': fail,
                'pod': scenarios.random_pod(rng, flavor, max_groups=2 if counter[0] % 3 else 3)}

    init = [new_pod() for _ in range(int(rng.integers(3, 10)))]
    steps = []
    for _ in range(n_steps):
        r = rng.random()
        if r < 0.30:
            steps += [new_pod() for _ in range(int(rng.integers(1, 7)))]
            steps.append({'op': 'idle'})
        elif r < 0.48:
            p = new_pod()
            steps.append(p)
            steps.append({'op': 'watch', 'type': 'NHD_WATCH_TYPE_TRIAD_POD_CREATE',
                          'pod': {'ns': p['ns'], 'name': p['name'], 'uid': p['uid']}})
        elif r < 0.54 and known:                          # a create event for a pod we already know
            ns, name = known[int(rng.integers(0, len(known)))]
            uid = 'u' + name[3:] if (name.startswith('pod') and rng.random() < 0.5) else 'uX'
            steps.append({'op': 'watch', 'type': 'NHD_WATCH_TYPE_TRIAD_POD_CREATE',
                          'pod': {'ns': ns, 'name': name, 'uid': uid}})
        elif r < 0.66 and known:
            ns, name = known[int(rng.integers(0, len(known)))]
            if rng.random() < 0.3:                        # the API object is gone before the event arrives
                steps.append({'op': 'delete_pod', 'ns': ns, 'name': name})
            steps.append({'op': 'watch', 'type': 'NHD_WATCH_TYPE_TRIAD_POD_DELETE',
                          'pod': {'ns': ns, 'name': name, 'uid': 'whatever'}})
            if rng.random() < 0.7:
                steps.append({'op': 'delete_pod', 'ns': ns, 'name': name})
        elif r < 0.76:
            t = str(rng.choice(['NHD_WATCH_TYPE_NODE_CORDON', 'NHD_WATCH_TYPE_NODE_UNCORDON',
                                'NHD_WATCH_TYPE_NODE_MAINT_START', 'NHD_WATCH_TYPE_NODE_MAINT_END']))
            steps.append({'op': 'watch', 'type': t, 'node': nodes[int(rng.integers(0, len(nodes)))]['name']})
        elif r < 0.80:
            k = int(rng.integers(1, 3))
            groups = '.'.join(scenarios.GROUP_NAMES[i] for i in rng.choice(4, size=k, replace=False))
            steps.append({'op': 'watch', 'type': 'NHD_WATCH_TYPE_GROUP_UPDATE', 'groups': groups,
                          'node': nodes[int(rng.integers(0, len(nodes)))]['name']})
        elif r < 0.90:
            steps.append({'op': 'clock', 'dt': float(rng.choice([1.0, 5.0, 31.0, 100.0]))})
        elif r < 0.94:
            steps.append({'op': 'rpc', 'msg': str(rng.choice(['TYPE_NODE_INFO', 'TYPE_SCHEDULER_INFO',
                                                              'TYPE_POD_INFO']))})
        elif r < 0.97 and known:
            ns, name = known[int(rng.integers(0, len(known)))]
            steps.append({'op': 'set_phase', 'ns': ns, 'name': name,
                          'phase': str(rng.choice(['Running', 'Failed', 'Succeeded']))})
        else:
            steps.append({'op': 'restart'})
    steps += [{'op': 'idle'}, {'op': 'rpc', 'msg': 'TYPE_NODE_INFO'}, {'op': 'rpc', 'msg': 'TYPE_POD_INFO'},
              {'op': 'rpc', 'msg': 'TYPE_SCHEDULER_INFO'}]
    return {'nodes': nodes, 'min_busy_secs': float(rng.choice([30.0, 30.0, 0.0])), 'clock0': 1000.0,
            'init': init, 'steps': steps, 'codec': codec}


# ----------------------------------------------------------------------------------------------
# shared pieces
# ----------------------------------------------------------------------------------------------
class Clock:
    def __init__(self, t):
        self.t = float(t)

    def __call__(self):
        return self.t


def apply_k8s_op(k8s, clock, st):
    op = st['op']
    if op == 'add_pod':
        k8s.add_pod(st['ns'], st['name'], st['pod'], uid=st['uid'], fail=st['fail'])
    elif op == 'delete_pod':
        k8s.delete_pod(st['ns'], st['name'])
    elif op == 'set_phase':
        if (st['ns'], st['name']) in k8s.pods:
            k8s.pods[(st['ns'], st['name'])]['phase'] = st['phase']
    elif op == 'clock':
        clock.t += st['dt']


class RpcSink:
    def __init__(self):
        self.answers = []

    def put(self, rsp):
        self.answers.append(json.loads(json.dumps(rsp)))


def state_document(sched, k8s, sink):
    nodes = {}
    for name, n in sched.nodes.items():
        st = scenarios.node_state(n)
        st.update({'active': bool(n.active), 'maintenance': bool(n.maintenance), 'groups': list(n.groups),
                   'pods': sorted(f'{ns}/{pod}' for (pod, ns) in n.pod_info)})
        nodes[name] = st
    return json.loads(json.dumps({
        'k8s': k8s.transcript(),
        'pod_state': {f'{ns}/{name}': [v['state'].name, v['uid']] for (ns, name), v in sched.pod_state.items()},
        'failed_schedule_count': sched.failed_schedule_count,
        'nodes': nodes,
        'rpc': sink.answers}))


# ----------------------------------------------------------------------------------------------
# the unmodified reference
# ----------------------------------------------------------------------------------------------
class _Stop(Exception):
    pass


class _StopItem(dict):
    def __getitem__(self, key):
        raise _Stop()


class _RefFeed:
    """Plays the part of ``qinst`` (watch queue) and of the gRPC queue for ``NHDScheduler.run``."""

    def __init__(self, ref, k8s, steps, sink, watch_enum=None, rpc_enum=None, clock=None):
        self.ref, self.k8s, self.steps, self.sink = ref, k8s, steps, sink
        self.watch_enum = watch_enum if watch_enum is not None else ref.sched.NHDWatchTypes
        self.rpc_enum = rpc_enum if rpc_enum is not None else ref.sched.RpcMsgType
        self.clock = clock if clock is not None else ref.clock
        self.i = 0
        self.checked = False
        self.armed = False
        self.rpcq = self._Rpc(self)

    def get(self, *args, **kw):                           # watch queue
        if 'timeout' in kw:                               # start-up flush (NHDScheduler.py:459-465)
            raise Empty()
        while True:
            if self.i >= len(self.steps):
                return _StopItem()
            st = self.steps[self.i]
            if st['op'] in K8S_OPS:
                apply_k8s_op(self.k8s, self.clock, st)
                self.i += 1
            elif st['op'] == 'restart':
                self.i += 1
                return _StopItem()
            elif st['op'] == 'watch':
                self.i += 1
                item = {k: v for k, v in st.items() if k != 'op'}
                item['type'] = self.watch_enum[st['type']]
                return item
            else:
                raise Empty()                             # rpc / idle: served by the other queue

    class _Rpc:
        def __init__(self, feed):
            self.f = feed

        def get(self, block, timeout):
            f = self.f
            st = f.steps[f.i]
            if st['op'] == 'rpc':
                f.i += 1
                return (f.rpc_enum[st['msg']], f.sink)
            assert st['op'] == 'idle'
            if not f.armed:
                f.armed, f.checked = True, False
            elif f.checked:                               # run() reached IDLE_CNT_THRESH and re-scanned (:483-486)
                f.armed = False
                f.i += 1
            raise Empty()


def run_reference(script):
    from oracle import ref_sched_loader
    ref = ref_sched_loader.load()
    ref.node.Node.MIN_BUSY_SECS = float(script['min_busy_secs'])
    ref.clock.t = float(script['clock0'])
    triad = script.get('codec', 'json') == 'triad'
    if triad:
        ref_sched_loader.load_codec()
    k8s = fake_k8s.FakeK8s(script['nodes'], codec=script.get('codec', 'json'))
    sink = RpcSink()
    for st in script['init']:
        apply_k8s_op(k8s, ref.clock, st)
    feed = _RefFeed(ref, k8s, script['steps'], sink)
    try:
        while True:
            # 'triad': the reference's own GetCfgParser -> nhd.TriadCfgParser reads the libconfig text
            s = ref_sched_loader.make_scheduler(
                ref, k8s, None if triad else (lambda cfgtype, cfgstr: fake_k8s.JsonCfgParser(cfgstr, ref.cfg)))
            s.nqueue, s.rpcq = feed, feed.rpcq
            orig = s.CheckPendingPods

            def checked(orig=orig):
                orig()
                feed.checked = True
            s.CheckPendingPods = checked
            try:
                import contextlib
                import io
                with contextlib.redirect_stdout(io.StringIO()):      # stray print at Matcher.py:329
                    s.run()
            except _Stop:
                pass
            if feed.i >= len(script['steps']):
                break
    finally:
        ref.node.Node.MIN_BUSY_SECS = 30.0
    return state_document(s, k8s, sink)


# ----------------------------------------------------------------------------------------------
# this repo's scheduler
# ----------------------------------------------------------------------------------------------
def run_mirror(script, solver_factory=None, stats=None):
    import nhd_b200.CfgTopology as cfg_mod
    import nhd_b200.Node as node_mod
    from nhd_b200.NHDScheduler import NHDScheduler
    node_mod.Node.MIN_BUSY_SECS = float(script['min_busy_secs'])
    clock = Clock(script['clock0'])
    k8s = fake_k8s.FakeK8s(script['nodes'], codec=script.get('codec', 'json'))
    sink = RpcSink()
    for st in script['init']:
        apply_k8s_op(k8s, clock, st)
    if script.get('codec', 'json') == 'triad':
        from nhd_b200.TriadCfgParser import TriadCfgParser

        def parser(cfgtype, cfgstr):
            return TriadCfgParser(cfgstr, False)
    else:
        def parser(cfgtype, cfgstr):
            return fake_k8s.JsonCfgParser(cfgstr, cfg_mod)

    def make():
        s = NHDScheduler(k8s, parser,
                         solver_factory=solver_factory, clock=clock)
        s.Startup()
        return s

    s = None
    try:
        s = make()
        for st in script['steps']:
            op = st['op']
            if op in K8S_OPS:
                apply_k8s_op(k8s, clock, st)
            elif op == 'watch':
                s.HandleWatchItem({k: v for k, v in st.items() if k != 'op'})
            elif op == 'rpc':
                s.ParseRPCReq(st['msg'], sink)
            elif op == 'idle':
                s.CheckPendingPods()
            elif op == 'restart':
                _collect(stats, s)
                s.close()
                s = make()
        _collect(stats, s)
        return state_document(s, k8s, sink)
    finally:
        node_mod.Node.MIN_BUSY_SECS = 30.0
        if s is not None:
            s.close()


def drop_speed_residue(doc, names):
    """NodeNic.speed_used of nodes on which an assignment failed is left out of a comparison: the
    reference's unwind leaves the Gb/s of the aborted pod there (Node.py:831-835 indexes self.nics with a
    speed), a residue in a statistic that nhd_b200 does not reproduce (nhd_b200/NHDScheduler.py)."""
    doc = json.loads(json.dumps(doc))
    for n in names:
        if n in doc['nodes']:
            doc['nodes'][n].pop('speed_used', None)
    for ans in doc['rpc']:
        if isinstance(ans, list):
            for row in ans:
                if isinstance(row, dict) and row.get('name') in names:
                    row.pop('nicstats', None)
    return doc


def fingerprint(doc, names=()):
    """A state document with its bulk replaced by digests (tests.helpers.digest): one per Kubernetes record
    kind, for pod_state, for all nodes and for the RPC answers, all without the fields drop_speed_residue
    drops, and one per node for those fields (its NodeNic.speed_used and the nicstats of its RPC answer
    rows), left out for the nodes in ``names``.  Two documents compare equal after drop_speed_residue(...,
    names) exactly when their fingerprints with those names do."""
    from tests.helpers import digest
    bare = drop_speed_residue(doc, list(doc['nodes']))
    rows = [r for ans in doc['rpc'] if isinstance(ans, list) for r in ans if isinstance(r, dict)]
    residue = {n: digest([st.get('speed_used'), [r.get('nicstats') for r in rows if r.get('name') == n]])
               for n, st in doc['nodes'].items() if n not in names}
    k8s = bare['k8s']
    return {'k8s': {k: digest(v) for k, v in k8s.items()} if isinstance(k8s, dict) else digest(k8s),
            'pod_state': digest(bare['pod_state']), 'failed_schedule_count': bare['failed_schedule_count'],
            'nodes': digest(bare['nodes']), 'rpc': digest(bare['rpc']), 'residue': residue}


def run_mirror_loop(script, solver_factory=None):
    """Like run_mirror, but through ``nhd_b200.NHDScheduler.run()`` — the thread function with its queue
    polling and idle counting — fed by the same fake queues that drive the reference's ``run()``."""
    import nhd_b200.CfgTopology as cfg_mod
    import nhd_b200.Node as node_mod
    from nhd_b200 import NHDScheduler as M
    node_mod.Node.MIN_BUSY_SECS = float(script['min_busy_secs'])
    clock = Clock(script['clock0'])
    k8s = fake_k8s.FakeK8s(script['nodes'], codec=script.get('codec', 'json'))
    sink = RpcSink()
    for st in script['init']:
        apply_k8s_op(k8s, clock, st)
    if script.get('codec', 'json') == 'triad':
        from nhd_b200.TriadCfgParser import TriadCfgParser
        parser = lambda cfgtype, cfgstr: TriadCfgParser(cfgstr, False)          # noqa: E731
    else:
        parser = lambda cfgtype, cfgstr: fake_k8s.JsonCfgParser(cfgstr, cfg_mod)  # noqa: E731
    feed = _RefFeed(None, k8s, script['steps'], sink, M.NHDWatchTypes, M.RpcMsgType, clock)
    s = None
    try:
        while True:
            if s is not None:
                s.close()
            s = M.NHDScheduler(k8s, parser, rpcq=feed.rpcq, solver_factory=solver_factory, clock=clock)
            orig = s.CheckPendingPods

            def checked(orig=orig):
                orig()
                feed.checked = True
            s.CheckPendingPods = checked
            try:
                s.run(feed)
            except _Stop:
                pass
            if feed.i >= len(script['steps']):
                break
        return state_document(s, k8s, sink)
    finally:
        node_mod.Node.MIN_BUSY_SECS = 30.0
        if s is not None:
            s.close()


def _collect(stats, s):
    if stats is not None:
        stats.setdefault('assign_failed_nodes', set()).update(s.assign_failed_nodes)
        for k in ('full_loads', 'delta_nodes', 'batches', 'rewinds'):
            stats[k] = stats.get(k, 0) + getattr(s.cluster, k)
        stats['pods'] = stats.get('pods', 0) + s.pods_solved


def first_difference(a, b, path=''):
    """Human-readable location of the first difference between two state documents."""
    if type(a) != type(b):
        return f'{path}: {a!r} != {b!r}'
    if isinstance(a, dict):
        for k in sorted(set(a) | set(b)):
            if k not in a or k not in b:
                return f'{path}/{k}: only on one side'
            d = first_difference(a[k], b[k], f'{path}/{k}')
            if d:
                return d
        return None
    if isinstance(a, list):
        if len(a) != len(b):
            return f'{path}: length {len(a)} != {len(b)}: {a!r} != {b!r}'
        for i, (x, y) in enumerate(zip(a, b)):
            d = first_difference(x, y, f'{path}[{i}]')
            if d:
                return d
        return None
    return None if a == b else f'{path}: {a!r} != {b!r}'
