"""``NHDScheduler`` — host-side mirror of the reference's scheduler loop (``nhd/NHDScheduler.py``)
with the pending set solved as ONE batch on the GPU (SURVEY 8f row 1).

What is kept from the reference, method for method and with the same names, arguments, return
values and side effects on ``Node`` / ``pod_state`` / Kubernetes:

* start-up: ``InitNHDNodes`` / ``BuildInitialNodeList`` (``NHDScheduler.py:63-105``),
  ``LoadDeployedConfigs`` / ``ClaimPodResources`` (``:107-144, 161-172``), ``ResetResources`` (``:146-159``);
* ``ReleasePodResources`` (``:174-205``) including its two odd exits — a pod that was never annotated
  triggers a full ``ResetResources``, a pod that was annotated but not bound keeps its resources;
* ``InitialNodeFilter`` (``:235-247``), ``AttemptScheduling`` (``:249-353``), ``CheckPendingPods``
  (``:425-441``), the watch-queue handlers of ``run`` (``:491-577``) as ``HandleWatchItem``;
* ``GetBasicNodeStats`` / ``GetPodStats`` / ``ParseRPCReq`` (``:355-423``).

What is different is *where the placement is computed*.  The reference calls
``Matcher.FindNode`` once per pod (``:277``) against Python ``Node`` objects.  Here the packed
cluster lives on the GPU (``DeviceCluster``): ``CheckPendingPods`` first does the Kubernetes reads
for every pending pod, hands all their ``CfgTopology`` requests to ``nhd_solve_batch`` in one call
(pod *i* sees pods *0..i-1*, exactly like the loop), then walks the bindings in pod order doing what
``AttemptScheduling`` does after ``FindNode``: events, ``SetBusy``, physical ids into the topology,
NIC claim, NAD / GPU-map / config annotations, bind.  Only nodes the host changed outside the
solver (release, re-claim, reset, cordon, maintenance, groups) are re-sent (``nhd_update_nodes``).

A Kubernetes write that fails half way makes the reference call ``ReleasePodResources``, which may
reset the whole cluster; the pods after it in the batch were solved on a state that no longer
exists.  The batch is then cut at that pod: the host objects (always the truth) are pushed to the
device for every node that differs and the rest of the pending set is solved again — the outcome
is the one the sequential loop produces (``tests/test_scheduler.py``, pinned to the unmodified
reference ``NHDScheduler`` driven through the same fake Kubernetes manager).

Kubernetes itself, the kopf controller and the gRPC server are not part of this module: ``k8s`` is
any object with ``K8SMgr``'s method surface, ``cfg_parser(cfgtype, cfgstr)`` returns an object with
``CfgToTopology / TopologyToCfg / TopologyToGpuMap`` (``TriadCfgParser``).  There is no CPU
placement path: without the CUDA library ``DeviceCluster`` raises.
"""
import re
import time
from enum import Enum
from queue import Queue
from typing import Callable, Dict, Iterable, List, Optional, Sequence

import numpy as np

from nhd_b200 import packing, wire
from nhd_b200.Node import Node

NHD_SCHED_NAME = "nhd-scheduler"                # NHDScheduler.py:23


class PodStatus(Enum):                          # NHDScheduler.py:29-34
    POD_STATUS_SCHEDULED = 0
    POD_STATUS_FAILED = 1
    POD_STATUS_SUCCEEDED = 2
    POD_STATUS_RUNNING = 3
    POD_STATUS_COMPLETED = 4


class K8SEventType(Enum):                       # K8SMgr.py:16-18
    EVENT_TYPE_NORMAL = 0
    EVENT_TYPE_WARNING = 1


class NHDWatchTypes(Enum):                      # NHDWatchQueue.py:6-15 (the trailing commas make tuples there)
    NHD_WATCH_TYPE_TRIADSET_CREATE = 1
    NHD_WATCH_TYPE_TRIADSET_DELETE = 2
    NHD_WATCH_TYPE_TRIAD_POD_CREATE = 3
    NHD_WATCH_TYPE_TRIAD_POD_DELETE = 4
    NHD_WATCH_TYPE_NODE_UNCORDON = 5
    NHD_WATCH_TYPE_NODE_CORDON = 6
    NHD_WATCH_TYPE_GROUP_UPDATE = 7
    NHD_WATCH_TYPE_NODE_MAINT_START = 8
    NHD_WATCH_TYPE_NODE_MAINT_END = 9


class RpcMsgType(Enum):                         # NHDCommon.py:69-73
    TYPE_NODE_INFO = 1
    TYPE_SCHEDULER_INFO = 2
    TYPE_POD_INFO = 3
    TYPE_NODE_DETAIL = 4


OUTSIDE_LIMITS = 'OUTSIDE_LIMITS'                    # failure_reasons key: active nodes beyond the packed limits


def unschedulable_message(reasons: Dict[str, int], n_nodes: int) -> str:
    """kube-scheduler style summary of ``{reason name: nodes}`` (``wire.WHY_NAMES`` plus ``OUTSIDE_LIMITS``), e.g.
    ``0/12 nodes are available: 3 not in the pod's node groups, 9 too few free CPU cores.``  Reasons in code order,
    the nodes outside the solver's limits last.  Feasible nodes can only appear when busy windows expired after the
    pod's attempt: the message says so."""
    parts = [f'{reasons[name]} {wire.WHY_TEXT[w]}' for w, name in enumerate(wire.WHY_NAMES)
             if w != wire.WHY_FEASIBLE and reasons.get(name)]
    if reasons.get(OUTSIDE_LIMITS):
        parts.append(f"{reasons[OUTSIDE_LIMITS]} outside the solver's limits")
    feasible = reasons.get(wire.WHY_NAMES[wire.WHY_FEASIBLE], 0)
    head = f'{feasible}/{n_nodes} nodes are available'
    if feasible:
        head += ' now (busy windows expired since the attempt)'
    return head + (': ' + ', '.join(parts) if parts else '') + '.'


def _type_name(t) -> str:
    """Watch / RPC types may arrive as this module's enums, the reference's, or plain names."""
    return t if isinstance(t, str) else t.name


class DeviceCluster:
    """The packed node records of ``NHDScheduler.nodes`` resident on the GPU.

    The Python ``Node`` objects stay the source of truth (the rest of the reference reads them);
    this class keeps the device copy equal to them: a full ``nhd_load_nodes`` when the node set or
    the solver constants change, ``nhd_update_nodes`` for the nodes named dirty, nothing for nodes
    only the solver itself changed (its own commit already holds what ``apply_binding`` writes
    into the objects — that equality is the parity the GPU tests establish)."""

    def __init__(self, solver_factory: Optional[Callable] = None, device: int = 0):
        self._factory = solver_factory
        self._device = device
        self._solver = None
        self._layout = packing.ClusterLayout()
        self._names: List[str] = []
        self._index: Dict[str, int] = {}
        self._speeds: List[float] = []
        self._min_busy = None
        self.full_loads = 0
        self.delta_nodes = 0
        self.batches = 0
        self.rewinds = 0
        self._last = None
        self.stubs = set()
        self.unsupported_nodes: Dict[str, str] = {}

    @property
    def layout(self):
        return self._layout

    def close(self):
        if self._solver is not None:
            self._solver.close()
            self._solver = None

    def _make_solver(self, min_busy):
        if self._solver is not None:
            self._solver.close()
        factory = self._factory
        if factory is None:
            from nhd_b200.solver import Solver          # raises without the CUDA library / a GPU
            factory = Solver
        self._speeds = list(self._layout.speeds)
        self._min_busy = min_busy
        self._solver = factory(self._layout.speed_table(), nic_bw_avail_percent=0.9,
                               min_busy_secs=min_busy, device=self._device)

    def _pack(self, nodes: Sequence) -> np.ndarray:
        recs = np.zeros(len(nodes), dtype=wire.NODE_DTYPE)
        for i, node in enumerate(nodes):
            try:
                packing.pack_node(node, self._layout, out=recs[i])
            except packing.UnsupportedError as err:
                # a node whose labels were refused stays in NHDScheduler.nodes, deactivated and half
                # initialised (NHDScheduler.py:88-100); it holds its place in the order as an inactive stub.
                # An ACTIVE node beyond the packed limits (> 256 logical cores, > 16 GPUs, ...) cannot be
                # described to the solver either: it is kept out of placement (never approximated) and named in
                # unsupported_nodes for the operator.
                if node.active:
                    if node.name not in self.unsupported_nodes:
                        packing._log.warning('node %s is outside the packed limits and is kept out of placement: %s', node.name, err)
                    self.unsupported_nodes[node.name] = str(err)
                packing.stub_record(recs[i])
                self.stubs.add(node.name)
        return recs

    def sync(self, nodes: Dict[str, object], dirty: Iterable[str]):
        """Make the device copy equal to ``nodes``; ``dirty`` names the nodes the host changed since
        the last call."""
        names = list(nodes)
        min_busy = float(getattr(type(nodes[names[0]]), 'MIN_BUSY_SECS', 30.0)) if names else 30.0
        full = self._solver is None or names != self._names or min_busy != self._min_busy
        recs = idx = None
        if not full:
            dirty = set(dirty)
            todo = [n for n in names if n in dirty]
            if todo:
                recs = self._pack([nodes[n] for n in todo])
                idx = np.asarray([self._index[n] for n in todo], dtype='<i4')
            full = self._layout.speeds != self._speeds      # a NIC speed the solver has no class for yet
        if full:
            recs = self._pack([nodes[n] for n in names])
            if self._solver is None or self._layout.speeds != self._speeds or min_busy != self._min_busy:
                self._make_solver(min_busy)
            self._solver.load_nodes(recs)
            self._names = names
            self._index = {n: i for i, n in enumerate(names)}
            self.full_loads += 1
        elif recs is not None:
            self._solver.update_nodes(idx, recs)
            self.delta_nodes += len(idx)

    def solve(self, tops: Sequence, pod_groups: Sequence[Iterable[str]], now: float, packed: Sequence = None):
        """Bindings of ``tops`` scheduled in order on the synced cluster (one GPU call).  ``packed``: records
        ``pack_pod`` already made of them; only the node-group mask is worked out again (``sync`` may have met new
        group names since)."""
        pods = np.zeros(len(tops), dtype=wire.POD_DTYPE)
        for i, top in enumerate(tops):
            if packed is not None and packed[i] is not None:
                pods[i] = packed[i]
                pods[i]['group_mask'] = self._layout.groups_mask(pod_groups[i], create=False)
            else:
                packing.pack_pod(top, pod_groups[i], self._layout, out=pods[i])
        self.batches += 1
        self._solver.snapshot()                       # so that rewind() can step back inside this batch
        self._last = (pods, np.full(len(tops), now, dtype='<f8'))
        return self._solver.solve_batch(*self._last)

    def explain(self, packed: Sequence, pod_groups: Sequence[Iterable[str]], now: float) -> np.ndarray:
        """Nodes per ``wire.WHY_*`` reason for each packed pod on the synced cluster at ``now`` (one
        ``nhd_explain`` call; the device state is left as it is)."""
        pods = np.zeros(len(packed), dtype=wire.POD_DTYPE)
        for i, rec in enumerate(packed):
            pods[i] = rec
            pods[i]['group_mask'] = self._layout.groups_mask(pod_groups[i], create=False)
        counts, _, _ = self._solver.explain(pods, np.full(len(packed), now, dtype='<f8'))
        return counts

    def rewind(self, k: int):
        """Put the device back to the state right after pod ``k`` of the last batch (restore the
        snapshot taken before it, solve pods ``0..k`` again: the solver is deterministic)."""
        pods, now = self._last
        self._solver.restore()
        self._solver.solve_batch(pods[:k + 1], now[:k + 1])
        self.rewinds += 1

    def read_records(self):
        return self._solver.read_nodes()

    def read_record(self, index: int):
        return self._solver.read_nodes(index, 1)[0]

    def name_of(self, index: int) -> str:
        return self._names[index]


class _Pending:
    """One pending pod between the Kubernetes reads and the Kubernetes writes."""
    __slots__ = ('pos', 'key', 'pobj', 'tcfg', 'top', 'groups', 'ready', 'unsupported', 'rec')

    def __init__(self, pos, key):
        self.pos, self.key = pos, key
        self.pobj = self.tcfg = self.top = self.groups = self.unsupported = self.rec = None
        self.ready = False


class NHDScheduler:
    def __init__(self, k8s, cfg_parser: Callable, rpcq: Queue = None, solver_factory: Callable = None,
                 device: int = 0, clock: Callable[[], float] = time.monotonic,
                 wall: Callable[[], float] = time.time, node_cls=Node, logger=None,
                 stats_from_device: bool = False, explain_failures: bool = False):
        """``explain_failures``: after each ``CheckPendingPods`` pass, explain on the GPU why every pod that found
        no candidate node is unschedulable (one ``Unschedulable`` Warning event per pod, counts kept in
        ``failure_reasons``).  Off by default: the event stream is then exactly the reference's."""
        self.nodes: Dict[str, Node] = {}
        self.k8s = k8s
        self.sched_name = NHD_SCHED_NAME
        self.pod_state = {}
        self.rpcq = rpcq
        self.failed_schedule_count = 0
        self.cluster = DeviceCluster(solver_factory, device)
        self._cfg_parser = cfg_parser
        self._clock, self._wall = clock, wall
        self._node_cls = node_cls
        self._dirty = set()
        self._log = logger
        self.pods_solved = 0
        self.assign_failed_nodes = set()
        self.unsupported_pods = []                   # (ns, pod, why): requests beyond the packed layout's limits
        self.stats_from_device = stats_from_device
        self.explain_failures = explain_failures
        self.failure_reasons: Dict[tuple, Dict[str, int]] = {}   # (ns, pod) -> {reason name: nodes}, last pass
        self._unplaced = None                        # pods of the current pass that found no node (explain_failures)

    # ---- small helpers --------------------------------------------------------------------
    def _info(self, msg):
        if self._log is not None:
            self._log.info(msg)

    def _error(self, msg):
        if self._log is not None:
            self._log.error(msg)

    def _touch(self, name):
        """The host changed node ``name`` outside the solver: re-send it before the next batch."""
        self._dirty.add(name)

    def _set_busy(self, node):                       # Node.SetBusy, Node.py:843-845, on the scheduler's clock
        node.busy_time = float(self._clock())

    def close(self):
        self.cluster.close()

    # ---- start-up (NHDScheduler.py:63-105) --------------------------------------------------
    def InitNHDNodes(self):
        for node in self.k8s.GetNodes():
            self.nodes[node] = self._node_cls(node, self.k8s.IsNodeActive(node))

    def BuildInitialNodeList(self):
        self.InitNHDNodes()
        for n, v in self.nodes.items():
            try:
                v.SetNodeAddr(self.k8s.GetNodeAddr(n))
                if not v.ParseLabels(self.k8s.GetNodeLabels(n)):
                    self._error(f'Error while parsing labels for node {n}, deactivating node')
                    v.active = False
                    continue
                (alloc, free) = self.k8s.GetNodeHugepageResources(n)
                if alloc == 0 or not v.SetHugepages(alloc, free):
                    self._error(f'Error while parsing allocatable resources for node {n}, deactivating node')
                    v.active = False
            except Exception as e:                   # the reference swallows everything here (:98-100)
                self._error(f'Caught exception while setting up node {n}:\n    {e}')
                v.active = False
        self._dirty.update(self.nodes)

    # ---- claim / release of deployed pods (NHDScheduler.py:107-205) ---------------------------
    def GetCfgParser(self, cfgtype: str, cfgstr: str):
        return self._cfg_parser(cfgtype, cfgstr)

    def ClaimPodResources(self, podname, ns, uid):
        cfgstr = self.k8s.GetCfgAnnotations(podname, ns)
        if cfgstr == False:                          # noqa: E712  (the reference's test, :112)
            self._error(f'Couldn\'t find pod resources for {ns}.{podname}')
            return
        cfgtype = self.k8s.GetCfgType(podname, ns)
        tcfg = self.GetCfgParser(cfgtype, cfgstr)
        top = tcfg.CfgToTopology(True)
        if top is not None:
            n = self.k8s.GetPodNode(podname, ns)
            if not n:
                return
            if n not in self.nodes:
                return
            if self.nodes[n].PodPresent(podname, ns):
                return
            self._touch(n)
            if not self.nodes[n].RemoveResourcesFromTopology(top):
                self._error('Failed removing resources')
                return
            self.nodes[n].AddScheduledPod(podname, ns, top)
            self.pod_state[(ns, podname)] = {'state': PodStatus.POD_STATUS_SCHEDULED, 'time': self._wall(),
                                             'uid': uid}

    def ResetResources(self):
        for name, n in self.nodes.items():
            n.ResetResources()
            self._touch(name)
        self.pod_state.clear()
        self.LoadDeployedConfigs()

    def LoadDeployedConfigs(self):
        for p in self.k8s.GetScheduledPods(self.sched_name):
            if p[3] in ('Running', 'CrashLoopBackOff', 'Pending'):
                self.ClaimPodResources(p[0], p[1], p[2])

    def ReleasePodResources(self, podname, ns):
        cfgstr = self.k8s.GetCfgAnnotations(podname, ns)
        if cfgstr == False:                          # noqa: E712  never annotated: full re-scan (:178-181)
            self.ResetResources()
            return
        cfgtype = self.k8s.GetCfgType(podname, ns)
        tcfg = self.GetCfgParser(cfgtype, cfgstr)
        top = tcfg.CfgToTopology(True)
        if top is not None:
            node = self.k8s.GetPodNode(podname, ns)
            if not node:                             # annotated but not bound: nothing is given back (:189-191)
                return
            if node not in self.nodes:
                return
            if not self.nodes[node].PodPresent(podname, ns):
                return
            self._touch(node)
            self.nodes[node].AddResourcesFromTopology(top)
            self.nodes[node].RemoveScheduledPod(podname, ns)
            self._set_busy(self.nodes[node])

    def ParsePodResources(self, pod: str, ns: str) -> Dict[str, int]:      # :214-224
        res = self.k8s.GetRequestedPodResources(pod, ns)
        trimmed = {}
        if 'hugepages-1Gi' in res:
            trimmed['hugepages-1Gi'] = int(res['hugepages-1Gi'][:res['hugepages-1Gi'].find('G')])
        return trimmed

    # ---- placement ------------------------------------------------------------------------------
    def InitialNodeFilter(self, podname: str, ns: str):
        """``NHDScheduler.py:235-247``.  Informational here: the batch path evaluates the same gate
        on the GPU from the pod's group list (group mask AND + active flag)."""
        ngroups = self.k8s.GetPodNodeGroups(podname, ns)
        return {n: v for n, v in self.nodes.items() if len(set(v.groups) & set(ngroups)) > 0 and v.active}

    def _prepare(self, e: _Pending):
        """The Kubernetes reads of ``AttemptScheduling`` up to ``FindNode`` (``:254-275``)."""
        ns, podname = e.key[0], e.key[1]
        e.ready = True
        e.pobj = self.k8s.GetPodObj(podname, ns)
        if e.pobj is None:
            self._error(f'Could not get pod object for pod {ns}.{podname}')
            return
        self.k8s.GeneratePodEvent(e.pobj, podname, ns, 'StartedScheduling', K8SEventType.EVENT_TYPE_NORMAL,
                                  f'Started scheduling {ns}/{podname}')
        _, cfgstr = self.k8s.GetCfgMap(podname, ns)
        cfgtype = self.k8s.GetCfgType(podname, ns)
        e.tcfg = self.GetCfgParser(cfgtype, cfgstr)
        e.top = e.tcfg.CfgToTopology(False)
        if e.top is None:
            self.k8s.GeneratePodEvent(e.pobj, podname, ns, 'FailedCfgParse', K8SEventType.EVENT_TYPE_WARNING,
                                      f'Error while processing config for pod {podname}')
            return
        e.groups = self.k8s.GetPodNodeGroups(podname, ns)
        try:                                         # a request beyond the packed layout (include/nhd_b200.h, NHD_MAX_*)
            e.rec = packing.pack_pod(e.top, e.groups, self.cluster.layout)     # kept for the solve (group mask aside)
        except packing.UnsupportedError as err:      # cannot be solved here and is never approximated: the pod fails,
            e.unsupported = str(err)                 # loudly, instead of taking the scheduler thread down

    def _finish(self, e: _Pending, binding, now: float) -> bool:
        """``AttemptScheduling`` from the result of ``FindNode`` on (``:278-353``)."""
        ns, podname = e.key[0], e.key[1]
        if e.pobj is None or e.top is None:
            return False
        k8s, pobj, top, tcfg = self.k8s, e.pobj, e.top, e.tcfg
        if e.unsupported is not None:
            self._error(f'Pod {ns}.{podname} is outside the solver\'s limits: {e.unsupported}')
            k8s.GeneratePodEvent(pobj, podname, ns, 'FailedScheduling', K8SEventType.EVENT_TYPE_WARNING,
                                 f'Pod {podname} cannot be placed by the B200 solver: {e.unsupported}')
            self.failed_schedule_count += 1
            self.unsupported_pods.append((ns, podname, e.unsupported))
            return False
        if binding is None or int(binding['node']) < 0:
            k8s.GeneratePodEvent(pobj, podname, ns, 'FailedScheduling', K8SEventType.EVENT_TYPE_WARNING,
                                 f'No valid candidate nodes found for scheduling pod {podname}')
            self.failed_schedule_count += 1
            return False
        nodename = self.cluster.name_of(int(binding['node']))
        k8s.GeneratePodEvent(pobj, podname, ns, 'Scheduling', K8SEventType.EVENT_TYPE_NORMAL,
                             f'Node {nodename} selected for scheduling')
        node = self.nodes[nodename]
        node.busy_time = float(now)                                           # SetBusy (:289)
        try:
            packing.apply_binding(node, top, binding)                         # SetPhysicalIdsFromMapping (:292)
        except IndexError:
            self._error('Failed to map physical resources from topology config!')
            # The reference's unwind (Node.py:825-837) gives cores and GPUs back but never the hugepages it
            # took at :794-796 (a failure at the last step, the top-level misc cores); the solver's record
            # holds the node as the reference leaves it.  Its NIC part indexes self.nics with a *speed* and
            # stops at the first entry (IndexError again, or a TypeError that ends the reference's thread:
            # status REF_WOULD_CRASH), leaving the Gb/s it had added in NodeNic.speed_used: that residue of a
            # statistic is not reproduced, the node is remembered in assign_failed_nodes instead.
            rec = self.cluster.read_record(int(binding['node']))
            node.mem.free_hugepages_gb = int(rec['free_hugepages_gb'])
            self.assign_failed_nodes.add(nodename)
            return False
        nidx = [int(x) for x in binding['claimed_nics'][:int(binding['n_claimed'])]]   # list({x[0] ...}) (:302)
        node.ClaimPodNICResources(nidx)
        if any(node.nics[i].pods_used <= 0 for i in nidx):
            # Release counts a NIC down once per RX/TX pairing but the claim counts it up once per pod
            # (Node.py:579,629 vs :644-646), so a counter can sit below zero and a claimed NIC still reads
            # as free (pods_used > 0, Node.py:292).  The device keeps one in-use bit: re-send this node.
            self._touch(nodename)
        nadlist = node.GetNADListFromIndices(nidx)
        csnad = ','.join([f'{x}@{x}' for x in nadlist])
        if not k8s.AddNADToPod(podname, ns, csnad):
            self._error('Failed to set NetworkAttachmentDefinition')
            self.ReleasePodResources(podname, ns)
            return False
        topstr = tcfg.TopologyToCfg()
        gpustr = tcfg.TopologyToGpuMap()
        if gpustr:
            if not k8s.AnnotatePodGpuMap(ns, podname, gpustr):
                k8s.GeneratePodEvent(pobj, podname, ns, 'PodCfgFailed', K8SEventType.EVENT_TYPE_WARNING,
                                     f'Failed to annotate pod\'s GPU configuration')
                self.ReleasePodResources(podname, ns)
                return False
        if not k8s.AnnotatePodConfig(ns, podname, topstr):
            k8s.GeneratePodEvent(pobj, podname, ns, 'PodCfgFailed', K8SEventType.EVENT_TYPE_WARNING,
                                 f'Failed to annotate pod\'s configuration')
            self.ReleasePodResources(podname, ns)
            return False
        else:
            k8s.GeneratePodEvent(pobj, podname, ns, 'PodCfgSuccess', K8SEventType.EVENT_TYPE_NORMAL,
                                 f'Successfully added pod\'s configuration to annotations')
        if not k8s.BindPodToNode(podname, nodename, ns):
            k8s.GeneratePodEvent(pobj, podname, ns, 'FailedScheduling', K8SEventType.EVENT_TYPE_WARNING,
                                 f'Failed to schedule {ns}/{podname} to {nodename}')
            self.ReleasePodResources(podname, ns)
            return False
        else:
            k8s.GeneratePodEvent(pobj, podname, ns, 'Scheduled', K8SEventType.EVENT_TYPE_NORMAL,
                                 f'Successfully assigned {ns}/{podname} to {nodename}')
        node.AddScheduledPod(podname, ns, top)
        return True

    def ScheduleBatch(self, keys: Sequence, wanted: Callable = None) -> Dict:
        """Schedule the pods ``keys`` = ``[(ns, name, uid), ...]`` in order, as if ``AttemptScheduling``
        were called for one after the other.  ``wanted(key)`` is asked again for the pods behind a cut
        (``CheckPendingPods`` re-reads ``pod_state``, which a reset clears).  Returns ``{key: bool}``."""
        results = {}
        entries = [_Pending(i, k) for i, k in enumerate(keys)]
        pos = 0
        while pos < len(entries):
            run = [e for e in entries[pos:] if wanted is None or wanted(e.key)]
            if not run:
                break
            for e in run:
                if not e.ready:
                    self._prepare(e)
            now = float(self._clock())
            solvable = [e for e in run if e.top is not None and e.unsupported is None]
            bindings = {}
            if solvable and self.nodes:
                self.cluster.sync(self.nodes, self._dirty)
                self._dirty.clear()
                out = []
                while solvable:
                    try:
                        out = self.cluster.solve([e.top for e in solvable], [e.groups for e in solvable], now,
                                                 packed=[e.rec for e in solvable])
                        break
                    except Exception as err:
                        # a limit that depends on the cluster as well (numa^(groups+1) tuples, include/nhd_b200.h):
                        # the library refuses the whole batch and names the pod; that pod fails loudly, the rest goes on
                        m = re.search(r'pod (\d+)', str(err)) if getattr(err, 'code', None) == wire.ERR_UNSUPPORTED else None
                        if m is None or int(m.group(1)) >= len(solvable):
                            raise
                        solvable.pop(int(m.group(1))).unsupported = str(err)
                self.pods_solved += len(solvable)
                bindings = {e.pos: out[i] for i, e in enumerate(solvable)}
            cut = None
            for e in run:
                b = bindings.get(e.pos)
                rewound = False
                if b is not None and int(b['status']) in (wire.ASSIGN_FAILED, wire.REF_WOULD_CRASH):
                    # what a failed assignment leaves on its node is read back from the solver (see _finish);
                    # for that the device must stand right after this pod, not at the end of the batch
                    self.cluster.rewind(solvable.index(e))
                    rewound = True
                results[e.key] = ok = self._finish(e, b, now)
                self._record(e.key, ok)
                if self._unplaced is not None and e.pobj is not None and b is not None and int(b['node']) < 0:
                    self._unplaced.append(e)
                if self._dirty or rewound:            # nodes changed behind the solver's back / device rewound
                    cut = e
                    break
            if cut is None:
                break
            # bindings not yet applied are void: their nodes on the device are ahead of the host objects
            for e in run:
                b = bindings.get(e.pos)
                if e.pos > cut.pos and b is not None and int(b['node']) >= 0:
                    self._touch(self.cluster.name_of(int(b['node'])))
            pos = cut.pos + 1
        return results

    def _record(self, key, ok: bool):                 # the two branches of CheckPendingPods (:431-436)
        podkey = (key[0], key[1])
        if ok:
            self.pod_state[podkey] = {'state': PodStatus.POD_STATUS_SCHEDULED, 'time': self._wall(), 'uid': key[2]}
            self.failure_reasons.pop(podkey, None)
        else:
            self._error(f'Failed scheduling pod {key[0]}.{key[1]} [{key[2]}]')
            self.pod_state[podkey] = {'state': PodStatus.POD_STATUS_FAILED, 'time': self._wall(), 'uid': '0'}

    def AttemptScheduling(self, podname, ns) -> bool:
        """Single pod, reference signature (``:249``): a batch of one."""
        saved = self.pod_state.get((ns, podname))
        key = (ns, podname, None)
        ok = self.ScheduleBatch([key])[key]
        if saved is None:                             # the caller owns pod_state for this entry point
            self.pod_state.pop((ns, podname), None)
        else:
            self.pod_state[(ns, podname)] = saved
        return ok

    def CheckPendingPods(self):
        """``NHDScheduler.py:425-441`` with the pending set solved as one batch."""
        podlist = self.k8s.ServicePods(self.sched_name)
        phase = {(k[0], k[1], k[2]): p for k, p in podlist.items()}

        def wanted(k):
            p = phase[k]
            podkey = (k[0], k[1])
            return (p[0] == 'Pending' and p[1] == None and                     # noqa: E711
                    ((podkey not in self.pod_state) or
                     self.pod_state[podkey]['state'] != PodStatus.POD_STATUS_SCHEDULED))

        self._unplaced = [] if self.explain_failures else None
        try:
            self.ScheduleBatch(list(phase), wanted)
            unplaced = self._unplaced
        finally:
            self._unplaced = None
        if unplaced:
            self._explain_unplaced(unplaced)
        # The reference's second branch (:437-440) compares the pod_state *dict* with an enum member and
        # therefore never runs; a pod reported 'Failed' keeps its resources until its delete event.

    def _explain_unplaced(self, entries: Sequence[_Pending]):
        """Why the pods of ``entries`` found no node, on the cluster as their next attempt will find it (the state
        after the pass, at the scheduler clock now): one ``nhd_explain`` call, one ``Unschedulable`` event each."""
        if not self.nodes:
            return
        self.cluster.sync(self.nodes, self._dirty)
        self._dirty.clear()
        counts = self.cluster.explain([e.rec for e in entries], [e.groups for e in entries], float(self._clock()))
        outside = sum(1 for n in self.cluster.unsupported_nodes if n in self.nodes)
        for e, row in zip(entries, counts):
            reasons = {wire.WHY_NAMES[w]: int(c) for w, c in enumerate(row) if c}
            if outside:
                # inactive stubs on the device (packing.stub_record: no node group), listed for what they are
                moved = min(outside, reasons.get('NOT_IN_GROUP', 0))
                if moved:
                    reasons['NOT_IN_GROUP'] -= moved
                    if not reasons['NOT_IN_GROUP']:
                        del reasons['NOT_IN_GROUP']
                    reasons[OUTSIDE_LIMITS] = moved
            ns, podname = e.key[0], e.key[1]
            self.failure_reasons[(ns, podname)] = reasons
            self.k8s.GeneratePodEvent(e.pobj, podname, ns, 'Unschedulable', K8SEventType.EVENT_TYPE_WARNING,
                                      unschedulable_message(reasons, int(row.sum())))

    # ---- the thread function (NHDScheduler.py:443-577) ------------------------------------------------
    def Startup(self):
        """What ``run`` does before its loop (``:448-455``)."""
        self.BuildInitialNodeList()
        self.LoadDeployedConfigs()
        self.CheckPendingPods()

    def run(self, nqueue, idle_thresh: int = 60, block_secs: float = 0.5, stop: Callable[[], bool] = None):
        """The reference's loop: watch items first, else one gRPC request, else count idleness and
        re-scan the pending pods every ``idle_thresh`` empty polls (``:468-489``)."""
        from queue import Empty
        self.Startup()
        try:                                           # drop what piled up during start-up (:459-465)
            while True:
                nqueue.get(block=False, timeout=0)
        except Empty:
            pass
        idle_cnt = 0
        while stop is None or not stop():
            try:
                item = nqueue.get(block=False)
            except Empty:
                try:
                    item = self.rpcq.get(True, block_secs)
                    self.ParseRPCReq(item[0], item[1])
                except Empty:
                    idle_cnt += 1
                    if idle_cnt >= idle_thresh:
                        idle_cnt = 0
                        self.CheckPendingPods()
                continue
            self.HandleWatchItem(item)

    # ---- watch queue (NHDScheduler.py:491-577) -----------------------------------------------------
    def HandleWatchItem(self, item):
        t = _type_name(item["type"])
        if t in ('NHD_WATCH_TYPE_TRIAD_POD_DELETE', 'NHD_WATCH_TYPE_TRIAD_POD_CREATE'):
            ns, pn, uid = item["pod"]["ns"], item["pod"]["name"], item["pod"]["uid"]
            if t == 'NHD_WATCH_TYPE_TRIAD_POD_DELETE':
                self.ReleasePodResources(pn, ns)
                self.pod_state.pop((ns, pn), None)
                self.failure_reasons.pop((ns, pn), None)
            else:
                if ((ns, pn) in self.pod_state) and \
                        (self.pod_state[(ns, pn)]['state'] == PodStatus.POD_STATUS_SCHEDULED):
                    if self.pod_state[(ns, pn)]['uid'] == uid:
                        return
                    self.ReleasePodResources(pn, ns)
                    self.pod_state.pop((ns, pn), None)
                key = (ns, pn, uid)
                if self.ScheduleBatch([key])[key]:
                    self.pod_state[(ns, pn)] = {'state': PodStatus.POD_STATUS_SCHEDULED, 'time': self._wall(),
                                                'uid': uid}
                else:
                    self.pod_state[(ns, pn)] = {'state': PodStatus.POD_STATUS_FAILED, 'time': 0, 'uid': '0'}
        elif t in ('NHD_WATCH_TYPE_NODE_CORDON', 'NHD_WATCH_TYPE_NODE_UNCORDON'):
            v = self.nodes.get(item["node"])
            if v is not None:
                want = t == 'NHD_WATCH_TYPE_NODE_UNCORDON'
                if v.active != want:
                    v.active = want
                    self._touch(item["node"])
        elif t in ('NHD_WATCH_TYPE_NODE_MAINT_START', 'NHD_WATCH_TYPE_NODE_MAINT_END'):
            v = self.nodes.get(item["node"])
            if v is not None:
                want = t == 'NHD_WATCH_TYPE_NODE_MAINT_START'
                if v.maintenance != want:
                    v.maintenance = want
                    self._touch(item["node"])
        elif t == 'NHD_WATCH_TYPE_GROUP_UPDATE':
            v = self.nodes.get(item["node"])
            if v is not None:
                v.SetGroups(item["groups"])
                self._touch(item["node"])

    # ---- statistics (NHDScheduler.py:355-423) --------------------------------------------------------
    def GetBasicNodeStats(self):
        nodes = []
        for k, v in self.nodes.items():
            nodes.append({'name': k,
                          'freegpu': v.GetFreeGpuCount(),
                          'totalgpu': v.GetTotalGPUs(),
                          'freecpu': v.GetFreeCpuCoreCount(),
                          'totalcpu': v.GetTotalCPUs(),
                          'freehuge_gb': v.GetFreeHugepages(),
                          'totalhuge_gb': v.GetTotalHugepages(),
                          'totalpods': v.GetTotalPods(),
                          'active': v.GetNodeActive(),
                          'nicstats': v.GetNICUsedSpeeds()})
        return nodes

    def GetBasicNodeStatsFromDevice(self):
        """The same rows with the counters that are placement state taken from the GPU's records
        (``nhd_read_nodes`` + ``nhd_node_stats_from_records``) instead of walking the Python objects;
        ``totalhuge_gb``, ``totalpods`` and ``nicstats`` are not placement state and come from the host."""
        from nhd_b200 import ingest
        self.cluster.sync(self.nodes, self._dirty)
        self._dirty.clear()
        st = ingest.node_stats(self.cluster.read_records())
        rows = []
        by_name = {r['name']: r for r in self.GetBasicNodeStats()} if self.cluster.stubs else {}
        for i, (k, v) in enumerate(self.nodes.items()):
            if k in self.cluster.stubs:              # no usable record: the half-initialised object answers
                rows.append(by_name[k])
                continue
            s = st[i]
            rows.append({'name': k,
                         'freegpu': int(s['freegpu']), 'totalgpu': int(s['totalgpu']),
                         'freecpu': int(s['freecpu']), 'totalcpu': int(s['totalcpu']),
                         'freehuge_gb': int(s['freehuge_gb']), 'totalhuge_gb': v.GetTotalHugepages(),
                         'totalpods': v.GetTotalPods(), 'active': bool(s['active']),
                         'nicstats': v.GetNICUsedSpeeds()})
        return rows

    def GetPodStats(self):
        pinfo = []
        for k, v in self.nodes.items():
            for pname, pval in v.pod_info.items():
                # pod_info is keyed (pod, ns) (Node.py:205-208); the reference passes the two in this order to
                # GetPodAnnotations(podname, ns) (NHDScheduler.py:388), i.e. swapped, so unless a pod's name
                # equals its namespace the lookup fails and the pod is skipped.  Kept as is.
                annots = self.k8s.GetPodAnnotations(pname[1], pname[0])
                if annots == None:                   # noqa: E711
                    continue
                pinfo.append({
                    'namespace': pname[1],
                    'podname': pname[0],
                    'node': k,
                    'annotations': annots,
                    'hugepages': pval.hugepages_gb,
                    'proc_cores': [pc.core for pg in pval.proc_groups for pc in pg.proc_cores],
                    'proc_helper_cores': [pc.core for pg in pval.proc_groups for pc in pg.misc_cores],
                    'misc_cores': [pc.core for pc in pval.misc_cores],
                    'gpus': [g.device_id for pg in pval.proc_groups for g in pg.group_gpus],
                    'nics': [np_.mac for np_ in pval.nic_core_pairing],
                })
        return pinfo

    def ParseRPCReq(self, msgid, q: Queue):
        t = _type_name(msgid)
        if t == 'TYPE_NODE_INFO':
            q.put(self.GetBasicNodeStatsFromDevice() if self.stats_from_device and self.nodes
                  else self.GetBasicNodeStats())
        elif t == 'TYPE_SCHEDULER_INFO':
            q.put(self.failed_schedule_count)
        elif t == 'TYPE_POD_INFO':
            q.put(self.GetPodStats())
