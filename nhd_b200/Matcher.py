"""``Matcher`` — drop-in replacement of the reference's ``nhd/Matcher.py`` backed by the
B200 solver.

Same surface as the reference (``Matcher()`` no-arg constructor, ``FindNode(nl, top)``
returning ``(nodename, mapping)`` or ``(None,)``, ``Matcher.py:22-63``), so
``NHDScheduler.AttemptScheduling`` (``NHDScheduler.py:277-304``) can call it unchanged;
plus ``FindNodesBatch`` which schedules a whole pending set (``CheckPendingPods``,
``NHDScheduler.py:425-441``) in one GPU call with the same sequential semantics.

``nl`` may hold this package's ``Node`` mirrors or the reference's own ``nhd.Node.Node``
objects (duck-typed packing).  The filter, the NUMA/PCI intersection, node selection,
mapping choice and the physical core/GPU/NIC assignment all run in CUDA; this module only
converts formats.  Without the CUDA library / a GPU it raises — there is no CPU path.
"""
import time
from typing import Dict, Iterable, List, Optional, Sequence

import numpy as np

from nhd_b200 import packing, tracking, wire
from nhd_b200.solver import Solver


class _Cluster:
    """What the device holds: every node handed in so far, in an order every ``nl`` seen is a sub-sequence of."""
    __slots__ = ('names', 'index', 'objs', 'vers', 'recs', 'member', 'force')

    def __init__(self, names):
        n = len(names)
        self.names = names
        self.index = {nm: i for i, nm in enumerate(names)}
        self.objs = [None] * n
        self.vers = [None] * n                      # _nhd_version the record was packed at; None: pack every time
        self.recs = np.zeros(n, dtype=wire.NODE_DTYPE)
        self.member = np.zeros(n, dtype=bool)       # in the node dict of the current call
        self.force = set()                          # device copy changed by the solver itself: upload again


class Matcher:
    def __init__(self, device: int = 0, track: bool = True):
        """``track``: instrument the ``Node`` classes met with a change counter (``nhd_b200/tracking.py``) so that
        later calls pack only the nodes that changed; without it every call packs every node."""
        self.device = device
        self.track = track
        self._solver: Optional[Solver] = None
        self._layout = packing.ClusterLayout()
        self._speeds: List[float] = []
        self._min_busy = None
        self._cl: Optional[_Cluster] = None
        self._history: List[List[str]] = []              # node-dict orders seen when the device order was rebuilt
        self.unsupported_nodes: Dict[str, str] = {}      # active nodes kept out of placement: name -> reason
        self.stats = {'calls': 0, 'packed': 0, 'uploaded': 0, 'full_loads': 0}

    # ------------------------------------------------------------------ internals
    def _ensure_solver(self, nodes: Sequence):
        """(Re)create the device handle when the solver constants changed; True when it is a new one."""
        min_busy = float(getattr(type(nodes[0]), 'MIN_BUSY_SECS', 30.0)) if nodes else 30.0
        if self._solver is None or self._speeds != self._layout.speeds or self._min_busy != min_busy:
            if self._solver is not None:
                self._solver.close()
            self._speeds = list(self._layout.speeds)
            self._min_busy = min_busy
            self._solver = Solver(self._layout.speed_table(), nic_bw_avail_percent=0.9,
                                  min_busy_secs=min_busy, device=self.device)
            return True
        return False

    def _pack_into(self, cl: _Cluster, i: int, node, tracked: bool):
        """Host record i from ``node``.  A node outside the packed limits becomes an inactive stub (logged, listed in
        unsupported_nodes) and the others stay schedulable, as with the reference."""
        d = getattr(node, '__dict__', None)
        ver = d.get(tracking.VERSION, 0) if (tracked and d is not None) else None
        try:
            packing.pack_node(node, self._layout, out=cl.recs[i])
        except packing.UnsupportedError as err:
            packing.stub_record(cl.recs[i])
            if getattr(node, 'active', True):
                name = getattr(node, 'name', cl.names[i])
                if name not in self.unsupported_nodes:
                    packing._log.warning('node %s is outside the packed limits and is kept out of placement: %s', name, err)
                self.unsupported_nodes[name] = str(err)
        cl.objs[i] = node
        cl.vers[i] = ver
        self.stats['packed'] += 1

    def _merge_order(self, known: List[str], index: Dict[str, int], seq: List[str]) -> List[str]:
        """A device order that has ``seq`` (this call's node dict) and the dicts of earlier calls as sub-sequences.
        The scheduler filters one ordered dict per pod (NHDScheduler.py:235-247), so everything it hands in is a
        sub-sequence of that one order, which the matcher never sees whole: the order is rebuilt as a topological
        sort of the sequences seen at rebuilds (old positions break ties, so what already fitted keeps fitting).
        Sequences that contradict each other mean the caller's order really changed: then ``seq`` alone counts."""
        import heapq
        self._history = (self._history + [list(seq)])[-16:]
        if not known:
            return list(seq)
        for attempt in (0, 1):
            succ, indeg = {}, {}
            for h in self._history:
                for n in h:
                    indeg.setdefault(n, 0)
                for a, b in zip(h, h[1:]):
                    ss = succ.setdefault(a, set())
                    if b not in ss:
                        ss.add(b)
                        indeg[b] += 1
            big = len(known)
            pref = {n: index.get(n, big + k) for k, n in enumerate(indeg)}
            heap = [(pref[n], n) for n, d in indeg.items() if d == 0]
            heapq.heapify(heap)
            out = []
            while heap:
                _, n = heapq.heappop(heap)
                out.append(n)
                for b in succ.get(n, ()):
                    indeg[b] -= 1
                    if indeg[b] == 0:
                        heapq.heappush(heap, (pref[b], b))
            if len(out) == len(indeg):
                placed = set(out)
                return out + [n for n in known if n not in placed]
            self._history = [list(seq)]                # a cycle: forget the older sequences
        raise AssertionError('unreachable: one sequence has no cycle')

    def _device_view(self, cl: _Cluster, idx) -> np.ndarray:
        """Records as the device gets them: a node that is not in the current node dict is not a candidate
        (InitialNodeFilter left it out, NHDScheduler.py:241-243) — its ACTIVE flag is cleared."""
        out = cl.recs[idx].copy()
        out['flags'] &= np.where(cl.member[idx], 0xFF, 0xFF & ~wire.NODE_ACTIVE).astype(out['flags'].dtype)
        return out

    def _load(self, nl: Dict[str, object]):
        """Make the device cluster equal to ``nl``: pack the nodes that changed since the last call (all of them the
        first time, or when their class carries no change counter), upload those and the ones whose membership
        changed.  Returns (names in device order, node objects in device order, solver)."""
        self.stats['calls'] += 1
        names_nl = list(nl)
        nodes_nl = [nl[n] for n in names_nl]
        tracked = {}
        for cls in set(map(type, nodes_nl)):
            tracked[cls] = tracking.track_changes(cls) if self.track else False
        cl = self._cl
        idxs = None
        if cl is not None:
            try:
                idxs = np.fromiter((cl.index[n] for n in names_nl), dtype=np.int64, count=len(names_nl))
                if len(idxs) > 1 and not bool((np.diff(idxs) > 0).all()):
                    idxs = None                      # the order changed: lay the cluster out again
            except KeyError:
                idxs = None                          # a node not seen before
        full = idxs is None
        if full:
            # new layout: this call's nodes in their order, then the known ones that are not part of it; records of
            # nodes that did not change are carried over
            old = cl
            cl = _Cluster(self._merge_order(old.names if old else [], old.index if old else {}, names_nl))
            idxs = np.fromiter((cl.index[n] for n in names_nl), dtype=np.int64, count=len(names_nl))
            if old is not None:
                for i, nm in enumerate(cl.names):
                    j = old.index.get(nm)
                    if j is not None:
                        cl.recs[i] = old.recs[j]
                        cl.objs[i], cl.vers[i] = old.objs[j], old.vers[j]
                cl.force = {cl.index[old.names[j]] for j in old.force}
            self._cl = cl
        member = np.zeros(len(cl.names), dtype=bool)
        member[idxs] = True
        objs, vers, VER = cl.objs, cl.vers, tracking.VERSION
        changed = []
        for i, node in zip(idxs.tolist(), nodes_nl):
            d = getattr(node, '__dict__', None)
            if objs[i] is not node or vers[i] is None or d is None or vers[i] != d.get(VER, 0):
                changed.append((i, node))
        for i in cl.force:
            if objs[i] is not None and not member[i]:
                changed.append((i, objs[i]))         # bound by the solver last time, not part of this call
        for i, node in changed:
            self._pack_into(cl, i, node, tracked.get(type(node), self.track and tracking.is_tracked(type(node))))
        flips = np.flatnonzero(member != cl.member)
        cl.member = member
        new_solver = self._ensure_solver(nodes_nl)   # packing may have met a new NIC speed class
        if full or new_solver:
            self._solver.load_nodes(self._device_view(cl, np.arange(len(cl.names))))
            self.stats['full_loads'] += 1
            self.stats['uploaded'] += len(cl.names)
        else:
            up = np.unique(np.concatenate([np.asarray([i for i, _ in changed], dtype=np.int64), np.asarray(sorted(cl.force), dtype=np.int64),
                                           flips.astype(np.int64)]))
            if len(up):
                self._solver.update_nodes(up.astype('<i4'), self._device_view(cl, up))
                self.stats['uploaded'] += len(up)
        cl.force = set()
        return cl.names, cl.objs, self._solver

    # ------------------------------------------------------------------ reference API
    def FindNode(self, nl, top, pod_groups: Iterable[str] = None, now: float = None):
        """Reference signature ``FindNode(nl, top)`` (``Matcher.py:27``).  ``nl`` is the node
        dict already narrowed by ``InitialNodeFilter``; therefore every node's groups match
        by construction unless ``pod_groups`` is given.

        Returns ``(nodename, mapping)`` or ``(None,)``.  ``mapping`` carries the complete
        device-computed binding under ``'_nhd_binding'`` for ``Node.SetPhysicalIdsFromMapping``
        of this package's ``Node`` mirror; the reference's own ``Node`` ignores that key and
        recomputes the identical assignment itself."""
        if len(nl) == 0:
            return (None,)
        names, nodes, solver = self._load(nl)
        pod = packing.pack_pod(top, [], self._layout)
        if pod_groups is None:
            pod['group_mask'] = np.uint64(0xFFFFFFFFFFFFFFFF)   # nl is pre-filtered (NHDScheduler.py:274)
        else:
            pod['group_mask'] = self._layout.groups_mask(pod_groups, create=False)
        now = time.monotonic() if now is None else now
        b = solver.solve_batch(pod.reshape(1), [now])[0]
        if int(b['node']) < 0:
            return (None,)
        self._cl.force.add(int(b['node']))       # the solver committed the pod there; the caller may or may not follow
        mapping = packing.binding_to_mapping(b)
        mapping['_nhd_binding'] = b
        return names[int(b['node'])], mapping

    def Explain(self, nl, top, pod_groups: Iterable[str] = None, now: float = None):
        """Why ``FindNode(nl, top)`` would drop each node of ``nl`` now — what the reference logs node by node
        (``Matcher.py:74-353``) — without placing anything.  Returns ``(nodename or None, {node name: reason name})``
        with the names of ``wire.WHY_NAMES``; the first element is what ``FindNode`` returns first on the same
        state."""
        if len(nl) == 0:
            return None, {}
        names, nodes, solver = self._load(nl)
        pod = packing.pack_pod(top, [], self._layout)
        if pod_groups is None:
            pod['group_mask'] = np.uint64(0xFFFFFFFFFFFFFFFF)
        else:
            pod['group_mask'] = self._layout.groups_mask(pod_groups, create=False)
        now = time.monotonic() if now is None else now
        _, first, reasons = solver.explain(pod.reshape(1), [now], detail=True)
        index = self._cl.index
        why = {n: wire.WHY_NAMES[int(reasons[0, index[n]])] for n in nl}
        return (names[int(first[0])] if first[0] >= 0 else None), why

    def FindNodesBatch(self, nl, tops: Sequence, pod_groups: Sequence[Iterable[str]] = None,
                       now=None, apply: bool = True):
        """Schedule ``tops`` in order on ``nl`` (all nodes of the cluster, NOT pre-filtered:
        the per-pod ``InitialNodeFilter`` runs on the GPU from ``pod_groups``).

        Returns one ``(nodename, mapping)`` / ``(None,)`` per pod.  With ``apply`` the bindings
        are also written into the ``Node`` / ``CfgTopology`` objects exactly as the scheduler's
        ``SetBusy`` + ``SetPhysicalIdsFromMapping`` + ``ClaimPodNICResources`` sequence would
        (``NHDScheduler.py:289-304``)."""
        n = len(tops)
        if n == 0:
            return []
        if len(nl) == 0:
            return [(None,)] * n
        names, nodes, solver = self._load(nl)
        pods = np.zeros(n, dtype=wire.POD_DTYPE)
        for i, top in enumerate(tops):
            groups = ['default'] if pod_groups is None else pod_groups[i]
            packing.pack_pod(top, groups, self._layout, out=pods[i])
        if now is None:
            now = time.monotonic()
        nows = np.full(n, now, dtype='<f8') if np.isscalar(now) else np.asarray(now, dtype='<f8')
        bindings = solver.solve_batch(pods, nows)
        self._cl.force.update(int(x) for x in np.unique(bindings['node']) if x >= 0)
        results = []
        failed = set()
        for i, (top, b) in enumerate(zip(tops, bindings)):
            if int(b['node']) < 0:
                results.append((None,))
                continue
            node = nodes[int(b['node'])]
            mapping = packing.binding_to_mapping(b)
            mapping['_nhd_binding'] = b
            results.append((names[int(b['node'])], mapping))
            if apply:
                node.busy_time = float(nows[i])                                  # SetBusy
                if int(b['status']) == wire.PLACED:
                    packing.apply_binding(node, top, b)                          # SetPhysicalIdsFromMapping
                    node.ClaimPodNICResources([int(x) for x in b['claimed_nics'][:int(b['n_claimed'])]])
                else:
                    failed.add(int(b['node']))
        # a failed assignment gives cores and GPUs back but not the hugepages taken before the last step
        # (Node.py:794-796 vs :825-837); the solver's records hold the nodes as the reference leaves them
        for idx in failed:
            nodes[idx].mem.free_hugepages_gb = int(solver.read_nodes(idx, 1)[0]['free_hugepages_gb'])
            tracking.bump(nodes[idx])
        return results
