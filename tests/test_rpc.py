"""SURVEY 8f row 4 — the statistics service (``nhd_b200.NHDRpcServer``): messages built without
generated code must be the reference's (``nhd/proto/nhd_stats.proto``), the handlers must fill them like
the UNMODIFIED reference ``NHDRpcHandler`` (``nhd/NHDRpcServer.py:47-137``), and a live server on the
loopback interface must answer the calls of the reference's ``test/RPCTest.py`` from a running scheduler,
from the Python objects or from the solver's records."""
import json
import re
import threading
from queue import Empty, Queue

import pytest

from nhd_b200 import NHDRpcServer as R
from tests import helpers, sched_harness as H

NODE_ROWS = [{'name': 'n0', 'freegpu': 3, 'totalgpu': 8, 'freecpu': 40, 'totalcpu': 96, 'freehuge_gb': 20,
              'totalhuge_gb': 64, 'totalpods': 3, 'active': True, 'nicstats': [[10, 20], [0, 0]]},
             {'name': 'n1', 'freegpu': 0, 'totalgpu': 0, 'freecpu': 0, 'totalcpu': 64, 'freehuge_gb': 0,
              'totalhuge_gb': 32, 'totalpods': 0, 'active': False, 'nicstats': []}]
POD_ROWS = [{'namespace': 'prod', 'podname': 'p0', 'node': 'n0', 'annotations': {'a': 'b', 'sigproc.viasat.io/x': 'y'},
             'hugepages': 4, 'proc_cores': [3, 4, 5], 'proc_helper_cores': [6], 'misc_cores': [7, 8], 'gpus': [0, 2],
             'nics': ['0C:42:A1:00:00:01']}]


def _feeder(q, answers, n):
    """Plays the scheduler thread: answers n requests from a table keyed by message type name."""
    def run():
        for _ in range(n):
            msg, reply = q.get(True, 10)
            reply.put(answers[msg.name])
    t = threading.Thread(target=run, daemon=True)
    t.start()
    return t


def _proto_fields(text):
    """Tiny reader for the subset of proto3 the reference's file uses -> comparable structure."""
    text = re.sub(r'//[^\n]*', '', text)
    out = {'messages': {}, 'enums': {}, 'rpcs': []}
    for kind, name, body in re.findall(r'\b(message|enum)\s+(\w+)\s*\{([^{}]*)\}', text):
        if kind == 'enum':
            out['enums'][name] = sorted((n, int(v)) for n, v in re.findall(r'(\w+)\s*=\s*(\d+)\s*;', body))
        else:
            fields = []
            for stmt in body.split(';'):
                m = re.fullmatch(r'\s*(repeated\s+)?(map\s*<[^>]*>|[\w.]+)\s+(\w+)\s*=\s*(\d+)\s*', stmt)
                if m:
                    rep, typ, fname, num = m.groups()
                    fields.append((fname, int(num), typ.replace(' ', ''), bool(rep) or typ.startswith('map')))
            out['messages'][name] = sorted(fields, key=lambda f: f[1])
    out['rpcs'] = sorted(re.findall(r'rpc\s+(\w+)\s*\(\s*(\w+)\s*\)\s*returns\s*\(\s*(\w+)\s*\)', text))
    return out


def test_descriptor_is_the_references_proto():
    """Against the reference's nhd/proto/nhd_stats.proto as _proto_fields reads it (golden/make_frozen_golden.py)."""
    want = helpers.frozen('rpc')['proto']
    fd = R.file_descriptor_proto()
    assert fd.package == 'NhdStats' and fd.syntax == 'proto3'
    T = R._T
    names = {T.TYPE_STRING: 'string', T.TYPE_UINT32: 'uint32', T.TYPE_BOOL: 'bool'}
    got = {'messages': {}, 'enums': {e.name: sorted((v.name, v.number) for v in e.value) for e in fd.enum_type}}
    for m in fd.message_type:
        fields = []
        for f in m.field:
            if f.type in names:
                typ = names[f.type]
            elif f.type_name.endswith('Entry'):
                typ = 'map<string,string>'
            else:
                typ = f.type_name.split('.')[-1]
            fields.append((f.name, f.number, typ, f.label == T.LABEL_REPEATED))
        got['messages'][m.name] = sorted(fields, key=lambda f: f[1])
    got['rpcs'] = sorted((m.name, m.input_type.split('.')[-1], m.output_type.split('.')[-1]) for m in fd.service[0].method)
    assert json.loads(json.dumps(got)) == want
    assert len(want['messages']) == 9 and len(want['rpcs']) == 4


def test_messages_round_trip_and_wire_format():
    pb = R.nhd_stats_pb2
    m = pb.NodeStats(status=pb.NHD_STATUS_OK)
    n = m.info.add()
    n.name, n.free_cpus, n.active = 'n0', 40, True
    n.nic_info.add(used_rx=10, used_tx=20)
    raw = m.SerializeToString()
    # status OK is the default (not sent); field 2 (info), length-delimited: name, free_cpus=40, nic_info, active
    assert raw == bytes([0x12, 14, 0x0a, 2]) + b'n0' + bytes([0x10, 40, 0x4a, 4, 0x08, 10, 0x10, 20, 0x50, 1])
    assert pb.NodeStats.FromString(raw) == m
    p = pb.PodInfo(name='p', namespace='ns')
    p.annotations['k'] = 'v'
    p.gpus.extend([0, 2])
    assert pb.PodInfo.FromString(p.SerializeToString()).annotations['k'] == 'v'
    with pytest.raises((TypeError, ValueError)):
        pb.NICInfoBrief().used_rx = 'x'


ANSWERS = {'TYPE_NODE_INFO': NODE_ROWS, 'TYPE_SCHEDULER_INFO': 17, 'TYPE_POD_INFO': POD_ROWS}
CALLS = ('GetBasicNodeStats', 'GetSchedulerStats', 'GetPodStats')
# a Gb/s that is not an integer cannot go into a uint32 field
BAD_ANSWERS = {'TYPE_NODE_INFO': [dict(NODE_ROWS[0], nicstats=[[22.5, 0]])]}


def handler_responses(handler_cls):
    """call -> serialized response of a handler fed ANSWERS; 'bad' -> name of the exception BAD_ANSWERS raise."""
    out = {}
    for call in CALLS:
        q = Queue()
        _feeder(q, ANSWERS, 1)
        out[call] = getattr(handler_cls(q), call)(R.nhd_stats_pb2.Empty(), None).SerializeToString(deterministic=True).hex()
    q = Queue()
    _feeder(q, BAD_ANSWERS, 1)
    try:
        handler_cls(q).GetBasicNodeStats(R.nhd_stats_pb2.Empty(), None)
        out['bad'] = None
    except Exception as e:                                      # noqa: BLE001 - which exception is the outcome
        out['bad'] = type(e).__name__
    return out


def test_handlers_match_the_reference_handler():
    """The unmodified ``nhd.NHDRpcServer.NHDRpcHandler`` (run on this module's message classes in place of its
    absent generated code, golden/make_frozen_golden.py) built these responses; this handler must build them
    byte for byte, and fail the same call the same way."""
    want = helpers.frozen('rpc')['handlers']
    got = handler_responses(R.NHDRpcHandler)
    assert got == want
    assert want['bad'] in ('TypeError', 'ValueError')
    for call in CALLS:
        m = getattr(R.nhd_stats_pb2, {'GetBasicNodeStats': 'NodeStats', 'GetSchedulerStats': 'SchedulerStats',
                                      'GetPodStats': 'PodStats'}[call]).FromString(bytes.fromhex(got[call]))
        assert m.status == R.nhd_stats_pb2.NHD_STATUS_OK


def test_handler_times_out_with_error_status():
    h = R.NHDRpcHandler(Queue(), reply_timeout=0.05)          # nobody answers (NHDRpcServer.py:78-79)
    assert h.GetSchedulerStats(None, None).status == R.nhd_stats_pb2.NHD_STATUS_ERR
    assert h.GetBasicNodeStats(None, None).status == R.nhd_stats_pb2.NHD_STATUS_ERR
    assert h.GetPodStats(None, None).status == R.nhd_stats_pb2.NHD_STATUS_ERR


@pytest.mark.parametrize('from_device', [False, True], ids=['objects', 'device_records'])
def test_live_server_serves_a_running_scheduler(oracle_lib, from_device):
    """test/RPCTest.py against a loopback server fed by ``NHDScheduler.ParseRPCReq``; node counters come from
    the Python objects or (stats_from_device) from the solver's records — same answer."""
    import grpc
    import nhd_b200.CfgTopology as cfg_mod
    from nhd_b200.NHDScheduler import NHDScheduler
    from tests import fake_k8s, scenarios
    nodes = [scenarios.make_node(f'n{i}', 2, 16, True, 1, gpus=[(d, d // 2, 0x10 * (d // 2 + 1)) for d in range(4)],
                                 nics=[('eth0', 100000, 0, 0x10), ('eth1', 100000, 1, 0x20)]) for i in range(4)]
    k8s = fake_k8s.FakeK8s(nodes)
    pod = scenarios.make_pod([scenarios.make_group(pairs=((10, 20),), workers=2, gpus=(1,), helpers=1)], misc=1,
                             hugepages=2, map_type='PCI')
    for i in range(3):
        k8s.add_pod('same', 'same' if i == 0 else f'p{i}', pod, uid=f'u{i}')   # ns == name: GetPodStats finds it
    k8s.add_pod('a', 'huge', scenarios.make_pod([scenarios.make_group(workers=60)]), uid='u9')    # cannot fit
    rpcq = Queue()
    sched = NHDScheduler(k8s, lambda t, c: fake_k8s.JsonCfgParser(c, cfg_mod), rpcq=rpcq, clock=H.Clock(1000.0),
                         solver_factory=helpers.OracleSolver, stats_from_device=from_device)
    sched.Startup()
    stop = threading.Event()

    def scheduler_thread():                                    # the RPC part of NHDScheduler.run (:476-479)
        while not stop.is_set():
            try:
                item = rpcq.get(True, 0.05)
            except Empty:
                continue
            sched.ParseRPCReq(item[0], item[1])
    th = threading.Thread(target=scheduler_thread, daemon=True)
    th.start()
    srv = R.NHDRpcServer(rpcq, listen='127.0.0.1:0')
    srv.start()
    assert srv.ready.wait(10) and srv.port
    try:
        with grpc.insecure_channel(f'127.0.0.1:{srv.port}') as channel:
            stub = R.NHDControlStub(channel)
            ns = stub.GetBasicNodeStats(R.nhd_stats_pb2.Empty(), timeout=10)
            assert ns.status == R.nhd_stats_pb2.NHD_STATUS_OK and [n.name for n in ns.info] == ['n0', 'n1', 'n2', 'n3']
            rows = {r['name']: r for r in sched.GetBasicNodeStats()}
            for n in ns.info:
                r = rows[n.name]
                assert (n.free_cpus, n.used_cpus, n.free_gpus, n.used_gpus, n.free_hugepages, n.total_pods, n.active) == \
                       (r['freecpu'], r['totalcpu'] - r['freecpu'], r['freegpu'], r['totalgpu'] - r['freegpu'],
                        r['freehuge_gb'], r['totalpods'], r['active'])
                assert [[x.used_rx, x.used_tx] for x in n.nic_info] == r['nicstats']
            assert sum(n.used_gpus for n in ns.info) == 3 and sum(n.total_pods for n in ns.info) == 3
            fs = stub.GetSchedulerStats(R.nhd_stats_pb2.Empty(), timeout=10)
            assert (fs.status, fs.failed_schedule_count) == (R.nhd_stats_pb2.NHD_STATUS_OK, 1)
            ps = stub.GetPodStats(R.nhd_stats_pb2.Empty(), timeout=10)
            assert ps.status == R.nhd_stats_pb2.NHD_STATUS_OK
            assert [(p.namespace, p.name) for p in ps.info] == [('same', 'same')]     # the swapped lookup, 8.3
            assert len(ps.info[0].proc_cores) == 4 and len(ps.info[0].gpus) == 1 and ps.info[0].nic_macs
            with pytest.raises(grpc.RpcError) as e:                                   # declared, not served
                stub.GetDetailedNodeStats(R.nhd_stats_pb2.NodeReq(name='n0'), timeout=10)
            assert e.value.code() == grpc.StatusCode.UNIMPLEMENTED
    finally:
        stop.set()
        srv.stop()
        sched.close()
