"""Freezes what the UNMODIFIED reference computes for the seeded cases of the differential tests (run where the
reference is importable, see oracle/ref_loader.py):

    python tests/golden/make_frozen_golden.py

One file per test module under tests/golden/frozen/.  The cases themselves are not stored: the test modules
regenerate them from their seeds (the functions imported below), and the files hold the reference's side in
the same order.  Small outcomes are stored as they are; records, state documents and codec outcomes as
digests (tests.helpers.digest, sched_harness.fingerprint), which the tests compare against the digests of
what this package computes.
"""
import contextlib
import io
import json
import os
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from nhd_b200 import packing                                     # noqa: E402
from oracle import ref_loader, ref_sched_loader                  # noqa: E402
from tests import helpers, ref_compare, sched_harness, scenarios  # noqa: E402
from tests import test_codec, test_ingest, test_oracle_vs_reference, test_rpc, test_scheduler  # noqa: E402
from tests.golden import make_ingest_golden                      # noqa: E402

OUT = helpers.FROZEN


def _stream(scn):
    outs, init, final, _, _ = ref_compare.run_reference(scn)
    return {'outcomes': ref_compare.freeze_outcomes(outs), 'init': helpers.digest(init), 'final': helpers.digest(final)}


def oracle_vs_reference(ref):
    t = test_oracle_vs_reference
    return {'flavors': {f: [_stream(scn) for _, scn in t.flavor_scenarios(f)] for f in t.FLAVORS},
            'limits': [_stream(scn) for _, scn in t.limit_scenarios()],
            'labels': [{name: helpers.digest(t.node_view(x)) for name, x in scenarios.build_nodes(scn, ref.node).items()}
                       for _, scn in t.label_scenarios()]}


def ingest(ref):
    layout = packing.ClusterLayout()            # one cluster dictionary across the cases, in case order
    fuzzed = []
    for case in test_ingest.fuzzed_cases():
        e = make_ingest_golden.reference_outcome(ref, case, layout)
        if e['parse'] != 'ok':
            fuzzed.append([e['parse']])
        elif e['record'] == 'unsupported':
            fuzzed.append(['unsupported'])
        else:
            aux = {k: e[k] for k in ('data_vlan', 'res_hugepages_gb', 'n_reserved_cores', 'gpu_device_id', 'nic_ifname')}
            fuzzed.append(['ok', helpers.digest(bytes.fromhex(e['record'])), helpers.digest(aux)])
    stats = []
    for _, scn in test_ingest.stats_scenarios():
        nodes = scenarios.build_nodes(scn, ref.node)
        matcher = ref.matcher.Matcher()
        for pod, t in zip(scn['pods'], scn['now']):
            top = scenarios.build_top(pod, ref.cfg)
            with contextlib.redirect_stdout(io.StringIO()):      # stray print at Matcher.py:329
                ref_loader.attempt_scheduling(ref, matcher, nodes, top, pod['groups'], t)
        order = list(nodes.values())
        stats.append({'records': packing.pack_nodes(order, packing.ClusterLayout()).tobytes().hex(),
                      'rows': test_ingest._stats_of_objects(order)})
    return {'fuzzed': fuzzed, 'fuzzed_speed_table': [float(x) for x in layout.speed_table()], 'stats': stats}


def rpc(ref):
    """The reference's NHDRpcHandler runs once nhd.proto.nhd_stats_pb2* (generated code, absent from the reference)
    resolve to nhd_b200.NHDRpcServer's message classes."""
    R = test_rpc.R
    with open(os.path.join(ref_loader.REFERENCE_ROOT, 'nhd', 'proto', 'nhd_stats.proto')) as f:
        proto = test_rpc._proto_fields(f.read())
    stub_pb = types.ModuleType('nhd.proto.nhd_stats_pb2')
    for k in dir(R.nhd_stats_pb2):
        if not k.startswith('_'):
            setattr(stub_pb, k, getattr(R.nhd_stats_pb2, k))
    stub_grpc = types.ModuleType('nhd.proto.nhd_stats_pb2_grpc')
    stub_grpc.NHDControlServicer = object
    stub_grpc.add_NHDControlServicer_to_server = R.add_NHDControlServicer_to_server
    pkg = types.ModuleType('nhd.proto')
    pkg.__path__ = []
    pkg.nhd_stats_pb2, pkg.nhd_stats_pb2_grpc = stub_pb, stub_grpc
    sys.modules.update({'nhd.proto': pkg, 'nhd.proto.nhd_stats_pb2': stub_pb, 'nhd.proto.nhd_stats_pb2_grpc': stub_grpc})
    try:
        import nhd.NHDRpcServer as ref_rpc
        handlers = test_rpc.handler_responses(ref_rpc.NHDRpcHandler)
    finally:
        for k in ('nhd.proto', 'nhd.proto.nhd_stats_pb2', 'nhd.proto.nhd_stats_pb2_grpc', 'nhd.NHDRpcServer'):
            sys.modules.pop(k, None)
    return {'proto': json.loads(json.dumps(proto)), 'handlers': handlers}


def scheduler(ref):
    return {f: [sched_harness.fingerprint(sched_harness.run_reference(script))
                for _, script in test_scheduler.flavor_scripts(f)] for f in ('mixed', 'vf', 'big', 'wild')}


def codec(ref):
    Ref = ref_sched_loader.load_codec().codec.TriadCfgParser
    out = []
    for seed, text, broken in test_codec.generated_cases():
        parsed = test_codec.run_case(Ref, text, False, seed)
        reparsed = test_codec.run_case(Ref, parsed['cfg'], True, seed)
        out.append({'parsed': helpers.digest(parsed), 'reparsed': helpers.digest(reparsed),
                    'broken': [helpers.digest(test_codec.run_case(Ref, bad, False, seed)) for bad in broken]})
    return out


def main():
    ref = ref_loader.load()
    os.makedirs(OUT, exist_ok=True)
    for fn in (oracle_vs_reference, ingest, rpc, scheduler, codec):
        path = os.path.join(OUT, fn.__name__ + '.json')
        with open(path, 'w') as f:
            json.dump(fn(ref), f, separators=(',', ':'))
            f.write('\n')
        print(fn.__name__, os.path.getsize(path) // 1024, 'KiB ->', path)


if __name__ == '__main__':
    main()
