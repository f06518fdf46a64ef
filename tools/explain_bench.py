"""Time nhd_explain on BASELINE config 4 (65 536 nodes, its 16 pod types) on the cluster after one solved batch.

    python tools/explain_bench.py --out DIR [--reps 300] [--warmup 20]

nhd_explain returns after a device synchronise, so a host clock around the call is its latency.  Two variants are
timed, counts only and with per-node detail (16 x 65 536 reason bytes copied back and expanded per pod); the filter,
sweep and total times of the solve on the same state (nhd_last_timing, CUDA events) are given for comparison.  The
card's name and power limit are read in the same run.  Writes DIR/explain_bench.json; needs a CUDA device.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np                    # noqa: E402

import workload                       # noqa: E402
from nhd_b200.solver import Solver    # noqa: E402


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        name, power = [x.strip() for x in out[0].split(',')]
        return {'name': name, 'power_limit': power}
    except Exception as e:            # the numbers stay, marked with what could not be read
        return {'name': None, 'power_limit': None, 'error': str(e)}


def stats(ms):
    ms = np.asarray(ms)
    return {'median_ms': float(np.median(ms)), 'p10_ms': float(np.percentile(ms, 10)),
            'p90_ms': float(np.percentile(ms, 90)), 'reps': int(len(ms))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--reps', type=int, default=300)
    ap.add_argument('--warmup', type=int, default=20)
    a = ap.parse_args()
    recs, speed, pods, now = workload.make_workload(4)
    types = workload.make_pod_types(4)
    s = Solver(speed)
    try:
        s.load_nodes(recs)
        s.solve_batch(pods, now)                     # the state after one solved batch
        s.snapshot()
        s.solve_batch(pods[:1024], now[:1024])      # a solve on that state, for its device timings
        solve = s.timing()
        s.restore()
        t = float(now[-1])
        tnow = np.full(len(types), t)
        res = {}
        for name, detail in (('counts_only', False), ('per_node_detail', True)):
            for _ in range(a.warmup):
                s.explain(types, tnow, detail=detail)
            ms = []
            for _ in range(a.reps):
                t0 = time.perf_counter()
                counts, first, _ = s.explain(types, tnow, detail=detail)
                ms.append((time.perf_counter() - t0) * 1e3)
            res[name] = stats(ms)
        res['feasible_nodes_per_type'] = counts[:, 0].tolist()
        res['first_fit'] = first.tolist()
    finally:
        s.close()
    doc = {'what': 'nhd_explain latency, host clock around the synchronous call',
           'workload': {'config': 4, 'nodes': int(len(recs)), 'explain_types': int(len(types)),
                        'state': f'after one solved batch of {len(pods)} pods', 'clock': t},
           'explain': res,
           'solve_on_same_state': {'pods': 1024, 'filter_ms': solve['filter_ms'], 'sweep_ms': solve['sweep_ms'],
                                   'total_ms': solve['total_ms'], 'n_types': solve['n_types'],
                                   'source': 'nhd_last_timing (CUDA events)'},
           'gpu': card()}
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, 'explain_bench.json'), 'w') as f:
        json.dump(doc, f, indent=1)
    print(json.dumps(doc))


if __name__ == '__main__':
    main()
