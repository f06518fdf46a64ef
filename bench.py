#!/usr/bin/env python
"""Benchmark of the NHD placement hot path (contract: see the task's bench.py section).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    torchrun --nproc-per-node N bench.py --gpus N ...        (N > 1, one rank per GPU)

A *step* is one pass of the hot path over one batch: 4 096 pending pods scheduled, with the
reference's sequential semantics, on the 65 536-node synthetic cluster of BASELINE config 4
(workload.py).  Every step starts from the same cluster state.

Own arm (CUDA):
  value   decisions/s with the batch and the cluster resident in HBM; the timed region is the
          solver's kernels (snapshot filter [+ NCCL all-reduce] + sweep), timed with CUDA events
          on the stream they are launched on; L2 is flushed between steps.
  e2e     the same metric through the C-ABI with HOST buffers: per step, upload of the cluster
          records and of the pod batch from host memory, the kernels, and the download of the
          bindings (wall clock around nhd_load_nodes + nhd_solve_batch).
  roofline / cpu_baseline / clocks: see DESIGN.md "Measurement".
Reference arm (--impl reference): the reference's algorithm on the host CPU — the C restatement
under oracle/ (the reference itself is Python and cannot travel to the GPU box), each pod's walk over
the nodes split over all host threads, on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import workload  # noqa: E402

CONFIG = 4
METRIC = 'placement decisions/sec (64k nodes x 4k pods)'
UNIT = 'decisions/s'
S_BYTES_PER_NODE = 64          # SURVEY.md 8(d): algorithmic bytes per node per decision (configs 2-4)
FIXED_BYTES_PER_DECISION = 256


def measured_peaks():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    except Exception:
        return 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler:
    """SM clock / throttle-reason sampler running DURING the timed region.  The timed region is short (20 steps of
    about 3 ms), so the samples come from NVML inside this process (a thread polling every 2 ms: dozens of samples
    under load); nvidia-smi in a loop is the fallback where NVML cannot be loaded."""
    FIELDS = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
              'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
    NAMES = ('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap')

    def __init__(self, index=0, uuid=None):
        self.index = index
        self.uuid = uuid
        self.proc = None
        self.path = None
        self.thread = None
        self.stop_flag = False
        self.sm, self.mx, self.reasons = [], [], set()
        self.source = None

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        if self.uuid:
            for u in (self.uuid, 'GPU-' + self.uuid):
                try:
                    return pynvml, pynvml.nvmlDeviceGetHandleByUUID(u.encode() if hasattr(u, 'encode') else u)
                except Exception:
                    pass
        idx = self.index
        vis = os.environ.get('CUDA_VISIBLE_DEVICES', '')
        if vis:
            ids = [x.strip() for x in vis.split(',') if x.strip()]
            if idx < len(ids) and ids[idx].isdigit():
                idx = int(ids[idx])
        return pynvml, pynvml.nvmlDeviceGetHandleByIndex(idx)

    def _poll(self, nv, h):
        bits = ((nv.nvmlClocksEventReasonHwSlowdown, 'hw_slowdown'),
                (nv.nvmlClocksEventReasonHwThermalSlowdown, 'hw_thermal_slowdown'),
                (nv.nvmlClocksEventReasonSwThermalSlowdown, 'sw_thermal_slowdown'),
                (nv.nvmlClocksEventReasonSwPowerCap, 'sw_power_cap'))
        try:
            mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        except Exception:
            mx = None
        while not self.stop_flag:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                if mx is not None:
                    self.mx.append(mx)
                r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
                for bit, nm in bits:
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        try:
            import threading
            nv, h = self._nvml_handle()
            nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)            # fails here, not in the thread
            self.thread = threading.Thread(target=self._poll, args=(nv, h), daemon=True)
            self.source = 'nvml, 2 ms period'
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            fd, self.path = tempfile.mkstemp(suffix='.csv')
            os.close(fd)
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.FIELDS,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=open(self.path, 'w'), stderr=subprocess.DEVNULL)
            self.source = 'nvidia-smi -lms 100'
        except Exception:
            self.proc = None

    def stop(self):
        out = {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0, 'source': self.source}
        sm, mx, reasons = self.sm, self.mx, self.reasons
        if self.thread is not None:
            self.stop_flag = True
            self.thread.join(timeout=2)
        elif self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
            try:
                for line in open(self.path):
                    parts = [x.strip() for x in line.split(',')]
                    if len(parts) < 6:
                        continue
                    try:
                        sm.append(float(parts[0]))
                        mx.append(float(parts[1]))
                    except ValueError:
                        continue
                    for nm, v in zip(self.NAMES, parts[2:6]):
                        if v.lower().startswith('active'):
                            reasons.add(nm)
                os.unlink(self.path)
            except Exception:
                pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)) if mx else None,
                       reasons=sorted(reasons), samples=len(sm))
        return out


def host_cpu_model():
    try:
        for ln in open('/proc/cpuinfo'):
            if ln.lower().startswith('model name'):
                return ln.split(':', 1)[1].strip()
    except Exception:
        pass
    return None


def pin_near_gpu(torch, local_rank):
    """One process per GPU, run on the CPUs next to that GPU (its PCIe root's NUMA node), as such a process is deployed:
    the pinned host buffers of the end-to-end leg are then allocated on that node.  Returns (previous affinity, cpus
    now allowed) or None when the topology cannot be read or nothing would change."""
    try:
        pr = torch.cuda.get_device_properties(local_rank)
        bus = '%04x:%02x:%02x.0' % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        cpus = set()
        for part in open(f'/sys/bus/pci/devices/{bus}/local_cpulist').read().strip().split(','):
            if part:
                lo, _, hi = part.partition('-')
                cpus.update(range(int(lo), int(hi or lo) + 1))
        old = os.sched_getaffinity(0)
        new = cpus & old
        if len(new) >= 2 and new != old:
            os.sched_setaffinity(0, new)
            return old, len(new)
    except Exception:
        pass
    return None


def host_threads():
    """Threads for the CPU arm: the host cores this process may really use (affinity mask, cgroup CPU quota)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        quota, period = open('/sys/fs/cgroup/cpu.max').read().split()[:2]
        if quota != 'max':
            n = min(n, max(1, int(float(quota) / float(period) + 0.999)))
    except Exception:
        pass
    return max(1, n)


def pick_threads(ob, recs, speed, pods, now, single_per_pod=None):
    """Times a few pods with all host threads and with fewer; returns (threads, seconds per pod) of the fastest.
    The walk over the nodes is barrier-synchronised per pod, so more threads than usable cores only hurt."""
    best = (1, single_per_pod) if single_per_pod else None
    T = host_threads()
    tried = []
    if T >= 2:
        ob.solve(recs, speed, pods[:2], now[:2], threads=T)          # untimed: thread stacks, TLS, page faults
    for t in sorted({T, max(1, T // 2), max(1, T // 4), min(T, 16)}, reverse=True):
        if t < 2:
            continue
        t0 = time.perf_counter()
        ob.solve(recs, speed, pods[:12], now[:12], threads=t)
        per_pod = (time.perf_counter() - t0) / 12
        tried.append((t, per_pod))
        if best is None or per_pod < best[1]:
            best = (t, per_pod)
        if per_pod > 2.0:                       # hopeless already: do not spend the budget on calibration
            break
    if best is None:
        t0 = time.perf_counter()
        ob.solve(recs, speed, pods[:4], now[:4])
        best = (1, (time.perf_counter() - t0) / 4)
    return best


def quick_value(Solver, recs, speed, pods, now, steps=3, pre_step=None, **kw):
    """decisions/s (device-timed total, batch resident) of a side workload: `steps` solves from the same snapshot."""
    s = Solver(speed, **kw)
    try:
        s.load_nodes(recs)
        s.snapshot()
        s.stage_batch(pods, now)
        best = None
        for _ in range(steps + 1):
            s.restore()
            s.sync()
            if pre_step is not None:
                pre_step()                     # several ranks: enter the step together (else the collective times their skew)
            s.solve_staged()
            s.sync()
            t = s.timing()
            best = t if best is None or t['total_ms'] < best['total_ms'] else best
        return {'value': len(pods) / (best['total_ms'] / 1e3), 'unit': UNIT, 'ms': best['total_ms'],
                'filter_ms': best['filter_ms'], 'exchange_ms': best['exchange_ms'], 'sweep_ms': best['sweep_ms'],
                'pod_types': best['n_types']}
    finally:
        s.close()


def python_reference_baseline(recs, speed, pods, now, n_pods=8):
    """The reference's own Python path (unmodified nhd/Matcher.py + Node.py through oracle/ref_loader) on the first
    pods of the stream at full N, one thread — only where the reference is reachable (NHD_REFERENCE_ROOT or
    /root/reference; never on the GPU box).  Returns None otherwise."""
    root = os.environ.get('NHD_REFERENCE_ROOT', '/root/reference')
    if not os.path.isfile(os.path.join(root, 'nhd', 'Matcher.py')):
        return None
    try:
        from tests import pyref
        return pyref.time_reference(recs, speed, pods[:n_pods], now[:n_pods])
    except Exception as e:                      # never let the optional leg take the bench down
        return {'error': str(e)[:200]}


def dump_outputs(out_dir, bindings, nodes):
    """One float64 .npy per field of the bindings (bindings_<field>) and of the node records the step left on the
    device (nodes_<field>), so that two builds can be compared output for output.  A 64-bit integer field becomes
    its [low, high] 32-bit words on a last axis of 2: float64 holds those exactly."""
    out = {}
    for prefix, arr in (('bindings', bindings), ('nodes', nodes)):
        for name in arr.dtype.names:
            if name == 'pad_':
                continue
            a = np.ascontiguousarray(arr[name])
            if a.dtype.kind in 'iu' and a.dtype.itemsize == 8:
                a = a.view('<u4').reshape(a.shape + (2,))
            out[f'{prefix}_{name}'] = a.astype(np.float64)
    total = sum(a.nbytes for a in out.values())
    assert total <= 64 << 20, f'outputs to dump are {total} bytes'
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)


def run_reference_arm(args, rank):
    """CPU arm: the oracle port of the reference path on the host cores.  The reference itself is one
    Python thread (NHDScheduler.py:43); its per-pod walk over all nodes is independent per node, so the
    port splits that walk over all host threads (pods stay strictly sequential).  Bounded sample per step."""
    if rank != 0:
        return
    from oracle import binding as ob
    ob.build()
    recs, speed, pods, now = workload.make_workload(CONFIG)
    N = len(recs)
    # size one step at roughly budget/(steps+warmup) seconds from a short calibration run
    T, per_pod = pick_threads(ob, recs, speed, pods, now)
    budget = 60.0
    per_step = budget / max(1, args.steps + args.warmup)
    n_sample = int(max(8, min(len(pods), per_step / per_pod)))
    times = []
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        ob.solve(recs, speed, pods[:n_sample], now[:n_sample], threads=T)
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
    value = n_sample * len(times) / sum(times)
    sample = f'first {n_sample} pods of the 4096-pod stream on all {N} nodes, per step, {T} host threads'
    line = {'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * sum(times) / len(times),
            'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'u64', 'data': 'synthetic',
            'config': {'workload': f'BASELINE config {CONFIG}: 65536 nodes x 4096 pods', 'sample': sample},
            'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': T, 'kind': 'port', 'sample': sample},
            'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0, 'host_cores_available': os.cpu_count()}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='nhd_b200', choices=['nhd_b200', 'reference'])
    ap.add_argument('--cpu-sample-pods', type=int, default=128)
    ap.add_argument('--no-extra', action='store_true', help='skip the side workloads (config 5, heterogeneous, moving clock)')
    ap.add_argument('--stop-after-e2e', action='store_true', help='developer switch: print value / e2e / clocks only and stop')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the last timed step computed (bindings, final node records) to DIR/<name>.npy')
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl != 'reference' else args.warmup

    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))

    if args.impl == 'reference':
        run_reference_arm(args, rank)
        return

    import torch
    import torch.distributed as dist
    from nhd_b200 import wire
    from nhd_b200.solver import Solver, nccl_unique_id, pinned_array, shard_min_pairs

    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device; the B200 solver has no CPU fallback')
    torch.cuda.set_device(local_rank)
    pinned = pin_near_gpu(torch, local_rank)          # before any host buffer is allocated; undone before the CPU legs
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
        idt = torch.zeros(128, dtype=torch.uint8, device='cuda')
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(nccl_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        nccl_id = bytes(idt.cpu().numpy().tobytes())
    else:
        nccl_id = None

    recs, speed, pods, now = workload.make_workload(CONFIG)
    N, P = len(recs), len(pods)
    solver = Solver(speed, device=local_rank, rank=rank, world_size=world, nccl_id=nccl_id)
    solver.load_nodes(recs)
    solver.snapshot()

    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')      # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---------------- value: batch + cluster resident in HBM, kernels only -----------------
    solver.stage_batch(pods, now)
    phase = {'filter_ms': [], 'exchange_ms': [], 'sweep_ms': [], 'total_ms': []}
    try:
        dev_uuid = str(torch.cuda.get_device_properties(local_rank).uuid)
    except Exception:
        dev_uuid = None
    sampler = ClockSampler(local_rank, dev_uuid)
    launches = 0
    barrier()
    t_wall0 = None
    for it in range(args.warmup + args.steps):
        if it == args.warmup:
            barrier()
            if rank == 0:
                sampler.start()
            t_wall0 = time.perf_counter()
        solver.restore()
        solver.sync()
        flush.zero_()                      # L2 flush between timed iterations
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()                 # ranks enter the step together (the collective would otherwise time their skew)
        solver.solve_staged()
        solver.sync()
        t = solver.timing()
        if it >= args.warmup:
            for k in phase:
                phase[k].append(t[k])
            launches += t['n_launches']
    barrier()
    wall_s = time.perf_counter() - t_wall0
    clocks = sampler.stop() if rank == 0 else None
    bindings = solver.fetch_bindings()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, bindings, solver.read_nodes())
    n_types = t['n_types']

    step_ms = float(np.sum(phase['total_ms']))
    if world > 1:
        tt = torch.tensor([step_ms], dtype=torch.float64, device='cuda')
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        step_ms = float(tt.item())
    value = P * args.steps / (step_ms / 1e3)

    # ---------------- e2e: host buffers in, host buffers out --------------------------------
    pin_recs = pinned_array(N, wire.NODE_DTYPE)           # inputs and outputs in pinned host memory
    pin_recs[:] = recs
    pin_pods = pinned_array(P, wire.POD_DTYPE)
    pin_pods[:] = pods
    pin_now = pinned_array(P, '<f8')
    pin_now[:] = now
    out = pinned_array(P, wire.BINDING_DTYPE)
    e2e_t = []
    for it in range(args.warmup + min(args.steps, 10)):
        barrier()
        t0 = time.perf_counter()
        solver.load_nodes(pin_recs)                       # H2D: cluster records
        solver.solve_batch(pin_pods, pin_now, out=out)    # H2D: pod batch; D2H: bindings
        dt = time.perf_counter() - t0
        if world > 1:
            tt = torch.tensor([dt], dtype=torch.float64, device='cuda')
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = float(tt.item())
        if it >= args.warmup:
            e2e_t.append(dt)
    e2e_value = P * len(e2e_t) / sum(e2e_t)
    if pinned is not None:
        try:
            os.sched_setaffinity(0, pinned[0])           # the CPU baseline legs use every host core again
        except Exception:
            pass
    same = all(np.array_equal(out[n], bindings[n]) for n in out.dtype.names if n != 'pad_')
    if args.stop_after_e2e and world == 1:
        print(json.dumps({'partial': True, 'value': value, 'e2e_value': e2e_value, 'e2e_ms': [round(1e3 * x, 3) for x in e2e_t],
                          'clocks': clocks, 'bindings_equal_resident_run': bool(same)}), flush=True)
        solver.close()
        return
    h2d = N * wire.NODE_DTYPE.itemsize + n_types * 176 + P * 12
    d2h = P * wire.BINDING_DTYPE.itemsize

    # side numbers on all ranks, a few solves each (every rank runs the same calls in the same order):
    #  * BASELINE config 5 (262 144 x 8 192, SR-IOV VFs + node groups): above the sharding threshold
    #  * config 4 forced onto the node-sharded path: what the exchange costs where the library chooses not to shard
    def multi_quick(r_, s_, p_, n_, min_pairs=None):
        idt = torch.zeros(128, dtype=torch.uint8, device='cuda')
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(nccl_unique_id()), dtype=torch.uint8))     # a fresh id: one per handle
        dist.broadcast(idt, 0)
        old = os.environ.pop('NHD_SHARD_MIN_PAIRS', None)
        if min_pairs is not None:
            os.environ['NHD_SHARD_MIN_PAIRS'] = str(min_pairs)          # read when the handle is created
        try:
            q = quick_value(Solver, r_, s_, p_, n_, pre_step=barrier, device=local_rank, rank=rank, world_size=world,
                            nccl_id=bytes(idt.cpu().numpy().tobytes()))
        finally:
            os.environ.pop('NHD_SHARD_MIN_PAIRS', None)
            if old is not None:
                os.environ['NHD_SHARD_MIN_PAIRS'] = old
        tt = torch.tensor([q['ms']], dtype=torch.float64, device='cuda')
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        q['ms'] = float(tt.item())
        q['value'] = len(p_) / (q['ms'] / 1e3)
        return q

    cfg5_multi = cfg4_forced = None
    if world > 1 and not args.no_extra:
        r5, s5, p5, n5 = workload.make_workload(5)
        cfg5_multi = multi_quick(r5, s5, p5, n5)
        del r5, p5
        cfg4_forced = multi_quick(recs, speed, pods, now, min_pairs=1)

    # every rank ran the identical replicated sweep: their bindings must be byte-identical (digest vs rank 0)
    ranks_agree = True
    if world > 1:
        import hashlib
        hsh = hashlib.sha256()
        for n in bindings.dtype.names:
            if n != 'pad_':
                hsh.update(np.ascontiguousarray(bindings[n]).tobytes())
        dig = torch.frombuffer(bytearray(hsh.digest()), dtype=torch.uint8).cuda()
        ref = dig.clone()
        dist.broadcast(ref, 0)
        diff = torch.tensor([0 if bool((dig == ref).all()) else 1], device='cuda')
        dist.all_reduce(diff)
        ranks_agree = int(diff.item()) == 0

    if rank != 0:
        solver.close()
        if world > 1:
            dist.destroy_process_group()
        return

    # ---------------- roofline of the dominant kernel (the sweep) ---------------------------
    peak, peak_src = measured_peaks()
    alg_bytes = P * (N * S_BYTES_PER_NODE + FIXED_BYTES_PER_DECISION)
    sweep_ms = float(np.mean(phase['sweep_ms']))
    filter_ms = float(np.mean(phase['filter_ms']))
    dominant = 'sweep_kernel' if sweep_ms >= filter_ms else 'filter_kernel'
    dom_ms = max(sweep_ms, filter_ms)
    achieved = alg_bytes / (dom_ms / 1e3) / 1e9
    traffic = traffic_at = None
    try:
        with open(os.path.join(ROOT, 'profiles', 'traffic.json')) as f:
            tj = json.load(f)
            traffic = tj.get(dominant)
            traffic_at = tj.get('captured_at')          # commit / date of the ncu capture the figure comes from
    except Exception:
        pass

    # ---------------- CPU baseline on this box's host cores (bounded sample) ------------------
    cpu = None
    parity_vs_oracle = None
    names = [n for n in bindings.dtype.names if n != 'pad_']
    if world > 1:
        # multi-rank: rank 0 checks a prefix of the stream against the oracle (the full comparison at N > 1 is
        # tests/test_gpu_multirank.py); the CPU baseline itself is reported by the N = 1 run
        from oracle import binding as ob
        ob.build()
        T, per_pod = pick_threads(ob, recs, speed, pods, now)
        ns = int(max(32, min(P, 6.0 / per_pod)))
        cb, _ = ob.solve(recs, speed, pods[:ns], now[:ns], threads=T)
        parity_vs_oracle = bool(all(np.array_equal(cb[n], bindings[:ns][n]) for n in names)) and ranks_agree
        parity_note = f'first {ns} pods vs the oracle on rank 0; all {world} ranks byte-identical: {ranks_agree}'
    if world == 1:
        from oracle import binding as ob
        ob.build()
        # (1) as the reference runs it: one thread (NHDScheduler.py:43), a short prefix of the stream
        n1 = min(args.cpu_sample_pods, 64)
        t0 = time.perf_counter()
        c1, _ = ob.solve(recs, speed, pods[:n1], now[:n1])
        dt1 = time.perf_counter() - t0
        par1 = all(np.array_equal(c1[n], bindings[:n1][n]) for n in names)
        # (2) all host threads: each pod's walk over the nodes split over them; ~15 s of the same stream
        T, per_pod = pick_threads(ob, recs, speed, pods, now, single_per_pod=dt1 / n1)
        ns = int(max(32, min(P, 15.0 / per_pod)))
        t0 = time.perf_counter()
        cb, _ = ob.solve(recs, speed, pods[:ns], now[:ns], threads=T)
        dt = time.perf_counter() - t0
        parity = all(np.array_equal(cb[n], bindings[:ns][n]) for n in names)
        parity_vs_oracle = bool(parity and par1)
        parity_note = f'first {ns} pods vs the oracle'
        cpu = {'value': ns / dt, 'unit': UNIT, 'cores': T, 'kind': 'port',
               'sample': f'first {ns} pods of the same stream on all {N} nodes, {T} host threads ({dt:.1f} s); '
                         f'bindings identical to the GPU run: {parity}',
               'single_thread': {'value': n1 / dt1, 'cores': 1,
                                 'sample': f'first {n1} pods ({dt1:.1f} s); bindings identical to the GPU run: {par1}'},
               'host_cores_available': os.cpu_count()}

    placed = int((bindings['status'] == 0).sum())
    min_pairs = shard_min_pairs()
    sharded = world > 1 and N * n_types >= min_pairs
    line = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': step_ms / args.steps, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None,
        'dtype': 'u64', 'data': 'synthetic',
        'config': {'workload': f'BASELINE config {CONFIG}: {N} nodes x {P} pods, 16 pod types (50% GPU/PCI), '
                               f'30% nodes pre-occupied, constant clock',
                   'parallelism': 'single GPU' if world == 1 else
                   f'node-sharded filter x{world} + one NCCL all-gather + replicated sweep' if sharded else
                   f'{world} replicas, no collective: {N} nodes x {n_types} pod types is below the sharding threshold '
                   f'({min_pairs} pairs) — the exchange would cost more than the shards save (extra.config4_forced_sharding)',
                   'l2': 'flushed between steps (256 MiB memset)', 'pods_placed': placed, 'pod_types': n_types},
        'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(d2h),
                'ms_per_step': 1e3 * sum(e2e_t) / len(e2e_t), 'steps': len(e2e_t),
                'includes': 'cluster records H2D + ingest, pod batch H2D, kernels, bindings D2H',
                'bindings_equal_resident_run': bool(same),
                'note': 'wall clock around host calls: moves with the host (CPU, NUMA placement of the pinned buffers, PCIe)',
                'host_cpu': host_cpu_model(),
                'cpu_affinity': f'the {pinned[1]} CPUs local to the GPU (sysfs local_cpulist)' if pinned else 'unchanged'},
        'gpu_launches': int(launches),
        'kernel_ms': {'filter': filter_ms, 'exchange': float(np.mean(phase['exchange_ms'])), 'sweep': sweep_ms,
                      'wall_per_step_incl_restore_and_flush': 1e3 * wall_s / args.steps},
        'roofline': {'bound': 'latency (1 SM, one warp: sequential first-fit chain)', 'bound_metric': 'hbm (algorithmic bytes)',
                     'kernel': dominant, 'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
                     'frac': achieved / peak, 'traffic': traffic, 'traffic_captured_at': traffic_at,
                     'peak_source': peak_src, 'frac_of_nominal_8000': achieved / 8000.0,
                     'algorithmic_bytes_per_launch': int(alg_bytes),
                     'note': 'achieved/frac use ALGORITHMIC bytes = reference-equivalent work (every eligible node '
                             'record read once per decision, SURVEY 8d), not DRAM traffic: the sweep keeps its working '
                             'set in shared memory / L2 (traffic = ncu dram bytes per launch) and is bound by the '
                             'latency of the dependent chain on one SM, not by HBM'},
        'roofline_filter': {
            'kernel': 'filter_kernel (+ fast_tables_kernel in front of it, inside the same pair of events)', 'bound': 'hbm',
            'bytes_per_launch': int(N * 128 + (n_types + 2) * N // 8 + N * 32),
            'achieved': (N * 128 + (n_types + 2) * N // 8 + N * 32) / (filter_ms / 1e3) / 1e9, 'peak': peak, 'unit': 'GB/s',
            'frac': (N * 128 + (n_types + 2) * N // 8 + N * 32) / (filter_ms / 1e3) / 1e9 / peak,
            'note': 'the one kernel that streams the node records: reads every 128-byte record once, writes the bitmaps and '
                    'the 32-byte summaries (physical = algorithmic bytes); one wave of CTAs, compute- and launch-bound at '
                    'this size, not bandwidth-bound'},
        'clocks': clocks,
    }
    # ---------------- side workloads (not the headline; a few solves each) -------------------
    extra = {}
    if world == 1 and not args.no_extra:
        try:
            r5, s5, p5, n5 = workload.make_workload(5)
            extra['config5_262144x8192_1gpu'] = quick_value(Solver, r5, s5, p5, n5, device=local_rank)
            del r5, p5
            rw, sw, pw, nw = workload.make_workload(CONFIG, wild=True)
            extra['heterogeneous_65536x4096'] = dict(quick_value(Solver, rw, sw, pw, nw, device=local_rank),
                                                     note='1-4 NICs per NUMA node at 25/40/100G in any mix: hundreds of '
                                                          'hardware classes, most outside the direct-path tables')
            del rw
            mv = now + 0.001 * np.arange(P)
            extra['moving_clock_65536x4096'] = dict(quick_value(Solver, recs, speed, pods, mv, device=local_rank),
                                                    note='per-pod clocks: the general one-warp sweep with busy-list upkeep')
        except Exception as e:
            extra['error'] = str(e)[:200]
    if cfg5_multi is not None:
        extra[f'config5_262144x8192_{world}gpu'] = cfg5_multi
    if cfg4_forced is not None:
        extra['config4_forced_sharding'] = dict(cfg4_forced, note='the headline workload with NHD_SHARD_MIN_PAIRS=1: filter shards + all-gather + unpack')
    total_ms = float(np.mean(phase['total_ms']))
    line['amdahl'] = {'filter_share': filter_ms / total_ms,
                      'limit_if_filter_were_free': total_ms / max(total_ms - filter_ms, 1e-9),
                      'note': 'only the filter shards over GPUs (and only above nhd_shard_min_pairs); the sweep (sequential first-fit) is replicated'}
    if extra:
        line['extra'] = extra
    if cpu is not None:
        pyb = python_reference_baseline(recs, speed, pods, now)
        if pyb is not None:
            cpu['python_reference'] = pyb
        line['cpu_baseline'] = cpu
    if parity_vs_oracle is not None:
        line['parity_vs_oracle'] = parity_vs_oracle
        line['parity_note'] = parity_note
    print(json.dumps(line), flush=True)
    solver.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
