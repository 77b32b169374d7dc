#!/usr/bin/env python
"""bench.py — one JSON line per run (driver contract, tier framing (4)).

Workload (N = 1): BASELINE.json configs[1] — GaussianUnknownMean inference compilation,
InferenceNetworkLSTM h=512, observe embeddings 32+32, minibatch 256 prior traces, one Adam step per batch.
A "step" = one pass of the hot path over one synthetic minibatch: encode image -> forward -> hand-written
backward -> (N>1: one NCCL all-reduce of the flat gradient arena) -> fused Adam.

  value : traces/s, whole job, batch image resident in HBM when the timed region starts (device events,
          L2 flushed between steps, max over ranks)
  e2e   : same metric through the C-ABI host-buffer call (ppb_ic_train_step_host): pinned host image ->
          H2D -> forward/backward/Adam -> D2H loss, every step
  roofline     : LSTM gate GEMM class (input projections + recurrent GEMMs, fwd+bwd), tensor-core bound
  cpu_baseline : the oracle port of the reference's _loss + backward + Adam on this box's host cores
  workloads    : the other BASELINE configurations, each with its own CPU baseline timed in the same run:
                 IS posterior (GUM, 64k particles), IC posterior (GUM and GUM-Marsaglia, LSTM h=512, 64k particles) —
                 the particles/s half of the metric — and the configs[3] shape (50 addresses, T=50, 512 traces per GPU)
                 with the roofline of its gate-GEMM class
  extra        : HBM rooflines of the scoring kernels, the gate GEMM at a saturating size

`--impl reference` times the CPU oracle port (the reference cannot travel to the GPU box) on the same config.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BATCH = 256
LSTM_DIM = 512
WORKLOAD = 'GaussianUnknownMean IC train, LSTM h=512, obs-embed 32+32, batch 256/GPU (BASELINE configs[1])'
GUM_ADDRESS = '98__forward__mu__Normal__1'
GUM_PARAMETERS = 1643583    # the reference's count for this configuration (BASELINE.md section 1)


def workload_config(n_gpus):
    """What is computed — identical on the b200 arm and on the reference arm for the same --gpus."""
    return {'workload': WORKLOAD, 'global_batch': BATCH * n_gpus, 'batch_per_gpu': BATCH, 'lstm_dim': LSTM_DIM,
            'trace_length': 1, 'observe_embeddings': 'obs0:32,obs1:32 (feed-forward, depth 2)', 'mixture_components': 10,
            'parameters': GUM_PARAMETERS, 'optimizer': 'Adam lr 1e-3', 'arithmetic': 'fp32 results (1e-4 of the reference)',
            'l2': 'GPU arm: L2 flushed between timed steps (256 MiB memset outside the timed spans); CPU arm: not applicable'}


def percentile_stats(ms):
    a = np.sort(np.asarray(ms, dtype=np.float64))
    return {'median': float(np.median(a)), 'p90': float(a[min(len(a) - 1, int(math.ceil(0.9 * len(a))) - 1)]),
            'min': float(a[0]), 'max': float(a[-1])}


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        p = json.load(open(path))
        return {'hbm_gbs': p['hbm_gbs'], 'bf16_tflops': p['bf16_tflops'],
                'bf16_tflops_sustained': p.get('bf16_tflops_sustained', p['bf16_tflops']), 'source': 'measured'}
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0, 'source': 'fallback'}


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region.  The region lasts tens of milliseconds, far
    below nvidia-smi's loop period, so NVML is polled directly every ~2 ms from a thread; `nvidia-smi -lms` is
    the fallback when the NVML binding is missing."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')
    NVML_REASONS = ((0x8, 'hw_slowdown'), (0x40, 'hw_thermal_slowdown'), (0x20, 'sw_thermal_slowdown'),
                    (0x4, 'sw_power_cap'), (0x80, 'hw_power_brake_slowdown'))

    def __init__(self, gpu_index, uuid=None):
        self.rows, self.proc, self.gpu, self.uuid = [], None, gpu_index, uuid
        self.nvml, self.handle, self.thread, self.halt = None, None, None, False
        self.sm, self.mask, self.sm_max = [], 0, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            handle = None
            if self.uuid is not None:
                try:
                    handle = pynvml.nvmlDeviceGetHandleByUUID('GPU-' + str(self.uuid))
                except Exception:
                    handle = None
            if handle is None:
                visible = os.environ.get('CUDA_VISIBLE_DEVICES', '')
                ids = [x for x in visible.split(',') if x.strip().isdigit()]
                phys = int(ids[self.gpu]) if self.gpu < len(ids) else self.gpu
                handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(handle, pynvml.NVML_CLOCK_SM))
            self.reasons_fn = getattr(pynvml, 'nvmlDeviceGetCurrentClocksEventReasons', None) or \
                pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
            self.nvml, self.handle = pynvml, handle
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '20'], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _poll(self):
        while not self.halt:
            try:
                self.sm.append(float(self.nvml.nvmlDeviceGetClockInfo(self.handle, self.nvml.NVML_CLOCK_SM)))
                self.mask |= int(self.reasons_fn(self.handle))
            except Exception:
                pass
            time.sleep(0.002)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(',')])

    def stop(self):
        if self.nvml is not None:
            self.halt = True
            self.thread.join(1.0)
            reasons = sorted(nm for bit, nm in self.NVML_REASONS if self.mask & bit)
            return {'sm_mhz': float(np.median(self.sm)) if self.sm else None, 'sm_max_mhz': self.sm_max,
                    'reasons': reasons, 'samples': len(self.sm), 'source': 'nvml, 2 ms period'}
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace('.', '').isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace('.', '').isdigit()]
        reasons = set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            if len(r) >= 9:
                for k, nm in enumerate(names):
                    if r[5 + k].lower().startswith('active'):
                        reasons.add(nm)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm), 'source': 'nvidia-smi -lms 20'}


# ---- CPU arm: the oracle port of the reference path -------------------------------------------------------
def cpu_reference_arm(steps, warmup, budget_s=20.0):
    """_loss + backward + Adam of the reference network (oracle restatement, torch CPU fp32, all host threads)
    on GUM minibatches of 256 traces (four pre-generated minibatches cycled, like the GPU arm).  Returns traces/s.
    Times `steps` steps, or fewer once `budget_s` seconds are spent (budget_s=None: exactly `steps`)."""
    from oracle import network as onet
    from oracle import params as oparams
    from pyprob_b200 import synthetic
    threads = os.cpu_count() or 1
    rng = np.random.default_rng(0)
    params = oparams.random_params([('obs0', 1, 32, 2), ('obs1', 1, 32, 2)], [(GUM_ADDRESS, 'Normal', 0)],
                                   lstm_dim=LSTM_DIM, K=10, seed=0)
    plist = {k: v.requires_grad_(True) for k, v in params.items()}
    opt = torch.optim.Adam(list(plist.values()), lr=1e-3)
    batches = []
    for _ in range(4):
        b = synthetic.gum_batch(rng, BATCH)
        batches.append([{k: (torch.from_numpy(v) if isinstance(v, np.ndarray) else v) for k, v in sb.items()}
                        for sb in b.subs])
    it = [0]

    def one_step():
        subs = batches[it[0] % 4]
        it[0] += 1
        opt.zero_grad()
        loss, _ = onet.loss(plist, subs, ['obs0', 'obs1'], [1, 1], 10)
        loss.backward()
        opt.step()
        return float(loss.detach())
    # "all the host threads it can use": pick the fastest intra-op thread count for this (small-GEMM) workload
    best = None
    for nt in sorted(set([1, 2, 4, 8, 16, 32, 64, threads])):
        if nt > threads:
            continue
        torch.set_num_threads(nt)
        one_step()
        dt = float('inf')
        for _ in range(3):   # best of three: a single step is too noisy to choose on
            t0 = time.perf_counter()
            one_step()
            dt = min(dt, time.perf_counter() - t0)
        if best is None or dt < best[1]:
            best = (nt, dt)
    threads = best[0]
    torch.set_num_threads(threads)
    tw, nw = time.perf_counter(), 0
    while nw < max(warmup, 1) or time.perf_counter() - tw < 1.0:   # thread pool and allocator settle for about a second
        one_step()
        nw += 1
    t0 = time.perf_counter()
    done = 0
    for _ in range(steps):
        one_step()
        done += 1
        if budget_s is not None and time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return {'value': done * BATCH / dt, 'unit': 'traces/s', 'cores': threads, 'kind': 'port',
            'sample': '{} steps of _loss+backward+Adam on {}-trace GUM minibatches (oracle/network.py, torch CPU fp32, '
                      '{} of {} host threads — the fastest setting for this small-GEMM step), {:.1f} s'.format(
                          done, BATCH, threads, os.cpu_count(), dt)}, dt / done


def dump_outputs(out_dir, tensors):
    """Write each tensor as out_dir/<name>.npy, float32."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in tensors.items():
        np.save(os.path.join(out_dir, name + '.npy'), t.detach().float().cpu().numpy())
    log('outputs of the last timed step written to {}'.format(out_dir))


def log(msg):
    """Progress on stderr (stdout carries exactly one JSON line)."""
    sys.stderr.write('[bench {:7.1f}s] {}\n'.format(time.perf_counter() - _T0, msg))
    sys.stderr.flush()


_T0 = time.perf_counter()


def main():
    import faulthandler
    faulthandler.dump_traceback_later(300, repeat=True, file=sys.stderr)   # a stuck phase shows where it is stuck
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--precision', type=int, default=0)
    ap.add_argument('--no-extra', action='store_true')
    ap.add_argument('--no-graph', action='store_true')
    ap.add_argument('--cpu-budget', type=float, default=15.0, help='seconds of CPU work for the cpu_baseline sample')
    ap.add_argument('--nccl-allreduce', action='store_true',
                    help='N>1: NCCL all-reduce + local Adam instead of the fused peer-memory optimiser step')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last one computed (loss, updated parameters, gradient, '
                         'Adam moments; rank 0) as DIR/<name>.npy in float32, to compare two builds output for output. '
                         'The inputs are seeded; the backward pass accumulates with atomics, so two runs agree to float '
                         'rounding, not bit for bit')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs writes the outputs of the b200 arm')
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    warmup = max(args.warmup, 3)

    if args.impl == 'reference':
        if rank != 0:
            return
        cb, s_per_step = cpu_reference_arm(args.steps, warmup, budget_s=None)
        print(json.dumps({'impl': 'reference', 'metric': 'ic_train_traces_per_sec', 'value': cb['value'],
                          'unit': 'traces/s', 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': warmup,
                          'ms_per_step': s_per_step * 1e3, 'higher_is_better': True, 'scaling': 'weak',
                          'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
                          'config': workload_config(args.gpus),
                          'impl_config': {'note': 'CPU oracle port of the reference path (the Python reference cannot travel '
                                          'to the GPU box); rank 0 only, one 256-trace minibatch per step whatever --gpus'},
                          'cpu_baseline': cb,
                          'e2e': {'value': cb['value'], 'unit': 'traces/s', 'h2d_bytes_per_step': 0,
                                  'd2h_bytes_per_step': 0}}))
        return

    import torch.distributed as dist
    from pyprob_b200 import _lib, synthetic
    from pyprob_b200._lib import call, ptr
    from pyprob_b200.util import Optimizer
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        # keep NCCL's debug log (if NCCL_DEBUG asks for one) off stdout; the JSON line is the LAST line of stdout either way
        # (the one-line version banner of NCCL_DEBUG=VERSION is printed before it)
        os.environ.setdefault('NCCL_DEBUG_FILE', '/dev/stderr')
        dist.init_process_group('nccl', device_id=dev)
    rng = np.random.default_rng(1234 + rank)
    net = synthetic.gum_network(lstm_dim=LSTM_DIM, precision=args.precision, seed=0)
    net._optimizer_type, net._learning_rate_init, net._weight_decay = Optimizer.ADAM, 1e-3, 0.0
    net._create_optimizer()
    net._sync_native()
    if world > 1:
        dist.broadcast(net._arena.data, 0)
    nparams = net._arena.numel()
    peer = None
    if world > 1 and not args.nccl_allreduce:
        # data-parallel step = ONE kernel over NVLink peer memory: reduce-scatter + Adam on the owned slice +
        # all-gather of the parameters (ppb_dp_adam_step); the arena and the gradient live in the peer block
        from pyprob_b200 import parallel
        peer = parallel.PeerAdam(nparams, dev)
        peer.params.copy_(net._arena.data)
        net._arena_store = peer.params
        net._arena = torch.nn.Parameter(peer.params)
        grad = peer.grad[:nparams]
    else:
        grad = torch.zeros(nparams, device=dev)
    net._arena.grad = grad
    batches = [synthetic.gum_batch(rng, BATCH) for _ in range(4)]
    encs = [b.encode(net) for b in batches]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    stream = torch.cuda.current_stream()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident step -----------------------------------------------------------------------------
    import ctypes as C
    from pyprob_b200.network import BatchStruct
    hyper = torch.tensor([1e-3, 0.9, 0.999, 1e-8, 0.0, 1.0 / world], dtype=torch.float32, device=dev)
    adam_state = torch.zeros(4, dtype=torch.int32, device=dev)
    # the loss rides in the gradient tail so that the fused collective sums it with the gradient
    loss = peer.grad[nparams:nparams + 1].view(()) if peer is not None else torch.empty((), device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    # all batches of the workload share one structure: one "current batch" image in HBM is refreshed (device to
    # device) from the resident batches, so the index/problem lists are built and uploaded once
    hosts = [torch.from_numpy(enc.pack().copy()).pin_memory() for enc in encs]
    resident = [h.to(dev) for h in hosts]
    cur = torch.empty_like(resident[0])
    bs = BatchStruct()
    call('ppb_batch_from_image', hosts[0].data_ptr(), cur.data_ptr(), hosts[0].numel(), C.byref(bs))
    need = net._ensure_workspace(encs[0])

    def device_step(i):
        cur.copy_(resident[i % 4], non_blocking=True)
        grad.zero_()
        call('ppb_ic_loss_forward', net._handle, ptr(net._arena.data), C.byref(bs), ptr(net._workspace), need,
             args.precision, ptr(loss), ptr(status), None, 1, torch.cuda.current_stream().cuda_stream)
        call('ppb_ic_loss_backward', net._handle, ptr(net._arena.data), ptr(grad), C.byref(bs), ptr(net._workspace), need,
             args.precision, 1.0, torch.cuda.current_stream().cuda_stream)
        if peer is not None:
            peer.step(net._exp_avg, net._exp_avg_sq, hyper, adam_state, torch.cuda.current_stream().cuda_stream)
            return
        if world > 1:
            dist.all_reduce(grad)
        call('ppb_adam_step_dev', ptr(net._arena.data), ptr(grad), ptr(net._exp_avg), ptr(net._exp_avg_sq), nparams,
             ptr(hyper), ptr(adam_state), torch.cuda.current_stream().cuda_stream)

    log('network built, {} parameters'.format(nparams))
    for i in range(warmup):
        device_step(i)
    barrier()
    log('eager warm-up done')
    use_graph = not args.no_graph
    graphs = []
    if use_graph:  # the whole step (incl. the NCCL all-reduce for N > 1) replays from one CUDA graph per resident batch
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for i in range(4):
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=side):
                    device_step(i)
                graphs.append(g)
        torch.cuda.current_stream().wait_stream(side)
        for i in range(warmup):
            graphs[i % 4].replay()
    barrier()

    def run_step(i):
        if use_graph:
            graphs[i % 4].replay()
        else:
            device_step(i)
    log('graphs captured' if use_graph else 'no graph')
    sampler = ClockSampler(local_rank, getattr(torch.cuda.get_device_properties(dev), 'uuid', None))
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    if peer is not None:
        peer.phase_totals_us(reset=True)
    for i in range(args.steps):
        flush.zero_()                      # L2 flush between timed iterations (outside the timed spans)
        if peer is not None:
            # every rank starts the timed step at the same moment: the flush (not part of the step) must not leak its
            # cross-rank skew into the span through the step's first cross-rank barrier
            peer.rendezvous(stream.cuda_stream)
        ev[i][0].record(stream)
        run_step(i)
        ev[i][1].record(stream)
    barrier()
    if args.dump_outputs and rank == 0:
        # taken before the launch count below runs one more step on the same parameters
        dump_outputs(args.dump_outputs, {'loss': loss, 'parameters': net._arena.data, 'gradient': grad,
                                         'adam_exp_avg': net._exp_avg, 'adam_exp_avg_sq': net._exp_avg_sq})
    # graph replays bypass the library's host-side launch counter: count the launches of one eager step
    l0 = _lib.call('ppb_launch_count')
    device_step(0)
    torch.cuda.synchronize()
    launches = (_lib.call('ppb_launch_count') - l0) * args.steps
    step_ms = [a.elapsed_time(b) for a, b in ev]
    dev_ms = sum(step_ms)
    dp_phases = peer.phase_totals_us() if peer is not None else None
    t = torch.tensor([dev_ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms = float(t.item())
    value = args.steps * BATCH * world / (dev_ms * 1e-3)

    log('device-resident: {:.4f} ms/step'.format(dev_ms / args.steps))
    # ---- e2e: C-ABI host-buffer call, H2D + D2H inside the timed region --------------------------------------
    loss_host = torch.zeros(1).pin_memory()
    status_host = torch.zeros(1, dtype=torch.int32).pin_memory()
    e2e_img_dev = cur
    ws_bytes = net._workspace.numel()
    step_no = [int(adam_state.view(torch.int64)[0].item())]

    def e2e_step(i):
        host = hosts[i % 4]
        if world == 1:
            step_no[0] += 1
            call('ppb_ic_train_step_host', net._handle, ptr(net._arena.data), ptr(grad), ptr(net._exp_avg),
                 ptr(net._exp_avg_sq), nparams, host.data_ptr(), host.numel(), ptr(e2e_img_dev), ptr(net._workspace),
                 ws_bytes, args.precision, 1e-3, 0.9, 0.999, 1e-8, 0.0, step_no[0], loss_host.data_ptr(),
                 status_host.data_ptr(), stream.cuda_stream)
        else:
            resident[i % 4].copy_(host, non_blocking=True)   # host -> device copy of this step's batch image
            device_step(i)
            loss_host.copy_(loss.view(1), non_blocking=True)
            torch.cuda.current_stream().synchronize()
    for i in range(warmup):
        e2e_step(i)
    barrier()
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(args.steps):
        e2e_step(i)
    e1.record(stream)
    wall_ms = (time.perf_counter() - t0) * 1e3   # every e2e step ends with a stream synchronize
    barrier()
    e2e_ms = max(e0.elapsed_time(e1), wall_ms)   # what the caller waits for: the slower of device and host clocks
    t = torch.tensor([e2e_ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item())
    e2e_value = args.steps * BATCH * world / (e2e_ms * 1e-3)
    clocks = sampler.stop() if rank == 0 else None
    if peer is not None and peer.timed_out():
        raise RuntimeError('fused data-parallel step: a cross-rank barrier timed out; the measurement is void')

    log('e2e: {:.4f} ms/step'.format(e2e_ms / args.steps))
    # ---- roofline of the gate-GEMM class: per-launch durations from CUDA events inside the step ---------------
    peaks = measured_peaks()
    roof = None
    # every rank runs the profiled steps (the step contains the collective); only rank 0 records and reports
    if rank == 0:
        call('ppb_prof_enable', 1)
    prof_steps = min(args.steps, 20)
    for i in range(prof_steps):
        flush.zero_()
        device_step(i)
    torch.cuda.synchronize()
    if rank == 0:
        ms, n, fl = C.c_double(), C.c_int64(), C.c_double()
        call('ppb_prof_read', C.byref(ms), C.byref(n), C.byref(fl))
        call('ppb_prof_enable', 0)
        # the gate-GEMM launches are timed one by one with CUDA events: the burst figure is the matching denominator
        tf32_peak = peaks['bf16_tflops'] / 2.0   # tf32 dense = 1/2 of the measured bf16 GEMM peak
        achieved = fl.value / (ms.value * 1e-3) / 1e12 if ms.value > 0 else 0.0
        issue = 3.0 if args.precision == 0 else 1.0
        roof = {'bound': 'tensor', 'kernel': 'LSTM gate GEMM class (P_obs/P_step/recurrent + their dX/dW)',
                'achieved': achieved, 'peak': tf32_peak, 'unit': 'TFLOP/s', 'frac': achieved / tf32_peak,
                'frac_issued_mma': achieved * issue / tf32_peak,
                'traffic': committed_traffic('gate_gemm_configs1'), 'launches': n.value,
                'avg_launch_us': ms.value * 1e3 / max(n.value, 1),
                'flops_per_step': fl.value / max(prof_steps, 1),
                'peak_source': '{} bf16_tflops (burst) / 2 = tf32 dense'.format(peaks['source']),
                'note': 'achieved counts each product once; in 3xTF32 mode the tensor pipe issues 3 MMAs per product '
                        '(frac_issued_mma). T = 1 at configs[1]: three 67-MFLOP GEMMs per step, launch-bound by construction; '
                        'see workloads.ic_train_synthetic50_b512.roofline for the T = 50 recurrence'}

    extra = {}
    workloads = {}
    cpu_baseline = None
    if rank == 0 and world == 1:
        log('cpu baseline ...')
        cpu_baseline, _ = cpu_reference_arm(10 ** 6, 2, budget_s=args.cpu_budget)
        log('cpu baseline: {:.0f} traces/s'.format(cpu_baseline['value']))
        if not args.no_extra:
            # secondary workloads: a failure here must not cost the headline line
            for key, fn in (('is_posterior_gum_n65536', lambda: posterior_is_workload(dev)),
                            ('ic_posterior_gum_n65536', lambda: posterior_ic_gum_workload(dev)),
                            ('ic_posterior_marsaglia_n65536', lambda: posterior_ic_marsaglia_workload(dev)),
                            ('ic_train_synthetic50_b512', lambda: synthetic50_workload(dev, peaks))):
                try:
                    log('workload ' + key)
                    workloads[key] = fn()
                except Exception as exc:   # noqa: BLE001 - reported in the JSON line
                    workloads[key] = {'error': '{}: {}'.format(type(exc).__name__, exc)}
            for key, fn in (('scoring_hbm_roofline', lambda: scoring_rooflines(dev, peaks)),
                            ('gate_gemm_saturating_4096x2048x512', lambda: gate_gemm_saturating(dev, peaks))):
                try:
                    log('extra ' + key)
                    extra[key] = fn()
                except Exception as exc:   # noqa: BLE001
                    extra[key + '_error'] = '{}: {}'.format(type(exc).__name__, exc)
            extra['hbm_peak_gbs'] = peaks['hbm_gbs']
    if rank == 0:
        out = {'metric': 'ic_train_traces_per_sec', 'value': value, 'unit': 'traces/s', 'n_gpus': world,
               'steps': args.steps, 'warmup': warmup, 'ms_per_step': dev_ms / args.steps, 'higher_is_better': True,
               'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
               'config': workload_config(world),
               'impl_config': {'arena_floats': nparams, 'parallelism': 'dp{}'.format(world),
                               'collective': None if world == 1 else (
                                   'fused reduce-scatter+Adam+all-gather over NVLink peer memory (ppb_dp_adam_step)'
                                   if peer is not None else 'nccl all-reduce'),
                               'precision': ['3xTF32', 'TF32', 'fp32-simt'][args.precision],
                               'l2': 'flushed between timed steps (256 MiB memset outside the timed spans'
                                     + ('; stream-ordered cross-rank rendezvous between flush and span' if peer is not None
                                        else '') + ')',
                               'cuda_graph': bool(use_graph)},
               'ms_per_step_stats_rank0': percentile_stats(step_ms),
               'e2e': {'value': e2e_value, 'unit': 'traces/s', 'h2d_bytes_per_step': int(hosts[0].numel()),
                       'd2h_bytes_per_step': 8, 'ms_per_step': e2e_ms / args.steps},
               'gpu_launches': int(launches), 'clocks': clocks, 'roofline': roof, 'cpu_baseline': cpu_baseline,
               'workloads': workloads, 'extra': extra}
        if dp_phases is not None:
            out['dp_step_phases_us_rank0'] = dp_phases
        print(json.dumps(out))
        sys.stdout.flush()
    if world > 1:
        # captured graphs keep NCCL work objects alive: drop them, drain, and leave without tearing the
        # communicator down (destroy_process_group can block on graph-owned resources)
        graphs.clear()
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        os._exit(0)


def scoring_rooflines(dev, peaks):
    """HBM roofline of the scoring / sampling / normalisation kernels at a saturating size (2^24 particles,
    per-particle parameters: every operand array is 64 MiB, the working set is far beyond the 126 MB L2).
    achieved = algorithmic bytes per particle (SURVEY 8d) x N / CUDA-event time."""
    from pyprob_b200 import ops
    n, K, C = 1 << 24, 10, 8
    g = torch.Generator(device=dev).manual_seed(0)
    v = torch.randn(n, device=dev, generator=g)
    mu = torch.randn(n, device=dev, generator=g)
    sd = torch.rand(n, device=dev, generator=g) + 0.5
    lo = mu - 2.0
    hi = mu + 2.0
    rate = sd * 4
    cnt = torch.poisson(rate, generator=g)
    probs = torch.rand(n, C, device=dev, generator=g) + 0.01
    cat = torch.randint(0, C, (n,), device=dev, generator=g).float()
    m = torch.randn(n, K, device=dev, generator=g)
    s = torch.rand(n, K, device=dev, generator=g) + 0.1
    p = torch.rand(n, K, device=dev, generator=g) + 0.01
    lw = torch.randn(n, device=dev, generator=g) * 5 - 40
    out = torch.empty(n, device=dev)
    cases = [
        ('normal_log_prob', 16, lambda: ops.normal_log_prob(v, mu, sd, lp_out=out)),
        ('uniform_log_prob', 16, lambda: ops.uniform_log_prob(v, lo, hi, lp_out=out)),
        ('poisson_log_prob', 12, lambda: ops.poisson_log_prob(cnt, rate, lp_out=out)),
        ('categorical_log_prob', 4 * C + 8, lambda: ops.categorical_log_prob(cat, probs, lp_out=out)),
        ('mixture_normal_log_prob', (3 * K + 2) * 4, lambda: ops.mixture_normal_log_prob(v, m, s, p, lp_out=out)),
        ('mixture_truncated_normal_log_prob', (3 * K + 4) * 4,
         lambda: ops.mixture_truncated_normal_log_prob(v, m, s, p, lo, hi, lp_out=out)),
        ('normal_sample', 12, lambda: ops.normal_sample(mu, sd, n, 1, 2)),
        ('weights_finalize', 16, lambda: ops.weights_finalize(lw)),
    ]
    res = []
    for name, bytes_per, fn in cases:
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        reps = 10
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        gbs = bytes_per * n / (ms * 1e-3) / 1e9
        res.append({'kernel': name, 'bytes_per_particle': bytes_per, 'particles': n, 'ms': ms, 'achieved_gbs': gbs,
                    'frac_of_hbm': gbs / peaks['hbm_gbs']})
    return res


def gate_gemm_saturating(dev, peaks):
    """The LSTM gate GEMM shape at a saturating batch (one recurrent step of 4096 traces: [4096,512] x [512,2048]^T)
    through the production tcgen05 kernel: achieved tensor throughput vs the tf32 roofline."""
    from pyprob_b200 import _lib
    from pyprob_b200._lib import call, ptr, stream
    M, N, K = 4096, 2048, 512
    a = torch.randn(M, K, device=dev)
    b = torch.randn(N, K, device=dev)
    c = torch.empty(M, N, device=dev)

    def pack(x):
        nfl = _lib.call('ppb_packed_floats', x.shape[0], x.shape[1])
        hi = torch.empty(nfl, device=dev)
        lo = torch.empty(nfl, device=dev)
        call('ppb_pack_tf32', ptr(x), x.shape[0], x.shape[1], x.stride(0), ptr(hi), ptr(lo), stream())
        return hi, lo
    ah, al = pack(a)
    bh, bl = pack(b)
    out = {}
    for prec, name in ((0, '3xTF32'), (1, 'TF32')):
        for _ in range(5):
            call('ppb_gemm_packed', ptr(ah), ptr(al), ptr(bh), ptr(bl), ptr(c), M, N, K, N, None, 0, prec, stream())
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        reps = 20
        for _ in range(reps):
            call('ppb_gemm_packed', ptr(ah), ptr(al), ptr(bh), ptr(bl), ptr(c), M, N, K, N, None, 0, prec, stream())
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        useful = 2.0 * M * N * K / (ms * 1e-3) / 1e12
        issued = useful * (3 if prec == 0 else 1)
        peak = peaks['bf16_tflops'] / 2.0
        out[name] = {'ms': ms, 'useful_tflops': useful, 'issued_tf32_tflops': issued, 'tf32_peak': peak,
                     'frac_issued': issued / peak}
    return out


def committed_traffic(key):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of a kernel class from the committed
    `ncu --set full` capture (profiles/ncu_traffic.json, written by scripts/summarise_ncu.py), or None."""
    path = os.path.join(ROOT, 'profiles', 'ncu_traffic.json')
    if not os.path.exists(path):
        return None
    try:
        return json.load(open(path)).get(key, {}).get('dram_bytes_per_launch')
    except Exception:   # noqa: BLE001
        return None


def _timed_cpu(fn, n_first, budget_s):
    """Run fn(n) on growing particle counts until ~budget_s of CPU time is spent; returns (particles, seconds)."""
    fn(max(n_first // 8, 4))   # warm-up
    done, spent, n = 0, 0.0, n_first
    while spent < budget_s:
        t0 = time.perf_counter()
        fn(n)
        dt = time.perf_counter() - t0
        done += n
        spent += dt
        n = int(min(max(n * (0.5 * budget_s / max(dt, 1e-3)), n), 8 * n))
    return done, spent


def _gum_model():
    import pyprob_b200 as pyprob
    from pyprob_b200 import Model
    from pyprob_b200.distributions import Normal

    class GUM(Model):
        def forward(self):
            mu = pyprob.sample(Normal(1, math.sqrt(5)))
            lik = Normal(mu, math.sqrt(2))
            pyprob.observe(lik, name='obs0')
            pyprob.observe(lik, name='obs1')
            return mu
    return GUM()


def _time_posterior(model, n, engine, reps):
    """Wall-clock seconds of `reps` posterior_results calls, one at a time (each ends with a device->host read of the ESS).
    Returns (particles/s at the median call time, ess, per-call stats in ms incl. mean and max)."""
    obs = {'obs0': 8, 'obs1': 9}
    for _ in range(2):
        model.posterior_results(n, engine, observe=obs)
    torch.cuda.synchronize()
    ess = 0.0
    ms = []
    for _ in range(reps):
        t0 = time.perf_counter()
        post = model.posterior_results(n, engine, observe=obs)
        ess = float(post.effective_sample_size)   # device->host read of the result
        ms.append((time.perf_counter() - t0) * 1e3)
    st = percentile_stats(ms)
    st['mean'] = float(sum(ms) / len(ms))
    # headline = particles per MEDIAN call: one call in twenty occasionally stalls on the host for 5-35 ms (allocator / GC;
    # the device is idle meanwhile), which would otherwise decide the number; mean and max are reported next to it
    return n / (st['median'] * 1e-3), ess, st


def _cpu_entry(done, spent, what):
    return {'value': done / spent, 'unit': 'particles/s', 'cores': 1, 'kind': 'port',
            'sample': '{} particles, {:.1f} s: {} (oracle/posterior.py — one particle at a time like pyprob/model.py:59-60, '
                      'without the reference\'s address extraction and Trace objects, i.e. faster than the reference)'.format(
                          done, spent, what)}


def posterior_is_workload(dev, budget_s=3.0):
    """BASELINE configs[0] at north_star's size: GaussianUnknownMean, IMPORTANCE_SAMPLING from the prior, 64k particles
    through Model.posterior_results (sample + 2 observe scores + fp64 weight normalisation + ESS read back)."""
    import pyprob_b200 as pyprob
    from oracle import posterior as opost
    from pyprob_b200 import InferenceEngine
    pyprob.seed(1)
    pyprob.set_verbosity(0)
    m = _gum_model()
    value, ess, stats = _time_posterior(m, 65536, InferenceEngine.IMPORTANCE_SAMPLING, 20)
    big, _, _ = _time_posterior(m, 1 << 24, InferenceEngine.IMPORTANCE_SAMPLING, 3)
    done, spent = _timed_cpu(lambda n: opost.gum_is(n), 2000, budget_s)
    cb = _cpu_entry(done, spent, 'prior draw + two Normal log_probs + float sum per particle')
    return {'metric': 'is_posterior_particles_per_sec', 'value': value, 'unit': 'particles/s', 'particles': 65536,
            'ess': ess, 'ms_per_call': stats, 'value_at_16M_particles': big, 'cpu_baseline': cb, 'ratio_to_cpu_baseline': value / cb['value'],
            'config': 'GaussianUnknownMean, observe obs0=8 obs1=9, Model.posterior_results (BASELINE configs[0] at 64k)'}


def posterior_ic_gum_workload(dev, budget_s=4.0):
    """north_star's posterior case: GaussianUnknownMean, IMPORTANCE_SAMPLING_WITH_INFERENCE_NETWORK (LSTM h=512), 64k."""
    import contextlib
    import io
    import pyprob_b200 as pyprob
    from oracle import posterior as opost
    from pyprob_b200 import InferenceEngine, InferenceNetwork
    pyprob.seed(2)
    pyprob.set_verbosity(0)
    m = _gum_model()
    with contextlib.redirect_stdout(io.StringIO()):
        m.learn_inference_network(num_traces=10 * 256, batch_size=256, inference_network=InferenceNetwork.LSTM,
                                  lstm_dim=512, observe_embeddings={'obs0': {'dim': 32}, 'obs1': {'dim': 32}})
    value, ess, stats = _time_posterior(m, 65536, InferenceEngine.IMPORTANCE_SAMPLING_WITH_INFERENCE_NETWORK, 20)
    net = m._inference_network
    P = {k: v.cpu() for k, v in net.reference_state_dict().items()}
    address = next(iter(net._addresses))
    torch.set_num_threads(1)
    done, spent = _timed_cpu(lambda n: opost.gum_ic(n, P, address), 100, budget_s)
    cb = _cpu_entry(done, spent, 'observe embedding once, then per particle one LSTM step (h=512) + mixture proposal '
                                 'draw + log p - log q + two observe scores')
    return {'metric': 'ic_posterior_particles_per_sec', 'value': value, 'unit': 'particles/s', 'particles': 65536,
            'ess': ess, 'ms_per_call': stats, 'cpu_baseline': cb, 'ratio_to_cpu_baseline': value / cb['value'],
            'config': 'GaussianUnknownMean, LSTM h=512 proposal network (same weights on both sides), 64k particles'}


def posterior_ic_marsaglia_workload(dev, budget_s=5.0):
    """BASELINE configs[2]: GaussianUnknownMeanMarsaglia (stochastic control flow), IC posterior, 64k particles through
    Model.posterior_results (lock-step while_loop; LSTM h=512).  Throughput does not depend on how well the proposals are
    trained, so the network is only trained long enough to create its layers."""
    import contextlib
    import io
    import re
    import pyprob_b200 as pyprob
    from oracle import posterior as opost
    from pyprob_b200 import InferenceEngine, InferenceNetwork, Model
    from pyprob_b200.distributions import Normal, Uniform

    class Marsaglia(Model):
        def forward(self):
            def body(s):
                x = pyprob.sample(Uniform(-1, 1))
                y = pyprob.sample(Uniform(-1, 1))
                return {'x': x, 'y': y, 's': x * x + y * y}
            st = pyprob.while_loop(lambda s: s['s'] >= 1, body, {'x': 0.0, 'y': 0.0, 's': 2.0})
            mu = 1 + math.sqrt(5) * (st['x'] * torch.sqrt(-2 * torch.log(st['s']) / st['s']))
            lik = Normal(mu, math.sqrt(2))
            pyprob.observe(lik, name='obs0')
            pyprob.observe(lik, name='obs1')
            return mu
    pyprob.seed(3)
    pyprob.set_verbosity(0)
    m = Marsaglia()
    import warnings
    with contextlib.redirect_stdout(io.StringIO()), warnings.catch_warnings():
        warnings.simplefilter('ignore')
        m.learn_inference_network(num_traces=20 * 1024, batch_size=1024, inference_network=InferenceNetwork.LSTM,
                                  lstm_dim=512, observe_embeddings={'obs0': {'dim': 32}, 'obs1': {'dim': 32}})
        value, ess, stats = _time_posterior(m, 65536, InferenceEngine.IMPORTANCE_SAMPLING_WITH_INFERENCE_NETWORK, 10)
    net = m._inference_network
    P = {k: v.cpu() for k, v in net.reference_state_dict().items()}
    table = {}
    for a in net._addresses:
        mt = re.search(r'__([xy])__Uniform__(\d+)$', a)
        if mt:
            table[(mt.group(1), int(mt.group(2)))] = a
    torch.set_num_threads(1)
    done, spent = _timed_cpu(lambda n: opost.marsaglia_ic(n, P, lambda var, k: table.get((var, k))), 50, budget_s)
    cb = _cpu_entry(done, spent, 'rejection loop, per site one LSTM step (h=512) + truncated-normal-mixture proposal '
                                 'draw + log p - log q')
    return {'metric': 'ic_posterior_particles_per_sec', 'value': value, 'unit': 'particles/s', 'particles': 65536,
            'ess': ess, 'ms_per_call': stats, 'addresses': len(net._addresses), 'cpu_baseline': cb, 'ratio_to_cpu_baseline': value / cb['value'],
            'config': 'GaussianUnknownMeanMarsaglia, LSTM h=512 (same weights on both sides), 64k particles (BASELINE configs[2])'}


def synthetic50_workload(dev, peaks, B=512, T=50, cpu_budget_s=8.0):
    """BASELINE configs[3] shape on one GPU: 50-address Normal/Categorical(4) model, LSTM h=512, observe FF dim 256, 512 traces
    per GPU (the per-GPU share of the 4096-trace global batch on 8 GPUs): device-resident training step, the roofline of
    its LSTM gate-GEMM class (recurrent GEMMs forward, their dX and dW backward, P_obs), and the oracle port on the CPU."""
    import ctypes as C
    from oracle import network as onet
    from oracle import params as oparams
    from pyprob_b200 import synthetic
    from pyprob_b200._lib import call, ptr
    from pyprob_b200.network import BatchStruct
    from pyprob_b200.util import Optimizer
    rng = np.random.default_rng(5)
    net = synthetic.synthetic50_network(precision=0, T=T)
    net._optimizer_type, net._learning_rate_init, net._weight_decay = Optimizer.ADAM, 1e-3, 0.0
    net._create_optimizer()
    net._sync_native()
    batch = synthetic.synthetic50_batch(rng, B, T=T)
    enc = batch.encode(net)
    grad = torch.zeros_like(net._arena.data)
    img = torch.from_numpy(enc.pack().copy()).pin_memory()
    dimg = img.to(dev)
    bs = BatchStruct()
    call('ppb_batch_from_image', img.data_ptr(), dimg.data_ptr(), img.numel(), C.byref(bs))
    need = net._ensure_workspace(enc)
    loss = torch.empty((), device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    hyper = torch.tensor([1e-3, 0.9, 0.999, 1e-8, 0.0, 1.0], dtype=torch.float32, device=dev)
    state = torch.zeros(4, dtype=torch.int32, device=dev)

    def step():
        st = torch.cuda.current_stream().cuda_stream
        grad.zero_()
        call('ppb_ic_loss_forward', net._handle, ptr(net._arena.data), C.byref(bs), ptr(net._workspace), need, 0, ptr(loss),
             ptr(status), None, 1, st)
        call('ppb_ic_loss_backward', net._handle, ptr(net._arena.data), ptr(grad), C.byref(bs), ptr(net._workspace), need, 0,
             1.0, st)
        call('ppb_adam_step_dev', ptr(net._arena.data), ptr(grad), ptr(net._exp_avg), ptr(net._exp_avg_sq),
             net._arena.numel(), ptr(hyper), ptr(state), st)
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    reps = 10
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in evs:
        a.record()
        step()
        b.record()
    torch.cuda.synchronize()
    ms = float(np.mean([a.elapsed_time(b) for a, b in evs]))
    # roofline of the gate-GEMM class: per-launch CUDA events inside the step
    call('ppb_prof_enable', 1)
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    pms, pn, pfl = C.c_double(), C.c_int64(), C.c_double()
    call('ppb_prof_read', C.byref(pms), C.byref(pn), C.byref(pfl))
    call('ppb_prof_enable', 0)
    tf32_peak = peaks['bf16_tflops_sustained'] / 2.0     # kernels timed inside a multi-millisecond step
    achieved = pfl.value / (pms.value * 1e-3) / 1e12 if pms.value > 0 else 0.0
    roof = {'bound': 'tensor', 'kernel': 'LSTM gate GEMM class at T=50 (recurrent h W_hh^T per step, BPTT dX, dW_hh, P_obs)',
            'achieved': achieved, 'peak': tf32_peak, 'unit': 'TFLOP/s', 'frac': achieved / tf32_peak,
            'frac_issued_mma': 3.0 * achieved / tf32_peak, 'traffic': committed_traffic('gate_gemm_synthetic50'),
            'launches_per_step': pn.value / 3, 'gate_gemm_ms_per_step': pms.value / 3,
            'flops_per_step': pfl.value / 3,
            'peak_source': '{} bf16_tflops_sustained / 2 = tf32 dense'.format(peaks['source'])}
    # CPU: the oracle port on minibatches of the same model (256 traces per step keeps the sample bounded)
    Bc = 256
    P = oparams.random_params([('obs', 1, 256, 2)], synthetic.synthetic50_addresses(T), lstm_dim=512, K=10, seed=0)
    plist = {k: v.requires_grad_(True) for k, v in P.items()}
    opt = torch.optim.Adam(list(plist.values()), lr=1e-3)
    sb = synthetic.synthetic50_batch(np.random.default_rng(6), Bc, T=T).subs
    subs = [{k: (torch.from_numpy(v) if isinstance(v, np.ndarray) else v) for k, v in x.items()} for x in sb]
    def cpu_step():
        opt.zero_grad()
        l, _ = onet.loss(plist, subs, ['obs'], [1], 10)
        l.backward()
        opt.step()
    # a step is thousands of small torch ops: more threads than the GEMMs can feed only add synchronisation cost
    ncpu = os.cpu_count() or 1
    best = None
    for nt in sorted(set(min(ncpu, x) for x in (8, 16, 32, 64))):
        torch.set_num_threads(nt)
        t0 = time.perf_counter()
        cpu_step()
        dt = time.perf_counter() - t0
        if best is None or dt < best[1]:
            best = (nt, dt)
        if dt > 20.0:
            break
    torch.set_num_threads(best[0])
    t0 = time.perf_counter()
    done = 0
    while done < 1 or time.perf_counter() - t0 < cpu_budget_s:
        cpu_step()
        done += 1
    dt = time.perf_counter() - t0
    cb = {'value': done * Bc / dt, 'unit': 'traces/s', 'cores': best[0], 'kind': 'port',
          'sample': '{} steps of _loss+backward+Adam on {}-trace minibatches of the 50-address model (oracle/network.py, torch '
                    'CPU fp32, {} of {} host threads — the fastest of 8/16/32/64), {:.1f} s'.format(done, Bc, best[0], ncpu, dt)}
    value = B / (ms * 1e-3)
    return {'metric': 'ic_train_traces_per_sec', 'value': value, 'unit': 'traces/s', 'ms_per_step': ms, 'batch': B,
            'trace_length': T, 'parameters': int(net.num_parameters()), 'roofline': roof, 'cpu_baseline': cb,
            'ratio_to_cpu_baseline': value / cb['value'],
            'config': 'synthetic 50-address Normal/Categorical(4) model, T=50, observe FF dim 256 depth 2, LSTM h=512, '
                      '512 traces (per-GPU share of BASELINE configs[3]), device-resident step, back to back'}


if __name__ == '__main__':
    main()
