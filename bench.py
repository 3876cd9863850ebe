#!/usr/bin/env python
"""Benchmark of the fused flow hot path (contract: see the task statement / DESIGN.md section "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload q256|r64|m128] [--impl ours|reference]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch: ``Flow.log_prob`` on B rows followed by ``Flow.sample`` of
B rows (inverse direction).  Default workload (BASELINE.json configs[2], the one the north-star target and the
1/2/4/8-GPU metric are quoted on): CouplingRQNSF(n_dim=256), B = 2^20 rows per GPU, fp32, random-init weights
from the constructor under seed 0 with ActNorm data-initialised on the benchmark data (state T of SURVEY 8d).
Multi-GPU: one process per GPU (torchrun), the batch is sharded, there is no data-path collective (weak scaling).

Prints ONE JSON line (rank 0).  `value` is measured with inputs resident in HBM; `e2e` goes through the public
API with pinned host buffers (H2D of x, D2H of log_prob and of the samples inside the timed region).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (preset, D, rows per GPU, cpu chunk rows, cpu rows per bounded sample)
    'q256': ('CouplingRQNSF', 256, 1 << 20, 8192, 32768),
    'r64': ('RealNVP', 64, 1 << 20, 65536, 1 << 20),
    'm128': ('MAF', 128, 1 << 18, 2048, 16384),
    'mq128': ('MaskedAutoregressiveRQNSF', 128, 1 << 18, 512, 1024),
}


# the kernel each workload's log_prob launch dispatches to (b2f_flow_apply: csrc/b2f_flow.cu)
KERNELS = {'q256': 'b2f::flow_tcq_kernel', 'mq128': 'b2f::flow_tcm_kernel', 'r64': 'b2f::flow_tca_kernel',
           'm128': 'b2f::flow_rows_kernel'}
KERNEL_IDS = {0: 'none', 1: 'generic (b2f_flow.cu)', 2: 'tc (b2f_flow_tc.cu)', 3: 'rows (b2f_flow_rows.cu)',
              4: 'tcq (b2f_flow_tcq.cu)', 5: 'tca (b2f_flow_tca.cu)', 6: 'tcm (b2f_flow_tcm.cu)'}


def algorithmic_bytes(D):
    """SURVEY 8d, whole-flow kernels: log_prob reads x (4D) and writes one float; Flow.sample writes x (4D): the base
    draws are made inside the launch (counter-based Philox stream), no noise tensor is read."""
    return 4 * D + 4, 4 * D


class ClockSampler(threading.Thread):
    """nvidia-smi clocks and throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False
        # NVML in-process (nvidia_ml_py), imported and initialised HERE, on the caller's thread and before the timed
        # region: importing the module holds the GIL for tens of milliseconds, and forking nvidia-smi out of a process
        # with a CUDA context stalls the launching thread just as long -- both are whole steps at this scale.
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get('CUDA_VISIBLE_DEVICES')
            idx = index
            if visible:
                try:
                    idx = int(visible.split(',')[index])
                except Exception:
                    idx = index
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            sm_max = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            get_reasons = getattr(pynvml, 'nvmlDeviceGetCurrentClocksEventReasons', None) or \
                pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
            get_reasons(h)
            self.nvml = (pynvml, h, sm_max, get_reasons)
        except Exception:
            self.nvml = None

    def run(self):
        if self.nvml is None:
            return self._run_smi()
        pynvml, h, sm_max, get_reasons = self.nvml
        bits = ((0x8, 3), (0x40, 4), (0x20, 5), (0x4, 6))       # hw_slowdown, hw_thermal, sw_thermal, sw_power_cap
        period = float(os.environ.get('B2F_CLOCK_PERIOD', '0.05'))
        while not self.stop_flag:
            try:
                row = [str(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)), str(sm_max),
                       str(pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0), 'Not Active', 'Not Active', 'Not Active', 'Not Active']
                mask = int(get_reasons(h))
                for bit, col in bits:
                    if mask & bit:
                        row[col] = 'Active'
                self.rows.append(row)
            except Exception:
                pass
            time.sleep(period)

    def _run_smi(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.Q}',
                                      '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(',')]
                if len(parts) >= 7:
                    self.rows.append(parts)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.rows:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        sm = [float(r[0]) for r in self.rows if r[0].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith('active') for r in self.rows)]
        return {'sm_mhz': statistics.median(sm) if sm else None, 'sm_max_mhz': float(self.rows[0][1]),
                'power_w_max': max(float(r[2]) for r in self.rows), 'reasons': reasons, 'samples': len(self.rows)}


def build_flow(preset, D, device=None, init_rows=None):
    """Random-init weights exactly as the constructor makes them under seed 0; ActNorm data-initialised by one
    training-mode pass over `init_rows` (state T)."""
    import torch
    from torchflows_b200 import Flow
    import torchflows_b200.architectures as arch
    torch.manual_seed(0)
    flow = Flow(getattr(arch, preset)(D))
    if device is not None:
        flow = flow.to(device)
        if init_rows is not None:
            flow.train()
            with torch.no_grad():
                flow.log_prob(init_rows)
        flow.eval()
    return flow


def cpu_oracle_throughput(preset, D, state_dict, chunk, rows, steps, warmup, seed=1, init_state_t=False, device='cpu'):
    """The reference's own op sequence (oracle/flow_oracle.py: the same ATen ops in the same order, validated bit for bit
    against the real reference on the CPU): log_prob + sample over `rows` rows in chunks of `chunk`.  device='cpu': all host
    cores (the reference's CPU path).  device='cuda:0': the same ops eagerly on the B200, TF32 off -- the reference's own
    "CUDA support" is nn.Module.cuda() (docs/source/guides/cuda.rst), i.e. this is the existing Blackwell path.
    init_state_t: data-initialise ActNorm by the oracle itself on 8192 synthetic rows (state T of SURVEY 8d)."""
    import torch
    from oracle.flow_oracle import OracleFlow
    torch.set_num_threads(os.cpu_count() or 1)
    if device != 'cpu':
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = False
    o = OracleFlow(preset, (D,), state_dict, device=device)
    g = torch.Generator().manual_seed(seed)
    if init_state_t:
        with torch.no_grad():
            o.actnorm_initialise(torch.randn(8192, D, generator=g).to(device))
    x = torch.randn(rows, D, generator=g).to(device)
    z = torch.randn(rows, D, generator=g).to(device)

    def sync():
        if device != 'cpu':
            torch.cuda.synchronize()
    times = []
    with torch.no_grad():
        for it in range(warmup + steps):
            sync()
            t0 = time.perf_counter()
            for s in range(0, rows, chunk):
                o.log_prob(x[s:s + chunk])
            for s in range(0, rows, chunk):
                o.sample_from_noise(z[s:s + chunk])
            sync()
            if it >= warmup:
                times.append(time.perf_counter() - t0)
    t = statistics.median(times)
    return rows / t, t, torch.get_num_threads()


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    preset, D, B, chunk, cpu_rows = WORKLOADS[args.workload]
    flow = build_flow(preset, D)           # CPU module: only a weight container here
    flow.eval()
    sd = flow.state_dict()
    value, t, cores = cpu_oracle_throughput(preset, D, sd, chunk, cpu_rows, args.steps, args.warmup, init_state_t=True)
    sample = (f'{cpu_rows} rows in chunks of {chunk} per step (log_prob + sample); weights: constructor under seed 0, ActNorm '
              f'data-initialised by the oracle on 8192 synthetic rows (state T, like the repo arm)')
    line = {
        'impl': 'reference', 'metric': 'log_prob+sample samples/s', 'value': value, 'unit': 'samples/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': t * 1e3,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': f'{preset} n_dim={D}: log_prob + sample, CPU (oracle port of the reference, torch CPU ops)',
                   'weights': 'random init (seed 0), ActNorm data-initialised (state T)', 'rows_per_step': cpu_rows,
                   'chunk': chunk},
        'cpu_baseline': {'value': value, 'unit': 'samples/s', 'cores': cores, 'kind': 'port', 'sample': sample},
        'e2e': {'value': value, 'unit': 'samples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


DUMP_BYTES = 48 << 20       # array data written by --dump-outputs, at most (plus a 128-byte header per .npy file)


def dump_outputs(out_dir, outputs):
    """Write the row-aligned outputs of the last timed step as <out_dir>/<name>.npy in float32.  When all of them
    together exceed DUMP_BYTES, every output keeps the same rows: a sorted sample drawn from a private generator under
    a fixed seed, so two runs with the same arguments write comparable files and torch's global RNG (which keys the
    library's base draws) is left untouched."""
    import numpy as np
    import torch
    rows = next(iter(outputs.values())).shape[0]
    row_bytes = sum(4 * t[:1].numel() for t in outputs.values())
    keep = min(rows, DUMP_BYTES // row_bytes)
    idx = None
    if keep < rows:
        idx = torch.randperm(rows, generator=torch.Generator().manual_seed(0))[:keep].sort().values
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        if idx is not None:
            t = t[idx.to(t.device)]
        np.save(os.path.join(out_dir, name + '.npy'), t.detach().float().cpu().numpy())


def transformer_kernel_roofline(torch, dev, hbm_peak):
    """Stand-alone rational-quadratic spline transformer (b2f_transformer_apply, dense parameters): 16384 x 512 elements,
    (23 + 2) * 4 algorithmic bytes per element, CUDA-event timing over 10 launches, operands (771 MB of h) larger than L2."""
    from torchflows_b200 import _native as N
    rows, E, P = 16384, 512, 23
    x = torch.randn(rows, E, device=dev) * 2
    h = torch.randn(rows, E * P, device=dev)
    for _ in range(3):
        N.transformer_apply(N.T_RQ_FWD, x, h, E * P, 8, 50.0)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        N.transformer_apply(N.T_RQ_FWD, x, h, E * P, 8, 50.0)
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / 10
    achieved = rows * E * (P + 2) * 4 / (ms * 1e-3) / 1e9
    return {'bound': 'hbm', 'kernel': 'b2f::transformer_kernel<RQ_FWD> (b2f_transformer_apply)', 'achieved': achieved,
            'peak': hbm_peak, 'unit': 'GB/s', 'frac': achieved / hbm_peak, 'algorithmic_bytes_per_element': (P + 2) * 4,
            'elements': rows * E, 'launch_ms': ms}


def run_ours(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device: the hot path has no CPU fallback')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)

    preset, D, B, chunk, cpu_rows = WORKLOADS[args.workload]
    if args.rows:
        B = args.rows
    g = torch.Generator(device=dev).manual_seed(1 + rank)
    x = torch.randn(B, D, device=dev, generator=g)
    flow = build_flow(preset, D, dev, init_rows=x[:65536])
    by_lp, by_s = algorithmic_bytes(D)

    def step():
        lp = flow.log_prob(x)
        xs = flow.sample(B, no_grad=True)       # the public call: base draws + inverse pass in one launch
        return lp, xs

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    stream = torch.cuda.current_stream()
    with torch.no_grad():
        for _ in range(args.warmup):
            lp, xs = step()        # bound like in the timed loop: the allocator ends warm-up holding both output buffers
        sync_all()
        sampler = ClockSampler(local_rank)
        sampler.start()
        import gc
        gc.collect()
        gc.disable()           # a collector pause on the launching thread is a bubble on the GPU at ~1 ms per step
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3 * args.steps + 1)]
        ev[0].record(stream)
        for i in range(args.steps):
            lp = flow.log_prob(x)
            ev[3 * i + 1].record(stream)
            xs = flow.sample(B, no_grad=True)
            ev[3 * i + 2].record(stream)
            ev[3 * i + 3].record(stream)
        sync_all()
        total_ms = ev[0].elapsed_time(ev[3 * args.steps])
        lp_ms = [ev[3 * i].elapsed_time(ev[3 * i + 1]) for i in range(args.steps)]
        s_ms = [ev[3 * i + 1].elapsed_time(ev[3 * i + 2]) for i in range(args.steps)]
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, {'log_prob': lp, 'sample': xs})
        del xs
        from torchflows_b200 import _native as N_
        flow.sample(4096, no_grad=True)
        k_s = N_.last_flow_kernel()
        # for comparison: the inverse pass alone on noise that already sits in HBM (8 D bytes per row; what round 1 timed)
        zz = N_.philox_normal(B, D, dev, 1234, 0)
        flow._sample_from_base(zz, no_grad=True)
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record(stream)
        for _ in range(3):
            flow._sample_from_base(zz, no_grad=True)
        g1.record(stream)
        torch.cuda.synchronize()
        given_noise_ms = g0.elapsed_time(g1) / 3
        del zz
        lp = flow.log_prob(x)
        k_lp_full = N_.last_flow_kernel()
        del lp

        # ---- end to end through the public API: pinned host buffers in, host buffers out -----------------------
        e2e_steps = max(2, min(args.steps, 5))
        nchunk = 8
        rows_c = (B + nchunk - 1) // nchunk
        x_host = torch.empty(B, D, pin_memory=True)
        x_host.copy_(x)
        lp_host = torch.empty(B, pin_memory=True)
        xs_host = torch.empty(B, D, pin_memory=True)
        h2d_stream = torch.cuda.Stream(device=dev)
        d2h_stream = torch.cuda.Stream(device=dev)

        import collections
        in_flight = collections.deque()      # (device tensors, main-stream event, d2h-stream event) of the last two steps

        def e2e_step():
            # Chunked and interleaved: while the kernels of chunk i run, chunk i+1 of x is on its way up (H2D) and the
            # samples of chunk i-1 are on their way down (D2H) -- the two PCIe directions are used at the same time, also
            # across step boundaries.  The device tensors of a step stay referenced until the step after the next one
            # starts (ordered by events), so the caching allocator sees the same allocation pattern every step: no
            # cudaMalloc and no cross-stream reuse hazards inside the timed region.
            if len(in_flight) == 2:
                old, ev_main, ev_d2h = in_flight.popleft()
                h2d_stream.wait_event(ev_main)          # its staging blocks are no longer read by kernels
                stream.wait_event(ev_d2h)               # its output blocks have been copied out
                del old
            chunks = list(range(0, B, rows_c))
            staged, keep = {}, []

            def stage(s):
                with torch.cuda.stream(h2d_stream):
                    xc = x_host[s:s + rows_c].to(dev, non_blocking=True)
                    e = torch.cuda.Event()
                    e.record(h2d_stream)
                staged[s] = (xc, e)

            stage(chunks[0])
            for i, s in enumerate(chunks):
                if i + 1 < len(chunks):
                    stage(chunks[i + 1])
                xc, e = staged.pop(s)
                stream.wait_event(e)
                lpc = flow.log_prob(xc)                                   # public API, device chunk
                n = min(rows_c, B - s)
                xsc = flow.sample(n, no_grad=True)                        # draws z on the device, inverse pass
                done = torch.cuda.Event()
                done.record(stream)
                with torch.cuda.stream(d2h_stream):
                    d2h_stream.wait_event(done)
                    lp_host[s:s + n].copy_(lpc, non_blocking=True)
                    xs_host[s:s + n].copy_(xsc, non_blocking=True)
                keep.append((xc, lpc, xsc))
            ev_main, ev_d2h = torch.cuda.Event(), torch.cuda.Event()
            ev_main.record(stream)
            ev_d2h.record(d2h_stream)
            in_flight.append((keep, ev_main, ev_d2h))

        for _ in range(3):
            e2e_step()
        stream.wait_stream(d2h_stream)
        sync_all()
        t0 = torch.cuda.Event(enable_timing=True)
        t1 = torch.cuda.Event(enable_timing=True)
        t0.record(stream)
        for _ in range(e2e_steps):
            e2e_step()
        stream.wait_stream(d2h_stream)         # the last step's results are in host memory
        t1.record(stream)
        sync_all()
        e2e_ms = t0.elapsed_time(t1) / e2e_steps
        # the copies alone, both directions at once, same buffers: what the host side of this box can move
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        xd_tmp = torch.empty(B, D, device=dev)
        sync_all()
        c0.record(stream)
        for _ in range(2):
            with torch.cuda.stream(h2d_stream):
                xd_tmp.copy_(x_host, non_blocking=True)
            with torch.cuda.stream(d2h_stream):
                xs_host.copy_(x, non_blocking=True)
        stream.wait_stream(h2d_stream)
        stream.wait_stream(d2h_stream)
        c1.record(stream)
        sync_all()
        copy_ms = c0.elapsed_time(c1) / 2
        del xd_tmp
        gc.enable()
        sampler.stop_flag = True           # clocks were sampled across the device-resident, fast-mode and e2e regions
        sampler.join(timeout=3)

    # max over ranks
    times = torch.tensor([total_ms, e2e_ms, copy_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    total_ms, e2e_ms, copy_ms = float(times[0]), float(times[1]), float(times[2])
    ms_per_step = total_ms / args.steps
    value = world * B / (ms_per_step * 1e-3)
    lp_avg_ms, s_avg_ms = statistics.mean(lp_ms), statistics.mean(s_ms)

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    hbm_peak = float(peaks.get('hbm_gbs', 6650.0))
    peak_src = 'measured (MEASURED_PEAKS.json)' if 'hbm_gbs' in peaks else 'fallback (B200_PROFILING.md)'
    achieved = by_lp * B / (lp_avg_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None
    try:        # dram__bytes_read.sum + dram__bytes_write.sum of the log_prob launch from the committed ncu capture
        tr = json.load(open(os.path.join(ROOT, 'profiles', 'traffic.json')))
        if args.workload in tr and not args.rows:
            traffic = tr[args.workload]['log_prob_launch_dram_bytes']
            traffic_src = 'committed ncu capture, not this run: ' + tr[args.workload].get('source', '') + ' @ ' + \
                str(tr[args.workload].get('captured_at_commit', '?'))
    except Exception:
        pass

    line = {
        'metric': 'log_prob+sample samples/s', 'value': value, 'unit': 'samples/s', 'n_gpus': world,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_per_step, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': f'{preset} n_dim={D}, {B} rows per GPU: Flow.log_prob + Flow.sample (base draws by the library + inverse pass)',
                   'weights': 'random init (seed 0), ActNorm data-initialised (state T)', 'rows_per_gpu': B,
                   'l2': f'inputs larger than L2 ({B * D * 4 >> 20} MiB per tensor)',
                   'precision_mode': 'default: TF32 conditioner GEMMs (tcgen05), SFU ex2/lg2/rcp in the spline epilogue'},
        'log_prob_samples_per_s': world * B / (lp_avg_ms * 1e-3), 'sample_samples_per_s': world * B / (s_avg_ms * 1e-3),
        'roofline': {'bound': 'hbm', 'kernel': KERNELS[args.workload] + ' (log_prob launch)', 'achieved': achieved,
                     'peak': hbm_peak, 'unit': 'GB/s', 'frac': achieved / hbm_peak, 'traffic': traffic,
                     'traffic_source': traffic_src,
                     'peak_source': peak_src, 'algorithmic_bytes_per_row': by_lp, 'launch_ms': lp_avg_ms,
                     'sample_launch': {'achieved': by_s * B / (s_avg_ms * 1e-3) / 1e9, 'algorithmic_bytes_per_row': by_s,
                                       'launch_ms': s_avg_ms,
                                       'noise': 'Philox4x32-10 + Box-Muller inside the launch (no noise tensor in HBM)',
                                       'inverse_pass_on_resident_noise_ms': given_noise_ms}},
        'e2e': {'value': world * B / (e2e_ms * 1e-3), 'unit': 'samples/s', 'h2d_bytes_per_step': B * D * 4,
                'd2h_bytes_per_step': B * 4 + B * D * 4, 'ms_per_step': e2e_ms, 'bound': 'host',
                'copies_only_ms': copy_ms, 'h2d_GBps_per_gpu': B * D * 4 / (copy_ms * 1e-3) / 1e9,
                'd2h_GBps_per_gpu': B * D * 4 / (copy_ms * 1e-3) / 1e9,
                'note': 'pinned host memory <-> HBM over PCIe, both directions concurrently; copies_only_ms is the same '
                        'traffic without any kernel (max over ranks): the end-to-end step is bound by the host side of the '
                        'box (one NUMA node shared by all ranks), not by the GPU'},
        'gpu_launches': (2 if k_s in (N_.KERNEL_TCQ, N_.KERNEL_TCA) else 3) * args.steps,       # log_prob; sample (+ the noise kernel when the
                                                                                # program's kernel does not draw in registers)
        'dispatch': {'log_prob': KERNEL_IDS.get(k_lp_full, str(k_lp_full)), 'sample': KERNEL_IDS.get(k_s, str(k_s)),
                     'note': 'kernel each call of the timed loop ran on (b2f_last_flow_kernel): 100 % on the fused path'},
        'clocks': sampler.summary(),
    }
    if rank == 0:
        # SURVEY 8d asks for the per-layer transformer kernel next to the whole-flow one: the stand-alone spline transformer
        # (b2f_transformer_apply given materialised parameters) is the genuinely HBM-bound kernel of this path
        try:
            line['per_layer_roofline'] = transformer_kernel_roofline(torch, dev, hbm_peak)
        except Exception as e:       # never let the side measurement take the headline down
            line['per_layer_roofline'] = {'error': str(e)[:200]}
    if rank == 0 and not args.no_cpu:
        # the reference's op sequence run eagerly on this B200 (TF32 off): the existing Blackwell path (SURVEY 8d,
        # BASELINE.md section 3), same weights (state T of this run), same chunking as the CPU arm
        try:
            sd = {k: v.detach().clone() for k, v in flow.state_dict().items()}
            rows_e = min(B, 8 * chunk)
            v, t, _ = cpu_oracle_throughput(preset, D, sd, chunk, rows_e, 3, 1, device=str(dev))
            line['gpu_eager_baseline'] = {
                'value': v, 'unit': 'samples/s', 'kind': 'port', 'device': torch.cuda.get_device_name(dev),
                'sample': f'{rows_e} rows in chunks of {chunk} (log_prob + sample), allow_tf32=False, median of 3',
                'speedup_of_this_repo': (B / (ms_per_step * 1e-3)) / v}
        except Exception as e:
            line['gpu_eager_baseline'] = {'error': str(e)[:200]}
    if rank == 0 and world == 1 and not args.no_cpu:
        sd = {k: v.cpu() for k, v in flow.state_dict().items()}
        v, t, cores = cpu_oracle_throughput(preset, D, sd, chunk, cpu_rows, 3, 1)
        line['cpu_baseline'] = {'value': v, 'unit': 'samples/s', 'cores': cores, 'kind': 'port',
                                'sample': f'{cpu_rows} rows in chunks of {chunk} (log_prob + sample), same weights as the '
                                          f'repo arm (state T), median of 3'}
    if args.workload == 'q256' and not args.rows and not args.no_fit:
        # the other single-GPU configurations of BASELINE.json, briefly (their own bench lines: --workload r64|m128|mq128)
        del x
        torch.cuda.empty_cache()
        others = {}
        for wl in ('r64', 'm128', 'mq128'):
            try:
                others[wl] = quick_probe(torch, dev, rank, wl, hbm_peak)
            except Exception as e:
                others[wl] = {'error': str(e)[:200]}
        if world > 1:
            dist.barrier()
        line['other_workloads'] = others
        x = None
    if not args.no_fit:
        # Flow.fit, data-parallel over the same ranks: the path of this repo that has a collective in it
        del x_host, xs_host, lp_host
        x = None
        in_flight.clear()
        torch.cuda.empty_cache()
        fit = {}
        for wl in ('q256fit', 'w1024fit'):
            try:
                fit[wl] = fit_probe(torch, dist, dev, rank, world, wl)
            except Exception as e:          # never let the side measurement take the headline down
                fit[wl] = {'error': str(e)[:200]}
        line['fit'] = fit
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def quick_probe(torch, dev, rank, workload, hbm_peak, reps=20):
    """Flow.log_prob / Flow.sample launch times of one of the other BASELINE configurations on this rank's GPU (device
    events, 3 warm-up calls, `reps` timed calls each): the numbers their own bench lines report at length."""
    from torchflows_b200 import _native as N_
    preset, D, B, _, _ = WORKLOADS[workload]
    g = torch.Generator(device=dev).manual_seed(11 + rank)
    x = torch.randn(B, D, device=dev, generator=g)
    flow = build_flow(preset, D, dev, init_rows=x[:65536])
    by_lp, by_s = algorithmic_bytes(D)
    out = {'workload': f'{preset} n_dim={D}, {B} rows'}
    with torch.no_grad():
        for name, fn in (('log_prob', lambda: flow.log_prob(x)), ('sample', lambda: flow.sample(B, no_grad=True))):
            for _ in range(3):
                fn()
            kernel = N_.last_flow_kernel()
            torch.cuda.synchronize()
            # one event pair around `reps` back-to-back calls: the queue stays ahead of the GPU as long as a launch takes
            # longer than issuing it (~0.1 ms of Python per call), which holds for every workload here
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / reps
            nbytes = by_lp if name == 'log_prob' else by_s
            out[name] = {'launch_ms': ms, 'samples_per_s': B / (ms * 1e-3), 'kernel': KERNEL_IDS.get(kernel, str(kernel)),
                         'hbm_frac': nbytes * B / (ms * 1e-3) / 1e9 / hbm_peak}
    del flow, x
    torch.cuda.empty_cache()
    return out


def wide_tensor_roofline(torch, flow, x, dev, reps=5):
    """Tensor-pipe roofline of the wide-conditioner layer (csrc/b2f_wide.cu), timed with CUDA events around the C-ABI calls
    of ONE coupling layer on this workload's rows: forward = conditioner GEMMs + spline epilogue, backward = recompute +
    spline backward + the four gradient GEMMs.  achieved = ALGORITHMIC flops (2 B (Dh H + H 23 Dh) forward, twice that
    for the backward: the recompute GEMM is our choice, not the algorithm's) / duration; peak = the measured sustained bf16
    rate / 2 (kind::tf32 runs at half the bf16 rate)."""
    from torchflows_b200 import _native as N
    layer = next(l for l in flow.bijection.layers if getattr(l, '_wide', False))
    seq = layer.conditioner_transform.sequential
    W1, b1, W2, b2 = (t.detach() for t in (seq[0].weight, seq[0].bias, seq[2].weight, seq[2].bias))
    B, D = x.shape
    Dh, H = D // 2, W1.shape[0]
    gy, gld = torch.randn_like(x), torch.randn(B, device=dev)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    peak = float(peaks.get('bf16_tflops_sustained', 1400.0)) / 2
    src = 'measured bf16_tflops_sustained / 2 (MEASURED_PEAKS.json)' if 'bf16_tflops_sustained' in peaks else \
        'fallback 1400 / 2 (B200_PROFILING.md)'

    def timed(fn):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    ms_f = timed(lambda: N.wide_coupling_forward(N.T_RQ_FWD, x, W1, b1, W2, b2))
    ms_b = timed(lambda: N.wide_coupling_backward(N.T_RQ_FWD, x, gy, gld, W1, b1, W2, b2))
    flops_f = 2.0 * B * (Dh * H + H * Dh * 23)
    out = {'bound': 'tensor', 'unit': 'TFLOP/s', 'peak': peak, 'peak_source': src, 'dtype': 'tf32 (fp32 accumulate)',
           'forward': {'kernel': 'b2f_wide_coupling_forward (wide_gemm_kernel: hidden GEMM, output GEMM + spline epilogue)',
                       'launch_ms': ms_f, 'algorithmic_gflop': flops_f / 1e9, 'achieved': flops_f / (ms_f * 1e-3) / 1e12},
           'backward': {'kernel': 'b2f_wide_coupling_backward (recompute GEMM + spline backward epilogue, wgrad, dgrad)',
                        'launch_ms': ms_b, 'algorithmic_gflop': 2 * flops_f / 1e9, 'executed_gflop': 3 * flops_f / 1e9,
                        'achieved': 2 * flops_f / (ms_b * 1e-3) / 1e12, 'executed': 3 * flops_f / (ms_b * 1e-3) / 1e12}}
    out['achieved'] = 3 * flops_f / ((ms_f + ms_b) * 1e-3) / 1e12
    out['frac'] = out['achieved'] / peak
    return out


def fit_path(flow):
    """Which kernels a Flow.fit step of this flow runs on, read off the layers' own dispatch flags."""
    layers = [l for l in flow.bijection.layers if hasattr(l, '_fusable') and hasattr(l, 'coupling')]
    if layers and all(getattr(l, '_wide', False) for l in layers):
        return 'fused (b2f_wide_coupling_forward / _backward: tcgen05 TF32 GEMM pipeline, spline in the GEMM epilogue)'
    if layers and all(l._fusable for l in layers):
        return 'fused (b2f_flow_apply_saving + b2f_flow_backward)'
    return 'composite (library GEMMs for the conditioner, b2f transformer kernels)'


def fit_probe(torch, dist, dev, rank, world, workload, steps=5, warmup=3, rows=0):
    """ms per optimisation step of Flow.fit's inner loop (Flow.train_step: forward, backward, gradient exchange, AdamW) on
    this rank's GPU, data-parallel over the visible ranks, plus the gradient all-reduce on its own (the same buckets, no
    compute to hide behind).  Part of the default bench line so that the driver's 1/2/4/8-GPU run records the path that
    has a collective in it (BASELINE.json configs[4])."""
    from torchflows_b200 import Flow
    from torchflows_b200.architectures import CouplingRQNSF
    if workload == 'w1024fit':
        D, H, per_gpu, kwargs = 1024, 1024, rows or 16384, {'conditioner_kwargs': {'n_hidden': 1024}}
    else:
        D, H, per_gpu, kwargs = 256, 17, rows or 131072, {}
    torch.manual_seed(0)
    flow = Flow(CouplingRQNSF(D, **kwargs)).to(dev)
    n_params = sum(p.numel() for p in flow.parameters() if p.requires_grad)
    g = torch.Generator(device=dev).manual_seed(1 + rank)
    x = torch.randn(per_gpu, D, device=dev, generator=g)
    flow.train()
    flow._optimizer = torch.optim.AdamW(flow.parameters(), lr=1e-3)
    for _ in range(warmup):
        flow.train_step(x, n_global=per_gpu * world)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = flow.train_step(x, n_global=per_gpu * world)
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t = [e0.elapsed_time(e1) / steps, 0.0]
    nbytes = 0
    if world > 1 and flow._buckets is not None:
        b = flow._buckets
        nbytes = b.nbytes
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dist.barrier()
        torch.cuda.synchronize()
        a0.record()
        for _ in range(steps):
            b.begin_step()
            b.finish()
        a1.record()
        torch.cuda.synchronize()
        t[1] = a0.elapsed_time(a1) / steps
        b.close()
    ms = torch.tensor(t, device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_step, ms_ar = float(ms[0]), float(ms[1])
    path = fit_path(flow)
    tensor = None
    if workload == 'w1024fit' and rank == 0:
        tensor = wide_tensor_roofline(torch, flow, x, dev)
    out = {'workload': f'CouplingRQNSF n_dim={D} n_hidden={H}, {per_gpu} rows per GPU', 'ms_per_step': ms_step,
           'samples_per_s': world * per_gpu / (ms_step * 1e-3), 'trainable_parameters': n_params, 'path': path,
           'allreduce_bytes_per_step': nbytes, 'allreduce_alone_ms': ms_ar, 'final_loss': float(loss)}
    if tensor is not None:
        out['tensor_roofline'] = tensor
    del flow, x
    torch.cuda.empty_cache()
    return out


def run_fit(args):
    """BASELINE.json configs[4]: CouplingRQNSF(1024, n_hidden=1024) maximum-likelihood training, data-parallel over the
    visible GPUs (16384 rows per GPU per step, NCCL all-reduce of the 25.2 M-parameter gradient every step).  A step is
    one optimisation step of Flow.fit's inner loop (Flow.train_step)."""
    import torch
    import torch.distributed as dist
    from torchflows_b200 import Flow
    from torchflows_b200.architectures import CouplingRQNSF
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)
    if args.workload == 'w1024fit':
        D, H, per_gpu = 1024, 1024, args.rows or 16384
        kwargs = {'conditioner_kwargs': {'n_hidden': H}}
    else:      # q256fit: default CouplingRQNSF(256) through the fused backward kernel
        D, H, per_gpu = 256, 17, args.rows or 131072
        kwargs = {}
    torch.manual_seed(0)
    flow = Flow(CouplingRQNSF(D, **kwargs)).to(dev)
    n_params = sum(p.numel() for p in flow.parameters() if p.requires_grad)
    g = torch.Generator(device=dev).manual_seed(1 + rank)
    x = torch.randn(per_gpu, D, device=dev, generator=g)
    flow.train()
    flow._optimizer = torch.optim.AdamW(flow.parameters(), lr=1e-3)
    for _ in range(args.warmup):
        flow.train_step(x, n_global=per_gpu * world)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss = flow.train_step(x, n_global=per_gpu * world)
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_per_step = float(ms) / args.steps
    if rank == 0:
        print(json.dumps({
            'metric': 'fit samples/s', 'value': world * per_gpu / (ms_per_step * 1e-3), 'unit': 'samples/s', 'n_gpus': world,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_per_step, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': f'CouplingRQNSF n_dim={D} n_hidden={H}: Flow.fit step (fwd + bwd + all-reduce + AdamW), '
                                   f'{per_gpu} rows per GPU', 'trainable_parameters': n_params,
                       'path': fit_path(flow)},
            'final_loss': float(loss)}), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='q256', choices=sorted(WORKLOADS) + ['w1024fit', 'q256fit'])
    ap.add_argument('--rows', type=int, default=0, help='override rows per GPU')
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline and gpu_eager_baseline legs')
    ap.add_argument('--no-fit', action='store_true', help='skip the Flow.fit probe (q256fit, w1024fit) of the default line')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write log_prob.npy and sample.npy of the last timed step (rank 0; a fixed row sample of '
                         f'at most {DUMP_BYTES >> 20} MiB in all) to DIR')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl != 'ours' or args.workload in ('w1024fit', 'q256fit')):
        ap.error('--dump-outputs applies to the log_prob + sample workloads of --impl ours')
    args.warmup = max(args.warmup, 3) if args.impl == 'ours' else max(args.warmup, 1)
    if args.workload in ('w1024fit', 'q256fit'):
        run_fit(args)
    elif args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
