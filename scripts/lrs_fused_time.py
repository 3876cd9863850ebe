"""Linear rational spline presets: fused flow programs against the same flows forced onto the composite path
(conditioner GEMMs + stand-alone transformer kernel, the sequential direction as the reference's D-step loop).

CUDA-event medians over repeated calls after a warm-up of every timed shape; inputs are larger than L2 where the shape
allows.  Prints one JSON object (and writes it to --out): per case the fused and composite medians in ms, their ratio,
the kernel the fused program ran on, and the card's name and power limit read in the same run.

    python scripts/lrs_fused_time.py --out profiles/lrs_fused_time.json
"""
import argparse
import copy
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def force_composite(flow):
    from torchflows_b200.bijections.finite.autoregressive.layers_base import AutoregressiveBijection
    other = copy.deepcopy(flow)
    for m in other.modules():
        if isinstance(m, AutoregressiveBijection):
            m._fusable = False
            if hasattr(m, '_fusable_ctx'):
                m._fusable_ctx = False
    return other


def median_ms(fn, reps, warmup=2):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return statistics.median(times)


def gpu_info():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else torch.cuda.get_device_name(0)
    except Exception:
        return torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--composite-reps', type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('lrs_fused_time.py measures on a GPU; none is visible')
    from torchflows_b200 import Flow, _native as N
    from torchflows_b200.architectures import CouplingLRS, InverseAutoregressiveLRS, MaskedAutoregressiveLRS
    dev = torch.device('cuda:0')
    kernel_names = {N.KERNEL_GENERIC: 'generic', N.KERNEL_ROWS: 'rows', N.KERNEL_NONE: 'none'}
    results = {'gpu': gpu_info(), 'cases': []}

    def case(name, flow, run, rows):
        comp = force_composite(flow)
        with torch.no_grad():
            fused = median_ms(lambda: run(flow), args.reps)
            kernel = kernel_names.get(N.last_flow_kernel(), str(N.last_flow_kernel()))
            composite = median_ms(lambda: run(comp), args.composite_reps, warmup=1)
        r = dict(case=name, rows=rows, fused_ms=round(fused, 3), composite_ms=round(composite, 3),
                 speedup=round(composite / fused, 2), fused_kernel=kernel)
        results['cases'].append(r)
        print(json.dumps(r), flush=True)

    torch.manual_seed(0)
    B = 1 << 20
    flow = Flow(CouplingLRS(256)).to(dev).eval()
    x = torch.randn(B, 256, device=dev)
    case('CouplingLRS(256) log_prob', flow, lambda f: f.log_prob(x), B)

    B = 1 << 18
    flow = Flow(MaskedAutoregressiveLRS(128)).to(dev).eval()
    x = torch.randn(B, 128, device=dev)
    case('MaskedAutoregressiveLRS(128) log_prob', flow, lambda f: f.log_prob(x), B)
    case('MaskedAutoregressiveLRS(128) sample', flow, lambda f: f._sample_from_base(x, no_grad=True), B)

    flow = Flow(InverseAutoregressiveLRS(128)).to(dev).eval()
    case('InverseAutoregressiveLRS(128) log_prob', flow, lambda f: f.log_prob(x), B)

    # one training step (loss, backward, Adam) at 16 384 rows; the sequential log-det is the exact one on both sides
    Bt = 16384
    xt = torch.randn(Bt, 128, device=dev)
    wt = torch.ones(Bt, device=dev)
    flow = Flow(InverseAutoregressiveLRS(128)).to(dev)
    for m in flow.modules():
        if hasattr(m, 'sequential_log_det_reference_quirk'):
            m.sequential_log_det_reference_quirk = False
    comp = force_composite(flow)
    for f in (flow, comp):
        for m in f.modules():
            if hasattr(m, 'first_training_batch_pass'):
                m.first_training_batch_pass = False
        f.train()
    opts = {id(flow): torch.optim.Adam(flow.parameters(), lr=1e-3), id(comp): torch.optim.Adam(comp.parameters(), lr=1e-3)}

    def step(f):
        opt = opts[id(f)]
        opt.zero_grad()
        f._base_batch_loss((xt, wt)).backward()
        opt.step()
    fused = median_ms(lambda: step(flow), args.reps)
    r = dict(case='InverseAutoregressiveLRS(128) fit step', rows=Bt, fused_ms=round(fused, 3), fused_kernel='generic (backward)')
    try:
        # autograd over the composite's 2 x 128 sequential steps keeps every step's conditioner output alive
        composite = median_ms(lambda: step(comp), args.composite_reps, warmup=1)
        r.update(composite_ms=round(composite, 3), speedup=round(composite / fused, 2))
    except torch.cuda.OutOfMemoryError:
        r.update(composite_ms=None, note='composite step ran out of device memory: not measured')
    results['cases'].append(r)
    print(json.dumps(r), flush=True)

    print(json.dumps(results))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as fh:
            json.dump(results, fh, indent=1)


if __name__ == '__main__':
    main()
