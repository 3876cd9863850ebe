#!/usr/bin/env python
"""A/B timing of the spline tensor-core kernel's specialisations on the benchmark workload (bench.py q256:
CouplingRQNSF(256), 2^20 rows, state T): Flow.log_prob and Flow.sample with

    default      output-only sampling kernel, polynomial knot derivative where admitted
    always_ld    B2F_TCQ_ALWAYS_LD=1 (sampling computes and drops the log-det)
    no_dpoly     B2F_TCQ_NO_DPOLY=1 (SFU softplus)
    general      both switches: the kernel variants that existed before the specialisation

The variants alternate round by round in one process (the switches are read per launch), so clock and neighbour drift
spread over all of them.  CUDA events; the input (1 GiB) and each sample (1 GiB) are larger than the 126 MB L2.

    python scripts/tcq_specialise_time.py [--rounds 10] [--iters 5] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

VARIANTS = {'default': {}, 'always_ld': {'B2F_TCQ_ALWAYS_LD': '1'}, 'no_dpoly': {'B2F_TCQ_NO_DPOLY': '1'},
            'general': {'B2F_TCQ_ALWAYS_LD': '1', 'B2F_TCQ_NO_DPOLY': '1'}}
SWITCHES = ('B2F_TCQ_ALWAYS_LD', 'B2F_TCQ_NO_DPOLY')


def gpu_info():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else None
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=10)
    ap.add_argument('--iters', type=int, default=5, help='calls per variant and round (timed one by one)')
    ap.add_argument('--rows', type=int, default=1 << 20)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    import bench
    from torchflows_b200 import _native as N
    if not torch.cuda.is_available():
        raise SystemExit('needs a CUDA device')
    dev = torch.device('cuda:0')
    D, B = 256, args.rows
    g = torch.Generator(device=dev).manual_seed(1)
    x = torch.randn(B, D, device=dev, generator=g)
    flow = bench.build_flow('CouplingRQNSF', D, dev, init_rows=x[:65536])
    from torchflows_b200 import _tcq
    P = D // 2 * 23
    ws = [p for p in flow.parameters() if p.dim() == 2 and p.shape[0] == P]
    bs = [p for p in flow.parameters() if p.dim() == 1 and p.shape[0] == P]
    bounds = [_tcq.derivative_logit_bound(w.detach(), b.detach(), D // 2).item() for w, b in zip(ws, bs)]
    for k in SWITCHES:
        os.environ.pop(k, None)
    times = {v: {'log_prob': [], 'sample': []} for v in VARIANTS}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * args.iters + 1)]
    with torch.no_grad():
        for rnd in range(args.rounds + 1):              # round 0 is warm-up
            for name, kv in VARIANTS.items():
                os.environ.update(kv)
                try:
                    for leg in ('log_prob', 'sample'):
                        ev[0].record()
                        for i in range(args.iters):
                            if leg == 'log_prob':
                                lp = flow.log_prob(x)
                            else:
                                xs = flow.sample(B, no_grad=True)
                            ev[i + 1].record()
                        torch.cuda.synchronize()
                        assert N.last_flow_kernel() == N.KERNEL_TCQ
                        if rnd > 0:
                            times[name][leg] += [ev[i].elapsed_time(ev[i + 1]) for i in range(args.iters)]
                finally:
                    for k in kv:
                        os.environ.pop(k, None)
    del lp, xs
    res = {'workload': f'CouplingRQNSF({D}), {B} rows, state T (bench.py q256)', 'gpu': gpu_info(),
           'torch_device': torch.cuda.get_device_name(dev), 'rounds': args.rounds, 'iters': args.iters,
           'derivative_logit_bounds': bounds, 'variants': {}}
    for name in VARIANTS:
        r = {}
        for leg, t in times[name].items():
            q = statistics.quantiles(t, n=20)
            r[leg] = {'median_ms': statistics.median(t), 'p5_ms': q[0], 'p95_ms': q[-1], 'min_ms': min(t), 'max_ms': max(t),
                      'n': len(t)}
        r['step_ms'] = r['log_prob']['median_ms'] + r['sample']['median_ms']
        res['variants'][name] = r
    base = res['variants']['general']
    for name, r in res['variants'].items():
        r['vs_general'] = {leg: r[leg]['median_ms'] / base[leg]['median_ms'] - 1 for leg in ('log_prob', 'sample')}
        r['vs_general']['step'] = r['step_ms'] / base['step_ms'] - 1
    line = json.dumps(res, indent=1)
    print(line)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
