"""Per-step cost of the pruning pass against the exact scan, on the benchmark's workload (bench.py --gpus 1:
bench.make_genome / make_problem at --sites, centres on every --stride-th site, every chromosome resident).

torch.profiler with CUDA activities, in a run of its own, over --steps steps after one warm-up step; reports per
step the summed device time of bound_kernel and of each scan_kernel instantiation, the pruned-item count
(counters_all()['pruned_items'], summed over chromosomes) and the card it ran on.  Writes JSON to --out and
prints it.

    python tools/bound_cost.py --out profiles/r7_bound_cost.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench                                                     # noqa: E402
from ballermixplus_b200.native import Scanner                   # noqa: E402


def gpu_info():
    q = 'name,power.limit,clocks.max.sm'
    try:
        line = subprocess.run(['nvidia-smi', f'--query-gpu={q}', '--format=csv,noheader'],
                              capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as exc:                                     # the numbers still stand, without the card
        return {'query': q, 'error': str(exc)}
    return {'query': q, 'value': line}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--sites', type=int, default=10_000_000)
    ap.add_argument('--stride', type=int, default=bench.BASE_STRIDE)
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--out', default=None)
    opt = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile

    problems = bench.make_problem(bench.make_genome(opt.sites))
    plans = bench.plan_centres(problems, opt.stride)
    scanners = [Scanner(device=0).load(p) for p in problems]

    def step():
        pruned = items = 0
        for sc, (t, lo, hi), p in zip(scanners, plans, problems):
            sc.scan(t, lo, hi)
            pruned += sc.counters_all()['pruned_items']
            items += len(t) * len(p.A)
        return pruned, items

    step()                                                       # module load, scratch allocations
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(opt.steps):
            pruned, items = step()
        torch.cuda.synchronize()
    kernels = {}
    for ev in prof.key_averages():
        name = ev.key
        if 'bound_kernel' in name or 'scan_kernel' in name:
            us = getattr(ev, 'device_time_total', None)
            if us is None:
                us = ev.cuda_time_total
            kernels[name] = {'ms_per_step': us / 1e3 / opt.steps, 'launches_per_step': ev.count / opt.steps}
    bound = sum(v['ms_per_step'] for k, v in kernels.items() if 'bound_kernel' in k)
    scan = sum(v['ms_per_step'] for k, v in kernels.items() if 'scan_kernel' in k)
    out = {'gpu': gpu_info(), 'sites': opt.sites, 'chromosomes': len(problems), 'centre_stride': opt.stride,
           'centres_per_step': int(sum(len(pl[0]) for pl in plans)), 'items_per_step': int(items),
           'pruned_items_per_step': int(pruned), 'frac_items_pruned': pruned / items, 'steps_profiled': opt.steps,
           'bound_kernel_ms_per_step': bound, 'scan_kernel_ms_per_step': scan, 'kernels': kernels,
           'timing': 'torch.profiler CUDA activity, device time summed over the profiled steps / steps; '
                     'synchronous per-chromosome scans (Scanner.scan), one stream'}
    for sc in scanners:
        sc.close()
    line = json.dumps(out, indent=1)
    print(line)
    if opt.out:
        os.makedirs(os.path.dirname(os.path.abspath(opt.out)), exist_ok=True)
        with open(opt.out, 'w') as fh:
            fh.write(line + '\n')


if __name__ == '__main__':
    main()
