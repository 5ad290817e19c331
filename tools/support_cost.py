"""Cost of the profiles: blmx_scan against blmx_scan_profile on the benchmark's problem.

A 500 k-site bench.make_chromosome with the bench grid (100 A x 510 (x, a) points), every STRIDE-th site a
centre with the whole chromosome as its window.  After a warm-up of both calls, the two are alternated
three times each; each call is synchronous (host buffers in and out), so a host clock around it measures the
whole call: upload, kernels, the per-launch profile copies and the row copies.  Prints the card's name and
power limit, every time, the medians and their ratio, as one JSON line.

    python tools/support_cost.py [--sites 500000] [--stride 10]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                         capture_output=True, text=True)
    return out.stdout.strip() if out.returncode == 0 else 'unknown'


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--sites', type=int, default=500000)
    ap.add_argument('--stride', type=int, default=10)
    ap.add_argument('--seed', type=int, default=1)
    args = ap.parse_args()
    import bench
    from ballermixplus_b200.native import Scanner
    prob = bench.make_problem([bench.make_chromosome(args.sites, seed=args.seed)])[0]
    n = len(prob.genpos)
    c = np.arange(0, n, args.stride)
    t, lo, hi = prob.genpos[c], np.zeros(len(c), np.int64), np.full(len(c), n - 1, np.int64)
    times = {'scan': [], 'scan_profile': []}
    with Scanner(device=0).load(prob) as sc:
        rows = sc.scan(t, lo, hi)                                  # warm-up of both paths
        prof = sc.scan_profile(t, lo, hi)
        same = all(np.array_equal(a, b) for a, b in zip(rows, prof[:5]))
        for _ in range(3):
            for name, fn in (('scan', sc.scan), ('scan_profile', sc.scan_profile)):
                t0 = time.perf_counter()
                fn(t, lo, hi)
                times[name].append(time.perf_counter() - t0)
    med = {k: float(np.median(v)) for k, v in times.items()}
    print(json.dumps({
        'card': card(), 'sites': n, 'centres': len(c), 'grid': [len(prob.A), prob.n_x, prob.n_a],
        'seconds': times, 'median_s': med, 'us_per_centre': {k: 1e6 * v / len(c) for k, v in med.items()},
        'overhead_ratio': med['scan_profile'] / med['scan'], 'rows_identical': same,
    }))


if __name__ == '__main__':
    main()
