"""Cost of --balPos: blmx_scan against blmx_scan_split and against two scans (the full grid, then the bal half alone).

A 500 k-site bench.make_chromosome with the bench grid (100 A x 510 (x, a) points, 51 alpha of which 44 are >= 1),
every STRIDE-th site a centre with the whole chromosome as its window.  After a warm-up of every arm, the three
arms are alternated three times each; each call is synchronous (host buffers in and out), so a host clock around
it measures the whole call.  The two-scan arm is what a user without --balPos runs to get a balancing score next
to the row: the default grid, then the --findBal grid (here: the same problem restricted to the bal alphas).
Checks that the split call's rows equal blmx_scan's exactly, and prints the card's name and power limit, every
time, the medians and their ratios, as one JSON line.

    python tools/balpos_cost.py [--sites 500000] [--stride 10]
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
    from ballermixplus_b200.balpos import half_of_a
    from ballermixplus_b200.grids import Grids
    from ballermixplus_b200.native import Scanner, ScanProblem
    from ballermixplus_b200.problem import GridOrder
    prob = bench.make_problem([bench.make_chromosome(args.sites, seed=args.seed)])[0]
    half = half_of_a(GridOrder(Grids(None, None, False, False, bench.RANGE_A, None)).a)
    assert len(half) == prob.n_a
    bal = np.flatnonzero(half == 0)
    SP_bal = prob.SP.reshape(prob.n_x, prob.n_a, -1)[:, bal].reshape(prob.n_x * len(bal), -1)
    prob_bal = ScanProblem(prob.genpos, prob.cls, prob.G, SP_bal, prob.A, prob.n_x, len(bal))
    n = len(prob.genpos)
    c = np.arange(0, n, args.stride)
    t, lo, hi = prob.genpos[c], np.zeros(len(c), np.int64), np.full(len(c), n - 1, np.int64)
    times = {'scan': [], 'scan_split': [], 'two_scans': []}
    with Scanner(device=0).load(prob) as sc, Scanner(device=0).load(prob_bal) as sb:
        def two_scans(t, lo, hi):
            return sc.scan(t, lo, hi), sb.scan(t, lo, hi)

        def split(t, lo, hi):
            return sc.scan_split(t, lo, hi, half)

        rows = sc.scan(t, lo, hi)                                  # warm-up of every arm
        main_rows, bal_rows, pos_rows = split(t, lo, hi)
        _, bal_ref = two_scans(t, lo, hi)
        same = all(np.array_equal(a, b) for a, b in zip(rows, main_rows))
        bal_T_rel = float(np.max(np.abs(bal_rows[0] - bal_ref[0]) / np.maximum(np.abs(bal_ref[0]), 1.)))
        for _ in range(3):
            for name, fn in (('scan', sc.scan), ('scan_split', split), ('two_scans', two_scans)):
                t0 = time.perf_counter()
                fn(t, lo, hi)
                times[name].append(time.perf_counter() - t0)
    med = {k: float(np.median(v)) for k, v in times.items()}
    print(json.dumps({
        'card': card(), 'sites': n, 'centres': len(c), 'grid': [len(prob.A), prob.n_x, prob.n_a],
        'bal_alphas': int(len(bal)), 'seconds': times, 'median_s': med,
        'us_per_centre': {k: 1e6 * v / len(c) for k, v in med.items()},
        'split_over_scan': med['scan_split'] / med['scan'], 'two_scans_over_split': med['two_scans'] / med['scan_split'],
        'rows_identical': same, 'bal_vs_bal_only_scan_max_rel_T': bal_T_rel,
        'rows_with_T_gt_0': {'main': int((rows[1] >= 0).sum()), 'bal': int((bal_rows[1] >= 0).sum()),
                             'pos': int((pos_rows[1] >= 0).sum())},
    }))


if __name__ == '__main__':
    main()
