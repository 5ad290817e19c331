"""Cost of local refinement: blmx_scan against blmx_refine at K = 2, 4 and 8 on the benchmark's problem.

A 500 k-site bench.make_chromosome with the bench grid (100 A x 510 (x, a) points), every STRIDE-th site a
centre with the whole chromosome as its window, as tools/support_cost.py.  The scan gives the rows; the rows with
T > 0 are refined.  The fine tables of each K are built once (host time reported as ``tables_s``) and loaded
before each timed refine call.  After a warm-up of every call, scan and the three refine calls are alternated
three times; each call is synchronous (host buffers in and out), so a host clock around it measures the whole
call.  Prints the card's name and power limit, every time, the medians, the time per refined centre and how many
rows moved, as one JSON line.

    python tools/refine_cost.py [--sites 500000] [--stride 10]
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


def bench_tables(chrom):
    """The NeutralSFS and NormalizedBetaBinom bench.make_problem builds for one chromosome."""
    import bench
    from ballermixplus_b200 import Grids, InputData, NeutralSFS, NormalizedBetaBinom
    n = chrom['n']
    counts = np.bincount(chrom['k'], minlength=n + 1)
    ks = np.flatnonzero(counts)
    spect = {(int(k), n): float(counts[k]) / float(counts.sum()) for k in ks}
    classes = InputData.from_arrays(np.arange(len(ks)), np.arange(len(ks)) * 1e-6, ks, np.full(len(ks), n))
    grid = Grids(None, None, False, False, bench.RANGE_A, None)
    return NeutralSFS.from_spect(spect), NormalizedBetaBinom(classes, grid, False, False, False)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--sites', type=int, default=500000)
    ap.add_argument('--stride', type=int, default=10)
    ap.add_argument('--seed', type=int, default=1)
    args = ap.parse_args()
    import bench
    from ballermixplus_b200 import refine
    from ballermixplus_b200.problem import GridOrder
    from ballermixplus_b200.scan import DeviceScan
    from ballermixplus_b200.grids import Grids
    chrom = bench.make_chromosome(args.sites, seed=args.seed)
    prob = bench.make_problem([chrom])[0]
    neutral, sel = bench_tables(chrom)
    order = GridOrder(Grids(None, None, False, False, bench.RANGE_A, None))
    n = len(prob.genpos)
    c = np.arange(0, n, args.stride)
    t, lo, hi = prob.genpos[c], np.zeros(len(c), np.int64), np.full(len(c), n - 1, np.int64)
    dev = DeviceScan.from_problem(prob, order)
    Ks = (2, 4, 8)
    times = {'scan': [], **{f'refine_K{k}': [] for k in Ks}}
    try:
        T, iA, ix, ia, ns = dev.run(t, lo, hi)
        live = np.flatnonzero(iA >= 0)
        setup, tables_s, moved = {}, {}, {}
        for K in Ks:
            t0 = time.perf_counter()
            g = refine.RefineGrid(order, K)
            box = g.boxes(iA[live], ix[live], ia[live])
            row_of, SP = refine.fine_tables(g, box, neutral, sel)
            tables_s[K] = time.perf_counter() - t0
            setup[K] = (g, box, row_of, SP)
        def run_refine(K):
            g, box, row_of, SP = setup[K]
            dev.load_refine(np.array([float(v) for v in g.A]), len(g.x), len(g.a), row_of, SP)
            t0 = time.perf_counter()
            got = dev.refine(t[live], lo[live], hi[live], box)
            return time.perf_counter() - t0, g, got
        for K in Ks:                                                # warm-up, and the moved rows
            _, g, got = run_refine(K)
            full = [np.full(len(c), -np.inf), *(np.full(len(c), -1, np.int32) for _ in range(3)),
                    np.zeros(len(c), np.int32)]
            for col, v in zip(full, got):
                col[live] = v
            moved[K] = int(refine.moved(g, T, iA, ix, ia, full).sum())
        for _ in range(3):
            t0 = time.perf_counter()
            dev.run(t, lo, hi)
            times['scan'].append(time.perf_counter() - t0)
            for K in Ks:
                times[f'refine_K{K}'].append(run_refine(K)[0])
    finally:
        dev.close()
    med = {k: float(np.median(v)) for k, v in times.items()}
    print(json.dumps({
        'card': card(), 'sites': n, 'centres': len(c), 'grid': [len(prob.A), prob.n_x, prob.n_a],
        'refined_centres': len(live), 'seconds': times, 'median_s': med,
        'us_per_centre_scan': 1e6 * med['scan'] / len(c),
        'us_per_refined_centre': {k: 1e6 * med[f'refine_K{k}'] / max(len(live), 1) for k in Ks},
        'fine_rows': {k: int(setup[k][3].shape[0]) for k in Ks}, 'tables_s': tables_s, 'moved_rows': moved,
    }))


if __name__ == '__main__':
    main()
