"""Cost of scanning an empirical null three ways, on the benchmark's grid (bench.py: n = 200, --rangeA
1000,10900,100, default x / alpha grids, default window mode):

  segmented   the replicates laid end to end, one blmx_load_segmented and one scan
  loop        one blmx_load and one scan per replicate, the same tables
  plain       the same concatenation loaded with plain blmx_load (genpos not monotone: the direct path)

Two shapes: many short replicates and fewer long ones.  Every centre's window is its whole replicate (the
default mode), centres on every 16th (short) or 64th (long replicates) site.  Host clock around load + scan (both synchronous); the rows of
segmented and plain are compared with the loop's.  Writes JSON to --out and prints it.

    python tools/null_cost.py --out profiles/r5_null_cost.json
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

import bench                                                     # noqa: E402
from ballermixplus_b200.native import ScanProblem, Scanner      # noqa: E402


def gpu_info():
    try:
        return subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                              capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as exc:                                     # the numbers still stand, without the card
        return f'unavailable: {exc}'


def shape(n_reps, n_sites, seed):
    probs = bench.make_problem([bench.make_chromosome(n_sites, seed + i) for i in range(n_reps)])
    seg = np.arange(n_reps, dtype=np.int64) * n_sites
    p0 = probs[0]
    g = np.concatenate([p.genpos for p in probs])
    c = np.concatenate([p.cls for p in probs])
    cat = ScanProblem(g, c, p0.G, p0.SP, p0.A, p0.n_x, p0.n_a, seg_start=seg)
    plain = ScanProblem(g, c, p0.G, p0.SP, p0.A, p0.n_x, p0.n_a)
    return probs, cat, plain, seg


def centres(probs, seg, stride):
    ts, los, his = [], [], []
    for p, b in zip(probs, seg):
        n = len(p.genpos)
        k = np.arange(0, n, stride)
        ts.append(p.genpos[k]); los.append(np.zeros(len(k), np.int64)); his.append(np.full(len(k), n - 1, np.int64))
    return ts, los, his


def timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return out, time.perf_counter() - t0


def run_shape(n_reps, n_sites, stride, seed, plain_too):
    probs, cat, plain, seg = shape(n_reps, n_sites, seed)
    ts, los, his = centres(probs, seg, stride)
    t = np.concatenate(ts)
    lo = np.concatenate([x + b for x, b in zip(los, seg)])
    hi = np.concatenate([x + b for x, b in zip(his, seg)])
    sc = Scanner(device=0)
    # warm-up: module load and every scratch allocation at this size
    sc.load(probs[0]); sc.scan(ts[0], los[0], his[0]); sc.load(cat); sc.scan(t, lo, hi)

    def segmented():
        sc.load(cat)
        return sc.scan(t, lo, hi)

    def loop():
        rows = []
        for p, a, b, c in zip(probs, ts, los, his):
            sc.load(p)
            rows.append(sc.scan(a, b, c))
        return tuple(np.concatenate([r[k] for r in rows]) for k in range(5))

    def plain_run():
        sc.load(plain)
        return sc.scan(t, lo, hi)

    res = {'replicates': n_reps, 'sites_per_replicate': n_sites, 'centres': int(len(t)), 'centre_stride': stride,
           'grid_points_per_centre': int(len(cat.A) * cat.n_x * cat.n_a)}
    rows = {}
    for name, fn in (('segmented', segmented), ('loop', loop)) + ((('plain', plain_run),) if plain_too else ()):
        times = []
        for _ in range(1 if name == 'plain' else 3):      # the direct path is slow: one run
            rows[name], s = timed(fn)
            times.append(s)
        k = sc.counters_all()
        res[name] = {'seconds_median': float(np.median(times)), 'seconds': times,
                     'pruned_items_last_scan': k['pruned_items'], 'far_sites_last_scan': k['far_sites']}
    ref = rows['loop']
    for name in rows:
        if name == 'loop':
            continue
        T = rows[name][0]
        rel = np.abs(T - ref[0]) / np.maximum(np.abs(ref[0]), 1.0)
        res[name]['vs_loop'] = {'max_rel_dT': float(rel.max()), 'rows_over_1e-9': int((rel > 1e-9).sum()),
                                'nsites_mismatch': int((rows[name][4] != ref[4]).sum()),
                                'argmax_mismatch': int(np.sum((rows[name][1] != ref[1]) | (rows[name][2] != ref[2])
                                                              | (rows[name][3] != ref[3])))}
    for name in ('segmented', 'plain'):
        if name in res:
            res[name]['speedup_vs_loop'] = res['loop']['seconds_median'] / res[name]['seconds_median']
    sc.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--small', action='store_true', help='tiny shapes, to rehearse the script')
    opt = ap.parse_args()
    # (replicates, sites each, centre stride)
    shapes = [(1000, 2000, 16), (100, 50000, 64)] if not opt.small else [(20, 300, 16), (3, 2000, 64)]
    out = {'gpu (name, power limit, max SM clock)': gpu_info(),
           'what': 'seconds of load + scan (host clock, both synchronous): medians of 3 runs for segmented and '
                   'loop, one run for plain; one Scanner, warmed up at the shape',
           'shapes': [run_shape(r, n, st, 1000 + i, True) for i, (r, n, st) in enumerate(shapes)]}
    text = json.dumps(out, indent=1)
    print(text)
    if opt.out:
        os.makedirs(os.path.dirname(os.path.abspath(opt.out)), exist_ok=True)
        with open(opt.out, 'w') as fh:
            fh.write(text + '\n')


if __name__ == '__main__':
    main()
