"""Cost of binned spectra on the scan: the pruner's slab path (bound_kernel<SLABS>, more than 256 classes).

A 500 k-site bench.make_chromosome split into BINS bins by position, every bin with the chromosome's own spectrum
(what --getSpect writes), so the statistic is the unbinned one while the problem has BINS times its classes
(about 400 for two bins).  The bench grid (100 A x 510 (x, a) points), every STRIDE-th site a centre with the whole
chromosome as its window.  Three arms: the binned problem with pruning (the slab path), the binned problem with
prune = 0, and the unbinned problem with pruning (the one-slab path).  After a warm-up of every arm, the arms are
alternated three times each; each call is synchronous, so a host clock around it measures the whole call.  Checks
that prune = 1 and prune = 0 give identical rows and compares the binned rows with the unbinned ones; prints the
card's name and power limit, every time, the medians and their ratios, and the pruned items, as one JSON line.

    python tools/binmap_cost.py [--sites 500000] [--stride 10] [--bins 2]
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


def binned_problem(chrom, n_bins, same=True):
    """The product's binned ScanProblem (bins.BinnedNeutral, problem.build_problem) of a bench chromosome cut into
    ``n_bins`` position bins: bin 0 the first stretch (--spect), bins 1.. the others.  ``same``: every bin has the
    chromosome's spectrum; else each bin has the spectrum of its own sites."""
    import bench
    from ballermixplus_b200 import Grids, InputData, NeutralSFS, NormalizedBetaBinom
    from ballermixplus_b200.bins import BinMap, BinnedNeutral
    from ballermixplus_b200.problem import build_problem
    n, pos, k = chrom['n'], chrom['pos'], chrom['k']
    data = InputData.from_arrays(pos, pos * bench.REC_RATE, k, np.full(len(k), n))
    edges = np.quantile(pos, np.linspace(0, 1, n_bins + 1))
    site_bin = np.clip(np.searchsorted(edges, pos, 'right') - 1, 0, n_bins - 1)

    def spect(mask):
        counts = np.bincount(k[mask], minlength=n + 1)
        return NeutralSFS.from_spect({(int(j), n): float(counts[j]) / float(counts.sum())
                                      for j in np.flatnonzero(counts)})

    labels = [f'bin{b}' for b in range(1, n_bins)]
    ivs = {'chr': [(float(pos[site_bin == b].min()), float(pos[site_bin == b].max()), b, b)
                   for b in range(1, n_bins)]}
    spects = [spect(np.ones(len(k), bool) if same else site_bin == b) for b in range(n_bins)]
    neutral = BinnedNeutral(spects[0], list(zip(labels, spects[1:])), BinMap('map', labels, ivs))
    data.siteBin = neutral.site_bins('chr', pos)
    grid = Grids(None, None, False, False, bench.RANGE_A, None)
    sel = NormalizedBetaBinom(data, grid, False, False, False)
    return build_problem(data, neutral, sel, grid)[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--sites', type=int, default=500000)
    ap.add_argument('--stride', type=int, default=10)
    ap.add_argument('--bins', type=int, default=2)
    ap.add_argument('--seed', type=int, default=1)
    args = ap.parse_args()
    import bench
    from ballermixplus_b200.native import Scanner
    chrom = bench.make_chromosome(args.sites, seed=args.seed)
    plain = bench.make_problem([chrom])[0]
    binned = binned_problem(chrom, args.bins)
    n = len(plain.genpos)
    c = np.arange(0, n, args.stride)
    t, lo, hi = plain.genpos[c], np.zeros(len(c), np.int64), np.full(len(c), n - 1, np.int64)
    times = {'binned_prune': [], 'binned_prune0': [], 'unbinned_prune': []}
    with Scanner(device=0).load(binned) as sb, Scanner(device=0).load(binned) as sb0, \
            Scanner(device=0).load(plain) as sp:
        sb0.set_option('prune', 0)
        arms = (('binned_prune', sb), ('binned_prune0', sb0), ('unbinned_prune', sp))
        rows, pruned = {}, {}
        for name, s in arms:                                       # warm-up, rows and counters of every arm
            rows[name] = s.scan(t, lo, hi)
            pruned[name] = int(s.counters_all()['pruned_items'])
        for _ in range(3):
            for name, s in arms:
                t0 = time.perf_counter()
                s.scan(t, lo, hi)
                times[name].append(time.perf_counter() - t0)
    med = {k: float(np.median(v)) for k, v in times.items()}
    Tb, Tu = rows['binned_prune'][0], rows['unbinned_prune'][0]
    print(json.dumps({
        'card': card(), 'sites': n, 'centres': len(c), 'grid': [len(plain.A), plain.n_x, plain.n_a],
        'classes': {'binned': int(len(binned.G)), 'unbinned': int(len(plain.G))},
        'seconds': times, 'median_s': med,
        'prune0_over_prune': med['binned_prune0'] / med['binned_prune'],
        'binned_over_unbinned': med['binned_prune'] / med['unbinned_prune'],
        'pruned_items': pruned, 'items': int(len(c) * len(plain.A)),
        'prune_rows_identical': all(np.array_equal(a, b) for a, b in zip(rows['binned_prune'],
                                                                          rows['binned_prune0'])),
        'binned_vs_unbinned_max_rel_T': float(np.max(np.abs(Tb - Tu) / np.maximum(np.abs(Tu), 1.))),
        'binned_vs_unbinned_argmax_or_ns_differ': int(sum(np.sum(a != b) for a, b in
                                                          zip(rows['binned_prune'][1:], rows['unbinned_prune'][1:]))),
    }))


if __name__ == '__main__':
    main()
