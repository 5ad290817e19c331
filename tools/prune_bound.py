"""Feasibility of pruning scan items by an upper bound on T (DESIGN.md §9).

For one (centre, A) item the scan reports a grid point only when its T > 0 (v1:451).  If an upper bound on
T is <= 0 at every grid point, the item's candidate is (T = 0, xa = -1) whatever its exact T, and the exact
evaluation could be skipped.  This tool measures, on the benchmark's own seeded workload (bench.make_genome /
make_problem, ~1 M sites), how many items such a bound proves, next to the exact item maximum from the C oracle
(report_all, one A at a time).

The bound, per class c and grid point (D = R_xa[c] - 1, alpha the site weights of class c in the window):
  log(1 + x) <= P_K(x) = sum_{m=1..K} (-1)^(m+1) x^m / m   for x > -1 and odd K
  log(1 + alpha D) <= log(1 + D) = log R                    for D >= 0, alpha <= 1
  log(1 + alpha D) <= alpha D                               always
Variant 'issue': tail sites (alpha < alpha*) take P_K from their power sums; near sites take
min(n_near log R, D S1_near) when D >= 0 and D S1_near when D < 0.
Variant 'best': P_K(x) <= x for x <= 0, so for D < 0 every site takes P_K; for D >= 0 the near sites take the
least of the three bounds.
Variant 'jensen' (what bound_kernel evaluates, DESIGN.md §3.8): log(1 + alpha D) is concave in alpha, so the n
sites of a class in one alpha bin give at most n log(1 + abar D); two bins split at alpha* (K unused).  The kernel's
decision margin (1e-4 of the sum of |terms| plus 1e-5, in log2 units) is applied here too.

Usage: python tools/prune_bound.py [--sites 1000000] [--centres 30] [--out profiles/r4_prune_bound.json]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def item_sites(p, t, A):
    """alpha and class of the sites of item (t, A) over the whole chromosome, the reference's tests."""
    g = p.genpos
    alpha = np.exp(-A * np.abs(g - t))
    keep = (alpha >= 1e-8) & (g != t)
    return alpha[keep], p.cls[keep]


def bound_per_grid_point(alpha, cls, D, logR, K, a_star, variant):
    """Upper bound on T/2 at every grid point: D, logR are [n_xa, C]."""
    C = D.shape[1]
    near = alpha >= a_star
    if variant == 'jensen':
        tot = np.zeros(D.shape[0])
        tot_abs = np.zeros(D.shape[0])
        for m in (~near, near):
            cnt = np.bincount(cls[m], minlength=C).astype(np.float64)
            s1 = np.bincount(cls[m], weights=alpha[m], minlength=C)
            with np.errstate(divide='ignore', invalid='ignore'):
                term = np.where(cnt > 0, cnt * np.log2(1.0 + D * (s1 / np.maximum(cnt, 1))), 0.0)
            tot += term.sum(-1)
            tot_abs += np.abs(term).sum(-1)
        return (tot + 1e-4 * tot_abs + 1e-5) * np.log(2.0)       # T/2 units; proved when < 0
    ms = np.arange(1, K + 1)
    pw = alpha[:, None] ** ms[None, :]                                  # [sites, K]
    S_tail = np.zeros((C, K))
    S_all = np.zeros((C, K))
    np.add.at(S_tail, cls[~near], pw[~near])
    np.add.at(S_all, cls, pw)
    S_near = S_all - S_tail
    n_near = np.bincount(cls[near], minlength=C).astype(np.float64)
    coef = ((-1.0) ** (ms + 1)) / ms                                     # P_K coefficients
    Dp = D[:, :, None] ** ms[None, None, :]                              # [n_xa, C, K]
    tail = (Dp * (S_tail * coef)[None]).sum(-1)
    near_pk = (Dp * (S_near * coef)[None]).sum(-1)
    lin = D * S_near[None, :, 0]
    with np.errstate(invalid='ignore'):
        logn = np.where(n_near[None] > 0, n_near[None] * logR, 0.0)
    pos = D >= 0
    if variant == 'issue':
        nb = np.where(pos, np.minimum(logn, lin), lin)
    else:
        nb = np.where(pos, np.minimum(np.minimum(logn, lin), near_pk), near_pk)
    return (tail + nb).sum(-1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--sites', type=int, default=1_000_000)
    ap.add_argument('--centres', type=int, default=30)
    ap.add_argument('--every-a', type=int, default=9, help='take every k-th A of the grid')
    ap.add_argument('--out', default=None)
    opt = ap.parse_args()
    import bench
    from oracle import oracle_c
    t0 = time.time()
    chroms = bench.make_genome(opt.sites)
    problems = bench.make_problem(chroms[:1])          # the largest chromosome: interior windows are full-size
    p = problems[0]
    n = len(p.genpos)
    G = p.G
    R = p.SP / G[None, :]
    assert np.all(np.isfinite(R)), 'class rows must be finite'
    D = R - 1.0
    with np.errstate(divide='ignore'):
        logR = np.log(R)
    centres = np.linspace(n // 8, n - n // 8, opt.centres).astype(np.int64)
    iAs = np.arange(0, len(p.A), opt.every_a)
    configs = [(v, K, a) for v in ('issue', 'best') for K in (3, 5) for a in (0.5, 0.9)] + [('jensen', 0, 0.5)]
    rec = {c: {'proved': 0, 'proved_pairs': 0, 'violations': 0, 'slack': []} for c in configs}
    items = pos_items = 0
    pairs_total = 0
    exact_max = []
    for ci in centres:
        t = p.genpos[ci]
        for iA in iAs:
            A = p.A[iA]
            T, _, _, ns, _ = oracle_c.scan(p.genpos, p.cls, p.G, p.SP, np.array([A]), np.array([t]),
                                           np.array([0]), np.array([n - 1]), report_all=True)
            Tex = float(T[0])
            alpha, cls = item_sites(p, t, A)
            assert len(alpha) == ns[0]
            items += 1
            pos_items += Tex > 0
            pairs_total += len(alpha)
            exact_max.append(Tex)
            for c in configs:
                b = 2.0 * bound_per_grid_point(alpha, cls, D, logR, c[1], c[2], c[0])
                bmax = float(np.max(b))
                r = rec[c]
                if bmax < Tex - 1e-9 * max(abs(Tex), 1.0):
                    r['violations'] += 1
                if bmax < 0:
                    r['proved'] += 1
                    r['proved_pairs'] += len(alpha)
                r['slack'].append(bmax - Tex)
    out = {'sites': opt.sites, 'chromosome_sites': n, 'items': items, 'centres': len(centres),
           'A_values': [float(p.A[i]) for i in iAs], 'items_exact_T_gt_0': int(pos_items),
           'items_exact_max_le_0': items - int(pos_items),
           'exact_item_max_quantiles': np.quantile(exact_max, [0, .1, .5, .9, 1]).tolist(),
           'bounds': []}
    for c, r in rec.items():
        s = np.array(r['slack'])
        out['bounds'].append({'variant': c[0], 'K': c[1], 'alpha_star': c[2],
                              'items_proved': r['proved'], 'frac_items_proved': r['proved'] / items,
                              'frac_site_pairs_proved': r['proved_pairs'] / pairs_total,
                              'bound_below_exact': r['violations'],
                              'slack_bound_minus_exact_quantiles': np.quantile(s, [0, .1, .5, .9, 1]).tolist()})
    out['seconds'] = time.time() - t0
    line = json.dumps(out, indent=1)
    print(line)
    if opt.out:
        with open(opt.out, 'w') as fh:
            fh.write(line + '\n')


if __name__ == '__main__':
    main()
