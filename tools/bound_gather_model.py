"""CPU model of bound_kernel's gather (DESIGN.md §3.8) on the benchmark's generator: a 1 M-site chromosome,
8 centres x all 100 A, the kernel's whole-block rules.  Per item: the sites left to the per-site path in each
class, and the warp passes they cost one class at a time, in 32-site chunks shared by all classes, or with a lane
per short class.

    python tools/bound_gather_model.py
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench                                                     # noqa: E402

ch = bench.make_chromosome(1_000_000, 7)
g = ch['pos'] * 1e-8
ks = np.unique(ch['k']); cls = np.searchsorted(ks, ch['k'])
C = len(ks)
order = np.lexsort((np.arange(len(g)), cls)); gs = g[order]; cs = cls[order]
coff = np.searchsorted(cs, np.arange(C + 1))
rng = np.random.default_rng(0)
cent = rng.choice(np.arange(100_000, 900_000), 8, replace=False)
KBS = 32
res = {T: [0, 0] for T in (8, 16, 32, 64)}
cur = [0, 0, 0]; items = 0
nterm_hist = np.zeros(4000, np.int64)
for ci in cent:
    t = g[ci]
    for A in np.arange(1000, 10901, 100.0):
        r = np.log(1e8) / A; r_in = r * (1 - 1e-9); dh = np.log(2) / A
        L = np.searchsorted(g, t - r * 1.001); H = np.searchsorted(g, t + r * 1.001, 'right') - 1
        rest = np.zeros(C, np.int64); items += 1
        for c in range(C):
            c0 = coff[c]; seg = gs[c0:coff[c+1]]
            rb = c0 + np.searchsorted(seg, g[L]); re = c0 + np.searchsorted(seg, g[H], 'right')
            if re <= rb: continue
            nblk = 0
            if re - rb >= KBS:
                ja = (rb - c0 + KBS - 1) // KBS; jb = (re - c0) // KBS; x = gs[rb:re]
                p1 = rb + np.searchsorted(x, t - r_in); p2 = rb + np.searchsorted(x, t - dh, 'right')
                p3 = rb + np.searchsorted(x, t + dh); p4 = rb + np.searchsorted(x, t + r_in, 'right')
                jl0 = max(ja, (p1 - c0 + KBS - 1) // KBS); nl = max(0, min(jb, (p2 - c0) // KBS) - jl0)
                jr0 = max(ja, (p3 - c0 + KBS - 1) // KBS); nr = max(0, min(jb, (p4 - c0) // KBS) - jr0)
                nblk = nl + nr
            rest[c] = re - rb - nblk * KBS
            al = np.exp(-A * np.abs(gs[rb:re] - t)); inn = (al >= 1e-8)
            near = inn & (al >= .5); tail = inn & ~near
            for m in (tail, near):
                if m.any():
                    nterm_hist[min(int(m.sum()), 3999)] += 1
        cur[0] += int(np.sum((rest + 31) // 32))            # today: one warp pass per 32 sites of each class
        cur[1] += int(np.count_nonzero(rest))
        cur[2] += (int(rest.sum()) + 31) // 32              # chunks of 32 concatenated sites
        for T in res:                                        # lane per class for runs <= T, warp-wide otherwise
            lane = np.where(rest <= T, rest, 0)
            it = sum(int(lane[i:i+32].max()) for i in range(0, C, 32))
            res[T][0] += it + int(np.sum(np.where(rest > T, (rest + 31) // 32, 0)))
            res[T][1] += int(np.count_nonzero(rest > T))
print('items', items)
print('today: site passes %.1f, class iterations %.1f per item' % (cur[0] / items, cur[1] / items))
print('chunked: %.1f chunk passes per item' % (cur[2] / items))
for T, (it, nw) in res.items():
    print('lane-per-class (run <= %d): %.1f lane-serial+warp passes, %.1f warp-wide classes per item' % (T, it / items, nw / items))
h = nterm_hist; tot = h.sum()
print('terms per item %.1f; share with count 1: %.2f, <=4: %.2f, <=16: %.2f' % (tot / items, h[1] / tot, h[:5].sum() / tot, h[:17].sum() / tot))
