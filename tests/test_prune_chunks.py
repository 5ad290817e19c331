"""bound_kernel's gather in shared 32-site chunks (DESIGN.md §3.8): the whole blocks and the other sites of the 32
classes of a round are concatenated and visited 32 at a time.  Cases built to put class runs across chunk
boundaries: runs of 31, 32 and 33 sites, rounds with one class or none, a long class whose three per-site
remainders are empty or not in every combination, exactly kPruneClasses classes, a segmented problem.  For each,
rows with pruning on equal rows with it off, and the pruned count lies in the band of a double-precision Jensen
model; the range-checked build sees no violation on all of them."""
import os
import subprocess
import sys

import numpy as np
import pytest

import util

sys.path.insert(0, util.ROOT)

K_PRUNE_CLASSES = 256
KBS = 32
LN_1E8 = 18.420680743952367


def _base(n_sites=20000, seed=12345):
    import bench
    return bench.make_problem([bench.make_chromosome(n_sites, seed=seed)])[0]


def _with(prob, g=None, cls=None, G=None, SP=None, seg=None):
    from ballermixplus_b200.native import ScanProblem
    return ScanProblem(prob.genpos if g is None else g, prob.cls if cls is None else cls,
                       prob.G if G is None else G, prob.SP if SP is None else SP, prob.A, prob.n_x, prob.n_a,
                       seg_start=seg)


def _case_runs():
    """Windows holding exactly 31, 32, 33, 63, 64, 65 or 97 sites of the long class, with the short runs of the
    other classes between them: runs that end just before, on and just after chunk boundaries, across one and
    several of them."""
    p = _base()
    lc = int(np.bincount(p.cls).argmax())
    ranks = np.flatnonzero(p.cls == lc)
    rng = np.random.default_rng(41)
    c, lo, hi = [], [], []
    for k, m in enumerate([31, 32, 33, 63, 64, 65, 97] * 4):
        r0 = int(rng.integers(10, len(ranks) - m - 10))
        a, b = ranks[r0], ranks[r0 + m - 1]
        c.append(int(rng.integers(a, b + 1)) if k % 4 else max(a - 1, 0))
        lo.append(a), hi.append(b)
    c = np.array(c)
    return 'runs', p, p.genpos[c], np.array(lo, np.int64), np.array(hi, np.int64)


def _case_rounds():
    """Windows whose sites are all of the long class (one class in its round, none in every other round), and
    windows with one site of another class besides."""
    p = _base()
    lc = int(np.bincount(p.cls).argmax())
    other = np.flatnonzero(p.cls != lc)
    gaps = np.flatnonzero(np.diff(other) >= 4)[:40]
    a, b = other[gaps] + 1, other[gaps + 1] - 1                       # runs of long-class sites only
    lo = np.where(np.arange(len(a)) % 2, a, a - 1).astype(np.int64)   # even: one other site at the left end
    hi = b.astype(np.int64)
    c = (a + b) // 2
    return 'rounds', p, p.genpos[c], lo, hi


def _case_long():
    """The long class of the benchmark's generator, duplicated positions, centres on its sites and between
    sites; windows whose ends fall on block boundaries of the long class or off them, around the centre or away
    from it, so that the three per-site remainders [b, xl0), [xl1, xr0), [xr1, e) are empty or not in every
    combination."""
    p = _base()
    g = p.genpos.copy()
    g[1::97] = g[0:-1:97]
    n = len(g)
    lc = int(np.bincount(p.cls).argmax())
    ranks = np.flatnonzero(p.cls == lc)
    rng = np.random.default_rng(47)
    # a gap wider than 2 ln2 / A at every A, on a block boundary of the long class: centres in it have whole
    # blocks on both sides that meet, and no middle remainder
    kg = len(ranks) // (2 * KBS)
    q = ranks[KBS * kg]
    g[q:] += 0.003
    c, lo, hi = [], [], []
    for k in range(48):
        k1 = int(rng.integers(4, len(ranks) // KBS - 40))
        k2 = k1 + int(rng.integers(3, 30))
        a = ranks[KBS * k1 - (0 if k % 2 else int(rng.integers(1, KBS)))]
        b = ranks[KBS * k2 - 1 + (0 if (k // 2) % 2 else int(rng.integers(1, KBS)))]
        kind = (k // 4) % 3
        if kind == 0:
            ctr = ranks[int(rng.integers(KBS * k1, KBS * k2))]                 # inside the window
        elif kind == 1:
            ctr = min(b + int(rng.integers(1, 600)), n - 1)                     # right of it
        else:
            ctr = max(a - int(rng.integers(1, 600)), 0)                         # left of it
        c.append(ctr), lo.append(a), hi.append(b)
    c = np.array(c)
    t = g[c].copy()
    t[3::5] += np.diff(g)[np.minimum(c[3::5], n - 2)] * 0.5
    for k in range(6):
        a = ranks[KBS * (kg - 2 - k) + int(rng.integers(1, KBS))]
        b = ranks[KBS * (kg + 2 + k) - 1 - int(rng.integers(1, KBS))]
        t = np.append(t, 0.5 * (g[q - 1] + g[q]))
        lo.append(a), hi.append(b)
    return 'long', _with(p, g=g), t, np.array(lo, np.int64), np.array(hi, np.int64)


def _case_256():
    """Exactly kPruneClasses classes: the generator's classes, the sites of the first 56 split in half with a
    second class of the same row (the likelihood does not change), whole and cut windows."""
    p = _base()
    C = len(p.G)
    extra = K_PRUNE_CLASSES - C
    idx = np.concatenate([np.arange(C), np.arange(extra)])
    cls = p.cls.copy()
    rng = np.random.default_rng(53)
    move = (cls < extra) & (rng.random(len(cls)) < 0.5)
    cls[move] += C
    n = len(p.genpos)
    c = np.linspace(100, n - 100, 20).astype(np.int64)
    lo = np.where(np.arange(len(c)) % 2, 0, c - 1500).astype(np.int64)
    hi = np.where(np.arange(len(c)) % 2, n - 1, c + 1500).astype(np.int64)
    return '256', _with(p, cls=cls, G=p.G[idx], SP=p.SP[:, idx]), p.genpos[c], lo, hi


def _case_segmented():
    """Three replicates end to end: windows inside one segment and windows across a boundary."""
    import bench
    probs = bench.make_problem([bench.make_chromosome(5000, seed=s) for s in (8, 9, 10)])
    g = np.concatenate([q.genpos for q in probs])
    cls = np.concatenate([q.cls for q in probs])
    seg = np.array([0, 5000, 10000], np.int64)
    c = np.arange(30, 15000, 331)
    s = c // 5000
    lo, hi = (s * 5000).astype(np.int64), (s * 5000 + 4999).astype(np.int64)
    cross = np.min(np.abs(c[:, None] - seg[None, 1:]), axis=1) < 700
    lo[cross] = c[cross] - 700
    hi[cross] = c[cross] + 700
    return 'segmented', _with(probs[0], g=g, cls=cls, seg=seg), g[c], lo, hi


def cases():
    return [_case_runs(), _case_rounds(), _case_long(), _case_256(), _case_segmented()]


def remainder_combos(prob, t, lo, hi, cls_id):
    """The kernel's split of class cls_id's run into whole blocks and the three per-site remainders, per item
    with at least one whole block: the set of (na > 0, nm > 0, n_last > 0) that occur."""
    g, cls = prob.genpos, prob.cls
    n = len(g)
    c0 = int(np.sum(cls < cls_id))
    mem = np.flatnonzero(cls == cls_id)
    gs = g[mem]
    seen = set()
    for tc, l0, h0 in zip(t, lo, hi):
        for A in prob.A:
            r = (LN_1E8 / A) * (1.0 + 1e-9)
            L = max(int(l0), 0, int(np.searchsorted(g, tc - r, 'left')))
            H = min(int(h0), n - 1, int(np.searchsorted(g, tc + r, 'right')) - 1)
            if L > H:
                continue
            rb = c0 + int(np.searchsorted(mem, L))
            re = c0 + int(np.searchsorted(mem, H + 1))
            if re - rb < KBS:
                continue
            r_in, d_half = (LN_1E8 / A) * (1.0 - 1e-9), 0.6931471805599453 / A
            run = gs[rb - c0:re - c0]
            p1 = rb + int(np.searchsorted(run, tc - r_in, 'left'))
            p2 = rb + int(np.searchsorted(run, tc - d_half, 'right'))
            p3 = rb + int(np.searchsorted(run, tc + d_half, 'left'))
            p4 = rb + int(np.searchsorted(run, tc + r_in, 'right'))
            p2, p3, p4 = max(p2, p1), max(p3, max(p2, p1)), max(p4, max(p3, max(p2, p1)))
            ja, jb = (rb - c0 + KBS - 1) // KBS, (re - c0) // KBS
            jl0 = max(ja, (p1 - c0 + KBS - 1) // KBS)
            nl = max(0, min(jb, (p2 - c0) // KBS) - jl0)
            jr0 = max(ja, (p3 - c0 + KBS - 1) // KBS)
            nr = max(0, min(jb, (p4 - c0) // KBS) - jr0)
            if nl + nr == 0:
                continue
            xl0, xl1 = (c0 + jl0 * KBS, c0 + (jl0 + nl) * KBS) if nl else (rb, rb)
            xr0, xr1 = (c0 + jr0 * KBS, c0 + (jr0 + nr) * KBS) if nr else (re, re)
            seen.add((xl0 > rb, xr0 > xl1, re > xr1))
    return seen


def jensen_band(prob, t, lo, hi):
    """(sure, unsure): items the double-precision Jensen model proves with room to spare, and items within the fp32
    evaluation's reach of the margin (test_prune_units.test_pruned_count_matches_the_cpu_jensen_model's rule, with
    the items' windows; a window across a segment boundary is never proved)."""
    g, cls = prob.genpos, prob.cls
    n, C = len(g), len(prob.G)
    D = prob.SP / prob.G[None, :] - 1.0
    seg = prob.seg_start
    sure = unsure = 0
    for tc, l0, h0 in zip(t, lo, hi):
        L, H = max(int(l0), 0), min(int(h0), n - 1)
        if seg is not None and L <= H and np.searchsorted(seg, L, 'right') != np.searchsorted(seg, H, 'right'):
            continue
        win = slice(L, H + 1) if L <= H else slice(0, 0)
        gw, cw = g[win], cls[win]
        for A in prob.A:
            alpha = np.exp(-A * np.abs(gw - tc))
            keep = (alpha >= 1e-8) & (gw != tc)
            al, cl = alpha[keep], cw[keep]
            Bl = np.zeros(D.shape[0])
            Al = np.zeros(D.shape[0])
            for m in (al < 0.5, al >= 0.5):
                cnt = np.bincount(cl[m], minlength=C).astype(np.float64)
                s1 = np.bincount(cl[m], weights=al[m], minlength=C)
                k = cnt > 0
                with np.errstate(divide='ignore', invalid='ignore'):
                    lg = cnt[k] * np.log2(1.0 + D[:, k] * (s1[k] / cnt[k]))
                Bl += lg.sum(-1)
                Al += np.abs(lg).sum(-1)
            v = Bl + 1.005e-4 * Al + 1.001e-6 * len(al) + 1e-5
            slack = 5e-5 * Al + 2e-6 * len(al) + 1e-4 * np.maximum(1.0, np.abs(Bl))
            if np.all(v < -slack):
                sure += 1
            elif np.all(v < slack):
                unsure += 1
    return sure, unsure


def test_long_class_remainders_take_every_combination():
    name, prob, t, lo, hi = _case_long()
    lc = int(np.bincount(prob.cls).argmax())
    assert len(remainder_combos(prob, t, lo, hi, lc)) == 8


def _scan(prob, t, lo, hi, prune):
    from ballermixplus_b200.native import Scanner
    with Scanner(device=0).load(prob) as sc:
        sc.set_option('prune', prune)
        rows = sc.scan(t, lo, hi)
        return rows, sc.counters_all()


@pytest.mark.gpu
@pytest.mark.parametrize('k', range(5))
def test_chunked_gather_keeps_rows_and_the_pruned_count(k):
    name, prob, t, lo, hi = cases()[k]
    r0, k0 = _scan(prob, t, lo, hi, 0)
    r1, k1 = _scan(prob, t, lo, hi, 1)
    for x, y in zip(r0, r1):
        assert np.array_equal(x, y), name
    assert k0['pairs'] == k1['pairs'], name
    sure, unsure = jensen_band(prob, t, lo, hi)
    assert sure > 0, name
    assert sure <= k1['pruned_items'] <= sure + unsure, (name, sure, unsure, k1['pruned_items'])


@pytest.mark.gpu
def test_range_checked_build_sees_no_violation_on_the_chunk_cases():
    lib = os.path.join(util.ROOT, 'ballermixplus_b200', 'libblmx_checked.so')
    assert os.path.exists(lib), 'run __graft_entry__.build() first'
    code = r'''
import sys, numpy as np
sys.path.insert(0, %r); sys.path.insert(0, %r)
from ballermixplus_b200.native import Scanner
import test_prune_chunks as tc
bad = pruned = 0
for name, prob, t, lo, hi in tc.cases():
    res = []
    for pr in (0, 1):
        with Scanner(device=0, batch=37).load(prob) as sc:
            sc.set_option('prune', pr)
            res.append(sc.scan(t, lo, hi))
            k = sc.counters_all()
            bad += k['range_violations']
            pruned += k['pruned_items']
    for a, b in zip(*res):
        assert np.array_equal(a, b), name
print('VIOLATIONS', bad, 'PRUNED', pruned)
''' % (util.ROOT, os.path.join(util.ROOT, 'tests'))
    env = dict(os.environ, BLMX_LIB=lib)
    out = subprocess.run([sys.executable, '-c', code], env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    assert 'VIOLATIONS 0 ' in out.stdout, out.stdout[-500:]
    assert 'PRUNED 0' not in out.stdout.split('\n')[-2], out.stdout[-500:]
