"""Pruning (option `prune`, DESIGN.md §3.8): items whose T is proved <= 0 at every grid point skip the exact
evaluation.  The CPU tests check the bound's maths; the GPU tests check that the rows do not change."""
import os
import subprocess
import sys

import numpy as np
import pytest

import util


def _bound_f32(alpha, D, split=0.5, lg2_err=0.0):
    """bound_kernel's upper bound on sum_i log2(1 + alpha_i D) for one class, evaluated in float32 as the kernel
    does; `lg2_err` is subtracted from every log2 to stand in for the worst error lg2.approx may make."""
    total = np.float32(0.0)
    for m in (alpha < split, alpha >= split):
        n = int(m.sum())
        if n == 0:
            continue
        a = np.float32(alpha[m].sum() / n)
        d = np.float32(D)
        y = np.float32(np.fabs(d) * (a * np.float32(3e-7)) + (d * a + np.float32(1.0)))
        y = max(y, np.float32(1.17549435e-38))
        with np.errstate(divide='ignore'):
            l2 = np.float32(np.log2(y)) - np.float32(lg2_err) * max(np.float32(1.0), np.fabs(np.log2(y)))
        lu = np.float32(np.fabs(l2) * np.float32(4.76837158e-7) + (l2 + np.float32(1e-6)))
        total = np.float32(total + np.float32(n) * lu)
    return float(total)


def test_bound_never_below_the_literal_log_sum():
    rng = np.random.default_rng(11)
    Ds = [-1.0, -1.0 + 1e-12, -0.999, -0.5, -1e-9, 0.0, 1e-9, 0.3, 5.0, 785.0, 1e6, 1e30]
    for trial in range(400):
        n = int(rng.integers(1, 300))
        kind = trial % 4
        if kind == 0:
            alpha = rng.random(n)
        elif kind == 1:
            alpha = np.exp(-rng.random(n) * 18.42)                    # the scan's 1e-8 .. 1 range
        elif kind == 2:
            alpha = 1.0 - rng.random(n) * 1e-6                          # sites next to the centre
        else:
            alpha = np.clip(rng.choice([1e-8, 0.4999999, 0.5, 0.9999999999], n), 1e-8, 1.0)
        for D in Ds + [float(rng.uniform(-1, 3))]:
            with np.errstate(divide='ignore'):
                exact = float(np.sum(np.log1p(alpha * D))) / np.log(2.0)
            bound = _bound_f32(alpha, D, lg2_err=2.0 ** -22)
            if np.isfinite(exact):
                assert bound >= exact - 1e-9 * abs(exact), (n, D, bound, exact)
            else:
                assert exact == -np.inf                                 # D = -1 next to the centre: any bound holds


def _synthetic():
    import bench
    chrom = bench.make_chromosome(20000, seed=12345)
    return bench.make_problem([chrom])[0]


def _scan(prob, t, lo, hi, prune, **opts):
    from ballermixplus_b200.native import Scanner
    with Scanner(device=0).load(prob) as sc:
        sc.set_option('prune', prune)
        for k, v in opts.items():
            sc.set_option(k, v)
        rows = sc.scan(t, lo, hi)
        return rows, sc.counters_all()


def _same_rows(a, b):
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


@pytest.mark.gpu
def test_prune_keeps_rows_on_the_n200_synthetic_problem():
    prob = _synthetic()
    n = len(prob.genpos)
    c = np.arange(0, n, 50)
    t, lo, hi = prob.genpos[c], np.zeros(len(c), np.int64), np.full(len(c), n - 1, np.int64)
    r0, k0 = _scan(prob, t, lo, hi, 0)
    r1, k1 = _scan(prob, t, lo, hi, 1)
    _same_rows(r0, r1)
    assert k0['pruned_items'] == 0
    assert k1['pruned_items'] > 0.3 * len(c) * len(prob.A)         # the pruner was actually used
    assert k0['pairs'] == k1['pairs']
    assert k1['far_sites'] >= k0['far_sites']


@pytest.mark.gpu
def test_prune_keeps_rows_on_ragged_windows():
    prob = _synthetic()
    n = len(prob.genpos)
    rng = np.random.default_rng(4)
    c = rng.integers(0, n, size=400)
    t = prob.genpos[c].copy()
    t[::7] += 3e-7
    lo = c - rng.integers(0, 3000, size=400)
    hi = c + rng.integers(0, 3000, size=400)
    lo[::11] = hi[::11] + 5
    lo[::13] = -50
    hi[::17] = n + 100
    r0, _ = _scan(prob, t, lo, hi, 0, batch=64)
    r1, k1 = _scan(prob, t, lo, hi, 1, batch=64)
    _same_rows(r0, r1)
    assert k1['pruned_items'] > 0


@pytest.mark.gpu
def test_pruner_stays_off_with_report_all_and_unsorted_input():
    from ballermixplus_b200.native import ScanProblem
    prob = _synthetic()
    n = len(prob.genpos)
    c = np.arange(0, n, 400)
    t, lo, hi = prob.genpos[c], np.zeros(len(c), np.int64), np.full(len(c), n - 1, np.int64)
    r0, _ = _scan(prob, t, lo, hi, 0, report_all=1)
    r1, k1 = _scan(prob, t, lo, hi, 1, report_all=1)
    _same_rows(r0, r1)
    assert k1['pruned_items'] == 0
    perm = np.random.default_rng(5).permutation(n)
    shuffled = ScanProblem(prob.genpos[perm], prob.cls[perm], prob.G, prob.SP, prob.A, prob.n_x, prob.n_a)
    c = c[:8]
    t = prob.genpos[c]
    r0, _ = _scan(shuffled, t, lo[:8], hi[:8], 0)
    r1, k1 = _scan(shuffled, t, lo[:8], hi[:8], 1)
    _same_rows(r0, r1)
    assert k1['pruned_items'] == 0


@pytest.mark.gpu
def test_range_checked_build_sees_no_violation_with_pruning():
    lib = os.path.join(util.ROOT, 'ballermixplus_b200', 'libblmx_checked.so')
    assert os.path.exists(lib), 'run __graft_entry__.build() first'
    code = r'''
import sys, numpy as np
sys.path.insert(0, %r); sys.path.insert(0, %r)
import bench
from ballermixplus_b200.native import Scanner
prob = bench.make_problem([bench.make_chromosome(20000, seed=7)])[0]
n = len(prob.genpos)
rng = np.random.default_rng(17)
c = rng.integers(0, n, size=120)
t = prob.genpos[c] + np.where(rng.random(120) < 0.2, 1e-7, 0.0)
lo = c - rng.integers(-20, 9000, size=120)
hi = c + rng.integers(-20, 9000, size=120)
bad = pruned = 0
res = []
for pr in (0, 1):
    with Scanner(device=0, batch=37).load(prob) as sc:
        sc.set_option('prune', pr)
        res.append(sc.scan(t, lo, hi))
        k = sc.counters_all()
        bad += k['range_violations']
        pruned += k['pruned_items']
for a, b in zip(*res):
    assert np.array_equal(a, b)
print('VIOLATIONS', bad, 'PRUNED', pruned)
''' % (util.ROOT, os.path.join(util.ROOT, 'tests'))
    env = dict(os.environ, BLMX_LIB=lib)
    out = subprocess.run([sys.executable, '-c', code], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    assert 'VIOLATIONS 0 ' in out.stdout, out.stdout[-500:]
    assert 'PRUNED 0' not in out.stdout.split('\n')[-2], out.stdout[-500:]
