"""Likelihood surface, profiles and --support on the GPU (run with -m gpu on a B200): blmx_scan_surface against
the literal surface of the CPU oracle, blmx_scan_profile against blmx_scan and the surface, and the CLI's
support file against intervals derived from oracle surfaces."""
import os
import subprocess
import sys

import numpy as np
import pytest

import surface_oracle
import util

pytestmark = pytest.mark.gpu

CASES = util.scan_cases()


def _problem(name):
    from ballermixplus_b200.problem import build_problem
    opt, data, neutral, grid, sel = util.host_objects(CASES[name][0])
    prob, order = build_problem(data, neutral, sel, grid)
    return data, prob, order


def _ragged(n_sites, n, seed):
    """Centres on sites and between them, ragged, empty and out-of-range windows."""
    rng = np.random.default_rng(seed)
    c = rng.integers(0, n_sites, size=n)
    lo = c - rng.integers(0, 400, size=n)
    hi = c + rng.integers(0, 400, size=n)
    lo[::5] = hi[::5] + 3                            # empty windows
    lo[::7] = -20                                    # clamped by the library
    hi[::9] = n_sites + 50
    return c, lo.astype(np.int64), hi.astype(np.int64)


def _pmax(a, axis):
    """max that NaN never wins; -inf where nothing is left."""
    return np.max(np.where(np.isnan(a), -np.inf, a), axis=axis)


def _profiles(S, nsA):
    """TA, Tx, Ta of a surface [n, n_A, n_x, n_a]: the maxima over the A with sites."""
    S = np.where((nsA > 0)[:, :, None, None], S, -np.inf)
    return _pmax(S, (2, 3)), _pmax(S, (1, 3)), _pmax(S, (1, 2))


def _rows_from_surface(S, nsA, report_all=False):
    """The reference's rule on a surface: A in visiting order, (x, a) in visiting order, strict '>' from 0
    (v1:451,501), or from -inf with report_all; an A without sites is skipped (v1:458)."""
    n, n_A = nsA.shape
    n_a = S.shape[3]
    flat = S.reshape(n, n_A, -1)
    floor = -np.inf if report_all else 0.
    T = np.zeros(n)
    iA, ix, ia = (np.full(n, -1, np.int32) for _ in range(3))
    ns = np.zeros(n, np.int32)
    for j in range(n):
        bT = floor
        for a in range(n_A):
            row = flat[j, a]
            ok = row > floor
            if nsA[j, a] == 0 or not ok.any():
                continue
            xa = int(np.flatnonzero(ok)[np.argmax(row[ok])])
            if row[xa] > bT:
                bT, iA[j], ix[j], ia[j], ns[j] = row[xa], a, xa // n_a, xa % n_a, nsA[j, a]
        T[j] = bT if iA[j] >= 0 else 0.
    return T, iA, ix, ia, ns


def _same(got, want):
    for g, w in zip(got, want):
        assert np.array_equal(g, w), (g, w)


def _check_surface(prob, t, lo, hi, **opts):
    """GPU surface against the oracle: finite values within 1e-9 * max(|T|, 1), non-finite ones identical,
    nsA equal.  Then the rows and profiles of the same scan, bit for bit."""
    from ballermixplus_b200.native import Scanner
    with Scanner(device=0, **opts).load(prob) as sc:
        S, nsA = sc.scan_surface(t, lo, hi)
        rows = sc.scan(t, lo, hi)
        prof = sc.scan_profile(t, lo, hi)
    R, rns = surface_oracle.problem_surface(prob, t, lo, hi)
    assert np.array_equal(nsA, rns)
    fin = np.isfinite(R)
    assert np.array_equal(np.isfinite(S), fin)
    assert np.array_equal(S[~fin], R[~fin], equal_nan=True)
    err = np.abs(S[fin] - R[fin]) / np.maximum(np.abs(R[fin]), 1.)
    assert err.size == 0 or err.max() <= 1e-9, err.max()
    _same(_rows_from_surface(S, nsA), rows)
    _same(prof[:5], rows)
    _same(prof[5:8], _profiles(S, nsA))
    assert np.array_equal(prof[8], nsA)
    return S, nsA


@pytest.mark.parametrize('group,farfield', [(1, 0), (4, 0), (4, 1)])
@pytest.mark.parametrize('name', ['Example1_B2', 'Example1_B1', 'ex2_B2maf_findBal_s60', 'ex2_B0_s5'])
def test_surface_matches_the_oracle(name, group, farfield):
    data, prob, order = _problem(name)
    c, lo, hi = _ragged(data.numSites, 40, seed=len(name))
    t = data.genPos[c].copy()
    t[::6] += 2e-7                                   # centres that are not sites
    S, nsA = _check_surface(prob, t, lo, hi, group=group, farfield=farfield, batch=13)
    assert np.all(nsA[lo > hi] == 0) and np.all(S[lo > hi] == -np.inf)


def test_surface_of_a_grid_wider_than_one_pass():
    """n_x * n_a > 512: the kernel sweeps the (x, a) grid in several passes, each writes its part."""
    from ballermixplus_b200.native import ScanProblem
    data, prob, order = _problem('ex2_B0_s5')
    SP = np.concatenate([prob.SP * (1 + 1e-3 * r) for r in range(3)])
    big = ScanProblem(prob.genpos, prob.cls, prob.G, SP, prob.A, prob.n_x * 3, prob.n_a)
    c = np.arange(0, data.numSites, 23)
    t, lo, hi = data.genPos[c], np.zeros(len(c), np.int64), np.full(len(c), data.numSites - 1, np.int64)
    for ff in (0, 1):
        _check_surface(big, t, lo, hi, farfield=ff)


def test_surface_with_far_field_and_superblocks():
    """150 k sites, the default A grid (from A = 100: windows of ~130 k sites, superblocks in use)."""
    import bench
    from ballermixplus_b200.native import Scanner
    prob = bench.make_problem([bench.make_chromosome(150000, seed=77)], range_a=None)[0]
    n = len(prob.genpos)
    c = np.array([0, 3, n // 3, n // 2, n - 1])
    t, lo, hi = prob.genpos[c], np.zeros(len(c), np.int64), np.full(len(c), n - 1, np.int64)
    S, nsA = _check_surface(prob, t, lo, hi, farfield=1)
    with Scanner(device=0).load(prob) as sc:
        sc.scan_surface(t, lo, hi)
        assert sc.counters_all()['far_sites'] > 0               # the far field did run


def test_profile_rows_equal_scan_rows_across_launches_and_the_scratch_budget():
    """Several launches (small batch) and the cut of the 1 GiB scratch budget (100 A x 512 x 8 B per centre:
    2621 centres per launch) give blmx_scan's rows bit for bit, report_all included."""
    import bench
    from ballermixplus_b200.native import Scanner
    prob = bench.make_problem([bench.make_chromosome(20000, seed=9)])[0]
    n = len(prob.genpos)
    assert len(prob.A) * 512 * 8 * 2621 <= 1 << 30 < len(prob.A) * 512 * 8 * 2622
    c = np.arange(0, n, 3)                                       # 6667 centres: three launches of the budget
    t, lo, hi = prob.genpos[c], np.maximum(c - 3000, 0), np.minimum(c + 3000, n - 1)
    profs = []
    for report_all in (0, 1):
        with Scanner(device=0) as sc:
            sc.set_option('report_all', report_all)
            sc.load(prob)
            rows = sc.scan(t, lo, hi)
            prof = sc.scan_profile(t, lo, hi)
            assert sc.counters_all()['launches'] == 3 * 3           # scan, reduce, profile per launch
            _same(prof[:5], rows)
            sc.set_option('batch', 997)
            small = sc.scan_profile(t, lo, hi)
        _same(small, prof)
        profs.append(prof)
    _same(profs[0][5:], profs[1][5:])                               # profiles never clamp at 0
    assert np.any(profs[0][5] < 0)
    # the winning A's profile is the row's CLR
    T, iA = profs[0][:2]
    r = np.flatnonzero(iA >= 0)
    assert len(r) and np.array_equal(profs[0][5][r, iA[r]], T[r])


def _support_from_oracle(argv, q):
    """The support file that support.py derives from oracle surfaces of the plan's centres."""
    from ballermixplus_b200 import support, windows
    from ballermixplus_b200.problem import build_problem
    opt, data, neutral, grid, sel = util.host_objects(argv)
    prob, order = build_problem(data, neutral, sel, grid)
    with util.quiet():
        plan = windows.make_plan(data, fixSize=opt.size, r=opt.w, s=opt.step, phys=opt.phys, noCenter=opt.noCenter)
    t, lo, hi, gap = plan.arrays()
    live = np.flatnonzero(~gap)
    n = len(plan)
    T = np.zeros(n)
    iA, ix, ia = (np.full(n, -1, np.int32) for _ in range(3))
    ns = np.zeros(n, np.int32)
    iv = {k: np.full(n, -1, np.int32) for k in ('A_lo', 'A_hi', 'x_lo', 'x_hi', 's_lo', 's_hi')}
    S, nsA = surface_oracle.problem_surface(prob, t[live], lo[live], hi[live])
    rows = _rows_from_surface(S, nsA)
    for col, v in zip((T, iA, ix, ia, ns), rows):
        col[live] = v
    for k, v in support.support_intervals(rows[0], rows[1], *_profiles(S, nsA), order, q).items():
        iv[k][live] = v
    return [support.SUPPORT_HEADER] + support.format_support(plan, order, T, iA, ix, ia, ns, iv)


@pytest.mark.parametrize('name,extra', [('Example1_B2', []), ('ex2_B0maf_noCenter_gaps', ['--supportDrop', '10'])])
def test_cli_support_file(name, extra, tmp_path):
    from ballermixplus_b200.cli import main
    from ballermixplus_b200.support import DEFAULT_DROP
    argv = CASES[name][0]
    plain, with_s, sup = tmp_path / 'plain.txt', tmp_path / 'with.txt', tmp_path / 'support.txt'
    with util.quiet():
        main(util.abs_paths(argv) + ['-o', str(plain)])
        main(util.abs_paths(argv) + ['-o', str(with_s), '--support', str(sup)] + extra)
    assert with_s.read_bytes() == plain.read_bytes()
    got = sup.read_text().splitlines()
    main_rows = plain.read_text().splitlines()
    q = float(extra[1]) if extra else DEFAULT_DROP
    want = [line.rstrip('\n') for line in _support_from_oracle(argv, q)]
    assert len(got) == len(main_rows) == len(want) and got[0] == want[0]
    for g, m, w in zip(got[1:], main_rows[1:], want[1:]):
        g, m, w = g.split('\t'), m.split('\t'), w.split('\t')
        assert g[:3] == m[:3]                            # the main file's text
        assert g[3:] == w[3:], (g, w)                    # the oracle's intervals
    assert sum('\tNA' not in line for line in got[1:]) > 0


def test_checked_build_sees_no_violation_in_surface_scans():
    """Profile and surface scans through the -DBLMX_CHECKED build: ragged windows, shuffled input, a grid wider
    than one pass, both kernel modes; the range-violation counter stays 0 and results do not change."""
    lib = os.path.join(util.ROOT, 'ballermixplus_b200', 'libblmx_checked.so')
    assert os.path.exists(lib), 'run __graft_entry__.build() first'
    code = r'''
import sys, numpy as np
sys.path.insert(0, %r); sys.path.insert(0, %r)
import util
from ballermixplus_b200.native import Scanner, ScanProblem
from ballermixplus_b200.problem import build_problem
rng = np.random.default_rng(29)
bad = 0
for name in ('Example2_B2', 'Example1_B1', 'ex2_B0_s5'):
    argv, _ = util.scan_cases()[name]
    opt, data, neutral, grid, sel = util.host_objects(argv)
    prob, order = build_problem(data, neutral, sel, grid)
    n = data.numSites
    perm = rng.permutation(n)
    shuffled = ScanProblem(prob.genpos[perm], prob.cls[perm], prob.G, prob.SP, prob.A, prob.n_x, prob.n_a)
    wide = ScanProblem(prob.genpos, prob.cls, prob.G, np.concatenate([prob.SP, prob.SP * 1.01]), prob.A,
                       prob.n_x * 2, prob.n_a)
    c = rng.integers(0, n, size=60)
    t = data.genPos[c] + np.where(rng.random(60) < 0.2, 1e-7, 0.0)
    lo = c - rng.integers(-20, 900, size=60)
    hi = c + rng.integers(-20, 900, size=60)
    for p in (prob, shuffled, wide):
        for ff in (0, 1):
            with Scanner(device=0, farfield=ff, batch=17).load(p) as sc:
                rows = sc.scan(t, lo, hi)
                prof = sc.scan_profile(t, lo, hi)
                bad += sc.counters_all()['range_violations']
                S, nsA = sc.scan_surface(t, lo, hi)
                bad += sc.counters_all()['range_violations']
            for a, b in zip(rows, prof[:5]):
                assert np.array_equal(a, b)
            assert np.array_equal(nsA, prof[8])
print('VIOLATIONS', bad)
''' % (util.ROOT, os.path.join(util.ROOT, 'tests'))
    env = dict(os.environ, BLMX_LIB=lib)
    out = subprocess.run([sys.executable, '-c', code], env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    assert 'VIOLATIONS 0' in out.stdout, out.stdout[-500:]
