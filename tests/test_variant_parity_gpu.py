"""The kernel variants against the literal surface at every kernel width (run with -m gpu on a B200).

The seeded problems of variant_problems (grids on both sides of every width edge, extreme class tables, A = 0 and
A < 0, sorted / shuffled / segmented layouts, ragged windows, small launches) go through blmx_scan_surface and
blmx_scan_profile, blmx_scan_split, blmx_refine and blmx_scan; each is compared with the literal T of
surface_oracle (refine_oracle for refine boxes).  Finite T agree within 1e-9 * max(|T|, 1), non-finite T are
identical, and every reported grid point is the oracle's, or a proved tie: the oracle's T at the GPU's point lies
within the same 1e-9 * max(|T|, 1) of the oracle's maximum, with the nSites of that A.  An exact tie (grid rows or
refine points that share one class row) is no excuse: the first point in visiting order must win, as in the
reference.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

import refine_oracle
import surface_oracle
import util
import variant_problems as vp
from test_balpos_gpu import _check_split, _half_rows
from test_support_gpu import _check_surface, _rows_from_surface

pytestmark = pytest.mark.gpu

TOL = 1e-9
KS = list(range(vp.N_PROBLEMS))
STATS = {}


def _stat(variant, problems=0, centres=0, worst=0.0, ties=0):
    s = STATS.setdefault(variant, [0, 0, 0.0, 0])
    s[0] += problems
    s[1] += centres
    s[2] = max(s[2], worst)
    s[3] += ties
    print(f'\n{variant}: {s[0]} problems, {s[1]} centres, worst |dT|/max(|T|,1) = {s[2]:.2e}, {s[3]} ties proved')


def _width(variant, case):
    J, passes = vp.scan_width(case['prob'].n_x * case['prob'].n_a)
    return f'{variant} J={J}' + (f' ({passes} passes)' if passes > 1 else '')


@pytest.fixture(scope='module')
def problems():
    return {}


@pytest.fixture
def case(problems, request, monkeypatch):
    """Problem k and its oracle surface, computed once per problem (the helpers of test_support_gpu and
    test_balpos_gpu ask for it again)."""
    k = request.param
    if k not in problems:
        p = vp.make_problem(k)
        p['oracle'] = surface_oracle.problem_surface(p['prob'], p['t'], p['lo'], p['hi'])
        problems[k] = p
    p = problems[k]
    real = surface_oracle.problem_surface

    def cached(prob, t, lo, hi):
        if prob is p['prob'] and np.array_equal(t, p['t']) and np.array_equal(lo, p['lo']) \
                and np.array_equal(hi, p['hi']):
            return p['oracle']
        return real(prob, t, lo, hi)

    monkeypatch.setattr(surface_oracle, 'problem_surface', cached)
    return p


def _rel(got, want):
    """Largest relative difference of the finite values; non-finite ones must be identical."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    fin = np.isfinite(want)
    assert np.array_equal(np.isfinite(got), fin), (got[~fin], want[~fin])
    assert np.array_equal(got[~fin], want[~fin], equal_nan=True)
    if not fin.any():
        return 0.0
    err = np.abs(got[fin] - want[fin]) / np.maximum(np.abs(want[fin]), 1.)
    assert err.max() <= TOL, err.max()
    return float(err.max())


def check_rows(got, want, S, nsA, floor):
    """Rows (T, iA, ix, ia, ns) of a scan against the reference's rule on the oracle surface S [n, n_A, n_x, n_a]:
    T by _rel, the grid point and nSites identical or a proved tie -> (worst, ties)."""
    worst = _rel(got[0], want[0])
    n_a = S.shape[3]
    ties = 0
    for j in np.flatnonzero(np.any([g != w for g, w in zip(got[1:], want[1:])], axis=0)):
        best = want[0][j] if want[1][j] >= 0 else floor

        def value(r):
            return S[j, r[1][j], r[2][j], r[3][j]] if r[1][j] >= 0 else floor

        v = value(got)
        # a tie within rounding; an exact tie (rows that are copies) is decided by the visiting order, as the
        # reference decides it
        assert np.isfinite(best) and np.isfinite(v) and abs(v - best) <= TOL * max(abs(best), 1.) and v != best, \
            (j, [g[j] for g in got], [w[j] for w in want], v, best)
        assert got[1][j] < 0 or got[4][j] == nsA[j, got[1][j]], (j, got[4][j])
        assert got[1][j] < 0 or got[2][j] * n_a + got[3][j] < S.shape[2] * n_a
        ties += 1
    return worst, ties


@pytest.mark.parametrize('case', KS, indirect=True, ids=vp.problem_name)
def test_surface_and_profile(case):
    """blmx_scan_surface and blmx_scan_profile in every kernel mode (test_support_gpu._check_surface), then the
    rows against the reference's rule on the oracle surface."""
    R, rns = case['oracle']
    want = _rows_from_surface(R, rns)
    worst = ties = 0
    for group, ff in ((1, 0), (4, 0), (4, 1)):
        S, nsA = _check_surface(case['prob'], case['t'], case['lo'], case['hi'], group=group, farfield=ff,
                                batch=case['batch'])
        fin = np.isfinite(R)
        if fin.any():
            worst = max(worst, float(np.max(np.abs(S[fin] - R[fin]) / np.maximum(np.abs(R[fin]), 1.))))
        rows = _rows_from_surface(S, nsA)
        w, t = check_rows(rows, want, R, rns, 0.0)
        ties += t
    _stat(_width('surface', case), 1, len(case['t']), worst, ties)


@pytest.mark.parametrize('case', KS, indirect=True, ids=vp.problem_name)
def test_split(case):
    """blmx_scan_split with four half patterns, prune on and off, report_all 0 and 1
    (test_balpos_gpu._check_split: exact indices on the oracle surface)."""
    rng = np.random.default_rng(case['batch'] + len(case['t']))
    group = 1 if case['layout'] == 'shuffled' else 4
    R, rns = case['oracle']
    n = 0
    worst = 0.0
    for name, half in vp.half_patterns(case['alphas'], rng).items():
        for prune in (0, 1):
            for report_all in (0, 1):
                got = _check_split(case['prob'], case['t'], case['lo'], case['hi'], half, report_all, group=group,
                                   farfield=1, prune=prune, batch=case['batch'])
                for h in (0, 1):
                    worst = max(worst, _rel(got[h][0], _half_rows(R, rns, half, h, bool(report_all))[0]))
                n += 1
    _stat(_width('split', case), 1, len(case['t']) * n, worst)


@pytest.mark.parametrize('case', KS, indirect=True, ids=vp.problem_name)
def test_scan(case):
    """blmx_scan in every kernel mode, prune on and off, report_all 0 and 1."""
    from ballermixplus_b200.native import Scanner
    R, rns = case['oracle']
    worst = ties = 0
    for group, ff, prune in ((1, 0, 0), (4, 0, 0), (4, 1, 0), (4, 1, 1)):
        for report_all in (0, 1):
            with Scanner(device=0, group=group, farfield=ff, batch=case['batch']) as sc:
                sc.set_option('prune', prune)
                sc.set_option('report_all', report_all)
                sc.load(case['prob'])
                got = sc.scan(case['t'], case['lo'], case['hi'])
            floor = -np.inf if report_all else 0.0
            w, t = check_rows(got, _rows_from_surface(R, rns, bool(report_all)), R, rns, floor)
            worst, ties = max(worst, w), ties + t
    _stat(_width('scan', case), 1, len(case['t']), worst, ties)


def check_refine(prob, r, t, lo, hi, got):
    """blmx_refine rows against refine_oracle.refine: T by _rel, point and nSites identical or a proved tie."""
    want = refine_oracle.refine(prob, r['fA'], r['n_fx'], r['n_fa'], r['row_of'], r['SP'], t, lo, hi, r['box'])
    worst = _rel(got[0], want[0])
    ties = 0
    for j in np.flatnonzero(np.any([g != w for g, w in zip(got[1:], want[1:])], axis=0)):
        b = r['box'][j]
        assert got[1][j] >= 0 and want[1][j] >= 0, (j, [g[j] for g in got], [w[j] for w in want])
        S, ns = refine_oracle.box_surface(prob, r['fA'], r['n_fa'], r['row_of'], r['SP'], t[j], lo[j], hi[j], b)
        v = S[got[1][j] - b[0], got[2][j] - b[2], got[3][j] - b[4]]
        best = want[0][j]
        assert np.isfinite(best) and np.isfinite(v) and abs(v - best) <= TOL * max(abs(best), 1.) and v != best, \
            (j, v, best)                                  # an exact tie is decided by the visiting order
        assert got[4][j] == ns[got[1][j] - b[0]]
        ties += 1
    return worst, ties


@pytest.mark.parametrize('case', KS, indirect=True, ids=vp.problem_name)
def test_refine(case):
    """blmx_refine with one box at a width edge and smaller boxes in the same call."""
    from ballermixplus_b200.native import Scanner
    r = vp.refine_case(case['k'], case)
    t, lo, hi = case['t'], case['lo'], case['hi']
    with Scanner(device=0, batch=case['batch']).load(case['prob']) as sc:
        sc.load_refine(r['fA'], r['n_fx'], r['n_fa'], r['row_of'], r['SP'])
        got = sc.refine(t, lo, hi, r['box'])
    worst, ties = check_refine(case['prob'], r, t, lo, hi, got)
    _stat(f'refine J={vp.refine_width(int(vp.box_points(r["box"]).max()))}', 1, len(t), worst, ties)


def test_negative_A_two_site_example():
    """Both factors negative (alpha > 1): the literal T is NaN, so nothing is reported, where the product of the
    two factors would give T = +1.302."""
    from ballermixplus_b200.native import Scanner, ScanProblem
    prob = ScanProblem(np.array([-0.03, 0.02]), np.array([0, 1], np.int32), np.array([0.2, 0.3]),
                       np.array([[0.05, 0.1]]), np.array([-50.0]), 1, 1)
    t, lo, hi = np.array([0.0]), np.array([0], np.int64), np.array([1], np.int64)
    for group in (1, 4):
        for report_all in (0, 1):
            with Scanner(device=0, group=group) as sc:
                sc.set_option('report_all', report_all)
                sc.load(prob)
                T, iA, ix, ia, ns = sc.scan(t, lo, hi)
                S, nsA = sc.scan_surface(t, lo, hi)
                main, bal, pos = sc.scan_split(t, lo, hi, np.array([0], np.int8))
                sc.load_refine(np.array([-50.0]), 1, 1, np.array([0], np.int32), prob.SP)
                rT, rA, rx, ra, rns = sc.refine(t, lo, hi, np.zeros((1, 6), np.int32))
            assert np.isnan(S[0, 0, 0, 0]) and nsA[0, 0] == 2
            assert T[0] == 0 and iA[0] == -1 and ns[0] == 0, (T, iA, ns)
            assert bal[0][0] == 0 and bal[1][0] == -1 and pos[1][0] == -1
            assert rA[0] == -1 and rns[0] == 0


def _cli_vs_oracle(tmp_path, argv, kw):
    """The CLI's file against oracle_cli.scan_file(**kw) (the same flags), every 4th row; argmax ties proved."""
    from ballermixplus_b200.cli import main
    from oracle import oracle_cli
    out = tmp_path / 'out.txt'
    with util.quiet():
        main(util.abs_paths(argv) + ['-o', str(out)])
    got = out.read_text().splitlines(keepends=True)
    want = oracle_cli.scan_file(**kw, centre_stride=4)
    gold = tmp_path / 'oracle.txt'
    gold.write_text(''.join(w if w is not None else g for w, g in zip(want, got)))
    ties = []
    n, same, worst, _ = util.compare_scan([g if w is not None else None for g, w in zip(got, want)], str(gold),
                                          tie_rows=ties)
    if ties:
        util.assert_ties(argv, ties, tol=TOL)
    return got, n, same, worst, len(ties)


@pytest.mark.parametrize('name', ['Example1_B2', 'Example2_B2'])
def test_cli_negative_listA_matches_oracle_cli(name, tmp_path):
    """--listA -20,0,500 on a shipped example: the reference's arithmetic (oracle_cli) row for row; --refine moves
    rows only upward and to points the reference's arithmetic confirms."""
    from oracle import oracle_cli
    kw = dict(util.oracle_kwargs(util.SHIPPED[name]), listA='-20,0,500')
    argv = list(util.SHIPPED[name]) + ['--listA=-20,0,500']           # a value that starts with '-' needs '='
    got, n, same, worst, ties = _cli_vs_oracle(tmp_path, argv, kw)
    assert n > 20 and any(float(r.split('\t')[2]) > 0 for r in got[1:])
    _stat('cli --listA -20,0,500', 1, n, worst, ties)
    ref = tmp_path / 'ref.txt'
    from ballermixplus_b200.cli import main
    with util.quiet():
        main(util.abs_paths(argv) + ['-o', str(tmp_path / 'main.txt'), '--refine', str(ref)])
    main_lines = (tmp_path / 'main.txt').read_text().splitlines(keepends=True)
    assert main_lines == got
    ref_lines = ref.read_text().splitlines(keepends=True)
    moved = [j for j, (a, b) in enumerate(zip(main_lines, ref_lines)) if a != b]
    for j in moved:
        assert float(ref_lines[j].split('\t')[2]) > float(main_lines[j].split('\t')[2])
    for j in moved[:: max(1, len(moved) // 3)][:3]:
        f = ref_lines[j].rstrip('\n').split('\t')
        one = dict(kw, x=repr(float(f[3])), abeta=float(f[4]), listA=repr(float(f[5])))
        g = oracle_cli.scan_file(**one)[j].rstrip('\n').split('\t')
        assert g[:2] == f[:2] and g[6] == f[6]
        assert abs(float(g[2]) - float(f[2])) <= TOL * max(abs(float(f[2])), 1.), (g, f)


def test_checked_build_sees_no_violation_at_the_width_edges():
    """Surface, split and refine scans of every width-edge problem through the -DBLMX_CHECKED build: the
    range-violation counter stays 0."""
    lib = os.path.join(util.ROOT, 'ballermixplus_b200', 'libblmx_checked.so')
    assert os.path.exists(lib), 'run __graft_entry__.build() first'
    code = r'''
import sys, numpy as np
sys.path.insert(0, %r); sys.path.insert(0, %r)
import variant_problems as vp
from ballermixplus_b200.native import Scanner
bad = 0
for k in range(vp.N_PROBLEMS):
    p = vp.make_problem(k)
    r = vp.refine_case(k, p)
    t, lo, hi = p['t'], p['lo'], p['hi']
    half = vp.half_patterns(p['alphas'], np.random.default_rng(k))['alternate']
    for group, ff in ((1, 0), (4, 1)):
        with Scanner(device=0, group=group, farfield=ff, batch=p['batch']).load(p['prob']) as sc:
            sc.scan_surface(t, lo, hi)
            bad += sc.counters_all()['range_violations']
            sc.scan_profile(t, lo, hi)
            bad += sc.counters_all()['range_violations']
            sc.scan_split(t, lo, hi, half)
            bad += sc.counters_all()['range_violations']
            sc.load_refine(r['fA'], r['n_fx'], r['n_fa'], r['row_of'], r['SP'])
            sc.refine(t, lo, hi, r['box'])
            bad += sc.counters_all()['range_violations']
print('VIOLATIONS', bad)
''' % (util.ROOT, os.path.join(util.ROOT, 'tests'))
    env = dict(os.environ, BLMX_LIB=lib)
    out = subprocess.run([sys.executable, '-c', code], env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    assert 'VIOLATIONS 0' in out.stdout, out.stdout[-500:]
