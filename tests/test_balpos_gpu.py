"""--balPos on the GPU (run with -m gpu on a B200): blmx_scan_split against the half-restricted reference rule on the
oracle surface, in every kernel mode, with and without report_all, on plain and segmented problems; the command
line against a --findBal run and the main file; two torchrun ranks against one GPU; the range-checked build."""
import os
import subprocess
import sys

import numpy as np
import pytest

import genome_data
import surface_oracle
import util
from test_genome_list_gpu import _torchrun
from test_support_gpu import _ragged, _rows_from_surface

pytestmark = pytest.mark.gpu

CASES = util.scan_cases()
MODES = [dict(group=1, farfield=0, prune=0), dict(group=4, farfield=0, prune=0), dict(group=4, farfield=1, prune=0),
         dict(group=4, farfield=1, prune=1)]


def _problem(name):
    from ballermixplus_b200.problem import build_problem
    opt, data, neutral, grid, sel = util.host_objects(CASES[name][0])
    prob, order = build_problem(data, neutral, sel, grid)
    return data, prob, order


def _half_rows(S, nsA, half_of_a, h, report_all=False):
    """The reference's rule on the grid points of half h only: ``_rows_from_surface`` with the other half's
    points at -inf (they then never pass the strict '>' from 0 or from -inf)."""
    mask = (np.asarray(half_of_a) == h)[None, None, None, :]
    return _rows_from_surface(np.where(mask, S, -np.inf), nsA, report_all)


def _check_split(prob, t, lo, hi, half, report_all=0, **opts):
    """blmx_scan_split against blmx_scan (bit for bit) and against the half rule on the oracle surface (T within
    1e-9 * max(|T|, 1), indices and nSites identical) -> the two half rows."""
    from ballermixplus_b200.native import Scanner
    prune = opts.pop('prune', 1)
    with Scanner(device=0, **opts) as sc:
        sc.set_option('prune', prune)
        sc.set_option('report_all', report_all)
        sc.load(prob)
        rows = sc.scan(t, lo, hi)
        main, bal, pos = sc.scan_split(t, lo, hi, half)
    for a, b in zip(main, rows):
        assert np.array_equal(a, b)
    S, nsA = surface_oracle.problem_surface(prob, t, lo, hi)
    for h, got in ((0, bal), (1, pos)):
        want = _half_rows(S, nsA, half, h, bool(report_all))
        fin = np.isfinite(want[0])                      # T = +inf (a class with G = 0) must be +inf
        assert np.array_equal(got[0][~fin], want[0][~fin])
        err = np.abs(got[0][fin] - want[0][fin]) / np.maximum(np.abs(want[0][fin]), 1.)
        assert err.size == 0 or err.max() <= 1e-9, err.max()
        for g, w in zip(got[1:], want[1:]):
            assert np.array_equal(g, w)
    # every row's CLR is the better half's (report_all: both halves start from -inf as the row does); a half that
    # reports no grid point (iA = -1, T = 0: no alpha in it, or nothing above the floor) takes no part
    best = np.maximum(np.where(bal[1] >= 0, bal[0], -np.inf), np.where(pos[1] >= 0, pos[0], -np.inf))
    assert np.array_equal(np.where(rows[1] >= 0, best, 0.0), rows[0])
    assert np.array_equal(rows[1] >= 0, (bal[1] >= 0) | (pos[1] >= 0))
    return bal, pos


@pytest.mark.parametrize('report_all', [0, 1])
@pytest.mark.parametrize('mode', range(len(MODES)))
@pytest.mark.parametrize('name', ['Example1_B2', 'Example2_B2', 'ex2_B0_s5'])
def test_split_matches_the_half_rule_on_the_oracle_surface(name, mode, report_all):
    from ballermixplus_b200.balpos import half_of_a
    data, prob, order = _problem(name)
    c, lo, hi = _ragged(data.numSites, 48, seed=len(name) + mode)
    t = data.genPos[c].copy()
    t[::6] += 2e-7
    half = half_of_a(order.a)
    assert 0 < half.sum() < len(half)
    bal, pos = _check_split(prob, t, lo, hi, half, report_all, batch=17, **MODES[mode])
    assert np.any(bal[1] >= 0) and np.any(pos[1] >= 0)


def test_split_on_a_segmented_problem():
    """Two copies of a sequence laid end to end (blmx_load_segmented), windows inside each and across the
    boundary."""
    from ballermixplus_b200.balpos import half_of_a
    from ballermixplus_b200.native import ScanProblem
    data, prob, order = _problem('Example1_B2')
    n = len(prob.genpos)
    seg = ScanProblem(np.concatenate([prob.genpos, prob.genpos]), np.concatenate([prob.cls, prob.cls]), prob.G,
                      prob.SP, prob.A, prob.n_x, prob.n_a, seg_start=[0, n])
    rng = np.random.default_rng(3)
    c = np.concatenate([rng.integers(0, 2 * n, 40), np.arange(n - 30, n + 30, 3)])
    lo, hi = c - rng.integers(0, 300, len(c)), c + rng.integers(0, 300, len(c))
    t = np.concatenate([prob.genpos, prob.genpos])[np.clip(c, 0, 2 * n - 1)]
    assert np.any((lo < n) & (hi >= n))                         # windows across the boundary
    for mode in (MODES[0], MODES[3]):
        _check_split(seg, t, lo.astype(np.int64), hi.astype(np.int64), half_of_a(order.a), **dict(mode))


def _cli(argv):
    from ballermixplus_b200.cli import main
    with util.quiet():
        main(argv)


def _table(path):
    with open(path) as fh:
        return [line.rstrip('\n').split('\t') for line in fh]


def _check_against_main(bp, main):
    """The --balPos file has the main file's rows and positions, max(CLR_bal, CLR_pos) == CLR, gap rows as the
    main file's."""
    b, m = _table(bp), _table(main)
    assert len(b) == len(m) and b[0][:2] == m[0][:2] and b[0][2:] == ['CLR_bal', 'x_bal', 's_bal', 'A_bal',
                                                                      'nSites_bal', 'CLR_pos', 'x_pos', 's_pos',
                                                                      'A_pos', 'nSites_pos']
    for fb, fm in zip(b[1:], m[1:]):
        assert fb[:2] == fm[:2]
        if fm[3] == 'NA':
            assert fb[2:] == ['0', 'NA', 'NA', 'NA', '0'] * 2
            continue
        Tb, Tp = float(fb[2]), float(fb[7])
        win = fb[2:7] if Tb >= Tp else fb[7:12]
        assert float(fm[2]) == max(Tb, Tp)
        if float(fm[2]) > 0:
            assert win[1:] == fm[3:], (fb, fm)                  # the winning half's grid point is the row's
    return b


@pytest.mark.parametrize('name', ['Example1_B2', 'Example2_B2'])
def test_cli_bal_half_equals_a_findBal_run(name, tmp_path):
    argv = util.abs_paths(CASES[name][0])
    plain, main, fb, bp = (str(tmp_path / f) for f in ('plain.txt', 'main.txt', 'findbal.txt', 'bp.txt'))
    _cli(argv + ['-o', plain])
    _cli(argv + ['-o', main, '--balPos', bp])
    _cli(argv + ['-o', fb, '--findBal'])
    with open(plain, 'rb') as a, open(main, 'rb') as b:
        assert a.read() == b.read()
    rows = _check_against_main(bp, main)
    ref = _table(fb)
    assert len(ref) == len(rows)
    for r, f in zip(rows[1:], ref[1:]):
        assert r[:2] == f[:2]
        T, Tr = float(r[2]), float(f[2])
        assert abs(T - Tr) <= 1e-9 * max(abs(Tr), 1.), (r, f)
        assert r[3:7] == f[3:], (r, f)                          # the test data hold no exact tie across the halves
    assert sum(float(r[2]) > 0 for r in rows[1:]) > 10 and any(float(r[7]) > 0 for r in rows[1:])


def test_cli_balpos_with_noCenter_support_and_targets(tmp_path):
    name = 'ex2_B0maf_noCenter_gaps'
    argv = util.abs_paths(CASES[name][0])
    d = str(tmp_path)
    full = {k: os.path.join(d, f'full_{k}.txt') for k in ('out', 'sup', 'bp')}
    _cli(argv + ['-o', full['out'], '--balPos', full['bp']])
    rows = _check_against_main(full['bp'], full['out'])
    assert any(r[3] == 'NA' for r in rows[1:])                 # gap rows
    _cli(argv + ['-o', os.path.join(d, 'sup_out.txt'), '--support', full['sup'], '--balPos', os.path.join(d, 'b2.txt')])
    with open(full['bp']) as a, open(os.path.join(d, 'b2.txt')) as b:
        assert a.read() == b.read()                             # the halves' second scan (--support) writes the same
    pos = [float(r[0]) for r in rows[1:]]
    tfile = os.path.join(d, 'targets.txt')
    with open(tfile, 'w') as fh:
        fh.write(f'{os.path.basename(argv[argv.index("-i") + 1])} {pos[len(pos) // 4]} {pos[len(pos) // 2]}\n')
    part = os.path.join(d, 'part_bp.txt')
    _cli(argv + ['-o', os.path.join(d, 'part.txt'), '--balPos', part, '--targets', tfile, '--support',
                 os.path.join(d, 'part_sup.txt')])
    keep = [pos[len(pos) // 4] <= p <= pos[len(pos) // 2] for p in pos]
    with open(full['bp']) as fh:
        lines = fh.readlines()
    with open(part) as fh:
        assert fh.readlines() == lines[:1] + [line for line, k in zip(lines[1:], keep) if k]


def _bytes(p):
    with open(p, 'rb') as fh:
        return fh.read()


def test_cli_input_list_and_torchrun(tmp_path):
    """--inputList writes DIR/<input> equal to the one-input run's file; two torchrun ranks sharing the GPU (gloo)
    write the one-GPU bytes, for one input and for --inputList."""
    d = str(tmp_path)
    lst, paths = genome_data.make_genome(d)
    for k in ('list', 'list2', 'one'):
        for sub in ('out', 'bp'):
            os.makedirs(os.path.join(d, k, sub))
    flags = ['--spect', genome_data.SPECT, '-w', '40']
    for p in paths:
        n = os.path.basename(p)
        _cli(['-i', p, '-o', os.path.join(d, 'one', 'out', n), '--balPos', os.path.join(d, 'one', 'bp', n)] + flags)
    _cli(['--inputList', '-i', lst, '-o', os.path.join(d, 'list', 'out'), '--balPos', os.path.join(d, 'list', 'bp')]
         + flags)
    for p in paths:
        n = os.path.basename(p)
        for sub in ('out', 'bp'):
            assert _bytes(os.path.join(d, 'list', sub, n)) == _bytes(os.path.join(d, 'one', sub, n))
        _check_against_main(os.path.join(d, 'one', 'bp', n), os.path.join(d, 'one', 'out', n))
    _torchrun(['--inputList', '-i', lst, '-o', os.path.join(d, 'list2', 'out'), '--balPos',
               os.path.join(d, 'list2', 'bp')] + flags, 29591)
    n = os.path.basename(paths[0])
    _torchrun(['-i', paths[0], '-o', os.path.join(d, 'two_out.txt'), '--balPos', os.path.join(d, 'two_bp.txt')]
              + flags, 29593)
    assert _bytes(os.path.join(d, 'two_bp.txt')) == _bytes(os.path.join(d, 'one', 'bp', n))
    assert _bytes(os.path.join(d, 'two_out.txt')) == _bytes(os.path.join(d, 'one', 'out', n))
    for p in paths:
        n = os.path.basename(p)
        for sub in ('out', 'bp'):
            assert _bytes(os.path.join(d, 'list2', sub, n)) == _bytes(os.path.join(d, 'one', sub, n))


def test_checked_build_sees_no_violation_in_split_scans():
    lib = os.path.join(util.ROOT, 'ballermixplus_b200', 'libblmx_checked.so')
    assert os.path.exists(lib), 'run __graft_entry__.build() first'
    code = r'''
import sys, numpy as np
sys.path.insert(0, %r); sys.path.insert(0, %r)
import util
from ballermixplus_b200.balpos import half_of_a
from ballermixplus_b200.native import Scanner, ScanProblem
from ballermixplus_b200.problem import build_problem
rng = np.random.default_rng(31)
bad = 0
for name in ('Example2_B2', 'Example1_B1', 'ex2_B0_s5'):
    argv, _ = util.scan_cases()[name]
    opt, data, neutral, grid, sel = util.host_objects(argv)
    prob, order = build_problem(data, neutral, sel, grid)
    n = data.numSites
    seg = ScanProblem(np.concatenate([prob.genpos, prob.genpos]), np.concatenate([prob.cls, prob.cls]), prob.G,
                      prob.SP, prob.A, prob.n_x, prob.n_a, seg_start=[0, n])
    wide = ScanProblem(prob.genpos, prob.cls, prob.G, np.concatenate([prob.SP, prob.SP * 1.01]), prob.A,
                       prob.n_x * 2, prob.n_a)
    c = rng.integers(0, n, size=60)
    t = data.genPos[c] + np.where(rng.random(60) < 0.2, 1e-7, 0.0)
    lo = c - rng.integers(-20, 900, size=60)
    hi = c + rng.integers(-20, 900, size=60)
    for p in (prob, seg, wide):
        for group, ff in ((1, 0), (4, 0), (4, 1)):
            for ra in (0, 1):
                with Scanner(device=0, group=group, farfield=ff, batch=17) as sc:
                    sc.set_option('report_all', ra)
                    sc.load(p)
                    rows = sc.scan(t, lo, hi)
                    main, bal, pos = sc.scan_split(t, lo, hi, half_of_a(order.a))
                    bad += sc.counters_all()['range_violations']
                for a, b in zip(rows, main):
                    assert np.array_equal(a, b)
print('VIOLATIONS', bad)
''' % (util.ROOT, os.path.join(util.ROOT, 'tests'))
    env = dict(os.environ, BLMX_LIB=lib)
    out = subprocess.run([sys.executable, '-c', code], env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    assert 'VIOLATIONS 0' in out.stdout, out.stdout[-500:]
